// fd_core.cuh -- K13: forward dynamics per state, the inverse of the torque test:
//   qdd = M(q)^-1 (tau - h(q, qd)),   h = rne(q, qd, 0)   (Coriolis, centrifugal and gravity torques)
// and, on request, M^-1 itself (exactly symmetric: one triangle computed, the mirror written).
//
// Built from the code the torque and dynamics kernels already run, so the model (compiled-in or RtParams) is theirs:
//   * M: K10's column passes (dynamics_core.cuh, mass_column<COL>).  Column COL's rows i >= COL are final when its pass
//     ends, which is the order a left-looking LDL^T consumes them: each column is factored as it arrives, into a
//     28-value register triangle, and M never goes to memory.
//   * h: one rne_body pass with qdd = 0 (panda_model.cuh), TOOL for dyn, as K1 / K3 / K1m evaluate it.
//   * qdd: forward substitution, scaling by D^-1, back substitution.  M^-1 = L^-T D^-1 L^-1 (X = L^-1 in place).
// LDL^T rather than the articulated-body algorithm: links 1..5 carry regrouped base parameters, not physical bodies,
// so their articulated inertias need not be positive definite; M itself is.
// The same source builds for the host (tests/native/fd_host.cpp) to check it against the oracle.
#pragma once
#include "dynamics_core.cuh"

namespace tcmp {

// Lower triangle, row-major packed: element (r, c), r >= c.
TCMP_FN constexpr int tri(int r, int c) { return r * (r + 1) / 2 + c; }

// Receives M's lower triangle from mass_column (every index a compile-time constant after inlining).
template <typename T> struct TriOut {
    T A[28];
    TCMP_FN void M(int r, int c, T v) { A[tri(r, c)] = v; }
};

// Left-looking LDL^T step for column J, whose rows J..6 of M are in A: afterwards A holds L_iJ (i > J) below the
// diagonal and d_J on it.  Returns d_J > 0 (false for a zero, negative or NaN pivot).
template <int J, typename T> TCMP_FN bool ldl_column(T (&A)[28], T (&inv_d)[7]) {
    T v[7];
    T d = A[tri(J, J)];
#pragma unroll
    for (int k = 0; k < J; ++k) {
        v[k] = A[tri(J, k)] * A[tri(k, k)];
        d = d - A[tri(J, k)] * v[k];
    }
    A[tri(J, J)] = d;
    inv_d[J] = T(1) / d;
#pragma unroll
    for (int i = J + 1; i < 7; ++i) {
        T x = A[tri(i, J)];
#pragma unroll
        for (int k = 0; k < J; ++k) x = x - A[tri(i, k)] * v[k];
        A[tri(i, J)] = x * inv_d[J];
    }
    return d > T(0);
}

template <int COL, typename T, typename P>
TCMP_FN bool ldl_columns(const T (&s)[7], const T (&c)[7], const P &p, T mp, TriOut<T> &m, T (&inv_d)[7]) {
    if constexpr (COL <= 6) {
        mass_column<COL>(s, c, p, mp, m);
        const bool ok = ldl_column<COL>(m.A, inv_d);
        return ldl_columns<COL + 1>(s, c, p, mp, m, inv_d) && ok;
    } else {
        return true;
    }
}

// x <- L^-T D^-1 L^-1 x
template <typename T> TCMP_FN void ldl_solve(const T (&A)[28], const T (&inv_d)[7], T (&x)[7]) {
#pragma unroll
    for (int i = 1; i < 7; ++i)
#pragma unroll
        for (int k = 0; k < i; ++k) x[i] = x[i] - A[tri(i, k)] * x[k];
#pragma unroll
    for (int i = 0; i < 7; ++i) x[i] = x[i] * inv_d[i];
#pragma unroll
    for (int i = 5; i >= 0; --i)
#pragma unroll
        for (int k = i + 1; k < 7; ++k) x[i] = x[i] - A[tri(k, i)] * x[k];
}

// M^-1 = X^T D^-1 X with X = L^-1 (unit lower; overwrites L in A): out.M(r, c, v) for r >= c, once each.
template <typename T, typename Out> TCMP_FN void ldl_inverse(T (&A)[28], const T (&inv_d)[7], Out &out) {
    // X_ij = -(L_ij + sum_{j<k<i} L_ik X_kj): ascending columns, ascending rows, so every L read is still in place
#pragma unroll
    for (int j = 0; j < 6; ++j)
#pragma unroll
        for (int i = j + 1; i < 7; ++i) {
            T x = A[tri(i, j)];
#pragma unroll
            for (int k = j + 1; k < i; ++k) x = x + A[tri(i, k)] * A[tri(k, j)];
            A[tri(i, j)] = -x;
        }
    // W = D^-1 X (diagonal of X is 1), then (M^-1)_rc = sum_{k >= r} X_kr W_kc
    T W[28];
#pragma unroll
    for (int k = 0; k < 7; ++k)
#pragma unroll
        for (int c = 0; c <= k; ++c) W[tri(k, c)] = c == k ? inv_d[k] : inv_d[k] * A[tri(k, c)];
#pragma unroll
    for (int r = 0; r < 7; ++r)
#pragma unroll
        for (int c = 0; c <= r; ++c) {
            T v = W[tri(r, c)];
#pragma unroll
            for (int k = r + 1; k < 7; ++k) v = v + A[tri(k, r)] * W[tri(k, c)];
            out.M(r, c, v);
        }
}

// Load state i, solve, store.  TOOL: dyn (M without the payload, h with the tool-point force m g for every m); else
// rne (the payload a rigid body on the flange iff m > 0, in M and h).  qd / tau NULL = zeros.  Either output may be
// NULL (uniform branches; qdd is stored before M^-1 is formed, so it is the same with or without it).
// Non-finite inputs, as include/tcmp.h states: a non-finite q (joint 1's too) or mass makes every output of the state
// NaN, a non-finite qd or tau every qdd entry; so does a pivot that is not > 0 (a singular caller record).
template <typename I, bool TOOL, typename P, bool GLOBAL = false>
TCMP_FN void fd_state(I n, I i, const double *__restrict__ q, const double *__restrict__ qd,
                      const double *__restrict__ tau, double mass, const P &p, const SinCos *__restrict__ tab,
                      double *__restrict__ qdd_out, double *__restrict__ Minv_out) {
    double qs[7], vs[7], b[7], s[7], c[7];
    double bad_q = mass * 0.0, bad_v = 0.0;   // +-0 for finite inputs, NaN otherwise
#pragma unroll
    for (int j = 0; j < 7; ++j) {
#ifdef __CUDA_ARCH__
        qs[j] = __ldcs(q + (I)j * n + i);
        vs[j] = qd ? __ldcs(qd + (I)j * n + i) : 0.0;
        b[j] = tau ? __ldcs(tau + (I)j * n + i) : 0.0;
#else
        qs[j] = q[(I)j * n + i];
        vs[j] = qd ? qd[(I)j * n + i] : 0.0;
        b[j] = tau ? tau[(I)j * n + i] : 0.0;
#endif
        bad_q += qs[j] * 0.0;
        bad_v += vs[j] * 0.0 + b[j] * 0.0;
    }
    if (!sincos6_table<GLOBAL>(qs, s, c, tab)) {
#pragma unroll
        for (int j = 1; j < 7; ++j) sincos_t<double>(qs[j], &s[j], &c[j]);
    }
    const double mp = TOOL ? 0.0 : (mass > 0.0 ? mass : 0.0);   // TCMP_PAYLOAD_THRESHOLD_RAW, as tcmp_dynamics_batch
    const double mt = TOOL ? mass : 0.0;
    TriOut<double> m;
    double inv_d[7];
    const bool ok = ldl_columns<0>(s, c, p, mp, m, inv_d) && bad_q == 0.0;
#pragma unroll
    for (int j = 0; j < 7; ++j) inv_d[j] = ok ? inv_d[j] : double(NAN);
    if (qdd_out) {
        double h[7];
        const double zero[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        rne_body<double, true, TOOL, P>(s, c, vs, zero, mp, mt, h, p, gravity_for(qs[0]));
#pragma unroll
        for (int j = 0; j < 7; ++j) b[j] = (b[j] - h[j]) + bad_v;
        ldl_solve(m.A, inv_d, b);
#pragma unroll
        for (int j = 0; j < 7; ++j) DynOut<I>::put(qdd_out + (I)j * n + i, b[j]);
    }
    if (Minv_out) {
        DynOut<I> out{Minv_out, nullptr, nullptr, nullptr, n, i};
        ldl_inverse(m.A, inv_d, out);
    }
}

}  // namespace tcmp
