// dynamics_core.cuh -- K10: the joint-space terms of the rigid-body model that K1 evaluates, per state:
//   g(q)       gravity torques                 = rne(q, 0, 0)
//   M(q)       joint-space inertia matrix       (exactly symmetric: one triangle computed, the mirror written)
//   C(q, qd)   Christoffel-consistent Coriolis matrix, C_ij = sum_k Gamma_ijk qd_k
//   J(q)       geometric Jacobian [linear; angular] of the grasp-target point, base frame
// such that M qdd + C qd + g == rne(q, qd, qdd) for every state (same payload rule: a rigid body on the flange
// iff m > 0).
//
// Built from panda_model.cuh's primitives (rot_in / rot_out, backward_link, link_const, RtParams), so the model is
// exactly K1's: the regrouped base parameters leave tau unchanged for every (q, qd, qdd), hence M, C and g too.
//   * M column j is a gravity-free Newton-Euler pass with qd = 0 and qdd = e_j.  Links before j do not move, so the
//     forward pass starts at link j, and rows i >= j are final once the backward pass reaches link j: the lower
//     triangle costs 28 link steps instead of 49.
//   * C column j is B(qd, e_j), where B is the symmetric bilinear form with B(v, v) = rne(q, v, 0) - g(q): the
//     gravity-free, qdd = 0 pass carrying two angular velocities (w_u from qd, w_v from e_j), with every product of
//     two velocity-linear quantities a(v) o b(v) replaced by (a(u) o b(v) + a(v) o b(u)) / 2 (Echeandia & Wensing
//     2021).  w_u is the same for the seven columns; w_v vanishes below link j, so the forward pass starts at link j.
//   * J: the DH chain's frames in the base frame, J_j = [z_j x (p_tool - p_j); z_j].
// Every output element is handed to `Out` as soon as it is final: no 49-value accumulator lives in registers.
// The same source builds for the host (tests/native/dynamics_host.cpp) to check it against the oracle.
#pragma once
#include "panda_model.cuh"

namespace tcmp {

template <typename T> TCMP_FN V3<T> vcross(const V3<T> &a, const V3<T> &b) {
    return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
template <typename T> TCMP_FN T vdot(const V3<T> &a, const V3<T> &b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

// Inertial parameters of link K about its frame origin (regrouped; link 6 carries link8, the hand and the payload).
// Links 1..5 have m = hz = jyy = 0 after the regrouping (kFull<K> == false): those terms are not evaluated.
template <typename T> struct LinkP {
    T m, hx, hy, hz, jxx, jxy, jxz, jyy, jyz, jzz;
};
template <int K> constexpr bool kFull = K == 6;

template <int K, typename T, typename P> TCMP_FN LinkP<T> link_params(const P &p, T mp) {
    static_assert(K >= 1 && K <= 6, "link 0 enters only through Jzz");
    if constexpr (kIsConst<P>) {
        constexpr LinkConst L = link_const(K);
        if constexpr (kFull<K>)
            return {T(L.m) + mp, T(L.hx), T(L.hy), T(L.hz) + mp * T(kPayloadHz), T(L.jxx) + mp * T(kPayloadJ),
                    T(L.jxy), T(L.jxz), T(L.jyy) + mp * T(kPayloadJ), T(L.jyz), T(L.jzz)};
        else
            return {T(0), T(L.hx), T(L.hy), T(0), T(L.jxx), T(L.jxy), T(L.jxz), T(0), T(L.jyz), T(L.jzz)};
    } else {
        if constexpr (kFull<K>) {
            const T *l = p.l6;
            return {l[0] + mp, l[1], l[2], l[3] + mp * p.payload_hz, l[4] + mp * p.payload_j, l[5], l[6],
                    l[7] + mp * p.payload_j, l[8], l[9]};
        } else {
            const T *l = p.l[K - 1];
            return {T(0), l[0], l[1], T(0), l[2], l[3], l[4], T(0), l[5], l[6]};
        }
    }
}
template <typename T, typename P> TCMP_FN T link0_jzz(const P &p) {
    if constexpr (kIsConst<P>) return T(link_const(0).jzz);
    else return p.jzz0;
}

// J w (origin inertia times a vector)
template <bool FULL, typename T> TCMP_FN V3<T> jmul(const LinkP<T> &L, const V3<T> &w) {
    V3<T> r = {L.jxx * w.x + L.jxy * w.y + L.jxz * w.z, L.jxy * w.x + L.jyz * w.z, L.jxz * w.x + L.jyz * w.y + L.jzz * w.z};
    if constexpr (FULL) r.y += L.jyy * w.y;
    return r;
}
template <bool FULL, typename T> TCMP_FN V3<T> hvec(const LinkP<T> &L) { return {L.hx, L.hy, FULL ? L.hz : T(0)}; }

// Link wrench of an M column (w = 0):  F = m a + al x h,  N = J al + h x a.
template <int K, typename T>
TCMP_FN void wrench_acc(const LinkP<T> &L, const V3<T> &al, const V3<T> &a, V3<T> &F, V3<T> &N) {
    constexpr bool FULL = kFull<K>;
    const V3<T> h = hvec<FULL>(L);
    F = vcross(al, h);
    N = jmul<FULL>(L, al);
    const V3<T> ha = vcross(h, a);
    N.x += ha.x; N.y += ha.y; N.z += ha.z;
    if constexpr (FULL) { F.x += L.m * a.x; F.y += L.m * a.y; F.z += L.m * a.z; }
}

// Polarised link wrench of a C column:
//   F = m a + al x h + (wu (wv.h) + wv (wu.h)) / 2 - (wu.wv) h
//   N = J al + (wu x J wv + wv x J wu) / 2 + h x a
template <int K, typename T>
TCMP_FN void wrench_bil(const LinkP<T> &L, const V3<T> &wu, const V3<T> &wv, const V3<T> &al, const V3<T> &a,
                        V3<T> &F, V3<T> &N) {
    constexpr bool FULL = kFull<K>;
    const V3<T> h = hvec<FULL>(L);
    const T uh = T(0.5) * vdot(wu, h), vh = T(0.5) * vdot(wv, h), uv = vdot(wu, wv);
    F = vcross(al, h);
    F.x += wu.x * vh + wv.x * uh - uv * h.x;
    F.y += wu.y * vh + wv.y * uh - uv * h.y;
    F.z += wu.z * vh + wv.z * uh - uv * h.z;
    if constexpr (FULL) { F.x += L.m * a.x; F.y += L.m * a.y; F.z += L.m * a.z; }
    N = jmul<FULL>(L, al);
    const V3<T> Ju = jmul<FULL>(L, wu), Jv = jmul<FULL>(L, wv);
    const V3<T> g1 = vcross(wu, Jv), g2 = vcross(wv, Ju), ha = vcross(h, a);
    N.x += T(0.5) * (g1.x + g2.x) + ha.x;
    N.y += T(0.5) * (g1.y + g2.y) + ha.y;
    N.z += T(0.5) * (g1.z + g2.z) + ha.z;
}

// u += al x P with P = origin of frame K in frame K-1 (compile-time, structural zeros dropped)
template <int K, typename T> TCMP_FN void add_cross_P(V3<T> &u, const V3<T> &al) {
    constexpr LinkConst L = link_const(K);
    static_assert(L.pz == 0.0, "links 1..6 have planar DH offsets");
    if constexpr (L.px != 0.0) { u.y += al.z * T(L.px); u.z -= al.y * T(L.px); }
    if constexpr (L.py != 0.0) { u.x -= al.z * T(L.py); u.z += al.x * T(L.py); }
}
// u += (wu (wv.P) + wv (wu.P)) / 2 - (wu.wv) P
template <int K, typename T> TCMP_FN void add_centripetal_P(V3<T> &u, const V3<T> &wu, const V3<T> &wv) {
    constexpr LinkConst L = link_const(K);
    if constexpr (L.px != 0.0 || L.py != 0.0) {
        T up = T(0), vp = T(0);
        if constexpr (L.px != 0.0) { up += wu.x * T(0.5 * L.px); vp += wv.x * T(0.5 * L.px); }
        if constexpr (L.py != 0.0) { up += wu.y * T(0.5 * L.py); vp += wv.y * T(0.5 * L.py); }
        const T uv = vdot(wu, wv);
        u.x += wu.x * vp + wv.x * up;
        u.y += wu.y * vp + wv.y * up;
        u.z += wu.z * vp + wv.z * up;
        if constexpr (L.px != 0.0) u.x -= uv * T(L.px);
        if constexpr (L.py != 0.0) u.y -= uv * T(L.py);
    }
}

// ---- M ------------------------------------------------------------------------------------------------------------
template <int K, typename T, typename P>
TCMP_FN void mass_forward(const T (&s)[7], const T (&c)[7], const P &p, T mp, V3<T> al, V3<T> a, V3<T> (&F)[7],
                          V3<T> (&N)[7]) {
    if constexpr (K <= 6) {
        constexpr int A = link_const(K).alpha;
        add_cross_P<K>(a, al);
        a = rot_in<A>(c[K], s[K], a);
        al = rot_in<A>(c[K], s[K], al);
        wrench_acc<K>(link_params<K, T>(p, mp), al, a, F[K], N[K]);
        mass_forward<K + 1>(s, c, p, mp, al, a, F, N);
    }
}
// backward from link K into K-1, down to link COL; M(K-1, COL) is final after each step
template <int K, int COL, typename T, typename Out>
TCMP_FN void mass_backward(const T (&s)[7], const T (&c)[7], V3<T> (&F)[7], V3<T> (&N)[7], Out &out) {
    if constexpr (K > COL) {
        backward_link<K, T>(c[K], s[K], F[K], N[K], F[K - 1], N[K - 1]);
        out.M(K - 1, COL, N[K - 1].z);
        mass_backward<K - 1, COL>(s, c, F, N, out);
    }
}
template <int COL, typename T, typename P, typename Out>
TCMP_FN void mass_column(const T (&s)[7], const T (&c)[7], const P &p, T mp, Out &out) {
    V3<T> F[7], N[7];
    const V3<T> al = {T(0), T(0), T(1)}, a = {T(0), T(0), T(0)};
    if constexpr (COL == 0) {
        F[0] = a;
        N[0] = {T(0), T(0), link0_jzz<T>(p)};   // only n_0.z is needed
        mass_forward<1>(s, c, p, mp, al, a, F, N);
    } else {
        wrench_acc<COL>(link_params<COL, T>(p, mp), al, a, F[COL], N[COL]);
        mass_forward<COL + 1>(s, c, p, mp, al, a, F, N);
    }
    out.M(6, COL, N[6].z);
    mass_backward<6, COL>(s, c, F, N, out);
}
template <int COL, typename T, typename P, typename Out>
TCMP_FN void mass_columns(const T (&s)[7], const T (&c)[7], const P &p, T mp, Out &out) {
    if constexpr (COL <= 6) {
        mass_column<COL>(s, c, p, mp, out);
        mass_columns<COL + 1>(s, c, p, mp, out);
    }
}

// ---- C ------------------------------------------------------------------------------------------------------------
// w_u of link K from w_u of link K-1 (both in their own frames)
template <int K, typename T> TCMP_FN V3<T> joint_velocity(const T (&s)[7], const T (&c)[7], const T (&qd)[7],
                                                          const V3<T> &wp) {
    V3<T> w = rot_in<link_const(K).alpha>(c[K], s[K], wp);
    w.z += qd[K];
    return w;
}
// Column `col` is a run-time index: unrolled over the columns, ptxas interleaves the seven independent passes and runs
// out of registers (255 and spills); a rolled loop over the columns keeps one pass live at a time.
//   wu: w_u of link K-1 on entry (carried along rather than stored per link);  wv, al, a: the polarised pass, zero
//   below the column.
template <int K, typename T, typename P>
TCMP_FN void coriolis_forward(int col, const T (&s)[7], const T (&c)[7], const T (&qd)[7], const P &p, T mp, V3<T> wu,
                              V3<T> wv, V3<T> al, V3<T> a, V3<T> (&F)[7], V3<T> (&N)[7]) {
    if constexpr (K <= 6) {
        constexpr int A = link_const(K).alpha;
        if (K < col) {                  // below the column: w_v = 0, so no polarised motion and no wrench
            wu = joint_velocity<K>(s, c, qd, wu);
            F[K] = {T(0), T(0), T(0)};
            N[K] = {T(0), T(0), T(0)};
        } else {
            if (K == col) {
                // w_v = z; al = (w_u,K-1 in frame K) x z / 2; a = 0
                wu = joint_velocity<K>(s, c, qd, wu);
                wv = {T(0), T(0), T(1)};
                al = {T(0.5) * wu.y, -T(0.5) * wu.x, T(0)};
            } else {
                add_cross_P<K>(a, al);
                add_centripetal_P<K>(a, wu, wv);
                a = rot_in<A>(c[K], s[K], a);
                wv = rot_in<A>(c[K], s[K], wv);
                al = rot_in<A>(c[K], s[K], al);
                // + (w_v x qd_K z) / 2: the joint-K rate of the u velocity against the carried v velocity
                const T hq = T(0.5) * qd[K];
                al.x += wv.y * hq;
                al.y -= wv.x * hq;
                wu = joint_velocity<K>(s, c, qd, wu);
            }
            wrench_bil<K>(link_params<K, T>(p, mp), wu, wv, al, a, F[K], N[K]);
        }
        coriolis_forward<K + 1>(col, s, c, qd, p, mp, wu, wv, al, a, F, N);
    }
}
template <int K, typename T, typename Out>
TCMP_FN void coriolis_backward(int col, const T (&s)[7], const T (&c)[7], V3<T> (&F)[7], V3<T> (&N)[7], Out &out) {
    if constexpr (K >= 1) {
        backward_link<K, T>(c[K], s[K], F[K], N[K], F[K - 1], N[K - 1]);
        out.C(K - 1, col, N[K - 1].z);
        coriolis_backward<K - 1>(col, s, c, F, N, out);
    }
}
template <typename T, typename P, typename Out>
TCMP_FN void coriolis_columns(const T (&s)[7], const T (&c)[7], const T (&qd)[7], const P &p, T mp, Out &out) {
    const V3<T> zero = {T(0), T(0), T(0)}, wu0 = {T(0), T(0), qd[0]};
#pragma unroll 1
    for (int col = 0; col < 7; ++col) {
        V3<T> F[7], N[7];
        // link 0 spins about its own axis only: no wrench with a z component in any column
        F[0] = zero;
        N[0] = zero;
        const V3<T> wv0 = {T(0), T(0), col == 0 ? T(1) : T(0)};
        coriolis_forward<1>(col, s, c, qd, p, mp, wu0, wv0, zero, zero, F, N);
        out.C(6, col, N[6].z);
        coriolis_backward<6>(col, s, c, F, N, out);
    }
}

// ---- J ------------------------------------------------------------------------------------------------------------
// row . P for P = origin of frame K in frame K-1 (pz = 0 for K >= 1)
template <int K, typename T> TCMP_FN T dot_P(const V3<T> &r) {
    constexpr LinkConst L = link_const(K);
    if constexpr (L.px != 0.0 && L.py != 0.0) return r.x * T(L.px) + r.y * T(L.py);
    else if constexpr (L.px != 0.0) return r.x * T(L.px);
    else return r.y * T(L.py);
}
// Frame K's rotation (as three rows: row i of R_K = rot_in(row i of R_K-1)) and origin in the base frame, K = 1..6.
template <int K, typename T>
TCMP_FN void tool_chain(const T (&s)[7], const T (&c)[7], V3<T> (&r)[3], V3<T> &o, V3<T> (&z)[7], V3<T> (&org)[7]) {
    if constexpr (K <= 6) {
        constexpr LinkConst L = link_const(K);
        if constexpr (L.px != 0.0 || L.py != 0.0) {
            o.x += dot_P<K>(r[0]);
            o.y += dot_P<K>(r[1]);
            o.z += dot_P<K>(r[2]);
        }
        r[0] = rot_in<L.alpha>(c[K], s[K], r[0]);
        r[1] = rot_in<L.alpha>(c[K], s[K], r[1]);
        r[2] = rot_in<L.alpha>(c[K], s[K], r[2]);
        z[K] = {r[0].z, r[1].z, r[2].z};
        org[K] = o;
        tool_chain<K + 1>(s, c, r, o, z, org);
    }
}
template <typename T, typename P> TCMP_FN T tool_height(const P &p) {
    if constexpr (kIsConst<P>) return T(kToolZ);
    else return p.tool_z;
}

// ---- table-driven sin / cos of one angle ------------------------------------------------------------------------------
// The arithmetic of sincos6_table (panda_model.cuh) for an angle x whose nearest table node k pi / 512 is given as
// kd = k and (sin, cos)(k pi / 512) = e.  Templated so the operation count can be instrumented on the host.
template <typename T> TCMP_FN void sincos_from_node(T x, T kd, T es, T ec, T &s, T &c) {
    T r = fma(-kd, T(1.57079632673412561417e+00 / 256), x);
    r = fma(-kd, T(6.07710050630396597660e-11 / 256), r);
    const T z = r * r;
    const T sl = fma(r * z, fma(z, T(1.0 / 120), T(-1.0 / 6)), r);
    const T cm = z * fma(z, T(1.0 / 24), T(-0.5));
    s = fma(ec, sl, fma(es, cm, es));
    c = fma(-es, sl, fma(ec, cm, ec));
}
// Joint 1's angle (sincos6_table covers joints 2..7; only J needs joint 1): table path below 4096 rad, libm beyond.
template <bool GLOBAL>
TCMP_FN void sincos_joint1(double x, double &s, double &c, const SinCos *__restrict__ tab) {
    if ((hi_word(x) & 0x7fffffff) < 0x40b00000) {
        const double kt = fma(x, 162.97466172610082 /* 512 / pi */, 6755399441055744.0);
        const int k = lo_word(kt) & (kSinCosTableSize - 1);
        double es, ec;
#ifdef __CUDA_ARCH__
        if constexpr (GLOBAL) {
            const double2 v = __ldg(reinterpret_cast<const double2 *>(tab) + k);
            es = v.x;
            ec = v.y;
        } else
#endif
        {
            es = tab[k].s;
            ec = tab[k].c;
        }
        sincos_from_node<double>(x, kt - 6755399441055744.0, es, ec, s, c);
    } else {
        sincos_t<double>(x, &s, &c);
    }
}

// ---- one state ----------------------------------------------------------------------------------------------------
// Out receives every element once: M(r, c, v) and C(r, c, v) (M mirrored by the caller), g(r, v), J(r, c, v).
// s[1..6], c[1..6]: joints 2..7; s0, c0: joint 1 (read only when want_J).  qd is read only when want_C.
// mp: payload mass already through the m > 0 rule.
template <typename T, typename P, typename Out>
TCMP_FN void dynamics_body(const T (&s)[7], const T (&c)[7], T s0, T c0, const T (&qd)[7], T mp, bool want_M,
                           bool want_C, bool want_g, bool want_J, const P &p, Out &out) {
    if (want_g) {
        T tau[7];
        const T zero[7] = {T(0), T(0), T(0), T(0), T(0), T(0), T(0)};
        rne_body<T, false, false, P>(s, c, zero, zero, mp, T(0), tau, p);
#pragma unroll
        for (int i = 0; i < 7; ++i) out.g(i, tau[i]);
    }
    if (want_M) mass_columns<0>(s, c, p, mp, out);
    if (want_C) {
        coriolis_columns(s, c, qd, p, mp, out);
    }
    if (want_J) {
        V3<T> r[3] = {{c0, -s0, T(0)}, {s0, c0, T(0)}, {T(0), T(0), T(1)}};   // Rz(q_1)
        V3<T> o = {T(0), T(0), T(link_const(0).pz)};
        V3<T> z[7], org[7];
        z[0] = {T(0), T(0), T(1)};
        org[0] = o;
        tool_chain<1>(s, c, r, o, z, org);
        const T tz = tool_height<T>(p);
        const V3<T> pt = {o.x + z[6].x * tz, o.y + z[6].y * tz, o.z + z[6].z * tz};
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            const V3<T> d = {pt.x - org[j].x, pt.y - org[j].y, pt.z - org[j].z};
            const V3<T> lin = vcross(z[j], d);
            out.J(0, j, lin.x);
            out.J(1, j, lin.y);
            out.J(2, j, lin.z);
            out.J(3, j, z[j].x);
            out.J(4, j, z[j].y);
            out.J(5, j, z[j].z);
        }
    }
}

// Streaming stores into the [7][7][n] / [7][n] / [6][7][n] outputs (NULL = not requested); I = index type.
template <typename I> struct DynOut {
    double *Mo, *Co, *go, *Jo;
    I n, i;
    TCMP_FN static void put(double *p, double v) {
#ifdef __CUDA_ARCH__
        __stcs(p, v);
#else
        *p = v;
#endif
    }
    TCMP_FN void M(int r, int c, double v) {
        put(Mo + (I)(r * 7 + c) * n + i, v);
        if (r != c) put(Mo + (I)(c * 7 + r) * n + i, v);
    }
    TCMP_FN void C(int r, int c, double v) { put(Co + (I)(r * 7 + c) * n + i, v); }
    TCMP_FN void g(int r, double v) { put(go + (I)r * n + i, v); }
    TCMP_FN void J(int r, int c, double v) { put(Jo + (I)(r * 7 + c) * n + i, v); }
};

// Load state i, evaluate the requested terms, store them.  tab: the sin/cos table (GLOBAL: read in place through the
// read-only data cache, as sincos6_table<true>).
template <typename I, typename P, bool GLOBAL = false>
TCMP_FN void dynamics_state(I n, I i, const double *__restrict__ q, const double *__restrict__ qd, double mass,
                            const P &p, const SinCos *__restrict__ tab, DynOut<I> &out) {
    double qs[7], vs[7], s[7], c[7], s0 = 0.0, c0 = 0.0;
    const bool want_C = out.Co != nullptr, want_J = out.Jo != nullptr;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
#ifdef __CUDA_ARCH__
        qs[j] = __ldcs(q + (I)j * n + i);
        vs[j] = want_C ? __ldcs(qd + (I)j * n + i) : 0.0;
#else
        qs[j] = q[(I)j * n + i];
        vs[j] = want_C ? qd[(I)j * n + i] : 0.0;
#endif
    }
    if (!sincos6_table<GLOBAL>(qs, s, c, tab)) {
#pragma unroll
        for (int j = 1; j < 7; ++j) sincos_t<double>(qs[j], &s[j], &c[j]);
    }
    if (want_J) sincos_joint1<GLOBAL>(qs[0], s0, c0, tab);
    const double mp = mass > 0.0 ? mass : 0.0;   // rne.add_payload: attached iff m > 0 (TCMP_PAYLOAD_THRESHOLD_RAW)
    dynamics_body<double, P>(s, c, s0, c0, vs, mp, out.Mo != nullptr, want_C, out.go != nullptr, want_J, p, out);
}

}  // namespace tcmp
