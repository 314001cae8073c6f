// payload_core.cuh -- K11 / K12: the payload masses a state can carry within the torque limits.
//
// Every joint torque the torque test evaluates is affine in the payload mass m: rne_body folds the payload into link 6
// as m times a fixed rigid body (rne / nov) or as m times a tool-point gravity force (dyn), and the backward pass is
// linear in the wrenches.  So, per state,
//   tau(m) = a + m b     a = the arm alone (rne_body with mp_inertial = mp_tool = 0),
//                        b = the torque one kilogram of payload adds,
// and the masses that pass form an open interval per joint, hence per state and per edge.  Both come from ONE forward
// pass (the kinematics are shared) and TWO backward passes: a's, and b's, which carries the single payload wrench down
// the chain.  Built from panda_model.cuh's primitives, so the model (compiled-in or RtParams) is exactly the torque
// kernels'.  The same source builds for the host (tests/native/payload_host.cpp) to check it against the oracle.
#pragma once
#include "panda_model.cuh"

namespace tcmp {

// child K -> parent frame of a wrench that has no parent contribution of its own (b's pass below link 6):
//   f_p = R f,  n_p = R n + P x (R f)
template <int K, typename T> TCMP_FN void carry_link(T c, T s, V3<T> &f, V3<T> &n) {
    constexpr LinkConst L = link_const(K);
    const V3<T> g = rot_out<L.alpha>(c, s, f);
    V3<T> r = rot_out<L.alpha>(c, s, n);
    if constexpr (L.px != 0.0) { r.y -= T(L.px) * g.z; r.z += T(L.px) * g.y; }
    if constexpr (L.py != 0.0) { r.x += T(L.py) * g.z; r.z -= T(L.py) * g.x; }
    if constexpr (L.pz != 0.0) { r.x -= T(L.pz) * g.y; r.y += T(L.pz) * g.x; }
    f = g;
    n = r;
}

// a (arm alone) and b (per kilogram of payload), joints 0..6, given sin / cos of joints 2..7 and the gravity
// magnitude (gravity_for(q[0])).
//   rne / nov (TOOL = false): b is the wrench of the payload body on link 6 -- unit mass at the flange origin, first
//     moment (0, 0, payload_hz), inertia diag(payload_j, payload_j, 0) about link 6's origin: exactly the terms
//     rne_body scales by mp_inertial.
//   dyn (TOOL = true): b is the tool-point gravity force g6 with moment arm tool_z: the terms rne_body scales by mp_tool.
template <typename T, bool DYN, bool TOOL, typename P = ConstParams>
TCMP_FN void payload_terms(const T (&s)[7], const T (&c)[7], const T (&qd)[7], const T (&qdd)[7], T gravity,
                           const P &p, T (&a)[7], T (&b)[7]) {
    V3<T> F[7], N[7];
    Kin<T> k;
    V3<T> gv;  // gravity direction * g in the current frame (only tracked when TOOL && DYN), as in rne_body

    // ---- forward pass (rne_body's, with mp = 0) ----
    if constexpr (DYN) {
        k.w = {-s[1] * qd[0], -c[1] * qd[0], qd[1]};
        k.wd = {-s[1] * qdd[0] + k.w.y * qd[1], -c[1] * qdd[0] - k.w.x * qd[1], qdd[1]};
    }
    k.vd = {-s[1] * gravity, -c[1] * gravity, T(0)};
    if constexpr (TOOL && DYN) gv = k.vd;
    link_wrench_const<1, T, DYN>(p, k, F[1], N[1]);
#define TCMP_PFWD(K)                                                       \
    forward_link<K, T, DYN>(c[K], s[K], qd[K], qdd[K], k);                 \
    if constexpr (TOOL && DYN) gv = rot_in<link_const(K).alpha>(c[K], s[K], gv);
    TCMP_PFWD(2) link_wrench_const<2, T, DYN>(p, k, F[2], N[2]);
    TCMP_PFWD(3) link_wrench_const<3, T, DYN>(p, k, F[3], N[3]);
    TCMP_PFWD(4) link_wrench_const<4, T, DYN>(p, k, F[4], N[4]);
    TCMP_PFWD(5) link_wrench_const<5, T, DYN>(p, k, F[5], N[5]);
    TCMP_PFWD(6)
#undef TCMP_PFWD

    // ---- link 6: the arm's wrench and the payload's unit wrench ----
    V3<T> Fb, Nb;
    if constexpr (kIsConst<P>) {
        constexpr LinkConst L = link_const(6);
        link_wrench<T, DYN, true, true, true>(k, T(L.m), T(L.hx), T(L.hy), T(L.hz), T(L.jxx), T(L.jxy), T(L.jxz),
                                              T(L.jyy), T(L.jyz), T(L.jzz), F[6], N[6]);
    } else {
        const T *l = p.l6;
        link_wrench<T, DYN, true, true, true>(k, l[0], l[1], l[2], l[3], l[4], l[5], l[6], l[7], l[8], l[9], F[6], N[6]);
    }
    if constexpr (TOOL) {
        T tz;
        if constexpr (kIsConst<P>) tz = T(kToolZ);
        else tz = p.tool_z;
        const V3<T> &g6 = DYN ? gv : k.vd;   // static: vd is exactly the rotated gravity vector
        Fb = g6;
        Nb = {-tz * g6.y, tz * g6.x, T(0)};
    } else {
        T hz, j;
        if constexpr (kIsConst<P>) { hz = T(kPayloadHz); j = T(kPayloadJ); }
        else { hz = p.payload_hz; j = p.payload_j; }
        const V3<T> &vd = k.vd;
        // link_wrench with m = 1, h = (0, 0, hz), J = diag(j, j, 0), the structural zeros dropped:
        //   F = vd [+ wd x h + w (w.h) - |w|^2 h],  N = h x vd [+ J wd + w x (J w)]
        Fb = vd;
        Nb = {-hz * vd.y, hz * vd.x, T(0)};
        if constexpr (DYN) {
            const V3<T> &w = k.w, &wd = k.wd;
            const T xz = w.x * w.z, yz = w.y * w.z;
            Fb.x += hz * (wd.y + xz);
            Fb.y += hz * (yz - wd.x);
            Fb.z -= hz * (w.x * w.x + w.y * w.y);
            Nb.x += j * (wd.x - yz);
            Nb.y += j * (wd.y + xz);
        }
    }

    // ---- backward pass of a (rne_body's) ----
    a[6] = N[6].z;
    backward_link<6, T>(c[6], s[6], F[6], N[6], F[5], N[5]); a[5] = N[5].z;
    backward_link<5, T>(c[5], s[5], F[5], N[5], F[4], N[4]); a[4] = N[4].z;
    backward_link<4, T>(c[4], s[4], F[4], N[4], F[3], N[3]); a[3] = N[3].z;
    backward_link<3, T>(c[3], s[3], F[3], N[3], F[2], N[2]); a[2] = N[2].z;
    backward_link<2, T>(c[2], s[2], F[2], N[2], F[1], N[1]); a[1] = N[1].z;
    T t0 = -(s[1] * N[1].x + c[1] * N[1].y);
    if constexpr (DYN) {
        if constexpr (kIsConst<P>) t0 += T(link_const(0).jzz) * qdd[0];
        else t0 += p.jzz0 * qdd[0];
    }
    a[0] = t0;

    // ---- backward pass of b: the one payload wrench carried down the chain ----
    b[6] = Nb.z;
    carry_link<6, T>(c[6], s[6], Fb, Nb); b[5] = Nb.z;
    carry_link<5, T>(c[5], s[5], Fb, Nb); b[4] = Nb.z;
    carry_link<4, T>(c[4], s[4], Fb, Nb); b[3] = Nb.z;
    carry_link<3, T>(c[3], s[3], Fb, Nb); b[2] = Nb.z;
    carry_link<2, T>(c[2], s[2], Fb, Nb); b[1] = Nb.z;
    b[0] = -(s[1] * Nb.x + c[1] * Nb.y);
}

template <typename T, typename P> TCMP_FN T limit_for(int j, const P &p) {
    if constexpr (kIsConst<P>) return T(torque_limit(j));
    else return p.limit[j];
}

// The masses m with every tested joint inside its limit: the open interval (lo, hi), empty iff lo >= hi, over all real
// m; ok = the verdict with no payload attached.
template <typename T> struct MassInterval {
    T lo, hi;
    bool ok;
};

// Joints 0..5 (joint 7 is never tested, as in within_limits).  Per joint, {m : |a + m b| < L}:
//   b > 0: ((-L - a) / b, (L - a) / b);  b < 0: the ends swap;  b == 0: everything if |a| < L, else nothing;
//   a or b NaN: no bound (NaN never compares >= a limit, so the torque test passes such a joint at every mass).
// The intersection keeps an end only when it compares larger (lo) / smaller (hi): a NaN quotient, which only a and b
// both infinite can produce, imposes no bound either, and lo / hi never hold NaN.
template <typename T, typename P> TCMP_FN MassInterval<T> payload_interval(const T (&a)[7], const T (&b)[7], const P &p) {
    const T inf = T(INFINITY);
    MassInterval<T> r = {-inf, inf, true};
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const T L = limit_for<T>(j, p);
        const bool in = fabs(a[j]) < L;
        r.ok = r.ok && !(fabs(a[j]) >= L);
        T lo, hi;
        if (a[j] != a[j] || b[j] != b[j]) {
            lo = -inf;
            hi = inf;
        } else if (b[j] == T(0)) {
            lo = in ? -inf : inf;
            hi = in ? inf : -inf;
        } else {
            const T u = (-L - a[j]) / b[j], v = (L - a[j]) / b[j];
            lo = b[j] > T(0) ? u : v;
            hi = b[j] > T(0) ? v : u;
        }
        r.lo = lo > r.lo ? lo : r.lo;
        r.hi = hi < r.hi ? hi : r.hi;
    }
    return r;
}

// Intersection of two samples' intervals (edges, segments): exact, so the result means what a state's does.
template <typename T> TCMP_FN void intersect(MassInterval<T> &r, const MassInterval<T> &x) {
    r.lo = x.lo > r.lo ? x.lo : r.lo;
    r.hi = x.hi < r.hi ? x.hi : r.hi;
    r.ok = r.ok && x.ok;
}

// One state end to end: table-driven sin / cos (libm beyond 4096 rad or for a non-finite angle, as rne_core_table),
// gravity_for(q[0]) so a non-finite joint-1 angle gives NaN a and b -- hence (-inf, +inf) and ok = 1, the verdict
// tcmp_rne_batch gives such a state at every mass.
template <bool DYN, bool TOOL, typename P, bool GLOBAL = false>
TCMP_FN MassInterval<double> payload_state(const double (&q)[7], const double (&qd)[7], const double (&qdd)[7],
                                           const P &p, const SinCos *__restrict__ tab, double (&a)[7], double (&b)[7]) {
    double c[7], s[7];
    if (!sincos6_table<GLOBAL>(q, s, c, tab)) {
#pragma unroll
        for (int j = 1; j < 7; ++j) sincos_t<double>(q[j], &s[j], &c[j]);
    }
    payload_terms<double, DYN, TOOL, P>(s, c, qd, qdd, gravity_for(q[0]), p, a, b);
    return payload_interval<double>(a, b, p);
}

}  // namespace tcmp
