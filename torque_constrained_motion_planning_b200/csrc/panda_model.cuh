// panda_model.cuh -- Franka Panda rigid-body constants and the register-resident
// recursive Newton-Euler core shared by every torque kernel (K1 rne, K2 nov, K3 dyn,
// K4 edge / trajectory).
//
// What it computes is what the reference's rne.py:198-254 computes -- joint torques of the
// 7-DOF arm + flange (link8) + hand (+ payload link) under gravity given as a +9.81 z base
// acceleration (rne.py:199,232) -- but NOT how: the reference multiplies dense 6x6 spatial
// matrices built with np.block for 9-10 links; here
//   * the three rigidly attached tail bodies (link8 rne.py:72/133, hand :73/134, payload
//     :181-188) are folded at compile time into link 7's inertial parameters, which become
//     affine in the payload mass (4 FMAs at run time instead of 3 more links);
//   * the recursion is the classical 3-vector Newton-Euler form about each link-frame origin
//     with first moments h = m c and origin inertias J = I_c + m(|c|^2 1 - c c^T), so no
//     c x (.) products are evaluated at run time;
//   * the modified-DH twists alpha in {0, +-pi/2} (rne.py:47-54) make R_x(alpha) a signed
//     permutation, so a frame change costs 2 FMA + 2 MUL; zero DH offsets are removed with
//     `if constexpr`; joint 1's angle is never needed (gravity is along its axis), so only six
//     sincos are evaluated;
//   * the inertial parameters are regrouped at compile time into base parameters (make_model below), so
//     links 1..6 carry no mass, no axial first moment and no J_yy;
//   * everything lives in registers: one thread owns one state.
// The result differs from the reference only by rounding (measured <= 2e-13 N.m over the
// config-2 distribution, budget 1e-9).  The reference leaves cos(+-pi/2) = 6.1e-17 unsnapped
// (rne.py:39-42); that contributes < 1e-15 N.m and is dropped here.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <type_traits>

#include "../../include/tcmp.h"
// The recursion is plain arithmetic, so the SAME source also builds for the host: tests/native/rne_host.cpp
// compiles it with g++ and checks it against the oracle on a CPU-only box (a test harness -- libtcmp.so contains
// only the device code, there is no CPU path in the product).
#ifdef __CUDACC__
#include <cuda_runtime.h>
#define TCMP_FN __host__ __device__ __forceinline__
#else
#define TCMP_FN inline
#endif

namespace tcmp {

// ---- compile-time model ------------------------------------------------------------------
struct LinkConst {
    int alpha;             // twist code of DH row k: 0, +1 (= +pi/2), -1 (= -pi/2)   rne.py:47-54
    double px, py, pz;     // origin of frame k in frame k-1: (a, -sin(alpha) d, cos(alpha) d)  rne.py:39-42
    double m;              // mass                                                   rne.py:125-136
    double hx, hy, hz;     // first moment m*c                                       rne.py:106-117
    double jxx, jxy, jxz, jyy, jyz, jzz;  // inertia about the frame origin          rne.py:16-19,65-75
};

constexpr double kGravity = 9.81;             // rne.py:199
constexpr double kFlangeZ = 0.107;            // DH row 7 d (rne.py:54): link7 -> link8 / hand / payload frames
constexpr double kPayloadR = 0.14 + 0.025;    // rne.py:182,186: new_inertia([0,0,hand_width+0.025], m)
constexpr double kToolOffset = 0.105;         // panda_grasptarget above the flange (panda_mod.urdf:87-91)
constexpr double kToolZ = kFlangeZ + kToolOffset;   // ... in the link-7 frame

constexpr LinkConst make_link(int alpha, double a, double d, double m, double cx, double cy, double cz,
                              double ixx, double ixy, double ixz, double iyy, double iyz, double izz) {
    LinkConst L{};
    L.alpha = alpha;
    L.px = a;
    L.py = alpha == 0 ? 0.0 : (alpha > 0 ? -d : d);
    L.pz = alpha == 0 ? d : 0.0;
    L.m = m;
    L.hx = m * cx; L.hy = m * cy; L.hz = m * cz;
    const double c2 = cx * cx + cy * cy + cz * cz;
    L.jxx = ixx + m * (c2 - cx * cx);
    L.jyy = iyy + m * (c2 - cy * cy);
    L.jzz = izz + m * (c2 - cz * cz);
    L.jxy = ixy - m * cx * cy;
    L.jxz = ixz - m * cx * cz;
    L.jyz = iyz - m * cy * cz;
    return L;
}

// DH row j (rne.py:47-53): alpha code, a along x (Khalil's d_j), d along z (Khalil's r_j)
constexpr int kAlpha[7] = {0, -1, +1, +1, -1, +1, +1};
constexpr double kA[7] = {0, 0, 0, 0.0825, -0.0825, 0, 0.088};
constexpr double kD[7] = {0.333, 0, 0.316, 0, 0.384, 0, 0};
// The reference's inertial tables: panda_link1..7, panda_link8, panda_hand (also what tcmp_model_default returns).
constexpr double kMass[9] = {4.970684, 0.646926, 3.228604, 3.587895, 1.225946,                     // rne.py:125-136
                             1.666555, 7.35522e-01, 0.0, 0.68};
constexpr double kCom[9][3] = {{3.875e-03, 2.081e-03, -0.1750},        {-3.141e-03, -2.872e-02, 3.495e-03},   // rne.py:106-117
                               {2.7518e-02, 3.9252e-02, -6.6502e-02},  {-5.317e-02, 1.04419e-01, 2.7454e-02},
                               {-1.1953e-02, 4.1065e-02, -3.8437e-02}, {6.0149e-02, -1.4117e-02, -1.0517e-02},
                               {1.0517e-02, -4.252e-03, 6.1597e-02},   {0, 0, 0}, {0, 0, 0}};
constexpr double kInertia[9][6] = {{7.0337e-01, -1.3900e-04, 6.7720e-03, 7.0661e-01, 1.9169e-02, 9.1170e-03},   // rne.py:65-75
                                   {7.9620e-03, -3.9250e-03, 1.0254e-02, 2.8110e-02, 7.0400e-04, 2.5995e-02},
                                   {3.7242e-02, -4.7610e-03, -1.1396e-02, 3.6155e-02, -1.2805e-02, 1.0830e-02},
                                   {2.5853e-02, 7.7960e-03, -1.3320e-03, 1.9552e-02, 8.6410e-03, 2.8323e-02},
                                   {3.5549e-02, -2.1170e-03, -4.0370e-03, 2.9474e-02, 2.2900e-04, 8.6270e-03},
                                   {1.9640e-03, 1.0900e-04, -1.1580e-03, 4.3540e-03, 3.4100e-04, 5.4330e-03},
                                   {1.2516e-02, -4.2800e-04, -1.1960e-03, 1.0027e-02, -7.4100e-04, 4.8150e-03},
                                   {0.001, 0.0, 0.0, 0.001, 0.0, 0.001},
                                   {0.1, 0.0, 0.0, 0.1, 0.0, 0.1}};

// Link k = panda_link(k+1).  Link 6 additionally carries link8 (m = 0, I = 0.001*1) and the hand
// (m = 0.68, c = 0, I = 0.1*1), both rigidly at (0,0,0.107) in its frame (rne.py:54,58-61).
constexpr LinkConst raw_link_const(int k) {
    LinkConst L = make_link(kAlpha[k], kA[k], kD[k], kMass[k], kCom[k][0], kCom[k][1], kCom[k][2], kInertia[k][0],
                            kInertia[k][1], kInertia[k][2], kInertia[k][3], kInertia[k][4], kInertia[k][5]);
    if (k == 6) {
        const double mh = kMass[8], z = kFlangeZ;   // hand; link8 has zero mass, both have c = 0 and diagonal I
        L.m += mh;
        L.hz += mh * z;
        L.jxx += kInertia[7][0] + kInertia[8][0] + mh * z * z;
        L.jyy += kInertia[7][3] + kInertia[8][3] + mh * z * z;
        L.jzz += kInertia[7][5] + kInertia[8][5];
    }
    return L;
}
// ---- regrouped (base) inertial parameters ---------------------------------------------------
// Joint torques of a serial chain depend on fewer parameters than 10 per link: for a revolute joint j the
// mass M_j, the first moment MZ_j along the joint axis and the inertia YY_j can be moved into link j-1's
// parameters without changing any joint torque (Gautier & Khalil's regrouping for modified-DH chains).  Done
// here at COMPILE TIME from link 6 down to link 1, it leaves links 1..6 with m = 0, hz = 0, jyy = 0 -- the
// wrench of each of those links then needs 11 fewer FP64 instructions.  (Internal link forces change, the
// joint torques do not: checked against the oracle to 4e-14 N.m.)  The payload's runtime terms are NOT
// regrouped: they stay on link 6, which therefore keeps the general wrench.
struct Model {
    LinkConst L[7];
};
// constexpr so the compiled-in Panda is regrouped by the compiler; the same function regroups a caller-supplied
// inertial set at run time on the host (model_from_desc below).
constexpr Model regroup_model(Model M) {
    for (int j = 6; j >= 1; --j) {
        LinkConst &c = M.L[j];
        LinkConst &p = M.L[j - 1];
        const double Sa = c.alpha, Ca = c.alpha == 0 ? 1.0 : 0.0;   // sin / cos of alpha in {0, +-pi/2}
        const double d = kA[j], r = kD[j];
        const double YY = c.jyy, MZ = c.hz, Mj = c.m;
        p.jxx += YY + 2 * r * MZ + r * r * Mj;
        p.jxy += d * Sa * MZ + d * r * Sa * Mj;
        p.jxz += -d * Ca * MZ - d * r * Ca * Mj;
        p.jyy += Ca * Ca * YY + 2 * r * Ca * Ca * MZ + (d * d + r * r * Ca * Ca) * Mj;
        p.jyz += Ca * Sa * YY + 2 * r * Ca * Sa * MZ + r * r * Ca * Sa * Mj;
        p.jzz += Sa * Sa * YY + 2 * r * Sa * Sa * MZ + (d * d + r * r * Sa * Sa) * Mj;
        p.hx += d * Mj;
        p.hy += -Sa * MZ - r * Sa * Mj;
        p.hz += Ca * MZ + r * Ca * Mj;
        p.m += Mj;
        c.jxx -= YY;
        c.jyy = 0.0;
        c.hz = 0.0;
        c.m = 0.0;
    }
    return M;
}
constexpr Model make_model() {
    Model M{};
    for (int k = 0; k < 7; ++k) M.L[k] = raw_link_const(k);
    return regroup_model(M);
}
constexpr Model kModel = make_model();
constexpr LinkConst link_const(int k) { return kModel.L[k]; }

// Payload link (rne.py:181-188): mass mp at the flange frame origin with
// I = diag(mp r^2, mp r^2, 0), r = 0.165 -> affine terms added to link 6's parameters.
constexpr double kPayloadHz = kFlangeZ;
constexpr double kPayloadJ = kPayloadR * kPayloadR + kFlangeZ * kFlangeZ;

// panda_mod.urdf:127,153,179,205,231,257,283 (effort), lower/upper, velocity.
constexpr double torque_limit(int i) { return i < 4 ? 87.0 : 12.0; }

// ---- where the inertial parameters come from ----------------------------------------------------------------
// ConstParams: the compiled-in Panda (kModel) -- every parameter is an immediate, structural zeros vanish.
// RtParams<T>: a caller-supplied inertial set (tcmp_rne_batch_model), regrouped on the host and passed to the
// kernel by value (constant bank).  The DH geometry stays compile-time in both.
struct ConstParams {};
template <typename T> struct RtParams {
    T jzz0;          // link 0 enters only through tau_0 = Jzz qdd_0
    T l[5][7];       // links 1..5 after regrouping (m = hz = jyy = 0): hx hy jxx jxy jxz jyz jzz
    T l6[10];        // link 6 + link8 + hand: m hx hy hz jxx jxy jxz jyy jyz jzz
    T payload_hz;    // payload mass mp adds mp * payload_hz to hz ...
    T payload_j;     // ... and mp * payload_j to jxx and jyy          (rne.py:181-188)
    T tool_z;        // grasp-target height in the link-7 frame        (dyn mode)
    T limit[6];      // torque limits of joints 1..6                   (joint 7 is never tested)
};
template <typename P> constexpr bool kIsConst = std::is_same<P, ConstParams>::value;

// ---- host side of RtParams ------------------------------------------------------------------------------------
// Caller's record -> per-link parameters about the link-frame origins, tail bodies folded, regrouped.
inline Model model_from_desc(const tcmp_model &d) {
    Model M{};
    for (int k = 0; k < 7; ++k)
        M.L[k] = make_link(kAlpha[k], kA[k], kD[k], d.mass[k], d.com[k][0], d.com[k][1], d.com[k][2], d.inertia[k][0],
                           d.inertia[k][1], d.inertia[k][2], d.inertia[k][3], d.inertia[k][4], d.inertia[k][5]);
    // link8 (DH row 8: pure translation d = 0.107 along z, rne.py:54) and the hand (identity on link8,
    // rne.py:58-61) move rigidly with link 7: shift each to link 7's origin (parallel-axis) and add it.
    LinkConst &L = M.L[6];
    for (int b = 7; b < 9; ++b) {
        const double m = d.mass[b], rx = d.com[b][0], ry = d.com[b][1], rz = d.com[b][2] + kFlangeZ;
        const double *I = d.inertia[b];
        const double r2 = rx * rx + ry * ry + rz * rz;
        L.m += m;
        L.hx += m * rx; L.hy += m * ry; L.hz += m * rz;
        L.jxx += I[0] + m * (r2 - rx * rx);
        L.jyy += I[3] + m * (r2 - ry * ry);
        L.jzz += I[5] + m * (r2 - rz * rz);
        L.jxy += I[1] - m * rx * ry;
        L.jxz += I[2] - m * rx * rz;
        L.jyz += I[4] - m * ry * rz;
    }
    return regroup_model(M);
}

template <typename T> inline RtParams<T> params_from_desc(const tcmp_model &d) {
    const Model M = model_from_desc(d);
    RtParams<T> P;
    P.jzz0 = (T)M.L[0].jzz;
    for (int k = 1; k <= 5; ++k) {
        const LinkConst &L = M.L[k];
        const double v[7] = {L.hx, L.hy, L.jxx, L.jxy, L.jxz, L.jyz, L.jzz};
        for (int j = 0; j < 7; ++j) P.l[k - 1][j] = (T)v[j];
    }
    const LinkConst &L = M.L[6];
    const double v6[10] = {L.m, L.hx, L.hy, L.hz, L.jxx, L.jxy, L.jxz, L.jyy, L.jyz, L.jzz};
    for (int j = 0; j < 10; ++j) P.l6[j] = (T)v6[j];
    P.payload_hz = (T)kFlangeZ;
    P.payload_j = (T)(d.payload_radius * d.payload_radius + kFlangeZ * kFlangeZ);
    P.tool_z = (T)(kFlangeZ + d.tool_z);
    for (int i = 0; i < 6; ++i) P.limit[i] = (T)d.torque_limit[i];
    return P;
}

template <typename T> struct V3 { T x, y, z; };

// parent -> child frame:  E u,  E = Rz(theta)^T Rx(alpha)^T
template <int ALPHA, typename T>
TCMP_FN V3<T> rot_in(T c, T s, const V3<T> &u) {
    T wy, wz;
    if constexpr (ALPHA == 0) { wy = u.y; wz = u.z; }
    else if constexpr (ALPHA > 0) { wy = u.z; wz = -u.y; }
    else { wy = -u.z; wz = u.y; }
    return {c * u.x + s * wy, c * wy - s * u.x, wz};
}
// child -> parent frame:  R u,  R = Rx(alpha) Rz(theta)
template <int ALPHA, typename T>
TCMP_FN V3<T> rot_out(T c, T s, const V3<T> &u) {
    const T wx = c * u.x - s * u.y, wy = s * u.x + c * u.y;
    if constexpr (ALPHA == 0) return {wx, wy, u.z};
    else if constexpr (ALPHA > 0) return {wx, -u.z, wy};
    else return {wx, u.z, -wy};
}

template <typename T> TCMP_FN void sincos_t(T x, T *s, T *c);
template <> TCMP_FN void sincos_t<double>(double x, double *s, double *c) { sincos(x, s, c); }
template <> TCMP_FN void sincos_t<float>(float x, float *s, float *c) { sincosf(x, s, c); }

// Kinematic state carried down the chain, expressed in the current link frame.
template <typename T> struct Kin {
    V3<T> w;   // angular velocity
    V3<T> wd;  // angular acceleration
    V3<T> vd;  // linear acceleration of the frame origin (includes the +g base acceleration)
};

// Forward step for link K >= 2 (and the generic form for K == 1 when the parent is a full Kin).
// DYN == false is the static specialisation (qd = qdd = 0): only vd is propagated.
template <int K, typename T, bool DYN>
TCMP_FN void forward_link(T c, T s, T qd, T qdd, Kin<T> &k) {
    constexpr LinkConst L = link_const(K);
    static_assert(L.pz == 0.0, "generic forward step assumes a planar DH offset");
    V3<T> u = k.vd;
    if constexpr (DYN) {
        // u = vd + wd x P + w (w.P) - |w|^2 P   with P = (px, py, 0)
        if constexpr (L.px != 0.0 || L.py != 0.0) {
            const T w2 = k.w.x * k.w.x + k.w.y * k.w.y + k.w.z * k.w.z;
            T wp = T(0);
            if constexpr (L.px != 0.0) wp += k.w.x * T(L.px);
            if constexpr (L.py != 0.0) wp += k.w.y * T(L.py);
            if constexpr (L.px != 0.0) {
                u.x += -w2 * T(L.px);
                u.y += k.wd.z * T(L.px);
                u.z += -k.wd.y * T(L.px);
            }
            if constexpr (L.py != 0.0) {
                u.x += -k.wd.z * T(L.py);
                u.y += -w2 * T(L.py);
                u.z += k.wd.x * T(L.py);
            }
            u.x += k.w.x * wp;
            u.y += k.w.y * wp;
            u.z += k.w.z * wp;
        }
        V3<T> w = rot_in<L.alpha>(c, s, k.w);
        V3<T> wd = rot_in<L.alpha>(c, s, k.wd);
        wd.x += w.y * qd;
        wd.y -= w.x * qd;
        wd.z += qdd;
        w.z += qd;
        k.w = w;
        k.wd = wd;
    }
    k.vd = rot_in<L.alpha>(c, s, u);
}

// Net inertial force F and moment N (about the frame origin) of a link with parameters (m, h, J) moving with k.
// HAS_M / HAS_HZ / HAS_JYY = false drop the terms of parameters that the regrouping made structurally zero.
// Static: F = m vd, N = h x vd.
template <typename T, bool DYN, bool HAS_M, bool HAS_HZ, bool HAS_JYY>
TCMP_FN void link_wrench(const Kin<T> &k, T m, T hx, T hy, T hz, T jxx, T jxy, T jxz, T jyy,
                                            T jyz, T jzz, V3<T> &F, V3<T> &N) {
    const V3<T> &vd = k.vd;
    if constexpr (HAS_HZ) N = {hy * vd.z - hz * vd.y, hz * vd.x - hx * vd.z, hx * vd.y - hy * vd.x};
    else N = {hy * vd.z, -hx * vd.z, hx * vd.y - hy * vd.x};
    if constexpr (!DYN) {
        if constexpr (HAS_M) F = {m * vd.x, m * vd.y, m * vd.z};
        else F = {T(0), T(0), T(0)};
    } else {
        const V3<T> &w = k.w, &a = k.wd;
        const T w2 = w.x * w.x + w.y * w.y + w.z * w.z;
        T wh = w.x * hx + w.y * hy;
        if constexpr (HAS_HZ) wh += w.z * hz;
        // F = m vd + wd x h + w (w.h) - |w|^2 h
        F.x = -a.z * hy + w.x * wh - w2 * hx;
        F.y = a.z * hx + w.y * wh - w2 * hy;
        F.z = a.x * hy - a.y * hx + w.z * wh;
        if constexpr (HAS_HZ) { F.x += a.y * hz; F.y -= a.x * hz; F.z -= w2 * hz; }
        if constexpr (HAS_M) { F.x += m * vd.x; F.y += m * vd.y; F.z += m * vd.z; }
        // N += J wd + w x (J w)
        const T lx = jxx * w.x + jxy * w.y + jxz * w.z;
        T ly = jxy * w.x + jyz * w.z;
        if constexpr (HAS_JYY) ly += jyy * w.y;
        const T lz = jxz * w.x + jyz * w.y + jzz * w.z;
        N.x += jxx * a.x + jxy * a.y + jxz * a.z + (w.y * lz - w.z * ly);
        N.y += jxy * a.x + jyz * a.z + (w.z * lx - w.x * lz);
        if constexpr (HAS_JYY) N.y += jyy * a.y;
        N.z += jxz * a.x + jyz * a.y + jzz * a.z + (w.x * ly - w.y * lx);
    }
}

template <int K, typename T, bool DYN, typename P>
TCMP_FN void link_wrench_const(const P &p, const Kin<T> &k, V3<T> &F, V3<T> &N) {
    if constexpr (kIsConst<P>) {
        constexpr LinkConst L = link_const(K);
        link_wrench<T, DYN, L.m != 0.0, L.hz != 0.0, L.jyy != 0.0>(k, T(L.m), T(L.hx), T(L.hy), T(L.hz), T(L.jxx),
                                                                   T(L.jxy), T(L.jxz), T(L.jyy), T(L.jyz), T(L.jzz),
                                                                   F, N);
    } else {
        static_assert(K >= 1 && K <= 5, "links 1..5 are the regrouped ones");
        const T *l = p.l[K - 1];
        link_wrench<T, DYN, false, false, false>(k, T(0), l[0], l[1], T(0), l[2], l[3], l[4], T(0), l[5], l[6], F, N);
    }
}

// Backward step: fold child K's accumulated wrench (f, n, in frame K) into its parent's
// (F, N in frame K-1):  f_p = F + R f,  n_p = N + R n + P x (R f).
template <int K, typename T>
TCMP_FN void backward_link(T c, T s, const V3<T> &f, const V3<T> &n, V3<T> &F, V3<T> &N) {
    constexpr LinkConst L = link_const(K);
    const V3<T> g = rot_out<L.alpha>(c, s, f);
    const V3<T> r = rot_out<L.alpha>(c, s, n);
    N.x += r.x; N.y += r.y; N.z += r.z;
    if constexpr (L.px != 0.0) { N.y -= T(L.px) * g.z; N.z += T(L.px) * g.y; }
    if constexpr (L.py != 0.0) { N.x += T(L.py) * g.z; N.z -= T(L.py) * g.x; }
    if constexpr (L.pz != 0.0) { N.x -= T(L.pz) * g.y; N.y += T(L.pz) * g.x; }
    F.x += g.x; F.y += g.y; F.z += g.z;
}

// The whole recursion for one state.
//   DYN        false: static (nov, or rne/dyn called without velocities): qd/qdd ignored.
//   mp_inertial  payload mass carried as a rigid body on the flange (rne/nov; 0 = none).
//   mp_tool      payload mass applied as a pure gravity force at the grasp-target point
//                (dyn: J^T [0,0,m g,0,0,0], panda_primitives.py:101-111; 0 = none).
// sin/cos of the six joint angles the recursion needs.  TCMP_SINCOS6 (fp64): when every angle is below 1e5 rad
// the six evaluations run TOGETHER through one branch-free Cody-Waite + fdlibm-kernel sequence, so each of the 19
// polynomial / reduction constants is materialised once per state instead of once per angle (CUDA's sincos(),
// inlined six times, re-creates its ~13 coefficients at every call site: ~150 UMOV per state).  Any larger or
// non-finite angle sends the whole state down CUDA's sincos() (exact Payne-Hanek reduction), so results for
// absurd inputs still follow libm.  Worst abs error of the fast path 1.8e-16 (checked against 200-bit arithmetic).
#ifndef TCMP_SINCOS6
#define TCMP_SINCOS6 1
#endif
TCMP_FN int hi_word(double x) {
#ifdef __CUDA_ARCH__
    return __double2hiint(x);
#else
    int64_t b;
    memcpy(&b, &x, 8);
    return (int)(b >> 32);
#endif
}
TCMP_FN int lo_word(double x) {
#ifdef __CUDA_ARCH__
    return __double2loint(x);
#else
    int64_t b;
    memcpy(&b, &x, 8);
    return (int)(b & 0xffffffff);
#endif
}
template <typename T>
TCMP_FN void sincos6(const T (&q)[7], T (&s)[7], T (&c)[7]) {
    if constexpr (sizeof(T) == 8 && TCMP_SINCOS6) {
        bool fast = true;
#pragma unroll
        for (int j = 1; j < 7; ++j) fast = fast && ((hi_word((double)q[j]) & 0x7fffffff) < 0x40f86a00);  // |x| < 1e5
        if (fast) {
            double r[7], r2[7], ps[7], pc[7];
            int k[7];
#pragma unroll
            for (int j = 1; j < 7; ++j) {
                const double kt = fma((double)q[j], 0.63661977236758134308, 6755399441055744.0);  // rint via 1.5 * 2^52
                k[j] = lo_word(kt);
                const double kd = kt - 6755399441055744.0;
                double t = fma(-kd, 1.57079632673412561417e+00, (double)q[j]);
                t = fma(-kd, 6.07710050630396597660e-11, t);
                r[j] = fma(-kd, 2.02226624871116645580e-21, t);
                r2[j] = r[j] * r[j];
                ps[j] = 1.58969099521155010221e-10;
                pc[j] = -1.13596475577881948265e-11;
            }
#define TCMP_HORNER(SC, CC)                                                         \
    _Pragma("unroll") for (int j = 1; j < 7; ++j) {                                 \
        ps[j] = fma(ps[j], r2[j], SC);                                              \
        pc[j] = fma(pc[j], r2[j], CC);                                              \
    }
            TCMP_HORNER(-2.50507602534068634195e-08, 2.08757232129817482790e-09)
            TCMP_HORNER(2.75573137070700676789e-06, -2.75573143513906633035e-07)
            TCMP_HORNER(-1.98412698298579493134e-04, 2.48015872894767294178e-05)
            TCMP_HORNER(8.33333333332248946124e-03, -1.38888888888741095749e-03)
            TCMP_HORNER(-1.66666666666666324348e-01, 4.16666666666666019037e-02)
#undef TCMP_HORNER
#pragma unroll
            for (int j = 1; j < 7; ++j) {
                const double sn = fma(r[j] * r2[j], ps[j], r[j]);
                const double cs = fma(r2[j] * r2[j], pc[j], fma(-0.5, r2[j], 1.0));
                const double a = (k[j] & 1) ? cs : sn, b = (k[j] & 1) ? sn : cs;   // odd quadrant swaps
                s[j] = (T)((k[j] & 2) ? -a : a);
                c[j] = (T)(((k[j] + 1) & 2) ? -b : b);
            }
            return;
        }
    }
#pragma unroll
    for (int j = 1; j < 7; ++j) sincos_t<T>(q[j], &s[j], &c[j]);
}

// Table-driven form of the same (K1 only; fp64).  x = k h + r with h = pi/512 and k = rint(x / h): (sin, cos)(k h)
// come from a 1024-entry table of correctly rounded values (csrc/sincos_table.inc, staged in shared memory -- the
// lookup runs on the LSU, not the FP64 pipe), and |r| <= 3.1e-3 needs only r - r^3/6 + r^5/120 and
// 1 - r^2/2 + r^4/24 (truncation < 2e-18).  14 FP64 instructions per angle instead of 21; worst abs error 2.3e-16
// (tests/test_rne_core_host.py).  Valid while k h1 is exact, i.e. |x| < 4096 rad; any larger or non-finite angle
// sends the whole state down CUDA's sincos() as before.
struct alignas(16) SinCos { double s, c; };
constexpr int kSinCosTableSize = 1024;
// GLOBAL = false: `tab` is the CTA's shared-memory copy; true: the table is read in place through the read-only
// data cache (kernels whose shared memory is spoken for, or whose torque tests are too sparse to pay for staging).
template <bool GLOBAL = false>
TCMP_FN bool sincos6_table(const double (&q)[7], double (&s)[7], double (&c)[7], const SinCos *__restrict__ tab) {
    bool fast = true;
#pragma unroll
    for (int j = 1; j < 7; ++j) fast = fast && ((hi_word(q[j]) & 0x7fffffff) < 0x40b00000);   // |x| < 4096
    if (!fast) return false;
#pragma unroll
    for (int j = 1; j < 7; ++j) {
        const double kt = fma(q[j], 162.97466172610082 /* 512 / pi */, 6755399441055744.0);   // rint via 1.5 * 2^52
        SinCos e;
#ifdef __CUDA_ARCH__
        if constexpr (GLOBAL) {
            const double2 v = __ldg(reinterpret_cast<const double2 *>(tab) + (lo_word(kt) & (kSinCosTableSize - 1)));
            e.s = v.x;
            e.c = v.y;
        } else
#endif
            e = tab[lo_word(kt) & (kSinCosTableSize - 1)];
        const double kd = kt - 6755399441055744.0;
        // pi/512 = h1 + h2 + ...: fdlibm's 33-bit pieces of pi/2 scaled by 2^-8 (k < 2^20 keeps k h1, k h2 exact)
        double r = fma(-kd, 1.57079632673412561417e+00 / 256, q[j]);
        r = fma(-kd, 6.07710050630396597660e-11 / 256, r);
        const double z = r * r;
        const double sl = fma(r * z, fma(z, 1.0 / 120, -1.0 / 6), r);      // sin r
        const double cm = z * fma(z, 1.0 / 24, -0.5);                      // cos r - 1
        s[j] = fma(e.c, sl, fma(e.s, cm, e.s));                            // sin(kh) cos r + cos(kh) sin r
        c[j] = fma(-e.s, sl, fma(e.c, cm, e.c));                           // cos(kh) cos r - sin(kh) sin r
    }
    return true;
}

// Gravity as rne_core applies it: g + 0 * q[0].  The product is +-0 for a finite joint-1 angle, so the value is g
// exactly, and NaN for a NaN or infinite one.  Joint 1's angle cannot change a torque, but the reference rotates
// by it (rne.py), so a non-finite q[0] gives it NaN torques -- and, since NaN never compares >= a limit, a feasible
// verdict.  Folding q[0] into the base acceleration makes every torque here NaN in the same cases (one FMA).
template <typename T> TCMP_FN T gravity_for(T q0) { return q0 * T(0) + T(kGravity); }

// The recursion proper, given sin / cos of joints 2..7 (s[0], c[0] are never read) and the gravity magnitude.
template <typename T, bool DYN, bool TOOL, typename P = ConstParams>
TCMP_FN void rne_body(const T (&s)[7], const T (&c)[7], const T (&qd)[7], const T (&qdd)[7], T mp_inertial,
                      T mp_tool, T (&tau)[7], const P &p = P(), T gravity = T(kGravity)) {

    V3<T> F[7], N[7];
    Kin<T> k;
    V3<T> gv;  // gravity direction * g in the current frame (only tracked when TOOL && DYN)

    // link 0: w = (0,0,qd0), wd = (0,0,qdd0), vd = (0,0,g) -- its own wrench only matters through
    // tau_0 = N_0.z = Jzz qdd0 (the w x Jw and h x vd terms have no z component).
    // link 1 (alpha = -pi/2, P = 0): E (0,0,z) = (-s z, -c z, 0)
    if constexpr (DYN) {
        k.w = {-s[1] * qd[0], -c[1] * qd[0], qd[1]};
        k.wd = {-s[1] * qdd[0] + k.w.y * qd[1], -c[1] * qdd[0] - k.w.x * qd[1], qdd[1]};
    }
    k.vd = {-s[1] * gravity, -c[1] * gravity, T(0)};
    if constexpr (TOOL && DYN) gv = k.vd;
    link_wrench_const<1, T, DYN>(p, k, F[1], N[1]);

#define TCMP_FWD(K)                                                        \
    forward_link<K, T, DYN>(c[K], s[K], qd[K], qdd[K], k);                 \
    if constexpr (TOOL && DYN) gv = rot_in<link_const(K).alpha>(c[K], s[K], gv);
    TCMP_FWD(2) link_wrench_const<2, T, DYN>(p, k, F[2], N[2]);
    TCMP_FWD(3) link_wrench_const<3, T, DYN>(p, k, F[3], N[3]);
    TCMP_FWD(4) link_wrench_const<4, T, DYN>(p, k, F[4], N[4]);
    TCMP_FWD(5) link_wrench_const<5, T, DYN>(p, k, F[5], N[5]);
    TCMP_FWD(6)
#undef TCMP_FWD
    {
        T tool_z;
        if constexpr (kIsConst<P>) {
            constexpr LinkConst L = link_const(6);
            const T m6 = T(L.m) + mp_inertial;
            const T hz6 = T(L.hz) + mp_inertial * T(kPayloadHz);
            const T jxx6 = T(L.jxx) + mp_inertial * T(kPayloadJ);
            const T jyy6 = T(L.jyy) + mp_inertial * T(kPayloadJ);
            link_wrench<T, DYN, true, true, true>(k, m6, T(L.hx), T(L.hy), hz6, jxx6, T(L.jxy), T(L.jxz), jyy6,
                                                  T(L.jyz), T(L.jzz), F[6], N[6]);
            tool_z = T(kToolZ);
        } else {
            const T *l = p.l6;
            link_wrench<T, DYN, true, true, true>(k, l[0] + mp_inertial, l[1], l[2], l[3] + mp_inertial * p.payload_hz,
                                                  l[4] + mp_inertial * p.payload_j, l[5], l[6],
                                                  l[7] + mp_inertial * p.payload_j, l[8], l[9], F[6], N[6]);
            tool_z = p.tool_z;
        }
        if constexpr (TOOL) {
            const V3<T> &g6 = DYN ? gv : k.vd;   // static: vd is exactly the rotated gravity vector
            const T fx = mp_tool * g6.x, fy = mp_tool * g6.y, fz = mp_tool * g6.z;
            F[6].x += fx; F[6].y += fy; F[6].z += fz;
            N[6].x -= tool_z * fy;   // r x f, r = (0,0,tool_z)
            N[6].y += tool_z * fx;
        }
    }

    // backward pass
    tau[6] = N[6].z;
    backward_link<6, T>(c[6], s[6], F[6], N[6], F[5], N[5]); tau[5] = N[5].z;
    backward_link<5, T>(c[5], s[5], F[5], N[5], F[4], N[4]); tau[4] = N[4].z;
    backward_link<4, T>(c[4], s[4], F[4], N[4], F[3], N[3]); tau[3] = N[3].z;
    backward_link<3, T>(c[3], s[3], F[3], N[3], F[2], N[2]); tau[2] = N[2].z;
    backward_link<2, T>(c[2], s[2], F[2], N[2], F[1], N[1]); tau[1] = N[1].z;
    // link 1 -> link 0: only n_0.z is needed; alpha_1 = -pi/2, P_1 = 0:  (R n).z = -(s n.x + c n.y)
    T t0 = -(s[1] * N[1].x + c[1] * N[1].y);
    if constexpr (DYN) {
        if constexpr (kIsConst<P>) t0 += T(link_const(0).jzz) * qdd[0];
        else t0 += p.jzz0 * qdd[0];
    }
    tau[0] = t0;
}

template <typename T, bool DYN, bool TOOL, typename P = ConstParams>
TCMP_FN void rne_core(const T (&q)[7], const T (&qd)[7], const T (&qdd)[7], T mp_inertial, T mp_tool, T (&tau)[7],
                      const P &p = P()) {
    T c[7], s[7];
    sincos6<T>(q, s, c);
    rne_body<T, DYN, TOOL, P>(s, c, qd, qdd, mp_inertial, mp_tool, tau, p, gravity_for(q[0]));
}

// K1's form: sin / cos from the table (shared-memory copy, or GLOBAL = in place) when every angle allows it.
template <bool DYN, bool TOOL, typename P = ConstParams, bool GLOBAL = false>
TCMP_FN void rne_core_table(const double (&q)[7], const double (&qd)[7], const double (&qdd)[7], double mp_inertial,
                            double mp_tool, double (&tau)[7], const SinCos *__restrict__ tab, const P &p = P()) {
    double c[7], s[7];
    if (!sincos6_table<GLOBAL>(q, s, c, tab)) {
#pragma unroll
        for (int j = 1; j < 7; ++j) sincos_t<double>(q[j], &s[j], &c[j]);
    }
    rne_body<double, DYN, TOOL, P>(s, c, qd, qdd, mp_inertial, mp_tool, tau, p, gravity_for(q[0]));
}

// |tau_i| < limit_i for i in 0..5 (panda_primitives.py:182-183; joint 7 is never tested).
template <typename T> TCMP_FN bool within_limits(const T (&tau)[7]) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 6; ++i) ok = ok && !(fabs(tau[i]) >= T(torque_limit(i)));
    return ok;
}
template <typename T> TCMP_FN bool within_limits(const T (&tau)[7], const RtParams<T> &p) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 6; ++i) ok = ok && !(fabs(tau[i]) >= p.limit[i]);
    return ok;
}

template <typename T, typename P> TCMP_FN bool limits_ok(const T (&tau)[7], const P &p) {
    if constexpr (kIsConst<P>) return within_limits<T>(tau);
    else return within_limits<T>(tau, p);
}

}  // namespace tcmp
