// collision_core.cuh -- the per-configuration and per-edge arithmetic of K8 (collision_kernel) and K9
// (extend_prefix_kernel): the scene record, the link-sphere model of collision.py, the joint-limit test and the
// extend-step generator of utils.get_extend_fn / get_refine_fn (utils.py:3031-3041, 3068-3077).
//
// It is plain arithmetic, so the same source also builds for the host: tests/native/collision_host.cpp compiles it
// with g++ (-ffp-contract=off) and checks it against a long-double reference on a CPU-only box.  libtcmp.so
// contains only the device code; there is no CPU path in the product.
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/tcmp.h"

// Under nvcc these are device functions: the sphere tables are __device__ arrays, which host code cannot read, and
// the library has no host caller.  g++ builds them as ordinary inline functions for the test harness.
#ifdef __CUDACC__
#define TCMP_CC __device__
#define TCMP_CC_INLINE __device__ __forceinline__
#define TCMP_CC_CONST __device__ constexpr
#else
#define TCMP_CC inline
#define TCMP_CC_INLINE inline
#define TCMP_CC_CONST constexpr
#endif

namespace tcmp {

struct Scene {
    int n_obs;
    int kind[TCMP_MAX_OBSTACLES];            // 0 = box, 1 = sphere
    double c[TCMP_MAX_OBSTACLES][3];         // centre
    double h[TCMP_MAX_OBSTACLES][3];         // box half extents; sphere: h[0] = radius
    double lo[7], hi[7];                     // joint limits (limits_fn, utils.py:3177)
    double payload_radius;                   // > 0: a sphere at the grasp target (held object)
};

// Fills S from the C-ABI arguments; the caller has checked 0 <= n_obs <= TCMP_MAX_OBSTACLES.  Unused slots are zero.
inline void fill_scene(int n_obs, const tcmp_obstacle *obs, const double *q_lo, const double *q_hi,
                       double payload_radius, Scene *S) {
    S->n_obs = n_obs;
    for (int o = 0; o < TCMP_MAX_OBSTACLES; ++o) {
        S->kind[o] = o < n_obs ? obs[o].kind : 0;
        for (int r = 0; r < 3; ++r) {
            S->c[o][r] = o < n_obs ? obs[o].center[r] : 0.0;
            S->h[o][r] = o < n_obs ? obs[o].half[r] : 0.0;
        }
    }
    for (int j = 0; j < 7; ++j) {
        S->lo[j] = q_lo[j];
        S->hi[j] = q_hi[j];
    }
    S->payload_radius = payload_radius;
}

// Operations rounded once each, in the order written (numpy's float64 arithmetic): the device intrinsics forbid
// contraction into an FMA; the host harness is built with -ffp-contract=off, so plain operators round the same way.
#ifdef __CUDA_ARCH__
__device__ __forceinline__ double rn_div(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ double rn_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double rn_add(double a, double b) { return __dadd_rn(a, b); }
#else
inline double rn_div(double a, double b) { return a / b; }
inline double rn_mul(double a, double b) { return a * b; }
inline double rn_add(double a, double b) { return a + b; }
#endif

// Link-sphere model of collision.py (_SEGMENTS): spheres strung between consecutive DH frame origins
// 1..7 and the grasp target (8).
TCMP_CC_CONST int kSegCount = 7;
TCMP_CC_CONST int kSegSamples[kSegCount] = {3, 2, 4, 2, 2, 2, 3};
TCMP_CC_CONST double kSegRadius[kSegCount] = {0.07, 0.07, 0.065, 0.06, 0.055, 0.05, 0.05};

TCMP_CC_INLINE bool sphere_hits(const Scene &S, double x, double y, double z, double r) {
    bool hit = false;
    for (int o = 0; o < S.n_obs; ++o) {
        const double dx = x - S.c[o][0], dy = y - S.c[o][1], dz = z - S.c[o][2];
        if (S.kind[o] == 1) {
            hit = hit || (sqrt(dx * dx + dy * dy + dz * dz) < r + S.h[o][0]);
        } else {
            // np.maximum(delta, 0.0): a NaN (non-finite joint angle) stays NaN and then hits nothing, as in the
            // stand-in.  fmax would return the 0.0 and report a hit.
            const double dxo = fabs(dx) - S.h[o][0], dyo = fabs(dy) - S.h[o][1], dzo = fabs(dz) - S.h[o][2];
            const double ex = dxo < 0.0 ? 0.0 : dxo, ey = dyo < 0.0 ? 0.0 : dyo, ez = dzo < 0.0 ? 0.0 : dzo;
            hit = hit || (sqrt(ex * ex + ey * ey + ez * ez) < r);
        }
    }
    return hit;
}

// collision.py get_collision_fn.batch for one configuration
TCMP_CC bool config_collides(const Scene &S, const double (&q)[7]) {
    bool out = false;
#pragma unroll
    for (int j = 0; j < 7; ++j) out = out || (q[j] < S.lo[j]) || (q[j] > S.hi[j]);
    if (out || S.n_obs == 0) return out;
    // origins of DH frames 0..7 and the grasp target (collision.link_frames)
    double O[9][3];
    double X[3] = {1, 0, 0}, Y[3] = {0, 1, 0}, Z[3] = {0, 0, 1}, p[3] = {0, 0, 0};
    const double A[7] = {0, 0, 0, 0.0825, -0.0825, 0, 0.088};
    const double D[7] = {0.333, 0, 0.316, 0, 0.384, 0, 0};
    const int AL[7] = {0, -1, 1, 1, -1, 1, 1};
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        double s, c;
        sincos(q[k], &s, &c);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const double y = AL[k] == 0 ? Y[r] : (AL[k] > 0 ? Z[r] : -Z[r]);
            const double z = AL[k] == 0 ? Z[r] : (AL[k] > 0 ? -Y[r] : Y[r]);
            p[r] += A[k] * X[r] + D[k] * z;
            const double x = X[r];
            X[r] = c * x + s * y;
            Y[r] = c * y - s * x;
            Z[r] = z;
            O[k][r] = p[r];
        }
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        O[7][r] = p[r] + 0.107 * Z[r];
        O[8][r] = O[7][r] + 0.105 * Z[r];
    }
    bool hit = false;
#pragma unroll
    for (int g = 0; g < kSegCount; ++g) {
        const int a = g + 1, b = g + 2, m = kSegSamples[g];
        for (int i = 0; i < m; ++i) {
            const double t = (double)i / (double)(m - 1);   // np.linspace(0, 1, m)
            const double x = (1 - t) * O[a][0] + t * O[b][0], y = (1 - t) * O[a][1] + t * O[b][1],
                         z = (1 - t) * O[a][2] + t * O[b][2];
            hit = hit || sphere_hits(S, x, y, z, kSegRadius[g]);
        }
    }
    if (S.payload_radius > 0) hit = hit || sphere_hits(S, O[8][0], O[8][1], O[8][2], S.payload_radius);
    return hit;
}

// Number of configurations on the edge a -> b: int(np.linalg.norm((b - a) / res)) + 1 (utils.py:3074), with the sum
// of squares rounded in joint order: nrm2 = extend_norm2_add(nrm2, a[j], b[j], res[j]) for j = 0..6 from 0.0, then
// extend_num_configs(nrm2).  A non-finite norm (NaN / inf end point) has no step count: 0 configurations, so the host
// never truncates a sequence with it (the cast of a NaN to int is undefined); a huge finite norm gives 0 for the same
// reason.
TCMP_CC_INLINE double extend_norm2_add(double nrm2, double a, double b, double res) {
    const double d = rn_div(rn_add(b, -a), res);   // np.divide(difference, resolutions)
    return rn_add(nrm2, rn_mul(d, d));
}

TCMP_CC_INLINE int extend_num_configs(double nrm2) {
    const double nrm = sqrt(nrm2);
    const bool sane = nrm == nrm && nrm < 1.0e6;
    return sane ? (int)nrm + 1 : 0;
}

// Configuration k (0-based, k < N) of the N-configuration edge a -> b, by the get_refine_fn recurrence
// (utils.py:3036-3039): q <- (1 / (N - i)) * (b - q) + q for i = 0..k, starting from q = a.
TCMP_CC_INLINE void extend_config(const double (&a)[7], const double (&b)[7], int N, int k, double (&q)[7]) {
#pragma unroll
    for (int j = 0; j < 7; ++j) q[j] = a[j];
    for (int i = 0; i <= k; ++i) {
        const double w = rn_div(1.0, (double)(N - i));
#pragma unroll
        for (int j = 0; j < 7; ++j) q[j] = rn_add(rn_mul(w, rn_add(b[j], -q[j])), q[j]);
    }
}

}  // namespace tcmp
