// collision_kernels.cu -- SURVEY.md 8f-1/8f-2: the synthetic-scene collision predicate on the GPU, fused IN
// FRONT of the torque test so that RRT* tree growth checks whole candidate edges in one launch.
//
// The reference's collision predicate is PyBullet's (utils.get_collision_fn, utils.py:3165-3218), out of scope
// and not installed; planner-level runs use the stand-in defined in collision.py (joint-limit test as in
// utils.py:3177-3178, then link spheres from the DH forward kinematics against axis-aligned boxes / spheres).
// These kernels implement exactly that stand-in, keep the reference's evaluation ORDER -- collision first,
// torque only for collision-free configurations (rrt_star.py:92-96) -- and generate the extend steps of
// utils.get_extend_fn / get_refine_fn (utils.py:3031-3041, 3068-3077) on the fly.
//
//   collision_kernel       1 thread = 1 configuration            -> hit[n]
//   extend_prefix_kernel   1 warp   = 1 candidate edge q1 -> q2; lanes = extend steps (32 per round);
//                          __ballot_sync / __ffs gives the safe-prefix length (safe_path_force_aware,
//                          rrt_star.py:90-98); the warp stops at the first round containing a failure.
#include "panda_model.cuh"
#include "tcmp_internal.h"

namespace tcmp {

// (sin, cos)(i pi / 512) for the table-driven sincos of the static torque tests (panda_model.cuh sincos6_table<GLOBAL>):
// read in place through the read-only cache -- this kernel's shared memory is spoken for, and its torque tests are
// too few per CTA to pay for staging 16 KB.  Own copy per translation unit (no relocatable device code in the build).
static __device__ const SinCos kExtSinCosTable[kSinCosTableSize] = {
#include "sincos_table.inc"
};

}  // namespace tcmp

// Included after kExtSinCosTable so that the table keeps the first slot of the kernels' global-address constant bank.
#include "collision_core.cuh"

namespace tcmp {

__global__ void __launch_bounds__(128)
collision_kernel(int64_t n, const double *__restrict__ q, Scene S, uint8_t *__restrict__ hit_out) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double qs[7];
#pragma unroll
        for (int j = 0; j < 7; ++j) qs[j] = __ldg(q + j * n + i);
        hit_out[i] = (uint8_t)config_collides(S, qs);
    }
}

template <bool TOOL, typename P>
__global__ void __launch_bounds__(128)
extend_prefix_kernel(int64_t n_edges, const double *__restrict__ q1, const double *__restrict__ q2, Scene S,
                     double r0, double r1, double r2, double r3, double r4, double r5, double r6, int check_torque,
                     double mass, double payload_threshold, int32_t *__restrict__ n_steps_out,
                     int32_t *__restrict__ prefix_out, const __grid_constant__ P prm) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const double res[7] = {r0, r1, r2, r3, r4, r5, r6};
    const double mp_inertial = TOOL ? 0.0 : (mass > payload_threshold ? mass : 0.0);
    const double mp_tool = TOOL ? mass : 0.0;
    for (int64_t e = warp; e < n_edges; e += n_warps) {
        double a[7], b[7];
        double nrm2 = 0.0;
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            a[j] = __ldg(q1 + j * n_edges + e);
            b[j] = __ldg(q2 + j * n_edges + e);
            nrm2 = extend_norm2_add(nrm2, a[j], b[j], res[j]);
        }
        const int N = extend_num_configs(nrm2);   // 0 for a non-finite or huge norm
        int prefix = N;
        for (int base = 0; base < N; base += 32) {
            const int k = base + lane;
            const bool active = k < N;
            double q[7];
            extend_config(a, b, N, active ? k : N - 1, q);
            bool bad = config_collides(S, q);
            if (!bad && check_torque) {   // torque only for collision-free configurations (rrt_star.py:92-96)
                double tau[7];
                const double z[7] = {0, 0, 0, 0, 0, 0, 0};
                rne_core_table<false, TOOL, P, true>(q, z, z, mp_inertial, mp_tool, tau, kExtSinCosTable, prm);   // table read in place (__ldg)
                bad = !limits_ok<double, P>(tau, prm);
            }
            const unsigned fails = __ballot_sync(0xffffffffu, active && bad);
            if (fails) {
                prefix = base + __ffs(fails) - 1;
                break;
            }
        }
        if (lane == 0) {
            n_steps_out[e] = N;
            prefix_out[e] = prefix;
        }
    }
}

static cudaError_t make_scene(int n_obs, const tcmp_obstacle *obs, const double *q_lo, const double *q_hi,
                              double payload_radius, Scene *S) {
    if (n_obs < 0 || n_obs > TCMP_MAX_OBSTACLES) return cudaErrorInvalidValue;
    fill_scene(n_obs, obs, q_lo, q_hi, payload_radius, S);
    return cudaSuccess;
}

cudaError_t launch_collision_batch(int64_t n, const double *q, int n_obs, const tcmp_obstacle *obs,
                                   const double *q_lo, const double *q_hi, double payload_radius, uint8_t *hit_out,
                                   cudaStream_t st) {
    Scene S;
    cudaError_t e = make_scene(n_obs, obs, q_lo, q_hi, payload_radius, &S);
    if (e != cudaSuccess) return e;
    const int grid = grid_for(reinterpret_cast<const void *>(collision_kernel), 128, n);
    collision_kernel<<<grid, 128, 0, st>>>(n, q, S, hit_out);
    return cudaGetLastError();
}

template <bool TOOL, typename P>
static cudaError_t launch_extend_p(int64_t n_edges, const double *q1, const double *q2, const Scene &S, const double *res,
                                   int check, double mass, double payload_threshold, int32_t *n_steps_out,
                                   int32_t *prefix_out, const P &prm, cudaStream_t st) {
    auto kern = extend_prefix_kernel<TOOL, P>;
    const int grid = grid_for(reinterpret_cast<const void *>(kern), 128, n_edges * 32);
    kern<<<grid, 128, 0, st>>>(n_edges, q1, q2, S, res[0], res[1], res[2], res[3], res[4], res[5], res[6], check, mass,
                               payload_threshold, n_steps_out, prefix_out, prm);
    return cudaGetLastError();
}

template <bool TOOL>
static cudaError_t launch_extend_t(int64_t n_edges, const double *q1, const double *q2, const Scene &S, const double *res,
                                   int check, double mass, double payload_threshold, int32_t *n_steps_out,
                                   int32_t *prefix_out, const tcmp_model *model, cudaStream_t st) {
    if (model)
        return launch_extend_p<TOOL>(n_edges, q1, q2, S, res, check, mass, payload_threshold, n_steps_out, prefix_out,
                                     params_from_desc<double>(*model), st);
    return launch_extend_p<TOOL>(n_edges, q1, q2, S, res, check, mass, payload_threshold, n_steps_out, prefix_out,
                                 ConstParams(), st);
}

cudaError_t launch_extend_prefix(int mode, int64_t n_edges, const double *q1, const double *q2,
                                 const double *res, int n_obs, const tcmp_obstacle *obs, const double *q_lo,
                                 const double *q_hi, double payload_radius, double mass, double payload_threshold,
                                 int32_t *n_steps_out, int32_t *prefix_out, cudaStream_t st, const tcmp_model *model) {
    Scene S;
    cudaError_t e = make_scene(n_obs, obs, q_lo, q_hi, payload_radius, &S);
    if (e != cudaSuccess) return e;
    const int check = mode != TCMP_MODE_BASE;
    if (mode == TCMP_MODE_DYN)
        return launch_extend_t<true>(n_edges, q1, q2, S, res, check, mass, payload_threshold, n_steps_out, prefix_out,
                                     model, st);
    return launch_extend_t<false>(n_edges, q1, q2, S, res, check, mass, payload_threshold, n_steps_out, prefix_out,
                                  model, st);
}

}  // namespace tcmp
