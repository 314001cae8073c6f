// track_kernels.cu -- K15 (tcmp_track_batch): closed-loop tracking rollouts, a computed-torque controller with torque
// saturation driving K14's RK4 plant.  The per-rollout code is csrc/track_core.cuh.  Launch pattern as K14
// (rollout_kernels.cu): one thread per rollout in 128-thread CTAs, no grid-stride loop, the sin/cos table read in
// place; each thread's state lives in its column of a [kTrackRows][128] shared array (45 KB per CTA).  One kernel per
// (index type, mode, parameter source).
#include "track_core.cuh"
#include "tcmp_internal.h"

namespace tcmp {

static __device__ const SinCos kTrackSinCosTable[kSinCosTableSize] = {
#include "sincos_table.inc"
};

template <typename I, bool TOOL, typename P>
__global__ void __launch_bounds__(128)
track_kernel(const __grid_constant__ TrackArgs a, const __grid_constant__ P p) {
    __shared__ double scratch[kTrackRows][128];
    const I i = (I)blockIdx.x * (I)blockDim.x + (I)threadIdx.x;
    if (i >= (I)a.roll.n) return;
    track_state<I, TOOL, P, true>(a, i, p, kTrackSinCosTable, &scratch[0][threadIdx.x], 128);
}

template <typename I, bool TOOL, typename P>
static cudaError_t launch_track_p(const TrackArgs &a, const P &p, cudaStream_t st) {
    const int64_t grid = (a.roll.n + 127) / 128;
    track_kernel<I, TOOL, P><<<(unsigned)grid, 128, 0, st>>>(a, p);
    return cudaGetLastError();
}

// 32-bit element offsets while the largest -- 7 n n_steps - 1 (a trajectory element) and, for per-rollout
// coefficients, 42 n_seg n - 1 -- fits in 31 bits
static bool fits_track_int(const TrackArgs &a) {
    const int64_t big = 0x7fffffff;
    if (a.roll.n > big / (7 * (int64_t)a.roll.n_steps)) return false;
    return a.coeffs_broadcast || a.roll.n <= big / (42 * (int64_t)a.n_seg);
}

template <typename P> static cudaError_t launch_mode_track(int mode, const TrackArgs &a, const P &p, cudaStream_t st) {
    const bool small = fits_track_int(a);
    if (mode == TCMP_MODE_DYN)
        return small ? launch_track_p<int, true>(a, p, st) : launch_track_p<int64_t, true>(a, p, st);
    return small ? launch_track_p<int, false>(a, p, st) : launch_track_p<int64_t, false>(a, p, st);
}

cudaError_t launch_track(const tcmp_model *model, int mode, int64_t n, int n_steps, double dt, int n_seg,
                         const double *coeffs, int coeffs_broadcast, const double *q0, const double *qd0,
                         const double *kp, const double *kd, const double *pm, double ps, const double *cm, double cs,
                         const double *q_lo, const double *q_hi, const double *qd_max, double *q_out, double *qd_out,
                         double *q_traj, double *qd_traj, double *tau_traj, int32_t *fv, int32_t *fs,
                         double *max_err, cudaStream_t st) {
    TrackArgs a{};
    a.roll = RollArgs{n, n_steps, dt, q0, qd0, nullptr, 0, pm, ps, {}, q_out, qd_out, q_traj, qd_traj, fv};
    a.roll.lim.check_q = q_lo != nullptr;
    a.roll.lim.check_qd = qd_max != nullptr;
    tcmp_model stock;
    if (!model) default_model_desc(&stock);
    const tcmp_model &m = model ? *model : stock;
    for (int j = 0; j < 7; ++j) {
        a.roll.lim.lo[j] = q_lo ? q_lo[j] : 0.0;
        a.roll.lim.hi[j] = q_hi ? q_hi[j] : 0.0;
        a.roll.lim.qd_max[j] = qd_max ? qd_max[j] : 0.0;
        a.kp[j] = kp[j];
        a.kd[j] = kd[j];
        a.tau_limit[j] = m.torque_limit[j];
    }
    a.n_seg = n_seg;
    a.coeffs_broadcast = coeffs_broadcast != 0;
    a.coeffs = coeffs;
    a.ctrl_mass = cm;
    a.ctrl_scalar = cs;
    a.tau_traj = tau_traj;
    a.max_err = max_err;
    a.first_saturation = fs;
    if (model) return launch_mode_track(mode, a, params_from_desc<double>(*model), st);
    return launch_mode_track(mode, a, ConstParams(), st);
}

}  // namespace tcmp
