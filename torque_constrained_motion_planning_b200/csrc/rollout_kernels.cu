// rollout_kernels.cu -- K14 (tcmp_rollout_batch): RK4 forward-dynamics rollouts under a held or per-step torque, with
// the first joint- or velocity-limit violation.  The per-rollout code is csrc/rollout_core.cuh.  Launch pattern as K13
// (fd_kernels.cu): one thread per rollout in 128-thread CTAs, no grid-stride loop, SoA inputs read with streaming
// loads, outputs stored with streaming stores, the sin/cos table read in place through the read-only cache.  Each
// thread's RK4 state lives in its column of a [kRollRows][128] shared array (44 KB per CTA).  One kernel per (index
// type, mode, parameter source).
#include "rollout_core.cuh"
#include "tcmp_internal.h"

namespace tcmp {

static __device__ const SinCos kRollSinCosTable[kSinCosTableSize] = {
#include "sincos_table.inc"
};

template <typename I, bool TOOL, typename P>
__global__ void __launch_bounds__(128)
rollout_kernel(const __grid_constant__ RollArgs a, const __grid_constant__ P p) {
    __shared__ double scratch[kRollRows][128];
    const I i = (I)blockIdx.x * (I)blockDim.x + (I)threadIdx.x;
    if (i >= (I)a.n) return;
    rollout_state<I, TOOL, P, true>(a, i, p, kRollSinCosTable, &scratch[0][threadIdx.x], 128);
}

template <typename I, bool TOOL, typename P>
static cudaError_t launch_roll(const RollArgs &a, const P &p, cudaStream_t st) {
    const int64_t grid = (a.n + 127) / 128;
    rollout_kernel<I, TOOL, P><<<(unsigned)grid, 128, 0, st>>>(a, p);
    return cudaGetLastError();
}

// 32-bit element offsets while the largest, 7 n n_steps - 1 (a trajectory or per-step torque element), fits in 31 bits
static bool fits_roll_int(int64_t n, int n_steps) { return n <= (int64_t)0x7fffffff / (7 * (int64_t)n_steps); }

template <typename P> static cudaError_t launch_mode_roll(int mode, const RollArgs &a, const P &p, cudaStream_t st) {
    const bool small = fits_roll_int(a.n, a.n_steps);
    if (mode == TCMP_MODE_DYN) return small ? launch_roll<int, true>(a, p, st) : launch_roll<int64_t, true>(a, p, st);
    return small ? launch_roll<int, false>(a, p, st) : launch_roll<int64_t, false>(a, p, st);
}

cudaError_t launch_rollout(const tcmp_model *model, int mode, int64_t n, int n_steps, double dt, const double *q0,
                           const double *qd0, const double *tau, int tau_per_step, const double *pm, double ps,
                           const double *q_lo, const double *q_hi, const double *qd_max, double *q_out,
                           double *qd_out, double *q_traj, double *qd_traj, int32_t *fv, cudaStream_t st) {
    RollArgs a{n, n_steps, dt, q0, qd0, tau, tau_per_step, pm, ps, {}, q_out, qd_out, q_traj, qd_traj, fv};
    a.lim.check_q = q_lo != nullptr;
    a.lim.check_qd = qd_max != nullptr;
    for (int j = 0; j < 7; ++j) {
        a.lim.lo[j] = q_lo ? q_lo[j] : 0.0;
        a.lim.hi[j] = q_hi ? q_hi[j] : 0.0;
        a.lim.qd_max[j] = qd_max ? qd_max[j] : 0.0;
    }
    if (model) return launch_mode_roll(mode, a, params_from_desc<double>(*model), st);
    return launch_mode_roll(mode, a, ConstParams(), st);
}

}  // namespace tcmp
