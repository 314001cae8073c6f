// fd_kernels.cu -- K13 (tcmp_forward_dynamics_batch): joint accelerations qdd = M^-1 (tau - h) and, on request, M^-1
// per state.  The per-state code is csrc/fd_core.cuh.  Launch pattern as K10 (dynamics_kernels.cu): one thread per
// state in 128-thread CTAs, no grid-stride loop, SoA inputs [7][n] read with streaming loads, outputs stored with
// streaming stores, the sin/cos table read in place through the read-only cache, and which outputs are computed a
// uniform run-time branch on the output pointers.  One kernel per (index type, mode, parameter source).
#include "fd_core.cuh"
#include "tcmp_internal.h"

namespace tcmp {

static __device__ const SinCos kFdSinCosTable[kSinCosTableSize] = {
#include "sincos_table.inc"
};

template <typename I, bool TOOL, typename P>
__global__ void __launch_bounds__(128)
forward_dynamics_kernel(I n, const double *__restrict__ q, const double *__restrict__ qd,
                        const double *__restrict__ tau, const double *__restrict__ payload_mass,
                        double payload_scalar, double *__restrict__ qdd_out, double *__restrict__ Minv_out,
                        const __grid_constant__ P p) {
    const I i = (I)blockIdx.x * (I)blockDim.x + (I)threadIdx.x;
    if (i >= n) return;
    const double mass = payload_mass ? __ldcs(payload_mass + i) : payload_scalar;
    fd_state<I, TOOL, P, true>(n, i, q, qd, tau, mass, p, kFdSinCosTable, qdd_out, Minv_out);
}

template <typename I, bool TOOL, typename P>
static cudaError_t launch_fd(int64_t n, const double *q, const double *qd, const double *tau, const double *pm,
                             double ps, double *qdd, double *Minv, const P &p, cudaStream_t st) {
    const int64_t grid = (n + 127) / 128;
    forward_dynamics_kernel<I, TOOL, P><<<(unsigned)grid, 128, 0, st>>>((I)n, q, qd, tau, pm, ps, qdd, Minv, p);
    return cudaGetLastError();
}

template <bool TOOL, typename P>
static cudaError_t launch_indexed_fd(int64_t n, const double *q, const double *qd, const double *tau,
                                     const double *pm, double ps, double *qdd, double *Minv, const P &p,
                                     cudaStream_t st) {
    if (fits_int49(n)) return launch_fd<int, TOOL, P>(n, q, qd, tau, pm, ps, qdd, Minv, p, st);
    return launch_fd<int64_t, TOOL, P>(n, q, qd, tau, pm, ps, qdd, Minv, p, st);
}

template <typename P>
static cudaError_t launch_mode_fd(int mode, int64_t n, const double *q, const double *qd, const double *tau,
                                  const double *pm, double ps, double *qdd, double *Minv, const P &p, cudaStream_t st) {
    if (mode == TCMP_MODE_DYN) return launch_indexed_fd<true, P>(n, q, qd, tau, pm, ps, qdd, Minv, p, st);
    return launch_indexed_fd<false, P>(n, q, qd, tau, pm, ps, qdd, Minv, p, st);
}

cudaError_t launch_forward_dynamics(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                    const double *tau, const double *pm, double ps, double *qdd, double *Minv,
                                    cudaStream_t st) {
    if (model) return launch_mode_fd(mode, n, q, qd, tau, pm, ps, qdd, Minv, params_from_desc<double>(*model), st);
    return launch_mode_fd(mode, n, q, qd, tau, pm, ps, qdd, Minv, ConstParams(), st);
}

}  // namespace tcmp
