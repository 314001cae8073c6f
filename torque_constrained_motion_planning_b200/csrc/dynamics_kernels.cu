// dynamics_kernels.cu -- K10 (tcmp_dynamics_batch): M(q), C(q, qd), g(q) and the tool-point Jacobian J(q) per state.
//
// Replaces what the reference's `dyn` torque test imports from panda_dynamics_model (get_mass_matrix,
// get_coriolis_matrix, get_gravity_vector; panda_primitives.py:86-91) and PyBullet's calculateJacobian (:93-99), for
// many states per launch.  The per-state code is csrc/dynamics_core.cuh.  One thread per state, SoA inputs [7][n]
// read with streaming loads, every output element stored with a streaming store as soon as it is final (the
// outputs, up to 1 176 B per state, are write-once).  Which terms are computed is a uniform run-time branch on the
// output pointers: one kernel per parameter source, not one per output subset.  Table-driven sincos as in K1.
#include "dynamics_core.cuh"
#include "tcmp_internal.h"

namespace tcmp {

static __device__ const SinCos kDynSinCosTable[kSinCosTableSize] = {
#include "sincos_table.inc"
};

// One state per thread and no grid-stride loop: with a loop, ptxas hoists the 147 loop-invariant output offsets
// (r*7 + c)*n out of it and spills; the table is read in place through the read-only cache (16 KB, L1-resident)
// instead of being staged per 128-thread CTA.
template <typename I, typename P>
__global__ void __launch_bounds__(128)
dynamics_kernel(I n, const double *__restrict__ q, const double *__restrict__ qd, const double *__restrict__ payload_mass,
                double payload_scalar, double *__restrict__ M_out, double *__restrict__ C_out,
                double *__restrict__ g_out, double *__restrict__ J_out, const __grid_constant__ P p) {
    const I i = (I)blockIdx.x * (I)blockDim.x + (I)threadIdx.x;
    if (i >= n) return;
    DynOut<I> out{M_out, C_out, g_out, J_out, n, i};
    const double mass = payload_mass ? __ldcs(payload_mass + i) : payload_scalar;
    dynamics_state<I, P, true>(n, i, q, qd, mass, p, kDynSinCosTable, out);
}

template <typename I, typename P>
static cudaError_t launch_dyn(int64_t n, const double *q, const double *qd, const double *pm, double ps, double *M,
                              double *C, double *g, double *J, const P &p, cudaStream_t st) {
    const int64_t grid = (n + 127) / 128;
    dynamics_kernel<I, P><<<(unsigned)grid, 128, 0, st>>>((I)n, q, qd, pm, ps, M, C, g, J, p);
    return cudaGetLastError();
}

template <typename P>
static cudaError_t launch_indexed_dyn(int64_t n, const double *q, const double *qd, const double *pm, double ps,
                                      double *M, double *C, double *g, double *J, const P &p, cudaStream_t st) {
    if (fits_int49(n)) return launch_dyn<int, P>(n, q, qd, pm, ps, M, C, g, J, p, st);
    return launch_dyn<int64_t, P>(n, q, qd, pm, ps, M, C, g, J, p, st);
}

cudaError_t launch_dynamics_batch(const tcmp_model *model, int64_t n, const double *q, const double *qd,
                                  const double *pm, double ps, double *M, double *C, double *g, double *J,
                                  cudaStream_t st) {
    if (model) return launch_indexed_dyn(n, q, qd, pm, ps, M, C, g, J, params_from_desc<double>(*model), st);
    return launch_indexed_dyn(n, q, qd, pm, ps, M, C, g, J, ConstParams(), st);
}

}  // namespace tcmp
