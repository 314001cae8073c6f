// tcmp_internal.h -- declarations shared by the kernel translation units and the C-ABI shim.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tcmp.h"

namespace tcmp {

// Persistent-style grid: `waves` x enough CTAs to fill every SM at the kernel's occupancy, never more than the
// work needs.  148 SMs on B200; the count is read from the device so a grid is always a whole number of waves.
// One wave minimises CTA launches; a few waves let retiring CTAs be replaced, which matters when units differ in
// cost (edges stop at their first failing waypoint, IK solves die at different gates) or warps run ahead.
int grid_for(const void *kernel, int block, int64_t n_threads_needed, int waves = 1);
// Measured (profiles/r01/ab_variants_aux_waves.log): edges +7 % and goal-IK selection +8 % at 16 waves; the IK
// sweep kernel LOSES with more waves (every retiring CTA flushes a partly filled survivor queue), as does the
// single-buffered model kernel, so those stay at one.
constexpr int kEdgeWaves = 16;
constexpr int kSelWaves = 16;
int sm_count();

// out[i] = v for i < n (used by the `base` torque test, which is constant-true).
template <typename T> __global__ void fill_kernel(int64_t n, T *out, T v) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = v;
}
template <typename T> inline cudaError_t launch_fill(int64_t n, T *out, T v, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const int64_t want = (n + 255) / 256;
    const int grid = (int)(want < 148 * 8 ? want : 148 * 8);
    fill_kernel<T><<<grid, 256, 0, st>>>(n, out, v);
    return cudaGetLastError();
}

cudaError_t launch_rne_batch(int mode, int dtype, int64_t n, const void *q, const void *qd, const void *qdd,
                             const void *payload_mass, double payload_scalar, double payload_threshold,
                             void *tau_out, uint8_t *feasible_out, cudaStream_t st);

// model_kernels.cu: caller-supplied inertial set (mode BASE is handled by the caller: nothing to compute)
cudaError_t launch_rne_batch_model(const tcmp_model &model, int mode, int dtype, int64_t n, const void *q,
                                   const void *qd, const void *qdd, const void *payload_mass, double payload_scalar,
                                   double payload_threshold, void *tau_out, uint8_t *feasible_out, cudaStream_t st);
void default_model_desc(tcmp_model *out);
const char *model_desc_problem(const tcmp_model &model);

// 32-bit element offsets of the [7][7][n] outputs while the largest, 48 n + n - 1, fits (with a margin)
inline bool fits_int49(int64_t n) { return n < ((int64_t)0x7fffffff - ((int64_t)1 << 24)) / 49; }

// dynamics_kernels.cu: M, C, g, J per state (any output may be NULL; model NULL = compiled-in Panda)
cudaError_t launch_dynamics_batch(const tcmp_model *model, int64_t n, const double *q, const double *qd,
                                  const double *payload_mass, double payload_scalar, double *M_out, double *C_out,
                                  double *g_out, double *J_out, cudaStream_t st);

// fd_kernels.cu: qdd = M^-1 (tau - h) and M^-1 per state (K13); mode RNE or DYN, either output may be NULL, qd / tau
// NULL = zeros; model NULL = compiled-in Panda
cudaError_t launch_forward_dynamics(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                    const double *tau, const double *payload_mass, double payload_scalar,
                                    double *qdd_out, double *Minv_out, cudaStream_t st);

// rollout_kernels.cu: RK4 forward-dynamics rollouts (K14); mode RNE or DYN, qd0 / tau NULL = zeros, limits are host
// arrays of 7 (NULL = not checked), each output may be NULL; model NULL = compiled-in Panda
cudaError_t launch_rollout(const tcmp_model *model, int mode, int64_t n, int n_steps, double dt, const double *q0,
                           const double *qd0, const double *tau, int tau_per_step, const double *payload_mass,
                           double payload_scalar, const double *q_lo, const double *q_hi, const double *qd_max,
                           double *q_out, double *qd_out, double *q_traj_out, double *qd_traj_out,
                           int32_t *first_violation_out, cudaStream_t st);

// track_kernels.cu: closed-loop tracking rollouts (K15); mode RNE or DYN, q0 / qd0 NULL = the reference's x(0) / v(0),
// gains and limits are host arrays of 7 (limits NULL = not checked), each output may be NULL; model NULL = compiled-in
// Panda
cudaError_t launch_track(const tcmp_model *model, int mode, int64_t n, int n_steps, double dt, int n_seg,
                         const double *coeffs, int coeffs_broadcast, const double *q0, const double *qd0,
                         const double *kp, const double *kd, const double *payload_mass, double payload_scalar,
                         const double *ctrl_payload_mass, double ctrl_payload_scalar, const double *q_lo,
                         const double *q_hi, const double *qd_max, double *q_out, double *qd_out, double *q_traj_out,
                         double *qd_traj_out, double *tau_traj_out, int32_t *first_violation_out,
                         int32_t *first_saturation_out, double *max_err_out, cudaStream_t st);

// payload_kernels.cu: payload-mass intervals per state (K11) and per min-jerk edge (K12); each output may be NULL,
// mode BASE fills (-inf, +inf, 1) and reads nothing; model NULL = compiled-in Panda
cudaError_t launch_payload_interval(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                    const double *qdd, double *m_lo_out, double *m_hi_out, uint8_t *unloaded_ok_out,
                                    cudaStream_t st);
cudaError_t launch_edge_payload_interval(const tcmp_model *model, int mode, int64_t n_edges, int n_waypoints,
                                         const double *qa, const double *qb, int static_only, double *m_lo_out,
                                         double *m_hi_out, uint8_t *unloaded_ok_out, cudaStream_t st);

// Per-rank sync block of the fused gathers (TCMP_PEER_SYNC_BYTES, allocated with tcmp_peer_alloc, zeroed once):
// arrived[r] = last epoch rank r has published here (written by rank r's kernels over NVLink); epoch / ticket are
// this rank's own.
struct PeerSync {
    unsigned long long arrived[TCMP_MAX_PEERS];
    unsigned long long epoch;
    unsigned int ticket;
    unsigned int pad[13];
};
static_assert(sizeof(PeerSync) == TCMP_PEER_SYNC_BYTES, "tcmp.h: TCMP_PEER_SYNC_BYTES");

cudaError_t launch_rne_batch_scatter(int mode, int dtype, int64_t n, const void *q, const void *qd, const void *qdd,
                                     const void *payload_mass, double payload_scalar, double payload_threshold,
                                     void *tau_out, int n_dest, void *const *dest_masks, int64_t dest_offset,
                                     cudaStream_t st, void *mc_masks = nullptr);
cudaError_t launch_peer_signal(int rank, int n_dest, void *const *dest_sync, cudaStream_t st);
cudaError_t launch_peer_push(const void *src, int64_t bytes, int n_dest, void *const *dests, int64_t dest_offset,
                             cudaStream_t st);
cudaError_t launch_peer_wait(void *own_sync, int world, cudaStream_t st);

cudaError_t launch_edge_feasibility(int mode, int dtype, int64_t n_edges, int n_waypoints, const void *qa,
                                    const void *qb, double payload_scalar, double payload_threshold,
                                    int static_only, int32_t *first_fail_out, cudaStream_t st,
                                    const tcmp_model *model = nullptr);

cudaError_t launch_edge_feasibility_scatter(int mode, int64_t n_edges, int n_waypoints, const void *qa, const void *qb,
                                            double payload_scalar, double payload_threshold, int static_only,
                                            int n_dest, void *const *dest_ff, int64_t dest_offset, cudaStream_t st);

cudaError_t launch_traj_feasibility(int mode, int dtype, int n_seg, int samples_per_segment,
                                    const double *coeffs, double payload_scalar, double payload_threshold,
                                    void *q_out, void *qd_out, void *qdd_out, void *tau_out,
                                    uint8_t *feasible_out, int32_t *first_fail_out, cudaStream_t st,
                                    const tcmp_model *model = nullptr);

cudaError_t launch_ik_batch(int64_t n, const double *rot9, const double *trans3, const double *free_vals,
                            int n_free, int free_broadcast, double *sols_out, int32_t *count_out,
                            uint8_t *status_out, cudaStream_t st);

cudaError_t launch_ik_select(int64_t n, const double *rot9, const double *trans3, const double *free_vals,
                             int n_free, int free_broadcast, const double *q_ref, int ref_broadcast,
                             const double *q_lo, const double *q_hi, int mode, double mass,
                             double payload_threshold, int use_max_norm, double *best_q, double *best_cost,
                             int32_t *n_valid, cudaStream_t st, const tcmp_model *model = nullptr);

cudaError_t launch_fk_batch(int64_t n, const double *q, double *trans3, double *rot9, cudaStream_t st);

cudaError_t launch_collision_batch(int64_t n, const double *q, int n_obs, const tcmp_obstacle *obs,
                                   const double *q_lo, const double *q_hi, double payload_radius, uint8_t *hit_out,
                                   cudaStream_t st);

cudaError_t launch_extend_prefix(int mode, int64_t n_edges, const double *q1, const double *q2,
                                 const double *res, int n_obs, const tcmp_obstacle *obs, const double *q_lo,
                                 const double *q_hi, double payload_radius, double mass, double payload_threshold,
                                 int32_t *n_steps_out, int32_t *prefix_out, cudaStream_t st,
                                 const tcmp_model *model = nullptr);

cudaError_t launch_fp64_peak(int iters, double *sink, int *grid_out, int *block_out, cudaStream_t st);

}  // namespace tcmp
