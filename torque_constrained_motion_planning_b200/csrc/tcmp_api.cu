// tcmp_api.cu -- the extern "C" boundary declared in include/tcmp.h.
// Argument validation, error strings, launch-geometry helpers, the host-staged (pinned host
// buffer -> chunked H2D / kernel / D2H pipeline) variants, and the FP64 peak microbenchmark.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>

#include "tcmp_internal.h"

namespace tcmp {

static thread_local char g_err[512] = "";

static int fail(int status, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return status;
}
static int cuda_fail(cudaError_t e, const char *what) {
    return fail(TCMP_ERR_CUDA, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
}
#define TCMP_CUDA(call)                                   \
    do {                                                  \
        cudaError_t e_ = (call);                          \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
    } while (0)

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (!cached[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

int grid_for(const void *kernel, int block, int64_t n_threads_needed, int waves) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, 0) != cudaSuccess || per_sm <= 0)
        per_sm = 1;
    const int64_t full = (int64_t)sm_count() * per_sm * (waves > 0 ? waves : 1);
    int64_t want = (n_threads_needed + block - 1) / block;
    if (want < 1) want = 1;
    return (int)(want < full ? want : full);
}

// ---- FP64 FMA peak: 8 independent dependent-chains per thread, 2 flops per DFMA -------------
__global__ void __launch_bounds__(256) fp64_peak_kernel(int iters, double *sink) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
           a7 = a0 + 7;
    const double m = 0.999999999, b = 1e-12;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
            a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
        }
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123.456) sink[0] = s;  // never true; keeps the chains alive
}

cudaError_t launch_fp64_peak(int iters, double *sink, int *grid_out, int *block_out, cudaStream_t st) {
    const int block = 256;
    const int grid = grid_for(reinterpret_cast<const void *>(fp64_peak_kernel), block, (int64_t)1 << 40);
    fp64_peak_kernel<<<grid, block, 0, st>>>(iters, sink);
    *grid_out = grid;
    *block_out = block;
    return cudaGetLastError();
}

}  // namespace tcmp

using namespace tcmp;

// ---- host-staged pipeline -------------------------------------------------------------------
struct tcmp_workspace {
    static constexpr int kStages = 3;
    int64_t chunk = 0;        // states (or edges / solves) per stage
    size_t bytes = 0;         // device bytes per stage
    void *dev[kStages] = {nullptr, nullptr, nullptr};
    cudaStream_t stream[kStages] = {nullptr, nullptr, nullptr};
    int device = 0;
};

// A workspace belongs to the device that was current when it was created; host-array calls made while another
// device is current switch to it for the duration of the call.
struct DeviceScope {
    int prev = -1;
    bool switched = false;
    explicit DeviceScope(int device) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != device) switched = cudaSetDevice(device) == cudaSuccess;
    }
    ~DeviceScope() {
        if (switched) cudaSetDevice(prev);
    }
    DeviceScope(const DeviceScope &) = delete;
    DeviceScope &operator=(const DeviceScope &) = delete;
};

// Drain the stage streams; used on the success path and before reporting a mid-pipeline failure so no copy into
// caller memory is still in flight when the call returns.
static cudaError_t ws_drain(tcmp_workspace *ws) {
    cudaError_t first = cudaSuccess;
    for (int s = 0; s < tcmp_workspace::kStages; ++s) {
        cudaError_t e = cudaStreamSynchronize(ws->stream[s]);
        if (first == cudaSuccess) first = e;
    }
    return first;
}
#define TCMP_CUDA_WS(ws, expr)                  \
    do {                                        \
        cudaError_t e__ = (expr);               \
        if (e__ != cudaSuccess) {               \
            ws_drain(ws);                       \
            return cuda_fail(e__, #expr);       \
        }                                       \
    } while (0)

static int ws_reserve(tcmp_workspace *ws, size_t bytes_per_stage) {
    if (bytes_per_stage <= ws->bytes) return TCMP_OK;
    for (int s = 0; s < tcmp_workspace::kStages; ++s) {
        if (ws->dev[s]) TCMP_CUDA(cudaFree(ws->dev[s]));
        ws->dev[s] = nullptr;
    }
    ws->bytes = 0;
    for (int s = 0; s < tcmp_workspace::kStages; ++s) TCMP_CUDA(cudaMalloc(&ws->dev[s], bytes_per_stage));
    ws->bytes = bytes_per_stage;
    return TCMP_OK;
}

extern "C" {

int tcmp_abi_version(void) { return TCMP_ABI_VERSION; }
const char *tcmp_last_error(void) { return g_err; }

int tcmp_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return fail(TCMP_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    int ok = 0;
    for (int d = 0; d < n; ++d) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ++ok;
    }
    return ok;
}

static int check_common(int mode, int dtype, int64_t n) {
    if (mode < TCMP_MODE_RNE || mode > TCMP_MODE_BASE) return fail(TCMP_ERR_INVALID_ARG, "bad mode %d", mode);
    if (dtype != TCMP_F64 && dtype != TCMP_F32) return fail(TCMP_ERR_INVALID_ARG, "bad dtype %d", dtype);
    if (n < 0) return fail(TCMP_ERR_INVALID_ARG, "negative count %lld", (long long)n);
    return TCMP_OK;
}

int tcmp_rne_batch(int mode, int dtype, int64_t n, const void *q, const void *qd, const void *qdd,
                   const void *payload_mass, double payload_scalar, double payload_threshold, void *tau_out,
                   uint8_t *feasible_out, void *stream) {
    if (int rc = check_common(mode, dtype, n)) return rc;
    if (n == 0) return TCMP_OK;
    if (!q && mode != TCMP_MODE_BASE) return fail(TCMP_ERR_INVALID_ARG, "q is NULL");
    if (!tau_out && !feasible_out) return fail(TCMP_ERR_INVALID_ARG, "both outputs are NULL");
    if ((qd == nullptr) != (qdd == nullptr))
        return fail(TCMP_ERR_INVALID_ARG, "qd and qdd must both be given or both be NULL");
    TCMP_CUDA(launch_rne_batch(mode, dtype, n, q, qd, qdd, payload_mass, payload_scalar, payload_threshold, tau_out,
                               feasible_out, (cudaStream_t)stream));
    return TCMP_OK;
}

static int check_model(const tcmp_model *model) {
    if (!model) return TCMP_OK;
    if (const char *why = model_desc_problem(*model)) return fail(TCMP_ERR_INVALID_ARG, "tcmp_model: %s", why);
    return TCMP_OK;
}

int tcmp_model_default(tcmp_model *out) {
    if (!out) return fail(TCMP_ERR_INVALID_ARG, "model is NULL");
    default_model_desc(out);
    return TCMP_OK;
}

int tcmp_rne_batch_model(const tcmp_model *model, int mode, int dtype, int64_t n, const void *q, const void *qd,
                         const void *qdd, const void *payload_mass, double payload_scalar, double payload_threshold,
                         void *tau_out, uint8_t *feasible_out, void *stream) {
    if (!model || mode == TCMP_MODE_BASE)   // base computes nothing, so no model enters
        return tcmp_rne_batch(mode, dtype, n, q, qd, qdd, payload_mass, payload_scalar, payload_threshold, tau_out,
                              feasible_out, stream);
    if (int rc = check_common(mode, dtype, n)) return rc;
    if (int rc = check_model(model)) return rc;
    if (n == 0) return TCMP_OK;
    if (!q) return fail(TCMP_ERR_INVALID_ARG, "q is NULL");
    if (!tau_out && !feasible_out) return fail(TCMP_ERR_INVALID_ARG, "both outputs are NULL");
    if ((qd == nullptr) != (qdd == nullptr))
        return fail(TCMP_ERR_INVALID_ARG, "qd and qdd must both be given or both be NULL");
    TCMP_CUDA(launch_rne_batch_model(*model, mode, dtype, n, q, qd, qdd, payload_mass, payload_scalar,
                                     payload_threshold, tau_out, feasible_out, (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_dynamics_batch(const tcmp_model *model, int64_t n, const double *q, const double *qd,
                        const double *payload_mass, double payload_scalar, double *M_out, double *C_out, double *g_out,
                        double *J_out, void *stream) {
    if (n < 0) return fail(TCMP_ERR_INVALID_ARG, "negative count %lld", (long long)n);
    if (int rc = check_model(model)) return rc;
    // an empty batch is a no-op whatever the buffers (empty arrays may have NULL data pointers), as in tcmp_rne_batch
    if (n == 0) return TCMP_OK;
    if (!q) return fail(TCMP_ERR_INVALID_ARG, "q is NULL");
    if (!M_out && !C_out && !g_out && !J_out) return fail(TCMP_ERR_INVALID_ARG, "every output is NULL");
    if (C_out && !qd) return fail(TCMP_ERR_INVALID_ARG, "C_out needs qd");
    TCMP_CUDA(launch_dynamics_batch(model, n, q, qd, payload_mass, payload_scalar, M_out, C_out, g_out, J_out,
                                    (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_forward_dynamics_batch(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                const double *tau, const double *payload_mass, double payload_scalar, double *qdd_out,
                                double *Minv_out, void *stream) {
    if (mode != TCMP_MODE_RNE && mode != TCMP_MODE_DYN)
        return fail(TCMP_ERR_INVALID_ARG, "forward dynamics needs mode rne or dyn, got %d", mode);
    if (n < 0) return fail(TCMP_ERR_INVALID_ARG, "negative count %lld", (long long)n);
    if (int rc = check_model(model)) return rc;
    if (n == 0) return TCMP_OK;
    if (!q) return fail(TCMP_ERR_INVALID_ARG, "q is NULL");
    if (!qdd_out && !Minv_out) return fail(TCMP_ERR_INVALID_ARG, "both outputs are NULL");
    TCMP_CUDA(launch_forward_dynamics(model, mode, n, q, qd, tau, payload_mass, payload_scalar, qdd_out, Minv_out,
                                      (cudaStream_t)stream));
    return TCMP_OK;
}

// What tcmp_rollout_batch and tcmp_track_batch reject alike.
static int check_rollout_common(const tcmp_model *model, int mode, int64_t n, int n_steps, double dt,
                                const double *q_lo_host, const double *q_hi_host, const double *qd_max_host) {
    if (mode != TCMP_MODE_RNE && mode != TCMP_MODE_DYN)
        return fail(TCMP_ERR_INVALID_ARG, "rollouts need mode rne or dyn, got %d", mode);
    if (n < 0) return fail(TCMP_ERR_INVALID_ARG, "negative count %lld", (long long)n);
    if (n_steps < 1) return fail(TCMP_ERR_INVALID_ARG, "n_steps must be >= 1, got %d", n_steps);
    if (!(dt > 0.0 && dt < INFINITY)) return fail(TCMP_ERR_INVALID_ARG, "dt must be finite and > 0");
    if (int rc = check_model(model)) return rc;
    if ((q_lo_host == nullptr) != (q_hi_host == nullptr))
        return fail(TCMP_ERR_INVALID_ARG, "q_lo and q_hi must both be given or both be NULL");
    for (int j = 0; j < 7; ++j) {
        if (q_lo_host && (q_lo_host[j] != q_lo_host[j] || q_hi_host[j] != q_hi_host[j]))
            return fail(TCMP_ERR_INVALID_ARG, "NaN joint limit on joint %d", j);
        if (qd_max_host && !(qd_max_host[j] >= 0.0))
            return fail(TCMP_ERR_INVALID_ARG, "qd_max[%d] must be >= 0 (and not NaN)", j);
    }
    return TCMP_OK;
}

int tcmp_rollout_batch(const tcmp_model *model, int mode, int64_t n, int n_steps, double dt, const double *q0,
                       const double *qd0, const double *tau, int tau_per_step, const double *payload_mass,
                       double payload_scalar, const double *q_lo_host, const double *q_hi_host,
                       const double *qd_max_host, double *q_out, double *qd_out, double *q_traj_out,
                       double *qd_traj_out, int32_t *first_violation_out, void *stream) {
    if (int rc = check_rollout_common(model, mode, n, n_steps, dt, q_lo_host, q_hi_host, qd_max_host)) return rc;
    if (n == 0) return TCMP_OK;
    if (!q0) return fail(TCMP_ERR_INVALID_ARG, "q0 is NULL");
    if (!q_out && !qd_out && !q_traj_out && !qd_traj_out && !first_violation_out)
        return fail(TCMP_ERR_INVALID_ARG, "every output is NULL");
    TCMP_CUDA(launch_rollout(model, mode, n, n_steps, dt, q0, qd0, tau, tau_per_step, payload_mass, payload_scalar,
                             q_lo_host, q_hi_host, qd_max_host, q_out, qd_out, q_traj_out, qd_traj_out,
                             first_violation_out, (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_track_batch(const tcmp_model *model, int mode, int64_t n, int n_steps, double dt, int n_seg,
                     const double *coeffs, int coeffs_broadcast, const double *q0, const double *qd0,
                     const double *kp_host, const double *kd_host, const double *payload_mass, double payload_scalar,
                     const double *ctrl_payload_mass, double ctrl_payload_scalar, const double *q_lo_host,
                     const double *q_hi_host, const double *qd_max_host, double *q_out, double *qd_out,
                     double *q_traj_out, double *qd_traj_out, double *tau_traj_out, int32_t *first_violation_out,
                     int32_t *first_saturation_out, double *max_err_out, void *stream) {
    if (int rc = check_rollout_common(model, mode, n, n_steps, dt, q_lo_host, q_hi_host, qd_max_host)) return rc;
    if (n_seg < 1) return fail(TCMP_ERR_INVALID_ARG, "n_seg must be >= 1, got %d", n_seg);
    if (!kp_host || !kd_host) return fail(TCMP_ERR_INVALID_ARG, "kp and kd are required");
    for (int j = 0; j < 7; ++j)
        if (!(kp_host[j] >= 0.0 && kp_host[j] < INFINITY && kd_host[j] >= 0.0 && kd_host[j] < INFINITY))
            return fail(TCMP_ERR_INVALID_ARG, "gains of joint %d must be finite and >= 0", j);
    if (n == 0) return TCMP_OK;
    if (!coeffs) return fail(TCMP_ERR_INVALID_ARG, "coeffs is NULL");
    if (!q_out && !qd_out && !q_traj_out && !qd_traj_out && !tau_traj_out && !first_violation_out &&
        !first_saturation_out && !max_err_out)
        return fail(TCMP_ERR_INVALID_ARG, "every output is NULL");
    TCMP_CUDA(launch_track(model, mode, n, n_steps, dt, n_seg, coeffs, coeffs_broadcast, q0, qd0, kp_host, kd_host,
                           payload_mass, payload_scalar, ctrl_payload_mass, ctrl_payload_scalar, q_lo_host, q_hi_host,
                           qd_max_host, q_out, qd_out, q_traj_out, qd_traj_out, tau_traj_out, first_violation_out,
                           first_saturation_out, max_err_out, (cudaStream_t)stream));
    return TCMP_OK;
}

static int check_payload_common(const tcmp_model *model, int mode, int64_t n) {
    if (mode < TCMP_MODE_RNE || mode > TCMP_MODE_BASE) return fail(TCMP_ERR_INVALID_ARG, "bad mode %d", mode);
    if (n < 0) return fail(TCMP_ERR_INVALID_ARG, "negative count %lld", (long long)n);
    return check_model(model);
}

int tcmp_payload_interval_batch(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                const double *qdd, double *m_lo_out, double *m_hi_out, uint8_t *unloaded_ok_out,
                                void *stream) {
    if (int rc = check_payload_common(model, mode, n)) return rc;
    if (n == 0) return TCMP_OK;
    if (!q && mode != TCMP_MODE_BASE) return fail(TCMP_ERR_INVALID_ARG, "q is NULL");
    if (!m_lo_out && !m_hi_out && !unloaded_ok_out) return fail(TCMP_ERR_INVALID_ARG, "every output is NULL");
    if ((qd == nullptr) != (qdd == nullptr))
        return fail(TCMP_ERR_INVALID_ARG, "qd and qdd must both be given or both be NULL");
    TCMP_CUDA(launch_payload_interval(model, mode, n, q, qd, qdd, m_lo_out, m_hi_out, unloaded_ok_out,
                                      (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_edge_payload_interval(const tcmp_model *model, int mode, int64_t n_edges, int n_waypoints, const double *qa,
                               const double *qb, int static_only, double *m_lo_out, double *m_hi_out,
                               uint8_t *unloaded_ok_out, void *stream) {
    if (int rc = check_payload_common(model, mode, n_edges)) return rc;
    if (n_waypoints < 1) return fail(TCMP_ERR_INVALID_ARG, "n_waypoints must be >= 1");
    if (n_edges == 0) return TCMP_OK;
    if ((!qa || !qb) && mode != TCMP_MODE_BASE) return fail(TCMP_ERR_INVALID_ARG, "NULL edge buffer");
    if (!m_lo_out && !m_hi_out && !unloaded_ok_out) return fail(TCMP_ERR_INVALID_ARG, "every output is NULL");
    TCMP_CUDA(launch_edge_payload_interval(model, mode, n_edges, n_waypoints, qa, qb, static_only, m_lo_out, m_hi_out,
                                           unloaded_ok_out, (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_rne_batch_scatter(int mode, int dtype, int64_t n, const void *q, const void *qd, const void *qdd,
                           const void *payload_mass, double payload_scalar, double payload_threshold, void *tau_out,
                           int n_dest, void *const *dest_masks, int64_t dest_offset, void *stream) {
    if (int rc = check_common(mode, dtype, n)) return rc;
    if (dtype != TCMP_F64) return fail(TCMP_ERR_UNSUPPORTED, "scatter form is fp64 only");
    if (n_dest < 1 || n_dest > TCMP_MAX_PEERS || !dest_masks || dest_offset < 0)
        return fail(TCMP_ERR_INVALID_ARG, "bad destination list");
    for (int i = 0; i < n_dest; ++i)
        if (!dest_masks[i]) return fail(TCMP_ERR_INVALID_ARG, "dest_masks[%d] is NULL", i);
    if (n == 0) return TCMP_OK;
    if (!q && mode != TCMP_MODE_BASE) return fail(TCMP_ERR_INVALID_ARG, "q is NULL");
    if ((qd == nullptr) != (qdd == nullptr))
        return fail(TCMP_ERR_INVALID_ARG, "qd and qdd must both be given or both be NULL");
    TCMP_CUDA(launch_rne_batch_scatter(mode, dtype, n, q, qd, qdd, payload_mass, payload_scalar, payload_threshold,
                                       tau_out, n_dest, dest_masks, dest_offset, (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_rne_batch_scatter_mc(int mode, int dtype, int64_t n, const void *q, const void *qd, const void *qdd,
                              const void *payload_mass, double payload_scalar, double payload_threshold, void *tau_out,
                              int n_dest, void *const *dest_masks, void *mc_masks, int64_t dest_offset, void *stream) {
    if (!mc_masks) return fail(TCMP_ERR_INVALID_ARG, "mc_masks is NULL (use tcmp_rne_batch_scatter)");
    if (int rc = check_common(mode, dtype, n)) return rc;
    if (dtype != TCMP_F64) return fail(TCMP_ERR_UNSUPPORTED, "scatter form is fp64 only");
    if (n_dest < 1 || n_dest > TCMP_MAX_PEERS || !dest_masks || dest_offset < 0)
        return fail(TCMP_ERR_INVALID_ARG, "bad destination list");
    for (int i = 0; i < n_dest; ++i)
        if (!dest_masks[i]) return fail(TCMP_ERR_INVALID_ARG, "dest_masks[%d] is NULL", i);
    if (n == 0) return TCMP_OK;
    if (!q && mode != TCMP_MODE_BASE) return fail(TCMP_ERR_INVALID_ARG, "q is NULL");
    if ((qd == nullptr) != (qdd == nullptr))
        return fail(TCMP_ERR_INVALID_ARG, "qd and qdd must both be given or both be NULL");
    TCMP_CUDA(launch_rne_batch_scatter(mode, dtype, n, q, qd, qdd, payload_mass, payload_scalar, payload_threshold,
                                       tau_out, n_dest, dest_masks, dest_offset, (cudaStream_t)stream, mc_masks));
    return TCMP_OK;
}

int tcmp_peer_push(const void *src, int64_t bytes, int n_dest, void *const *dests, int64_t dest_offset, void *stream) {
    if (bytes < 0 || n_dest < 1 || n_dest > TCMP_MAX_PEERS || !dests || dest_offset < 0)
        return fail(TCMP_ERR_INVALID_ARG, "bad push arguments");
    for (int i = 0; i < n_dest; ++i)
        if (!dests[i]) return fail(TCMP_ERR_INVALID_ARG, "dests[%d] is NULL", i);
    if (bytes == 0) return TCMP_OK;
    if (!src) return fail(TCMP_ERR_INVALID_ARG, "src is NULL");
    TCMP_CUDA(launch_peer_push(src, bytes, n_dest, dests, dest_offset, (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_peer_signal(int rank, int n_dest, void *const *dest_sync, void *stream) {
    if (n_dest < 1 || n_dest > TCMP_MAX_PEERS || !dest_sync || rank < 0 || rank >= n_dest)
        return fail(TCMP_ERR_INVALID_ARG, "bad sync list");
    for (int i = 0; i < n_dest; ++i)
        if (!dest_sync[i]) return fail(TCMP_ERR_INVALID_ARG, "dest_sync[%d] is NULL", i);
    TCMP_CUDA(launch_peer_signal(rank, n_dest, dest_sync, (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_peer_wait(void *own_sync, int n_ranks, void *stream) {
    if (!own_sync || n_ranks < 1 || n_ranks > TCMP_MAX_PEERS) return fail(TCMP_ERR_INVALID_ARG, "bad sync block");
    TCMP_CUDA(launch_peer_wait(own_sync, n_ranks, (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_peer_alloc(void **dev_ptr, int64_t bytes, unsigned char *handle_out) {
    if (!dev_ptr || bytes <= 0 || !handle_out) return fail(TCMP_ERR_INVALID_ARG, "bad peer alloc");
    static_assert(sizeof(cudaIpcMemHandle_t) == TCMP_IPC_HANDLE_BYTES, "IPC handle size");
    TCMP_CUDA(cudaMalloc(dev_ptr, (size_t)bytes));
    TCMP_CUDA(cudaMemset(*dev_ptr, 0, (size_t)bytes));   // sync blocks (TCMP_PEER_SYNC_BYTES) start at epoch 0
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, *dev_ptr);
    if (e != cudaSuccess) {
        cudaFree(*dev_ptr);
        *dev_ptr = nullptr;
        return cuda_fail(e, "cudaIpcGetMemHandle");
    }
    memcpy(handle_out, &h, sizeof(h));
    return TCMP_OK;
}
int tcmp_peer_free(void *dev_ptr) {
    if (dev_ptr) TCMP_CUDA(cudaFree(dev_ptr));
    return TCMP_OK;
}
int tcmp_peer_open(const unsigned char *handle, void **peer_ptr) {
    if (!handle || !peer_ptr) return fail(TCMP_ERR_INVALID_ARG, "bad peer open");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    TCMP_CUDA(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return TCMP_OK;
}
int tcmp_peer_close(void *peer_ptr) {
    if (peer_ptr) TCMP_CUDA(cudaIpcCloseMemHandle(peer_ptr));
    return TCMP_OK;
}

int tcmp_edge_feasibility_model(const tcmp_model *model, int mode, int dtype, int64_t n_edges, int n_waypoints,
                                const void *qa, const void *qb, double payload_scalar, double payload_threshold,
                                int static_only, int32_t *first_fail_out, void *stream) {
    if (int rc = check_common(mode, dtype, n_edges)) return rc;
    if (int rc = check_model(model)) return rc;
    if (n_waypoints < 1) return fail(TCMP_ERR_INVALID_ARG, "n_waypoints must be >= 1");
    if (n_edges == 0) return TCMP_OK;
    if (!qa || !qb || !first_fail_out) return fail(TCMP_ERR_INVALID_ARG, "NULL edge buffer");
    TCMP_CUDA(launch_edge_feasibility(mode, dtype, n_edges, n_waypoints, qa, qb, payload_scalar, payload_threshold,
                                      static_only, first_fail_out, (cudaStream_t)stream, model));
    return TCMP_OK;
}

int tcmp_edge_feasibility(int mode, int dtype, int64_t n_edges, int n_waypoints, const void *qa, const void *qb,
                          double payload_scalar, double payload_threshold, int static_only,
                          int32_t *first_fail_out, void *stream) {
    return tcmp_edge_feasibility_model(nullptr, mode, dtype, n_edges, n_waypoints, qa, qb, payload_scalar,
                                       payload_threshold, static_only, first_fail_out, stream);
}

int tcmp_edge_feasibility_scatter(int mode, int64_t n_edges, int n_waypoints, const void *qa, const void *qb,
                                  double payload_scalar, double payload_threshold, int static_only, int n_dest,
                                  void *const *dest_first_fail, int64_t dest_offset, void *stream) {
    if (int rc = check_common(mode, TCMP_F64, n_edges)) return rc;
    if (n_waypoints < 1) return fail(TCMP_ERR_INVALID_ARG, "n_waypoints must be >= 1");
    if (n_dest < 1 || n_dest > TCMP_MAX_PEERS || !dest_first_fail || dest_offset < 0)
        return fail(TCMP_ERR_INVALID_ARG, "bad destination list");
    for (int i = 0; i < n_dest; ++i)
        if (!dest_first_fail[i]) return fail(TCMP_ERR_INVALID_ARG, "dest_first_fail[%d] is NULL", i);
    if (n_edges == 0) return TCMP_OK;
    if (!qa || !qb) return fail(TCMP_ERR_INVALID_ARG, "NULL edge buffer");
    TCMP_CUDA(launch_edge_feasibility_scatter(mode, n_edges, n_waypoints, qa, qb, payload_scalar, payload_threshold,
                                              static_only, n_dest, dest_first_fail, dest_offset, (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_traj_feasibility(int mode, int dtype, int n_seg, int samples_per_segment, const double *coeffs,
                          double payload_scalar, double payload_threshold, void *q_out, void *qd_out, void *qdd_out,
                          void *tau_out, uint8_t *feasible_out, int32_t *first_fail_out, void *stream) {
    return tcmp_traj_feasibility_model(nullptr, mode, dtype, n_seg, samples_per_segment, coeffs, payload_scalar,
                                       payload_threshold, q_out, qd_out, qdd_out, tau_out, feasible_out,
                                       first_fail_out, stream);
}

int tcmp_traj_feasibility_model(const tcmp_model *model, int mode, int dtype, int n_seg, int samples_per_segment,
                                const double *coeffs, double payload_scalar, double payload_threshold, void *q_out,
                                void *qd_out, void *qdd_out, void *tau_out, uint8_t *feasible_out,
                                int32_t *first_fail_out, void *stream) {
    if (int rc = check_common(mode, dtype, n_seg)) return rc;
    if (int rc = check_model(model)) return rc;
    if (samples_per_segment < 1) return fail(TCMP_ERR_INVALID_ARG, "samples_per_segment must be >= 1");
    if (n_seg == 0) return TCMP_OK;
    if (!coeffs) return fail(TCMP_ERR_INVALID_ARG, "coeffs is NULL");
    TCMP_CUDA(launch_traj_feasibility(mode, dtype, n_seg, samples_per_segment, coeffs, payload_scalar,
                                      payload_threshold, q_out, qd_out, qdd_out, tau_out, feasible_out,
                                      first_fail_out, (cudaStream_t)stream, model));
    return TCMP_OK;
}

int tcmp_ik_batch(int64_t n, const double *rot9, const double *trans3, const double *free_vals, int n_free,
                  int free_broadcast, double *sols_out, int32_t *count_out, uint8_t *status_out, void *stream) {
    if (n < 0 || n_free < 1) return fail(TCMP_ERR_INVALID_ARG, "bad n / n_free");
    if (n == 0) return TCMP_OK;
    if (!rot9 || !trans3 || !free_vals || !count_out) return fail(TCMP_ERR_INVALID_ARG, "NULL IK buffer");
    TCMP_CUDA(launch_ik_batch(n, rot9, trans3, free_vals, n_free, free_broadcast, sols_out, count_out, status_out,
                              (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_ik_select(int64_t n, const double *rot9, const double *trans3, const double *free_vals, int n_free,
                   int free_broadcast, const double *q_ref, int ref_broadcast, const double *q_lo_host,
                   const double *q_hi_host, int mode, double payload_scalar, double payload_threshold, int use_max_norm,
                   double *best_q, double *best_cost, int32_t *n_valid, void *stream) {
    return tcmp_ik_select_model(nullptr, n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast,
                                q_lo_host, q_hi_host, mode, payload_scalar, payload_threshold, use_max_norm, best_q,
                                best_cost, n_valid, stream);
}

int tcmp_ik_select_model(const tcmp_model *model, int64_t n, const double *rot9, const double *trans3,
                         const double *free_vals, int n_free, int free_broadcast, const double *q_ref,
                         int ref_broadcast, const double *q_lo_host, const double *q_hi_host, int mode,
                         double payload_scalar, double payload_threshold, int use_max_norm, double *best_q,
                         double *best_cost, int32_t *n_valid, void *stream) {
    if (int rc = check_model(model)) return rc;
    if (n < 0 || n_free < 1) return fail(TCMP_ERR_INVALID_ARG, "bad n / n_free");
    if (mode < TCMP_MODE_RNE || mode > TCMP_MODE_BASE) return fail(TCMP_ERR_INVALID_ARG, "bad mode %d", mode);
    if (n == 0) return TCMP_OK;
    if (!rot9 || !trans3 || !free_vals || !q_ref || !q_lo_host || !q_hi_host || !best_q || !best_cost || !n_valid)
        return fail(TCMP_ERR_INVALID_ARG, "NULL IK-select buffer");
    TCMP_CUDA(launch_ik_select(n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast, q_lo_host,
                               q_hi_host, mode, payload_scalar, payload_threshold, use_max_norm, best_q, best_cost,
                               n_valid, (cudaStream_t)stream, model));
    return TCMP_OK;
}

int tcmp_collision_batch(int64_t n, const double *q, int n_obs, const tcmp_obstacle *obstacles_host,
                         const double *q_lo_host, const double *q_hi_host, double payload_radius, uint8_t *hit_out,
                         void *stream) {
    if (n < 0) return fail(TCMP_ERR_INVALID_ARG, "negative count");
    if (n_obs < 0 || n_obs > TCMP_MAX_OBSTACLES) return fail(TCMP_ERR_UNSUPPORTED, "0..%d obstacles", TCMP_MAX_OBSTACLES);
    if (n == 0) return TCMP_OK;
    if (!q || !hit_out || !q_lo_host || !q_hi_host || (n_obs > 0 && !obstacles_host))
        return fail(TCMP_ERR_INVALID_ARG, "NULL collision buffer");
    TCMP_CUDA(launch_collision_batch(n, q, n_obs, obstacles_host, q_lo_host, q_hi_host, payload_radius, hit_out,
                                     (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_extend_prefix(int mode, int64_t n_edges, const double *q1, const double *q2, const double *resolution_host,
                       int n_obs, const tcmp_obstacle *obstacles_host, const double *q_lo_host, const double *q_hi_host,
                       double payload_radius, double payload_scalar, double payload_threshold, int32_t *n_steps_out,
                       int32_t *prefix_out, void *stream) {
    return tcmp_extend_prefix_model(nullptr, mode, n_edges, q1, q2, resolution_host, n_obs, obstacles_host, q_lo_host,
                                    q_hi_host, payload_radius, payload_scalar, payload_threshold, n_steps_out,
                                    prefix_out, stream);
}

int tcmp_extend_prefix_model(const tcmp_model *model, int mode, int64_t n_edges, const double *q1, const double *q2,
                             const double *resolution_host, int n_obs, const tcmp_obstacle *obstacles_host,
                             const double *q_lo_host, const double *q_hi_host, double payload_radius,
                             double payload_scalar, double payload_threshold, int32_t *n_steps_out,
                             int32_t *prefix_out, void *stream) {
    if (int rc = check_common(mode, TCMP_F64, n_edges)) return rc;
    if (int rc = check_model(model)) return rc;
    if (n_obs < 0 || n_obs > TCMP_MAX_OBSTACLES) return fail(TCMP_ERR_UNSUPPORTED, "0..%d obstacles", TCMP_MAX_OBSTACLES);
    if (n_edges == 0) return TCMP_OK;
    if (!q1 || !q2 || !resolution_host || !q_lo_host || !q_hi_host || !n_steps_out || !prefix_out ||
        (n_obs > 0 && !obstacles_host))
        return fail(TCMP_ERR_INVALID_ARG, "NULL extend buffer");
    for (int j = 0; j < 7; ++j)
        if (!(resolution_host[j] > 0)) return fail(TCMP_ERR_INVALID_ARG, "resolution[%d] must be > 0", j);
    TCMP_CUDA(launch_extend_prefix(mode, n_edges, q1, q2, resolution_host, n_obs, obstacles_host, q_lo_host, q_hi_host,
                                   payload_radius, payload_scalar, payload_threshold, n_steps_out, prefix_out,
                                   (cudaStream_t)stream, model));
    return TCMP_OK;
}

int tcmp_fk_batch(int64_t n, const double *q, double *trans3, double *rot9, void *stream) {
    if (n < 0) return fail(TCMP_ERR_INVALID_ARG, "negative count");
    if (n == 0) return TCMP_OK;
    if (!q || !trans3 || !rot9) return fail(TCMP_ERR_INVALID_ARG, "NULL FK buffer");
    TCMP_CUDA(launch_fk_batch(n, q, trans3, rot9, (cudaStream_t)stream));
    return TCMP_OK;
}

int tcmp_workspace_create(tcmp_workspace **out, int64_t chunk_states) {
    if (!out) return fail(TCMP_ERR_INVALID_ARG, "ws is NULL");
    if (chunk_states < 0) return fail(TCMP_ERR_INVALID_ARG, "negative chunk");
    tcmp_workspace *ws = new tcmp_workspace();
    ws->chunk = chunk_states > 0 ? chunk_states : ((int64_t)1 << 18);
    cudaError_t e = cudaGetDevice(&ws->device);
    for (int s = 0; e == cudaSuccess && s < tcmp_workspace::kStages; ++s)
        e = cudaStreamCreateWithFlags(&ws->stream[s], cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        for (int s = 0; s < tcmp_workspace::kStages; ++s)      // streams created before the failure (ADVICE r01)
            if (ws->stream[s]) cudaStreamDestroy(ws->stream[s]);
        delete ws;
        return cuda_fail(e, "tcmp_workspace_create");
    }
    *out = ws;
    return TCMP_OK;
}

int tcmp_workspace_destroy(tcmp_workspace *ws) {
    if (!ws) return TCMP_OK;
    DeviceScope scope(ws->device);
    for (int s = 0; s < tcmp_workspace::kStages; ++s) {
        if (ws->stream[s]) {
            cudaStreamSynchronize(ws->stream[s]);
            cudaStreamDestroy(ws->stream[s]);
        }
        if (ws->dev[s]) cudaFree(ws->dev[s]);
    }
    delete ws;
    return TCMP_OK;
}

// Rows of a host SoA array [rows][n] restricted to columns [off, off+len) are `rows` separate
// contiguous runs; each is one cudaMemcpyAsync into a dense [rows][len] device tile.
static cudaError_t h2d_rows(void *dst, const void *src, int rows, int64_t n, int64_t off, int64_t len, size_t esz,
                            cudaStream_t st) {
    return cudaMemcpy2DAsync(dst, (size_t)len * esz, (const char *)src + (size_t)off * esz, (size_t)n * esz,
                             (size_t)len * esz, rows, cudaMemcpyHostToDevice, st);
}
static cudaError_t d2h_rows(void *dst, const void *src, int rows, int64_t n, int64_t off, int64_t len, size_t esz,
                            cudaStream_t st) {
    return cudaMemcpy2DAsync((char *)dst + (size_t)off * esz, (size_t)n * esz, src, (size_t)len * esz,
                             (size_t)len * esz, rows, cudaMemcpyDeviceToHost, st);
}

// Chunk schedule of the host pipelines: full chunks, then a tapered tail (C/2, C/4, C/4).  The host->device copies of
// all chunks run back to back whatever their size, so the only part of the pipeline that is NOT hidden is the last
// chunk's kernel and device->host copy: the smaller the last chunk the shorter that tail -- but every copy carries ~5 us
// of fixed cost on the copy engine, so small chunks everywhere lose (measured, 1 M states: 3.85 ms at 256 k uniform,
// 4.29 ms at 64 k uniform).
static int64_t next_chunk(int64_t remaining, int64_t C) {
    if (remaining > C) return C;
    if (remaining > C / 2 && C >= 4096) return C / 2;
    if (remaining > C / 4 && C >= 4096) return (remaining + 1) / 2;
    return remaining;
}

static int rne_batch_host_impl(tcmp_workspace *ws, int mode, int dtype, int64_t n, const void *q, const void *qd,
                               const void *qdd, const void *payload_mass, double payload_scalar,
                               double payload_threshold, void *tau_out, uint8_t *feasible_out, bool drain);

int tcmp_rne_batch_host(tcmp_workspace *ws, int mode, int dtype, int64_t n, const void *q, const void *qd,
                        const void *qdd, const void *payload_mass, double payload_scalar, double payload_threshold,
                        void *tau_out, uint8_t *feasible_out) {
    return rne_batch_host_impl(ws, mode, dtype, n, q, qd, qdd, payload_mass, payload_scalar, payload_threshold, tau_out,
                               feasible_out, true);
}

int tcmp_rne_batch_host_async(tcmp_workspace *ws, int mode, int dtype, int64_t n, const void *q, const void *qd,
                              const void *qdd, const void *payload_mass, double payload_scalar,
                              double payload_threshold, void *tau_out, uint8_t *feasible_out) {
    return rne_batch_host_impl(ws, mode, dtype, n, q, qd, qdd, payload_mass, payload_scalar, payload_threshold, tau_out,
                               feasible_out, false);
}

int tcmp_workspace_sync(tcmp_workspace *ws) {
    if (!ws) return fail(TCMP_ERR_INVALID_ARG, "workspace is NULL");
    DeviceScope scope(ws->device);
    TCMP_CUDA(ws_drain(ws));
    return TCMP_OK;
}

static int rne_batch_host_impl(tcmp_workspace *ws, int mode, int dtype, int64_t n, const void *q, const void *qd,
                               const void *qdd, const void *payload_mass, double payload_scalar,
                               double payload_threshold, void *tau_out, uint8_t *feasible_out, bool drain) {
    if (!ws) return fail(TCMP_ERR_INVALID_ARG, "workspace is NULL");
    DeviceScope scope(ws->device);
    if (int rc = check_common(mode, dtype, n)) return rc;
    if (n == 0) return TCMP_OK;
    if (!q && mode != TCMP_MODE_BASE) return fail(TCMP_ERR_INVALID_ARG, "q is NULL");
    if (!tau_out && !feasible_out) return fail(TCMP_ERR_INVALID_ARG, "both outputs are NULL");
    if ((qd == nullptr) != (qdd == nullptr))
        return fail(TCMP_ERR_INVALID_ARG, "qd and qdd must both be given or both be NULL");
    const size_t esz = dtype == TCMP_F64 ? 8 : 4;
    const int64_t C = ws->chunk;
    // per-stage tile: q[7][C] qd[7][C] qdd[7][C] mass[C] tau[7][C] mask[C]
    const size_t row = (size_t)C * esz;
    if (int rc = ws_reserve(ws, row * (7 * 4 + 1) + (size_t)C + 256)) return rc;
    int stage = 0;
    int64_t len = 0;
    for (int64_t off = 0; off < n; off += len, stage = (stage + 1) % tcmp_workspace::kStages) {
        len = next_chunk(n - off, C);
        cudaStream_t st = ws->stream[stage];
        char *base = (char *)ws->dev[stage];
        char *dq = base, *dqd = base + 7 * row, *dqdd = base + 14 * row, *dm = base + 21 * row, *dtau = base + 22 * row;
        uint8_t *dmask = (uint8_t *)(base + 29 * row);
        // the tile is dense [7][len]: the kernel sees n == len
        if (q) TCMP_CUDA_WS(ws, h2d_rows(dq, q, 7, n, off, len, esz, st));
        if (qd && mode != TCMP_MODE_NOV) {
            TCMP_CUDA_WS(ws, h2d_rows(dqd, qd, 7, n, off, len, esz, st));
            TCMP_CUDA_WS(ws, h2d_rows(dqdd, qdd, 7, n, off, len, esz, st));
        }
        if (payload_mass) TCMP_CUDA_WS(ws, h2d_rows(dm, payload_mass, 1, n, off, len, esz, st));
        const bool dyn_in = qd && mode != TCMP_MODE_NOV;
        TCMP_CUDA_WS(ws, launch_rne_batch(mode, dtype, len, dq, dyn_in ? dqd : nullptr, dyn_in ? dqdd : nullptr,
                                   payload_mass ? dm : nullptr, payload_scalar, payload_threshold,
                                   tau_out ? dtau : nullptr, feasible_out ? dmask : nullptr, st));
        if (tau_out) TCMP_CUDA_WS(ws, d2h_rows(tau_out, dtau, 7, n, off, len, esz, st));
        if (feasible_out) TCMP_CUDA_WS(ws, d2h_rows(feasible_out, dmask, 1, n, off, len, 1, st));
    }
    if (drain) TCMP_CUDA(ws_drain(ws));
    return TCMP_OK;
}

int tcmp_edge_feasibility_host(tcmp_workspace *ws, int mode, int dtype, int64_t n_edges, int n_waypoints,
                               const void *qa, const void *qb, double payload_scalar, double payload_threshold,
                               int static_only, int32_t *first_fail_out) {
    if (!ws) return fail(TCMP_ERR_INVALID_ARG, "workspace is NULL");
    DeviceScope scope(ws->device);
    if (int rc = check_common(mode, dtype, n_edges)) return rc;
    if (n_waypoints < 1) return fail(TCMP_ERR_INVALID_ARG, "n_waypoints must be >= 1");
    if (n_edges == 0) return TCMP_OK;
    if (!qa || !qb || !first_fail_out) return fail(TCMP_ERR_INVALID_ARG, "NULL edge buffer");
    const size_t esz = dtype == TCMP_F64 ? 8 : 4;
    const int64_t C = ws->chunk;
    const size_t row = (size_t)C * esz;
    if (int rc = ws_reserve(ws, row * 14 + (size_t)C * 4 + 256)) return rc;
    int stage = 0;
    for (int64_t off = 0; off < n_edges; off += C, stage = (stage + 1) % tcmp_workspace::kStages) {
        const int64_t len = (n_edges - off) < C ? (n_edges - off) : C;
        cudaStream_t st = ws->stream[stage];
        char *base = (char *)ws->dev[stage];
        char *da = base, *db = base + 7 * row;
        int32_t *dff = (int32_t *)(base + 14 * row);
        TCMP_CUDA_WS(ws, h2d_rows(da, qa, 7, n_edges, off, len, esz, st));
        TCMP_CUDA_WS(ws, h2d_rows(db, qb, 7, n_edges, off, len, esz, st));
        TCMP_CUDA_WS(ws, launch_edge_feasibility(mode, dtype, len, n_waypoints, da, db, payload_scalar, payload_threshold,
                                          static_only, dff, st));
        TCMP_CUDA_WS(ws, d2h_rows(first_fail_out, dff, 1, n_edges, off, len, 4, st));
    }
    TCMP_CUDA(ws_drain(ws));
    return TCMP_OK;
}

int tcmp_ik_batch_host(tcmp_workspace *ws, int64_t n, const double *rot9, const double *trans3,
                       const double *free_vals, int n_free, int free_broadcast, double *sols_out, int32_t *count_out,
                       uint8_t *status_out) {
    if (!ws) return fail(TCMP_ERR_INVALID_ARG, "workspace is NULL");
    DeviceScope scope(ws->device);
    if (n < 0 || n_free < 1) return fail(TCMP_ERR_INVALID_ARG, "bad n / n_free");
    if (n == 0) return TCMP_OK;
    if (!rot9 || !trans3 || !free_vals || !count_out) return fail(TCMP_ERR_INVALID_ARG, "NULL IK buffer");
    // chunk over poses; a stage holds rot[9][C] trans[3][C] free[n_free][C] sols[C*n_free*56] counts status
    int64_t C = ws->chunk / n_free;
    if (C < 1) C = 1;
    const size_t row = (size_t)C * 8;
    const size_t solves = (size_t)C * n_free;
    const size_t bytes = row * (12 + n_free) + solves * (56 * 8 + 4 + 1) + 512;
    if (int rc = ws_reserve(ws, bytes)) return rc;
    int stage = 0;
    for (int64_t off = 0; off < n; off += C, stage = (stage + 1) % tcmp_workspace::kStages) {
        const int64_t len = (n - off) < C ? (n - off) : C;
        cudaStream_t st = ws->stream[stage];
        char *base = (char *)ws->dev[stage];
        double *dr = (double *)base, *dt = (double *)(base + 9 * row), *df = (double *)(base + 12 * row);
        double *dsol = (double *)(base + (12 + n_free) * row);
        int32_t *dcnt = (int32_t *)((char *)dsol + solves * 56 * 8);
        uint8_t *dstat = (uint8_t *)((char *)dcnt + solves * 4);
        TCMP_CUDA_WS(ws, h2d_rows(dr, rot9, 9, n, off, len, 8, st));
        TCMP_CUDA_WS(ws, h2d_rows(dt, trans3, 3, n, off, len, 8, st));
        if (free_broadcast)
            TCMP_CUDA_WS(ws, cudaMemcpyAsync(df, free_vals, (size_t)n_free * 8, cudaMemcpyHostToDevice, st));
        else
            TCMP_CUDA_WS(ws, h2d_rows(df, free_vals, n_free, n, off, len, 8, st));
        TCMP_CUDA_WS(ws, launch_ik_batch(len, dr, dt, df, n_free, free_broadcast, sols_out ? dsol : nullptr, dcnt,
                                  status_out ? dstat : nullptr, st));
        const size_t s0 = (size_t)off * n_free, sl = (size_t)len * n_free;
        if (sols_out)
            TCMP_CUDA_WS(ws, cudaMemcpyAsync(sols_out + s0 * 56, dsol, sl * 56 * 8, cudaMemcpyDeviceToHost, st));
        TCMP_CUDA_WS(ws, cudaMemcpyAsync(count_out + s0, dcnt, sl * 4, cudaMemcpyDeviceToHost, st));
        if (status_out) TCMP_CUDA_WS(ws, cudaMemcpyAsync(status_out + s0, dstat, sl, cudaMemcpyDeviceToHost, st));
    }
    TCMP_CUDA(ws_drain(ws));
    return TCMP_OK;
}

int tcmp_host_alloc(void **ptr, int64_t bytes) {
    if (!ptr || bytes < 0) return fail(TCMP_ERR_INVALID_ARG, "bad host alloc");
    TCMP_CUDA(cudaHostAlloc(ptr, (size_t)bytes, cudaHostAllocDefault));
    return TCMP_OK;
}
int tcmp_host_free(void *ptr) {
    if (ptr) TCMP_CUDA(cudaFreeHost(ptr));
    return TCMP_OK;
}

int tcmp_fp64_peak(int iters, double *flops_out, void *stream) {
    if (iters < 1 || !flops_out) return fail(TCMP_ERR_INVALID_ARG, "bad fp64 peak args");
    cudaStream_t st = (cudaStream_t)stream;
    double *sink = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int grid = 0, block = 0;
    float ms = 0;
    cudaError_t e = cudaMalloc(&sink, 8);
    if (e == cudaSuccess) e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    if (e == cudaSuccess) e = launch_fp64_peak(iters / 8 + 1, sink, &grid, &block, st);  // warm-up
    if (e == cudaSuccess) e = cudaEventRecord(e0, st);
    if (e == cudaSuccess) e = launch_fp64_peak(iters, sink, &grid, &block, st);
    if (e == cudaSuccess) e = cudaEventRecord(e1, st);
    if (e == cudaSuccess) e = cudaEventSynchronize(e1);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (sink) cudaFree(sink);
    if (e != cudaSuccess) return cuda_fail(e, "tcmp_fp64_peak");
    *flops_out = 2.0 * 8 * 16 * (double)iters * (double)grid * block / (ms * 1e-3);
    return TCMP_OK;
}

int tcmp_get_limits(double *torque7, double *q_lo7, double *q_hi7, double *qd_max7) {
    // panda_mod.urdf:127,153,179,205,231,257,283
    static const double lo[7] = {-2.8973, -1.7628, -2.8973, -3.0718, -2.8973, -0.0175, -2.8973};
    static const double hi[7] = {2.8973, 1.7628, 2.8973, -0.0698, 2.8973, 3.7525, 2.8973};
    static const double vm[7] = {2.175, 2.175, 2.175, 2.175, 2.61, 2.61, 2.61};
    static const double tq[7] = {87, 87, 87, 87, 12, 12, 12};
    for (int i = 0; i < 7; ++i) {
        if (torque7) torque7[i] = tq[i];
        if (q_lo7) q_lo7[i] = lo[i];
        if (q_hi7) q_hi7[i] = hi[i];
        if (qd_max7) qd_max7[i] = vm[i];
    }
    return TCMP_OK;
}

}  // extern "C"
