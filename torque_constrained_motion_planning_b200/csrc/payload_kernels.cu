// payload_kernels.cu -- K11 (tcmp_payload_interval_batch) and K12 (tcmp_edge_payload_interval): the open interval of
// payload masses that keep a state, or every waypoint of a min-jerk edge, within the torque limits -- the inverse of
// the torque test, in one launch instead of a bisection over the mass.  The per-state code is csrc/payload_core.cuh.
//
//  * K11: one thread per state, SoA inputs [7][n] read with streaming loads, m_lo / m_hi / unloaded_ok stored with
//    streaming stores (any of them may be NULL: a uniform run-time branch).  No grid-stride loop, 32-bit offsets while
//    7 n fits, and the sin / cos table read in place through the read-only cache, as K10.
//  * K12: one warp per edge, lanes over waypoints (K4's layout, sampling and table staging).  Each lane keeps a running
//    intersection of its waypoints' intervals; a __shfl_xor_sync butterfly combines the 32 lanes at the end.  The warp
//    visits every waypoint: unlike K4's first failure, the interval's ends keep moving after it has become empty.
#include "payload_core.cuh"
#include "tcmp_internal.h"

namespace tcmp {

// (sin, cos)(i pi / 512): this translation unit's read-only copy (no relocatable device code in the build)
static __device__ const SinCos kPayloadSinCosTable[kSinCosTableSize] = {
#include "sincos_table.inc"
};

template <typename I>
__device__ __forceinline__ void store_interval(I i, const MassInterval<double> &r, double *__restrict__ lo_out,
                                               double *__restrict__ hi_out, uint8_t *__restrict__ ok_out) {
    if (lo_out) __stcs(lo_out + i, r.lo);
    if (hi_out) __stcs(hi_out + i, r.hi);
    if (ok_out) __stcs(ok_out + i, (uint8_t)r.ok);
}

template <typename I, bool DYN, bool TOOL, typename P>
__global__ void __launch_bounds__(128)
payload_interval_kernel(I n, const double *__restrict__ q, const double *__restrict__ qd,
                        const double *__restrict__ qdd, double *__restrict__ lo_out, double *__restrict__ hi_out,
                        uint8_t *__restrict__ ok_out, const __grid_constant__ P p) {
    const I i = (I)blockIdx.x * (I)blockDim.x + (I)threadIdx.x;
    if (i >= n) return;
    double qs[7], vs[7], as[7], a[7], b[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) {
        qs[j] = __ldcs(q + (I)j * n + i);
        if constexpr (DYN) {
            vs[j] = __ldcs(qd + (I)j * n + i);
            as[j] = __ldcs(qdd + (I)j * n + i);
        }
    }
    const MassInterval<double> r = payload_state<DYN, TOOL, P, true>(qs, vs, as, p, kPayloadSinCosTable, a, b);
    store_interval<I>(i, r, lo_out, hi_out, ok_out);
}

// np.linspace(1/W, 1, W)[w], as K4's linspace_sample
__device__ __forceinline__ double edge_time(int w, int W, double interval, double step) {
    return (w == W - 1 && W > 1) ? 1.0 : __dadd_rn(interval, __dmul_rn((double)w, step));
}

__device__ __forceinline__ double max_of(double x, double y) { return x > y ? x : y; }
__device__ __forceinline__ double min_of(double x, double y) { return x < y ? x : y; }

template <bool DYN, bool TOOL, typename P>
__global__ void __launch_bounds__(128)
edge_payload_kernel(int64_t n_edges, int W, double interval, double step, const double *__restrict__ qa,
                    const double *__restrict__ qb, double *__restrict__ lo_out, double *__restrict__ hi_out,
                    uint8_t *__restrict__ ok_out, const __grid_constant__ P prm) {
    __shared__ SinCos tab[kSinCosTableSize];
    for (int t = threadIdx.x; t < kSinCosTableSize; t += blockDim.x) tab[t] = kPayloadSinCosTable[t];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const double inf = INFINITY;
    for (int64_t e = warp; e < n_edges; e += n_warps) {
        double a0[7], A[7];
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            a0[j] = __ldg(qa + j * n_edges + e);
            A[j] = __ldg(qb + j * n_edges + e) - a0[j];      // min_jerk_v2.py:121 with x = qa, v = a = 0, t = 1
        }
        MassInterval<double> acc = {-inf, inf, true};
        for (int base = 0; base < W; base += 32) {
            const int w = base + lane;
            if (w < W) {
                const double t = edge_time(w, W, interval, step);
                double qs[7], vs[7], as[7], a[7], b[7];
                const double t2 = t * t;
                const double px = t2 * t * (10.0 + t * (-15.0 + 6.0 * t));
                const double pv = t2 * (30.0 + t * (-60.0 + 30.0 * t));
                const double pa = t * (60.0 + t * (-180.0 + 120.0 * t));
#pragma unroll
                for (int j = 0; j < 7; ++j) {
                    qs[j] = a0[j] + A[j] * px;
                    if constexpr (DYN) {
                        vs[j] = A[j] * pv;
                        as[j] = A[j] * pa;
                    }
                }
                intersect(acc, payload_state<DYN, TOOL, P>(qs, vs, as, prm, tab, a, b));
            }
        }
        // butterfly: every lane ends with the whole edge's intersection (never NaN, so plain compares suffice)
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            acc.lo = max_of(acc.lo, __shfl_xor_sync(0xffffffffu, acc.lo, off));
            acc.hi = min_of(acc.hi, __shfl_xor_sync(0xffffffffu, acc.hi, off));
        }
        acc.ok = __all_sync(0xffffffffu, acc.ok);
        if (lane == 0) store_interval<int64_t>(e, acc, lo_out, hi_out, ok_out);
    }
}

// ---- launch ------------------------------------------------------------------------------------------------------
// 32-bit element offsets while the largest, 6 n + n - 1, fits
static inline bool fits_int7(int64_t n) { return n < (int64_t)(0x7fffffff / 7); }

template <bool DYN, bool TOOL, typename P>
static cudaError_t launch_states_p(int64_t n, const double *q, const double *qd, const double *qdd, double *lo,
                                   double *hi, uint8_t *ok, const P &p, cudaStream_t st) {
    const int64_t grid = (n + 127) / 128;
    if (fits_int7(n))
        payload_interval_kernel<int, DYN, TOOL, P><<<(unsigned)grid, 128, 0, st>>>((int)n, q, qd, qdd, lo, hi, ok, p);
    else
        payload_interval_kernel<int64_t, DYN, TOOL, P><<<(unsigned)grid, 128, 0, st>>>(n, q, qd, qdd, lo, hi, ok, p);
    return cudaGetLastError();
}

template <bool DYN, bool TOOL, typename P>
static cudaError_t launch_edges_p(int64_t n_edges, int W, const double *qa, const double *qb, double *lo, double *hi,
                                  uint8_t *ok, const P &p, cudaStream_t st) {
    const double interval = 1.0 / W, step = W > 1 ? (1.0 - interval) / (W - 1) : 0.0;
    auto kern = edge_payload_kernel<DYN, TOOL, P>;
    const int grid = grid_for(reinterpret_cast<const void *>(kern), 128, n_edges * 32, kEdgeWaves);
    kern<<<grid, 128, 0, st>>>(n_edges, W, interval, step, qa, qb, lo, hi, ok, p);
    return cudaGetLastError();
}

// mode -> (DYN, TOOL) as the torque kernels dispatch it, model -> ConstParams / RtParams<double>
template <bool DYN, bool TOOL, typename F>
static cudaError_t with_params(const tcmp_model *model, F &&f) {
    if (model) return f.template operator()<DYN, TOOL>(params_from_desc<double>(*model));
    return f.template operator()<DYN, TOOL>(ConstParams());
}
template <typename F> static cudaError_t dispatch(int mode, bool dynamic, const tcmp_model *model, F &&f) {
    const bool tool = mode == TCMP_MODE_DYN;
    if (dynamic) return tool ? with_params<true, true>(model, f) : with_params<true, false>(model, f);
    return tool ? with_params<false, true>(model, f) : with_params<false, false>(model, f);
}

static cudaError_t fill_everything(int64_t n, double *lo, double *hi, uint8_t *ok, cudaStream_t st) {
    cudaError_t e = cudaSuccess;
    if (lo) e = launch_fill<double>(n, lo, -INFINITY, st);
    if (hi && e == cudaSuccess) e = launch_fill<double>(n, hi, INFINITY, st);
    if (ok && e == cudaSuccess) e = launch_fill<uint8_t>(n, ok, 1, st);
    return e;
}

struct StatesLaunch {
    int64_t n;
    const double *q, *qd, *qdd;
    double *lo, *hi;
    uint8_t *ok;
    cudaStream_t st;
    template <bool DYN, bool TOOL, typename P> cudaError_t operator()(const P &p) const {
        return launch_states_p<DYN, TOOL>(n, q, qd, qdd, lo, hi, ok, p, st);
    }
};

struct EdgesLaunch {
    int64_t n;
    int W;
    const double *qa, *qb;
    double *lo, *hi;
    uint8_t *ok;
    cudaStream_t st;
    template <bool DYN, bool TOOL, typename P> cudaError_t operator()(const P &p) const {
        return launch_edges_p<DYN, TOOL>(n, W, qa, qb, lo, hi, ok, p, st);
    }
};

cudaError_t launch_payload_interval(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                    const double *qdd, double *lo, double *hi, uint8_t *ok, cudaStream_t st) {
    if (mode == TCMP_MODE_BASE) return fill_everything(n, lo, hi, ok, st);
    // without both velocity arrays the torque test tests the static state; nov always does
    const bool dynamic = mode != TCMP_MODE_NOV && qd && qdd;
    return dispatch(mode, dynamic, model, StatesLaunch{n, q, qd, qdd, lo, hi, ok, st});
}

cudaError_t launch_edge_payload_interval(const tcmp_model *model, int mode, int64_t n_edges, int W, const double *qa,
                                         const double *qb, int static_only, double *lo, double *hi, uint8_t *ok,
                                         cudaStream_t st) {
    if (mode == TCMP_MODE_BASE) return fill_everything(n_edges, lo, hi, ok, st);
    const bool dynamic = mode != TCMP_MODE_NOV && !static_only;
    return dispatch(mode, dynamic, model, EdgesLaunch{n_edges, W, qa, qb, lo, hi, ok, st});
}

}  // namespace tcmp
