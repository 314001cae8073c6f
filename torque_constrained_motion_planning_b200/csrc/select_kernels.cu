// select_kernels.cu -- goal-IK post-filter fused behind the IK solver (SURVEY.md 8f-4).
//
// Per target pose the reference planner sweeps the free joint (ikfast.py:153-161), solves IK for each
// value, drops solutions outside the joint limits (ikfast.py:167, franka_ik_fast.py:55-57), keeps the
// one nearest to the current configuration (closest_inverse_kinematics, ikfast.py:172-188, max-norm by
// default; select_solution, ik_utils.py:43-52) and then requires the static torque test of that grasp
// configuration (panda_primitives.py:263).  Here one warp owns one pose and its lanes the values of the sweep: each lane
// solves, filters by limits, runs the STATIC torque test (rne_core<double, false, TOOL>) on every
// surviving solution and keeps the nearest feasible one -- no solution set ever leaves the SM.
#include "ik_core.cuh"
#include "panda_model.cuh"
#include "select_core.cuh"
#include "tcmp_internal.h"

namespace tcmp {

// (sin, cos)(i pi / 512) for the table-driven sincos of the static torque tests (panda_model.cuh sincos6_table<GLOBAL>):
// read in place through the read-only cache -- this kernel's shared memory is spoken for, and its torque tests are
// too few per CTA to pay for staging 16 KB.  Own copy per translation unit (no relocatable device code in the build).
static __device__ const SinCos kSelSinCosTable[kSinCosTableSize] = {
#include "sincos_table.inc"
};

// One warp per pose, two dense phases (the first version ran the torque test inside the per-lane solution loop:
// with 0 / 4 / 8 solutions per lane and ~1 in 4 inside the joint limits the warp executed 8 sparse RNE rounds
// per sweep and the kernel took 6x longer than the IK alone).
//   A. lanes own the free-joint values of the sweep (32 per round): solve, filter by joint limits, and append
//      every survivor (q, cost, key = f*8 + s) to a per-warp shared-memory candidate list with a ballot/popc
//      prefix -- the list is in sweep order.
//   B. lanes own CANDIDATES: one static torque test each (dense), then a shuffle arg-min over (cost, key) picks
//      the nearest feasible configuration; ties go to the earliest key, as a serial scan in sweep order would.
// Round 2 (profiles/r02/select_variants.log): one 8-warp CTA per SM with CTA barriers at the phase boundaries, so that
// all warps of the SM walk the solver's ~60 KB of code together (as the CTA-wide IK sweep kernel does), against
// 4 independent 2-warp CTAs per SM at the same occupancy: 0.89 -> 1.10 G solves/s (rne, 25 free values), outputs
// bit-identical.  Barriers alone at 2 / 4 warps: 0.99 / 1.03; 4 warps without barriers: 0.91.
#ifndef TCMP_SEL_WARPS
#define TCMP_SEL_WARPS 8
#endif
#ifndef TCMP_SEL_ALIGN
#define TCMP_SEL_ALIGN 1
#endif
constexpr int kSelWarps = TCMP_SEL_WARPS;   // warps per CTA (8: 147 KB of candidate lists, dynamic shared memory)
constexpr bool kSelAlign = TCMP_SEL_ALIGN;  // CTA barriers at the phase boundaries
constexpr int kSelCap = 256;            // 32 lanes x 8 solutions: a round can never overflow the list
constexpr int kSelRow = 9;              // q[7], cost, key (as double) -- odd stride, conflict-free 64-bit rows

template <bool TOOL, typename P>
__global__ void __launch_bounds__(kSelWarps * 32)
ik_select_kernel(int64_t n, int n_free, int free_broadcast, const double *__restrict__ rot9,
                 const double *__restrict__ trans3, const double *__restrict__ free_vals,
                 const double *__restrict__ q_ref, int ref_broadcast, JointLimits lim, int check_torque,
                 double mass, double payload_threshold, int use_max_norm, double *__restrict__ best_q,
                 double *__restrict__ best_cost, int32_t *__restrict__ n_valid, const __grid_constant__ P prm) {
    extern __shared__ double cand_all[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    double *cand = cand_all + wib * (kSelCap * kSelRow);
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const double mp_inertial = TOOL ? 0.0 : (mass > payload_threshold ? mass : 0.0);
    const double mp_tool = TOOL ? mass : 0.0;
    const unsigned lt_mask = (1u << lane) - 1u;
    // kSelAlign: the trip count is CTA-uniform (a warp past the end repeats the last pose and writes nothing), so the
    // barriers below are reached by every thread.
    const int64_t p_end = kSelAlign ? ((n + n_warps - 1) / n_warps) * n_warps : n;
    for (int64_t p0 = warp; p0 < p_end; p0 += n_warps) {
        const bool act = p0 < n;
        const int64_t p = act ? p0 : n - 1;
        double R[9], ref[7];
#pragma unroll
        for (int i = 0; i < 9; ++i) R[i] = __ldg(rot9 + i * n + p);
#pragma unroll
        for (int j = 0; j < 7; ++j) ref[j] = ref_broadcast ? __ldg(q_ref + j) : __ldg(q_ref + j * n + p);
        const double tx = __ldg(trans3 + p), ty = __ldg(trans3 + n + p), tz = __ldg(trans3 + 2 * n + p);
        double wc = INFINITY;     // this lane's best feasible candidate so far: cost, key, configuration
        int wk = kNoKey, valid = 0;
        double bq[7] = {0, 0, 0, 0, 0, 0, 0};
        for (int fbase = 0; fbase < n_free; fbase += 32) {
            // ---- phase A: IK + joint-limit filter for up to 32 free values ----
            if (kSelAlign) __syncthreads();
            const int f = fbase + lane;
            double sols[56];
            int cnt = 0;
            if (f < n_free) {
                const double j6 = free_broadcast ? __ldg(free_vals + f) : __ldg(free_vals + (int64_t)f * n + p);
                ik::Pose P;
                ik::prepare_pose(R, tx, ty, tz, j6, P);
                ik::Emit out;
                out.sols = sols;
                out.count = 0;
                out.status = 0;
                ik::solve_one_t<false>(P, out);
                if (out.status & ik::kStatusRedo) {   // elbow singularity: redo with the complete tree (cold region)
                    out.count = 0;
                    ik::solve_one_t<true>(P, out);
                }
                cnt = out.count < 8 ? out.count : 8;
            }
            int ncand = 0;
            for (int sidx = 0; sidx < 8; ++sidx) {       // warp-synchronous: every lane walks all 8 slots
                bool keep = sidx < cnt;
                double q[7], c2 = 0.0, cmax = 0.0;
                if (keep) keep = scan_candidate(sols + sidx * 7, ref, lim, q, c2, cmax);
                const unsigned m = __ballot_sync(0xffffffffu, keep);
                if (keep) {
                    // the list order is irrelevant: the KEY (f*8 + s) carries the sweep order for tie-breaks
                    double *row = cand + (ncand + __popc(m & lt_mask)) * kSelRow;
#pragma unroll
                    for (int j = 0; j < 7; ++j) row[j] = q[j];
                    row[7] = candidate_cost(c2, cmax, use_max_norm);
                    row[8] = (double)(f * 8 + sidx);
                }
                ncand += __popc(m);
            }
            if (kSelAlign) __syncthreads(); else __syncwarp();
            // ---- phase B: one candidate per lane, dense static torque tests ----
            for (int c = lane; c < ncand; c += 32) {
                const double *row = cand + c * kSelRow;
                double q[7];
#pragma unroll
                for (int j = 0; j < 7; ++j) q[j] = row[j];
                bool ok = true;
                if (check_torque) {
                    double tau[7];
                    const double z[7] = {0, 0, 0, 0, 0, 0, 0};
                    rne_core_table<false, TOOL, P, true>(q, z, z, mp_inertial, mp_tool, tau, kSelSinCosTable, prm);   // table read in place (__ldg)
                    ok = limits_ok<double, P>(tau, prm);
                }
                if (ok) {
                    ++valid;
                    const double cost = row[7];
                    const int key = (int)row[8];
                    if (better(cost, key, wc, wk)) {
                        wc = cost;
                        wk = key;
#pragma unroll
                        for (int j = 0; j < 7; ++j) bq[j] = q[j];
                    }
                }
            }
            __syncwarp();   // the list is rewritten by the next sweep round
        }
        // warp arg-min over (cost, key), sum of survivors
        double bc = wc;
        int bk = wk, bl = lane;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double oc = __shfl_xor_sync(0xffffffffu, bc, off);
            const int ok2 = __shfl_xor_sync(0xffffffffu, bk, off);
            const int ol = __shfl_xor_sync(0xffffffffu, bl, off);
            valid += __shfl_xor_sync(0xffffffffu, valid, off);
            if (better(oc, ok2, bc, bk) || (oc == bc && ok2 == bk && ol < bl)) { bc = oc; bk = ok2; bl = ol; }
        }
        if (lane == bl && act) {       // with no survivor every lane ties at (inf, kNoKey): lane 0 writes zeros
#pragma unroll
            for (int j = 0; j < 7; ++j) best_q[j * n + p] = bq[j];
            best_cost[p] = bc;
            n_valid[p] = valid;
        }
    }
}

template <bool TOOL, typename P>
static cudaError_t launch_select_p(int64_t n, const double *rot9, const double *trans3, const double *free_vals,
                                   int n_free, int free_broadcast, const double *q_ref, int ref_broadcast,
                                   const JointLimits &lim, int check, double mass, double payload_threshold,
                                   int use_max_norm, double *best_q, double *best_cost, int32_t *n_valid, const P &prm,
                                   cudaStream_t st) {
    auto kern = ik_select_kernel<TOOL, P>;
    constexpr int smem = kSelWarps * kSelCap * kSelRow * (int)sizeof(double);
    if (smem > 48 * 1024) {   // wider CTAs only (per device, so set on the launching one)
        const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
    }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSelWarps * 32, smem) != cudaSuccess || per_sm <= 0)
        per_sm = 1;
    const int64_t full = (int64_t)sm_count() * per_sm * kSelWaves, want = (n + kSelWarps - 1) / kSelWarps;
    const int grid = (int)(want < full ? want : full);
    kern<<<grid, kSelWarps * 32, smem, st>>>(n, n_free, free_broadcast, rot9, trans3, free_vals, q_ref, ref_broadcast, lim,
                                          check, mass, payload_threshold, use_max_norm, best_q, best_cost, n_valid, prm);
    return cudaGetLastError();
}

template <bool TOOL>
static cudaError_t launch_select_t(int64_t n, const double *rot9, const double *trans3, const double *free_vals,
                                   int n_free, int free_broadcast, const double *q_ref, int ref_broadcast,
                                   const JointLimits &lim, int check, double mass, double payload_threshold,
                                   int use_max_norm, double *best_q, double *best_cost, int32_t *n_valid,
                                   const tcmp_model *model, cudaStream_t st) {
    if (model)
        return launch_select_p<TOOL>(n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast, lim,
                                     check, mass, payload_threshold, use_max_norm, best_q, best_cost, n_valid,
                                     params_from_desc<double>(*model), st);
    return launch_select_p<TOOL>(n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast, lim, check,
                                 mass, payload_threshold, use_max_norm, best_q, best_cost, n_valid, ConstParams(), st);
}

cudaError_t launch_ik_select(int64_t n, const double *rot9, const double *trans3, const double *free_vals,
                             int n_free, int free_broadcast, const double *q_ref, int ref_broadcast,
                             const double *q_lo, const double *q_hi, int mode, double mass,
                             double payload_threshold, int use_max_norm, double *best_q, double *best_cost,
                             int32_t *n_valid, cudaStream_t st, const tcmp_model *model) {
    JointLimits lim;
    for (int j = 0; j < 7; ++j) {
        lim.lo[j] = q_lo[j];
        lim.hi[j] = q_hi[j];
    }
    const int check = mode != TCMP_MODE_BASE;
    if (mode == TCMP_MODE_DYN)
        return launch_select_t<true>(n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast, lim,
                                     check, mass, payload_threshold, use_max_norm, best_q, best_cost, n_valid, model, st);
    return launch_select_t<false>(n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast, lim, check,
                                  mass, payload_threshold, use_max_norm, best_q, best_cost, n_valid, model, st);
}

}  // namespace tcmp
