// tests/native/select_host.cpp -- TEST HARNESS: runs K7's goal-IK selection for the HOST from the sources the kernel
// uses (csrc/ik_core.cuh, csrc/select_core.cuh, the static torque test of csrc/panda_model.cuh), one pose at a time
// and its candidates serially in (free value, solver order), so the selection can be checked against the composed
// reference on a CPU-only box.  Never linked into libtcmp.so; not a fallback path.
#include <cmath>
#include <cstdint>

#include "../../torque_constrained_motion_planning_b200/csrc/ik_core.cuh"
#include "../../torque_constrained_motion_planning_b200/csrc/select_core.cuh"

using namespace tcmp;

static const SinCos kTable[kSinCosTableSize] = {
#include "../../torque_constrained_motion_planning_b200/csrc/sincos_table.inc"
};

template <bool TOOL, typename P>
static void run(int64_t n, const double *rot9, const double *trans3, const double *free_vals, int n_free,
                int free_broadcast, const double *q_ref, int ref_broadcast, const JointLimits &lim, int check,
                double mass, double payload_threshold, int use_max_norm, double *best_q, double *best_cost,
                int32_t *n_valid, int32_t *n_redo, const P &prm) {
    // the kernel's payload rule (select_kernels.cu)
    const double mp_inertial = TOOL ? 0.0 : (mass > payload_threshold ? mass : 0.0);
    const double mp_tool = TOOL ? mass : 0.0;
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t p = 0; p < n; ++p) {
        double R[9], ref[7];
        for (int i = 0; i < 9; ++i) R[i] = rot9[i * n + p];
        for (int j = 0; j < 7; ++j) ref[j] = ref_broadcast ? q_ref[j] : q_ref[j * n + p];
        double wc = INFINITY, bq[7] = {0, 0, 0, 0, 0, 0, 0};
        int wk = kNoKey, valid = 0, redo = 0;
        for (int f = 0; f < n_free; ++f) {
            double sols[56];
            ik::Pose Pz;
            ik::prepare_pose(R, trans3[p], trans3[n + p], trans3[2 * n + p],
                             free_broadcast ? free_vals[f] : free_vals[(int64_t)f * n + p], Pz);
            ik::Emit out;
            out.sols = sols;
            out.count = 0;
            out.status = 0;
            ik::solve_one_t<false>(Pz, out);
            if (out.status & ik::kStatusRedo) {
                ++redo;
                out.count = 0;
                ik::solve_one_t<true>(Pz, out);
            }
            const int cnt = out.count < 8 ? out.count : 8;
            for (int s = 0; s < cnt; ++s) {
                double q[7], c2 = 0.0, cmax = 0.0;
                if (!scan_candidate(sols + s * 7, ref, lim, q, c2, cmax)) continue;
                if (check) {
                    double tau[7];
                    const double z[7] = {0, 0, 0, 0, 0, 0, 0};
                    rne_core_table<false, TOOL, P>(q, z, z, mp_inertial, mp_tool, tau, kTable, prm);
                    if (!limits_ok<double, P>(tau, prm)) continue;
                }
                ++valid;
                const double cost = candidate_cost(c2, cmax, use_max_norm);
                if (better(cost, f * 8 + s, wc, wk)) {
                    wc = cost;
                    wk = f * 8 + s;
                    for (int j = 0; j < 7; ++j) bq[j] = q[j];
                }
            }
        }
        for (int j = 0; j < 7; ++j) best_q[j * n + p] = bq[j];
        best_cost[p] = wc;
        n_valid[p] = valid;
        if (n_redo) n_redo[p] = redo;
    }
}

template <bool TOOL>
static void with_model(const tcmp_model *model, int64_t n, const double *rot9, const double *trans3,
                       const double *free_vals, int n_free, int free_broadcast, const double *q_ref, int ref_broadcast,
                       const JointLimits &lim, int check, double mass, double thr, int use_max_norm, double *best_q,
                       double *best_cost, int32_t *n_valid, int32_t *n_redo) {
    if (model)
        run<TOOL>(n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast, lim, check, mass, thr,
                  use_max_norm, best_q, best_cost, n_valid, n_redo, params_from_desc<double>(*model));
    else
        run<TOOL>(n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast, lim, check, mass, thr,
                  use_max_norm, best_q, best_cost, n_valid, n_redo, ConstParams());
}

// tcmp_ik_select_model on the host, plus n_redo [n] (may be NULL): the solves per pose that took the elbow-singular
// redo path.  model == NULL: the compiled-in Panda.
extern "C" void host_select(const tcmp_model *model, int64_t n, const double *rot9, const double *trans3,
                            const double *free_vals, int n_free, int free_broadcast, const double *q_ref,
                            int ref_broadcast, const double *q_lo, const double *q_hi, int mode, double mass,
                            double payload_threshold, int use_max_norm, double *best_q, double *best_cost,
                            int32_t *n_valid, int32_t *n_redo) {
    JointLimits lim;
    for (int j = 0; j < 7; ++j) {
        lim.lo[j] = q_lo[j];
        lim.hi[j] = q_hi[j];
    }
    const int check = mode != TCMP_MODE_BASE;
    if (mode == TCMP_MODE_DYN)
        with_model<true>(model, n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast, lim, check,
                         mass, payload_threshold, use_max_norm, best_q, best_cost, n_valid, n_redo);
    else
        with_model<false>(model, n, rot9, trans3, free_vals, n_free, free_broadcast, q_ref, ref_broadcast, lim, check,
                          mass, payload_threshold, use_max_norm, best_q, best_cost, n_valid, n_redo);
}
