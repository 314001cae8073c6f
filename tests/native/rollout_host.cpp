// tests/native/rollout_host.cpp -- TEST HARNESS: compiles K14's per-rollout code (csrc/rollout_core.cuh, the same source
// rollout_kernels.cu instantiates) for the HOST, so rollouts can be checked against a NumPy RK4 over K13's host build
// on a CPU-only box, and counts the FP64 operations of one step.  It includes fd_host.cpp, so the same library also
// exports K13's host build (host_forward_dynamics_batch) and K10's (host_dynamics_batch).  Never linked into
// libtcmp.so.
#include "fd_host.cpp"

#include "../../torque_constrained_motion_planning_b200/csrc/rollout_core.cuh"

template <bool TOOL, typename P> static void run_rollouts(const RollArgs &a, const P &p) {
    double S[kRollRows];
    for (int64_t i = 0; i < a.n; ++i) rollout_state<int64_t, TOOL, P>(a, i, p, kTable, S, 1);
}

// Arguments as tcmp_rollout_batch (validated by the caller); mode TCMP_MODE_RNE or TCMP_MODE_DYN, model NULL = the
// compiled-in Panda.
extern "C" void host_rollout_batch(const tcmp_model *model, int mode, int64_t n, int n_steps, double dt,
                                   const double *q0, const double *qd0, const double *tau, int tau_per_step,
                                   const double *pm, double ps, const double *q_lo, const double *q_hi,
                                   const double *qd_max, double *q_out, double *qd_out, double *q_traj,
                                   double *qd_traj, int32_t *first_violation) {
    RollArgs a{n, n_steps, dt, q0, qd0, tau, tau_per_step, pm, ps, {}, q_out, qd_out, q_traj, qd_traj,
               first_violation};
    a.lim.check_q = q_lo != nullptr;
    a.lim.check_qd = qd_max != nullptr;
    for (int j = 0; j < 7; ++j) {
        a.lim.lo[j] = q_lo ? q_lo[j] : 0.0;
        a.lim.hi[j] = q_hi ? q_hi[j] : 0.0;
        a.lim.qd_max[j] = qd_max ? qd_max[j] : 0.0;
    }
    const bool dyn = mode == TCMP_MODE_DYN;
    if (model) {
        const RtParams<double> p = params_from_desc<double>(*model);
        if (dyn) run_rollouts<true>(a, p);
        else run_rollouts<false>(a, p);
    } else {
        if (dyn) run_rollouts<true>(a, ConstParams());
        else run_rollouts<false>(a, ConstParams());
    }
}

// FP64 operations of one RK4 step's combination (everything but the four evaluations of qdd), per joint, counted on
// the formulas of rollout_core.cuh: the stage states, the two weighted sums and the update.
extern "C" int64_t host_rollout_combination_flops(void) {
    Cnt q(0.1), v(0.2), h2(0.5), dt(1.0), h6(1.0 / 6), two(2.0), a1(0.3), a2(0.4), a3(0.5), a4(0.6);
    g_flops = 0;
    const Cnt q2 = q + h2 * v, v2 = v + h2 * a1;
    const Cnt q3 = q + h2 * v2, v3 = v + h2 * a2;
    const Cnt q4 = q + dt * v3, v4 = v + dt * a3;
    const Cnt qn = q + h6 * (((v + two * v2) + two * v3) + v4);
    const Cnt vn = v + h6 * (((a1 + two * a2) + two * a3) + a4);
    (void)q2; (void)q3; (void)q4; (void)qn; (void)vn;
    return 7 * g_flops;
}
