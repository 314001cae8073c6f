// tests/native/track_host.cpp -- TEST HARNESS: compiles K15's per-rollout code (csrc/track_core.cuh, the same source
// track_kernels.cu instantiates) for the HOST, so tracking rollouts can be checked against a NumPy composition of the
// controller torque and K14's host build on a CPU-only box, and counts the FP64 operations K15 adds to a K14 step.
// It includes rollout_host.cpp, so the same library also exports K14's host build (host_rollout_batch) and K13's / K10's.
// Never linked into libtcmp.so.
#include "rollout_host.cpp"

#include "../../torque_constrained_motion_planning_b200/csrc/track_core.cuh"

template <bool TOOL, typename P> static void run_tracks(const TrackArgs &a, const P &p) {
    double S[kTrackRows];
    for (int64_t i = 0; i < a.roll.n; ++i) track_state<int64_t, TOOL, P>(a, i, p, kTable, S, 1);
}

static const double *stock_limits() {
    static tcmp_model m;
    static bool init = false;
    if (!init) {
        for (int j = 0; j < 7; ++j) m.torque_limit[j] = torque_limit(j);
        init = true;
    }
    return m.torque_limit;
}

// Arguments as tcmp_track_batch (validated by the caller); mode TCMP_MODE_RNE or TCMP_MODE_DYN, model NULL = the
// compiled-in Panda.
extern "C" void host_track_batch(const tcmp_model *model, int mode, int64_t n, int n_steps, double dt, int n_seg,
                                 const double *coeffs, int coeffs_broadcast, const double *q0, const double *qd0,
                                 const double *kp, const double *kd, const double *pm, double ps, const double *cm,
                                 double cs, const double *q_lo, const double *q_hi, const double *qd_max,
                                 double *q_out, double *qd_out, double *q_traj, double *qd_traj, double *tau_traj,
                                 int32_t *first_violation, int32_t *first_saturation, double *max_err) {
    TrackArgs a{};
    a.roll = RollArgs{n, n_steps, dt, q0, qd0, nullptr, 0, pm, ps, {}, q_out, qd_out, q_traj, qd_traj,
                      first_violation};
    a.roll.lim.check_q = q_lo != nullptr;
    a.roll.lim.check_qd = qd_max != nullptr;
    const double *L = model ? model->torque_limit : stock_limits();
    for (int j = 0; j < 7; ++j) {
        a.roll.lim.lo[j] = q_lo ? q_lo[j] : 0.0;
        a.roll.lim.hi[j] = q_hi ? q_hi[j] : 0.0;
        a.roll.lim.qd_max[j] = qd_max ? qd_max[j] : 0.0;
        a.kp[j] = kp[j];
        a.kd[j] = kd[j];
        a.tau_limit[j] = L[j];
    }
    a.n_seg = n_seg;
    a.coeffs_broadcast = coeffs_broadcast != 0;
    a.coeffs = coeffs;
    a.ctrl_mass = cm;
    a.ctrl_scalar = cs;
    a.tau_traj = tau_traj;
    a.max_err = max_err;
    a.first_saturation = first_saturation;
    const bool dyn = mode == TCMP_MODE_DYN;
    if (model) {
        const RtParams<double> p = params_from_desc<double>(*model);
        if (dyn) run_tracks<true>(a, p);
        else run_tracks<false>(a, p);
    } else {
        if (dyn) run_tracks<true>(a, ConstParams());
        else run_tracks<false>(a, ConstParams());
    }
}

template <bool TOOL, typename P>
static void run_control(int64_t n, const double *q, const double *qd, const double *acmd, const double *cm, double cs,
                        double *tau, const P &p) {
    for (int64_t i = 0; i < n; ++i) {
        double qs[7], vs[7], as[7], t[7];
        for (int j = 0; j < 7; ++j) {
            qs[j] = q[j * n + i];
            vs[j] = qd[j * n + i];
            as[j] = acmd[j * n + i];
        }
        track_control<TOOL, P>(qs, vs, as, cm ? cm[i] : cs, p, kTable, t);
        for (int j = 0; j < 7; ++j) tau[j * n + i] = t[j];
    }
}

// K15's controller torque, unsaturated: [7][n] states and commanded accelerations, controller mass [n] or scalar.
extern "C" void host_track_control(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                   const double *acmd, const double *cm, double cs, double *tau) {
    const bool dyn = mode == TCMP_MODE_DYN;
    if (model) {
        const RtParams<double> p = params_from_desc<double>(*model);
        if (dyn) run_control<true>(n, q, qd, acmd, cm, cs, tau, p);
        else run_control<false>(n, q, qd, acmd, cm, cs, tau, p);
    } else {
        if (dyn) run_control<true>(n, q, qd, acmd, cm, cs, tau, ConstParams());
        else run_control<false>(n, q, qd, acmd, cm, cs, tau, ConstParams());
    }
}

// FP64 operations K15 adds to a K14 step (rne mode, compiled-in Panda, payload attached), counted on the formulas of
// track_core.cuh: part 0 = the controller's rne_body (its sincos of joints 2..7 excluded), 1 = the reference at t_k
// (x, v, a) and a_cmd, 2 = the reference x at t_{k+1} and the error.  Saturation and the maximum are compares.
extern "C" int64_t host_track_flops(int part) {
    g_flops = 0;
    if (part == 0) {
        Cnt s[7], c[7], qd[7], acmd[7], tau[7];
        for (int j = 0; j < 7; ++j) { s[j] = 0.3; c[j] = 0.9; qd[j] = 0.5; acmd[j] = 1.0; }
        rne_body<Cnt, true, false, ConstParams>(s, c, qd, acmd, Cnt(1.0), Cnt(0.0), tau, ConstParams(), Cnt(9.81));
        return g_flops;
    }
    const Cnt u(0.25), c0(0.1), c1(0.2), c2(0.3), c3(0.4), c4(0.5), c5(0.6), two(2), three(3), four(4), five(5), six(6),
        twelve(12), twenty(20), q(0.1), qd(0.2), kp(1), kd(1);
    const Cnt x = c0 + u * (c1 + u * (c2 + u * (c3 + u * (c4 + u * c5))));
    if (part == 1) {
        const Cnt v = c1 + u * (two * c2 + u * (three * c3 + u * (four * c4 + u * (five * c5))));
        const Cnt a = two * c2 + u * (six * c3 + u * (twelve * c4 + u * (twenty * c5)));
        const Cnt acmd = (a + kp * (x - q)) + kd * (v - qd);
        (void)acmd;
    } else {
        const Cnt d = q - x;
        (void)d;
    }
    return 7 * g_flops;
}
