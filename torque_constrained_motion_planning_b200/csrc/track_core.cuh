// track_core.cuh -- K15: closed-loop tracking rollouts per state.  A computed-torque controller follows a piecewise
// quintic reference at a zero-order hold of dt; its torque saturates at the joint limits and drives K14's RK4 plant
// (rollout_core.cuh), in the order include/tcmp.h pins.  Step k, t_k = k dt:
//   a_cmd = (a(t_k) + kp (x(t_k) - q)) + kd (v(t_k) - qd)
//   tau_cmd = rne_body(q, qd, a_cmd) with the controller's payload mass (K13's payload rule)
//   tau = |tau_cmd| > L ? copysign(L, tau_cmd) : tau_cmd      on all seven joints
//   (q, qd) <- one K14 RK4 step under tau held, with the plant's payload mass
// K14's rollout_state runs the loop; TrackControl is its policy: it evaluates the reference and the controller into
// the kRollU rows before each step, and observes the tracking error after it.  The same source builds for the host
// (tests/native/track_host.cpp).
#pragma once
#include "rollout_core.cuh"

namespace tcmp {

// Rows after K14's: the controller's mass, and the running maximum error and first saturation (-1 = none yet), which
// kept in registers through the RK4 stages would spill.
enum : int { kTrackCtrlMass = kRollRows, kTrackErr = kRollRows + 1, kTrackSat = kRollRows + 2, kTrackRows = kRollRows + 3 };

// One call's arguments beyond K14's, by value in the launch parameters.
struct TrackArgs {
    RollArgs roll;                  // q0 / qd0 NULL = the reference's x(0) / v(0); tau NULL (the controller's)
    int n_seg, coeffs_broadcast;
    const double *coeffs;           // [n_seg][7][6] shared, or [n_seg][7][6][n]
    double kp[7], kd[7], tau_limit[7];
    const double *ctrl_mass;        // [n] or NULL (then ctrl_scalar)
    double ctrl_scalar;
    double *tau_traj, *max_err;     // each may be NULL
    int32_t *first_saturation;
};

// Coefficients are re-read every step: through the read-only cache, not evicted first as the streamed inputs are.
TCMP_FN double track_ldg(const double *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

template <typename I> TCMP_FN double track_coeff(const TrackArgs &a, I i, int s, int j, int c) {
    if (a.coeffs_broadcast) return track_ldg(a.coeffs + ((int64_t)s * 7 + j) * 6 + c);
    return track_ldg(a.coeffs + (((I)s * 7 + j) * 6 + c) * (I)a.roll.n + i);
}

// The reference at time t >= 0: segment s = (int)t at local time u = t - s; from t = n_seg on, the end held (x on the
// last segment at u = 1, v = a = 0).
struct TrackTime {
    int s;
    double u;
    bool hold;
};
TCMP_FN TrackTime track_time(const TrackArgs &a, double t) {
    const bool hold = !(t < (double)a.n_seg);
    const int s = hold ? a.n_seg - 1 : (int)t;
    return {s, hold ? 1.0 : t - (double)s, hold};
}

// Joint j of the reference at tt, by traj_kernel's Horner formulas.  V / A false skip v / a.
template <bool V, bool A, typename I>
TCMP_FN void track_reference(const TrackArgs &a, I i, const TrackTime &tt, int j, double &x, double &v, double &acc) {
    const int s = tt.s;
    const double u = tt.u;
    const double c0 = track_coeff(a, i, s, j, 0), c1 = track_coeff(a, i, s, j, 1), c2 = track_coeff(a, i, s, j, 2),
                 c3 = track_coeff(a, i, s, j, 3), c4 = track_coeff(a, i, s, j, 4), c5 = track_coeff(a, i, s, j, 5);
    x = c0 + u * (c1 + u * (c2 + u * (c3 + u * (c4 + u * c5))));
    if (V) v = tt.hold ? 0.0 : c1 + u * (2.0 * c2 + u * (3.0 * c3 + u * (4.0 * c4 + u * (5.0 * c5))));
    if (A) acc = tt.hold ? 0.0 : 2.0 * c2 + u * (6.0 * c3 + u * (12.0 * c4 + u * (20.0 * c5)));
}

// The controller's inverse dynamics: rne_body at (q, qd, a_cmd) with mass m.  TOOL (dyn): the tool-point force m g for
// every m; else (rne) the payload a rigid body on the flange iff m > 0.  A non-finite m makes every torque NaN.
template <bool TOOL, typename PV, bool GLOBAL = false>
TCMP_FN void track_control(const double (&q)[7], const double (&qd)[7], const double (&acmd)[7], double m, const PV &p,
                           const SinCos *__restrict__ tab, double (&tau)[7]) {
    double s[7], c[7];
    fd_sincos<GLOBAL>(q, s, c, tab);
    const double mp = TOOL ? 0.0 : (m > 0.0 ? m : 0.0), mt = TOOL ? m : 0.0;
    rne_body<double, true, TOOL, PV>(s, c, qd, acmd, mp, mt, tau, p, gravity_for(q[0]));
    const bool bad = !(m * 0.0 == 0.0);
#pragma unroll
    for (int j = 0; j < 7; ++j) tau[j] = bad ? double(NAN) : tau[j];
}

// |tau_cmd| > L saturates to +-L; a NaN passes unchanged.  Returns whether any joint saturated.
TCMP_FN bool track_saturate(double (&tau)[7], const double (&L)[7]) {
    bool sat = false;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
        const bool over = fabs(tau[j]) > L[j];
        sat = sat || over;
        tau[j] = over ? copysign(L[j], tau[j]) : tau[j];
    }
    return sat;
}

// The rollout index as the step hooks use it, offset by roll_fresh's zero: addresses derived from it (coefficients,
// tau_traj) are then formed at each use, not hoisted ahead of the step loop, where they would stay live through the
// RK4 stages and spill.
template <typename I> TCMP_FN I track_fresh(I i, const double *S, int ld) {
#ifdef __CUDA_ARCH__
    return i + (I)*reinterpret_cast<const volatile long long *>(&S[kRollZero * ld]);
#else
    (void)S;
    (void)ld;
    return i;
#endif
}

// K15's policy for rollout_state: the initial state (q0 / qd0, or the reference at t = 0), the controller's saturated
// torque before each step, and the running maximum tracking error and first saturation.
template <bool TOOL, typename P, bool GLOBAL> struct TrackControl {
    const TrackArgs &a;
    const P &p;
    const SinCos *__restrict__ tab;

    template <typename I> TCMP_FN void init(const RollArgs &r, I i, double *__restrict__ S, int ld) {
        const I n = (I)r.n;
        S[kTrackCtrlMass * ld] = a.ctrl_mass ? roll_load<I>(a.ctrl_mass + i) : a.ctrl_scalar;
        S[kTrackErr * ld] = 0.0;
        S[kTrackSat * ld] = -1.0;
        const TrackTime t0 = track_time(a, 0.0);
#pragma unroll 1
        for (int j = 0; j < 7; ++j) {
            double x = 0.0, v = 0.0, unused;
            if (!r.q0 || !r.qd0) track_reference<true, false>(a, i, t0, j, x, v, unused);
            S[(kRollQ + j) * ld] = r.q0 ? roll_load<I>(r.q0 + (I)j * n + i) : x;
            S[(kRollV + j) * ld] = r.qd0 ? roll_load<I>(r.qd0 + (I)j * n + i) : v;
        }
    }

    template <typename I> TCMP_FN void torque(const RollArgs &r, int k, I i0, double *__restrict__ S, int ld) {
        const I i = track_fresh(i0, S, ld);
        // a_cmd into the kRollU rows, one joint at a time: the 42 coefficients are never live together
        const TrackTime tk = track_time(a, (double)k * r.dt);
        double bad = 0.0;
#pragma unroll 1
        for (int j = 0; j < 7; ++j) {
            double x, v, acc;
            track_reference<true, true>(a, i, tk, j, x, v, acc);
            acc = (acc + a.kp[j] * (x - S[(kRollQ + j) * ld])) + a.kd[j] * (v - S[(kRollV + j) * ld]);
            bad += x * 0.0 + acc * 0.0;   // a non-finite reference value poisons every torque (saturation would
            S[(kRollU + j) * ld] = acc;   // otherwise turn it into a limit)
        }
        double q[7], qd[7], acmd[7], tau[7];
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            q[j] = S[(kRollQ + j) * ld];
            qd[j] = S[(kRollV + j) * ld];
            acmd[j] = S[(kRollU + j) * ld];
        }
        const volatile long long *zero = reinterpret_cast<const volatile long long *>(&S[kRollZero * ld]);
        track_control<TOOL, decltype(roll_view(p, zero)), GLOBAL>(q, qd, acmd, S[kTrackCtrlMass * ld],
                                                                  roll_view(p, zero), tab, tau);
#pragma unroll
        for (int j = 0; j < 7; ++j) tau[j] = bad == 0.0 ? tau[j] : double(NAN);
        if (track_saturate(tau, a.tau_limit) && S[kTrackSat * ld] < 0.0) S[kTrackSat * ld] = (double)k;
        const I n = (I)r.n;
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            S[(kRollU + j) * ld] = tau[j];
            if (a.tau_traj) DynOut<I>::put(a.tau_traj + ((I)k * 7 + j) * n + i, tau[j]);
        }
    }

    // the stored state after step k against x(t_{k+1}); a NaN term makes the maximum NaN for good
    template <typename I>
    TCMP_FN void observe(int k, I i0, const double (&q)[7], double *__restrict__ S, int ld) {
        if (!a.max_err) return;
        const I i = track_fresh(i0, S, ld);
        const TrackTime tk = track_time(a, (double)(k + 1) * a.roll.dt);
        double err = S[kTrackErr * ld];
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            double x, unused;
            track_reference<false, false>(a, i, tk, j, x, unused, unused);
            const double d = fabs(q[j] - x);
            err = d > err || d != d ? d : err;
        }
        S[kTrackErr * ld] = err;
    }

    template <typename I> TCMP_FN void finish(I i, double *__restrict__ S, int ld) {
        if (a.max_err) DynOut<I>::put(a.max_err + i, S[kTrackErr * ld]);
        const double sat = S[kTrackSat * ld];
        if (a.first_saturation) a.first_saturation[i] = sat < 0.0 ? a.roll.n_steps : (int)sat;
    }
};

// Rollout i of tcmp_track_batch.
template <typename I, bool TOOL, typename P, bool GLOBAL = false>
TCMP_FN void track_state(const TrackArgs &a, I i, const P &p, const SinCos *__restrict__ tab, double *__restrict__ S,
                         int ld) {
    rollout_state<I, TOOL, P, GLOBAL>(a.roll, i, p, tab, S, ld, TrackControl<TOOL, P, GLOBAL>{a, p, tab});
}

}  // namespace tcmp
