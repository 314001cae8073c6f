// rollout_core.cuh -- K14: forward-dynamics rollouts per state.  Classical RK4 on qdd = f(q, qd) = K13's joint
// accelerations (fd_core.cuh: fd_sincos, fd_bias, fd_factor, ldl_solve) under a zero-order-hold torque, n_steps
// steps, in the order include/tcmp.h pins:
//   a1 = f(q, v);  q2 = q + h2 v;   v2 = v + h2 a1;  a2 = f(q2, v2);  q3 = q + h2 v2;  v3 = v + h2 a2;  a3 = f(q3, v3)
//   q4 = q + dt v3;  v4 = v + dt a3;  a4 = f(q4, v4)
//   q' = q + h6 (((v + 2 v2) + 2 v3) + v4);   v' = v + h6 (((a1 + 2 a2) + 2 a3) + a4)      h2 = dt / 2, h6 = dt / 6
// and, per stored state, the joint- and velocity-limit checks whose first failure is returned.
//
// Registers are the constraint: the four stages are one rolled loop around one inlined evaluation, h is formed before
// M's columns (so qd is dead while the factor is built), a caller record is read afresh at every use (FreshRt), and
// everything that outlives a stage -- the step's base state, the two RK4 sums, the next stage's position, the held
// torque and the mass -- lives in a per-thread column of scratch `S` (row r at S[r * ld]): shared memory
// [kRollRows][128] on the device (conflict-free: a warp reads 32 consecutive doubles of one row), a local array with
// ld = 1 in the host build (tests/native/rollout_host.cpp).
#pragma once
#include "fd_core.cuh"

namespace tcmp {

// Limit checks of a stored state, by value in the launch parameters (tcmp_collision_batch's convention).
struct RollLimits {
    double lo[7], hi[7], qd_max[7];
    int check_q, check_qd;
};

enum : int {
    kRollQ = 0, kRollV = 7, kRollSQ = 14, kRollSV = 21, kRollQN = 28, kRollU = 35, kRollMass = 42, kRollZero = 43,
    kRollRows = 44
};

// A record parameter as seen from one use: offset by a zero read from the scratch column through a volatile load,
// which neither the compiler nor ptxas can fold, hoist or share between uses.  Read directly, the record's ~50 values
// are loaded once into uniform registers ahead of the RK4 loop, and their live ranges through every stage overflow
// the register files (140-148 B of spills).  A zero from an inline-asm mov does not work: ptxas folds it.
template <typename T> TCMP_FN const T *roll_fresh(const T *p, const volatile long long *zero) {
#ifdef __CUDA_ARCH__
    return reinterpret_cast<const T *>(reinterpret_cast<const char *>(p) + *zero);
#else
    return p;
#endif
}

// A caller record as the rollout's dynamics read it: the members of RtParams<double> that rne_body and the mass
// columns use, each fetched afresh at every use.
struct FreshRt {
    using R = RtParams<double>;
    struct Rows {
        const R *r;
        const volatile long long *z;
        TCMP_FN const double *operator[](int k) const { return roll_fresh(r, z)->l[k]; }
    };
    struct Link6 {
        const R *r;
        const volatile long long *z;
        TCMP_FN operator const double *() const { return roll_fresh(r, z)->l6; }
    };
    template <double R::*M> struct Scalar {
        const R *r;
        const volatile long long *z;
        TCMP_FN operator double() const { return roll_fresh(r, z)->*M; }
    };
    Rows l;
    Link6 l6;
    Scalar<&R::jzz0> jzz0;
    Scalar<&R::payload_hz> payload_hz;
    Scalar<&R::payload_j> payload_j;
    Scalar<&R::tool_z> tool_z;
};
TCMP_FN ConstParams roll_view(const ConstParams &p, const volatile long long *) { return p; }
TCMP_FN FreshRt roll_view(const RtParams<double> &p, const volatile long long *z) {
    return FreshRt{{&p, z}, {&p, z}, {&p, z}, {&p, z}, {&p, z}, {&p, z}};
}

// lo <= q <= hi and |qd| <= qd_max on every joint, as requested; a NaN fails.
TCMP_FN bool roll_state_ok(const double (&q)[7], const double (&v)[7], const RollLimits &lim) {
    bool ok = true;
    if (lim.check_q) {
#pragma unroll
        for (int j = 0; j < 7; ++j) ok = ok && q[j] >= lim.lo[j] && q[j] <= lim.hi[j];
    }
    if (lim.check_qd) {
#pragma unroll
        for (int j = 0; j < 7; ++j) ok = ok && fabs(v[j]) <= lim.qd_max[j];
    }
    return ok;
}

template <typename I> TCMP_FN double roll_load(const double *p) {
#ifdef __CUDA_ARCH__
    return __ldcs(p);
#else
    return *p;
#endif
}

// One call's arguments, by value in the launch parameters.
struct RollArgs {
    int64_t n;
    int n_steps;
    double dt;
    const double *q0, *qd0, *tau;   // [7][n]; qd0 / tau NULL = zeros; tau [n_steps][7][n] when tau_per_step
    int tau_per_step;
    const double *payload_mass;     // [n] or NULL (then payload_scalar)
    double payload_scalar;
    RollLimits lim;
    double *q_out, *qd_out, *q_traj, *qd_traj;   // each may be NULL
    int32_t *first_violation;
};

// K14's torque source: the initial state from q0 / qd0 (qd0 NULL = zeros), and the torque held ([7][n]) or given per
// step ([n_steps][7][n]), NULL = zero; nothing else observed.  rollout_state calls a policy's init once, torque before
// each step (it leaves the step's torque in the kRollU rows), observe on each stored state and finish at the end, each
// with the scratch column.  K15 (track_core.cuh) supplies a controller instead.
struct RollHeldTorque {
    template <typename I> TCMP_FN void init(const RollArgs &a, I i, double *__restrict__ S, int ld) {
        const I n = (I)a.n;
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            S[(kRollQ + j) * ld] = roll_load<I>(a.q0 + (I)j * n + i);
            S[(kRollV + j) * ld] = a.qd0 ? roll_load<I>(a.qd0 + (I)j * n + i) : 0.0;
            S[(kRollU + j) * ld] = 0.0;
        }
    }
    template <typename I> TCMP_FN void torque(const RollArgs &a, int k, I i, double *__restrict__ S, int ld) {
        if (a.tau && (a.tau_per_step || k == 0)) {
            const I n = (I)a.n;
            const double *t = a.tau_per_step ? a.tau + (I)k * 7 * n : a.tau;
#pragma unroll
            for (int j = 0; j < 7; ++j) S[(kRollU + j) * ld] = roll_load<I>(t + (I)j * n + i);
        }
    }
    template <typename I> TCMP_FN void observe(int, I, const double (&)[7], double *__restrict__, int) {}
    template <typename I> TCMP_FN void finish(I, double *__restrict__, int) {}
};

// Rollout i.  The first violation is n_steps when no stored state fails (or nothing is checked).
template <typename I, bool TOOL, typename P, bool GLOBAL = false, typename Pol = RollHeldTorque>
TCMP_FN void rollout_state(const RollArgs &args, I i, const P &p, const SinCos *__restrict__ tab,
                           double *__restrict__ S, int ld, Pol pol = Pol()) {
#define TCMP_ROW(r) S[(r) * ld]
    {
        const RollArgs &a = args;
        const double mass = a.payload_mass ? roll_load<I>(a.payload_mass + i) : a.payload_scalar;
        TCMP_ROW(kRollMass) = mass;
        TCMP_ROW(kRollZero) = 0.0;   // all-zero bits: roll_fresh's offset
        pol.init(a, i, S, ld);
    }
    int first = -1;
#pragma unroll 1
    for (int k = 0; k < args.n_steps; ++k) {
        pol.torque(args, k, i, S, ld);
        double qs[7], vs[7];
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            qs[j] = TCMP_ROW(kRollQ + j);
            vs[j] = TCMP_ROW(kRollV + j);
        }
#pragma unroll 1
        for (int st = 0; st < 4; ++st) {
            {
                const double dt = args.dt;
                const double cs = st < 2 ? 0.5 * dt : dt;
                // position side, from this stage's velocity: the sum, and the next stage's (or the step's final) q
#pragma unroll
                for (int j = 0; j < 7; ++j) {
                    const double sq = st == 0 ? vs[j] : TCMP_ROW(kRollSQ + j) + 2.0 * vs[j];
                    if (st < 3) {
                        TCMP_ROW(kRollSQ + j) = sq;
                        TCMP_ROW(kRollQN + j) = TCMP_ROW(kRollQ + j) + cs * vs[j];
                    } else {
                        TCMP_ROW(kRollQ + j) = TCMP_ROW(kRollQ + j) + dt / 6.0 * (TCMP_ROW(kRollSQ + j) + vs[j]);
                    }
                }
            }
            const double mass = TCMP_ROW(kRollMass);
            double b[7], bad_q = mass * 0.0, bad_v = 0.0;   // +-0 for finite inputs, NaN otherwise (K13's rule)
#pragma unroll
            for (int j = 0; j < 7; ++j) {
                b[j] = TCMP_ROW(kRollU + j);
                bad_q += qs[j] * 0.0;
                bad_v += vs[j] * 0.0 + b[j] * 0.0;
            }
            // K13's steps (fd_core.cuh), h first so that qd is dead while M is factored
            double s[7], c[7];
            fd_sincos<GLOBAL>(qs, s, c, tab);
            const double mp = TOOL ? 0.0 : (mass > 0.0 ? mass : 0.0), mt = TOOL ? mass : 0.0;
            const volatile long long *zero = reinterpret_cast<const volatile long long *>(&TCMP_ROW(kRollZero));
            using PV = decltype(roll_view(p, zero));
            fd_bias<TOOL, PV>(s, c, qs[0], vs, mp, mt, bad_v, roll_view(p, zero), b);
            TriOut<double> m;
            double inv_d[7];
            fd_factor<PV>(s, c, roll_view(p, zero), mp, bad_q, m, inv_d);
            ldl_solve(m.A, inv_d, b);
            // velocity side, from this stage's acceleration
            const double dt = args.dt;
            const double cs = st < 2 ? 0.5 * dt : dt;
#pragma unroll
            for (int j = 0; j < 7; ++j) {
                if (st < 3) {
                    TCMP_ROW(kRollSV + j) = st == 0 ? b[j] : TCMP_ROW(kRollSV + j) + 2.0 * b[j];
                    vs[j] = TCMP_ROW(kRollV + j) + cs * b[j];
                    qs[j] = TCMP_ROW(kRollQN + j);
                } else {
                    TCMP_ROW(kRollV + j) = TCMP_ROW(kRollV + j) + dt / 6.0 * (TCMP_ROW(kRollSV + j) + b[j]);
                }
            }
        }
        const RollArgs &a = args;
        const I n = (I)a.n;
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            qs[j] = TCMP_ROW(kRollQ + j);
            vs[j] = TCMP_ROW(kRollV + j);
        }
        if (a.q_traj) {
#pragma unroll
            for (int j = 0; j < 7; ++j) DynOut<I>::put(a.q_traj + ((I)k * 7 + j) * n + i, qs[j]);
        }
        if (a.qd_traj) {
#pragma unroll
            for (int j = 0; j < 7; ++j) DynOut<I>::put(a.qd_traj + ((I)k * 7 + j) * n + i, vs[j]);
        }
        if (first < 0 && !roll_state_ok(qs, vs, a.lim)) first = k;
        pol.observe(k, i, qs, S, ld);
    }
    const RollArgs &a = args;
    const I n = (I)a.n;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
        if (a.q_out) DynOut<I>::put(a.q_out + (I)j * n + i, TCMP_ROW(kRollQ + j));
        if (a.qd_out) DynOut<I>::put(a.qd_out + (I)j * n + i, TCMP_ROW(kRollV + j));
    }
    if (a.first_violation) a.first_violation[i] = first < 0 ? a.n_steps : first;
    pol.finish(i, S, ld);
#undef TCMP_ROW
}

}  // namespace tcmp
