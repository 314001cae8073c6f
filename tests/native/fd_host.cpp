// tests/native/fd_host.cpp -- TEST HARNESS: compiles K13's per-state code (csrc/fd_core.cuh, the same source
// fd_kernels.cu instantiates) for the HOST, so forward dynamics can be checked against the oracle on a CPU-only box,
// and counts its FP64 operations.  It includes dynamics_host.cpp, so the same library also exports K10's host build
// (host_dynamics_batch: M to check M^-1 against) and its operation counter.  Never linked into libtcmp.so.
#include "dynamics_host.cpp"

#include "../../torque_constrained_motion_planning_b200/csrc/fd_core.cuh"

template <bool TOOL, typename P>
static void run_fd(int64_t n, const double *q, const double *qd, const double *tau, const double *pm, double ps,
                   double *qdd, double *Minv, const P &p) {
    for (int64_t i = 0; i < n; ++i)
        fd_state<int64_t, TOOL, P>(n, i, q, qd, tau, pm ? pm[i] : ps, p, kTable, qdd, Minv);
}

// mode: TCMP_MODE_RNE or TCMP_MODE_DYN; model == NULL: the compiled-in Panda.
extern "C" void host_forward_dynamics_batch(const tcmp_model *model, int mode, int64_t n, const double *q,
                                            const double *qd, const double *tau, const double *pm, double ps,
                                            double *qdd, double *Minv) {
    const bool dyn = mode == TCMP_MODE_DYN;
    if (model) {
        const RtParams<double> p = params_from_desc<double>(*model);
        if (dyn) run_fd<true>(n, q, qd, tau, pm, ps, qdd, Minv, p);
        else run_fd<false>(n, q, qd, tau, pm, ps, qdd, Minv, p);
    } else {
        if (dyn) run_fd<true>(n, q, qd, tau, pm, ps, qdd, Minv, ConstParams());
        else run_fd<false>(n, q, qd, tau, pm, ps, qdd, Minv, ConstParams());
    }
}

// ---- operation count (Cnt from dynamics_host.cpp; a division counts 1) --------------------------------------------
static inline Cnt operator/(Cnt a, Cnt b) { ++g_flops; return Cnt(a.v / b.v); }
static inline bool operator>(Cnt a, Cnt b) { return a.v > b.v; }

struct NullTri {
    void M(int, int, Cnt) {}
};

// FP64 operations per state of the compiled-in Panda in rne mode with the payload attached, sincos and the
// non-finite-input checks excluded: part 0 = M and its LDL^T factor, 1 = h and the solve for qdd, 2 = M^-1.
extern "C" int64_t host_fd_flops(int part) {
    Cnt s[7], c[7], qd[7], qdd0[7], b[7], h[7], inv_d[7];
    for (int j = 0; j < 7; ++j) { s[j] = 0.3; c[j] = 0.9; qd[j] = 0.5; qdd0[j] = 0.0; b[j] = 1.0; }
    TriOut<Cnt> m;
    ldl_columns<0>(s, c, ConstParams(), Cnt(1.0), m, inv_d);
    g_flops = 0;
    if (part == 0) {
        ldl_columns<0>(s, c, ConstParams(), Cnt(1.0), m, inv_d);
    } else if (part == 1) {
        rne_body<Cnt, true, false, ConstParams>(s, c, qd, qdd0, Cnt(1.0), Cnt(0.0), h, ConstParams(), Cnt(9.81));
        for (int j = 0; j < 7; ++j) b[j] = b[j] - h[j];
        ldl_solve(m.A, inv_d, b);
    } else {
        NullTri out;
        ldl_inverse(m.A, inv_d, out);
    }
    return g_flops;
}
