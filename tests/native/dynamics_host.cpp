// tests/native/dynamics_host.cpp -- TEST HARNESS: compiles K10's per-state code (csrc/dynamics_core.cuh, the same
// source dynamics_kernels.cu instantiates, table-driven sincos included) for the HOST, so M, C, g and J can be
// checked against the oracle on a CPU-only box, and counts the FP64 operations of the algorithm with an
// instrumented scalar type.  Never linked into libtcmp.so; not a fallback path.
#include <cstdint>

#include "../../torque_constrained_motion_planning_b200/csrc/dynamics_core.cuh"

using namespace tcmp;

static const SinCos kTable[kSinCosTableSize] = {
#include "../../torque_constrained_motion_planning_b200/csrc/sincos_table.inc"
};

template <typename P>
static void run(int64_t n, const double *q, const double *qd, const double *pm, double ps, double *M, double *C,
                double *g, double *J, const P &p) {
    for (int64_t i = 0; i < n; ++i) {
        DynOut<int64_t> out{M, C, g, J, n, i};
        dynamics_state<int64_t, P>(n, i, q, qd, pm ? pm[i] : ps, p, kTable, out);
    }
}

// model == NULL: the compiled-in Panda (ConstParams), else the record folded and regrouped at run time.
extern "C" void host_dynamics_batch(const tcmp_model *model, int64_t n, const double *q, const double *qd,
                                    const double *pm, double ps, double *M, double *C, double *g, double *J) {
    if (model) run(n, q, qd, pm, ps, M, C, g, J, params_from_desc<double>(*model));
    else run(n, q, qd, pm, ps, M, C, g, J, ConstParams());
}

// ---- operation count -------------------------------------------------------------------------------------------------
// A double that counts the FP64 operations applied to it: add / sub / mul = 1, fma = 2; negation and constants free.
static int64_t g_flops = 0;
struct Cnt {
    double v;
    Cnt() : v(0) {}
    Cnt(double x) : v(x) {}
};
static inline Cnt operator+(Cnt a, Cnt b) { ++g_flops; return Cnt(a.v + b.v); }
static inline Cnt operator-(Cnt a, Cnt b) { ++g_flops; return Cnt(a.v - b.v); }
static inline Cnt operator*(Cnt a, Cnt b) { ++g_flops; return Cnt(a.v * b.v); }
static inline Cnt operator-(Cnt a) { return Cnt(-a.v); }
static inline Cnt &operator+=(Cnt &a, Cnt b) { return a = a + b; }
static inline Cnt &operator-=(Cnt &a, Cnt b) { return a = a - b; }
static inline Cnt fma(Cnt a, Cnt b, Cnt c) { g_flops += 2; return Cnt(a.v * b.v + c.v); }

struct NullOut {
    void M(int, int, Cnt) {}
    void C(int, int, Cnt) {}
    void g(int, Cnt) {}
    void J(int, int, Cnt) {}
};

// FP64 operations per state of the compiled-in Panda for the output subset (want_* = 0 / 1), payload attached,
// sincos excluded (sincos_flops gives those per angle).
extern "C" int64_t host_dynamics_flops(int want_M, int want_C, int want_g, int want_J) {
    Cnt s[7], c[7], qd[7];
    for (int j = 0; j < 7; ++j) { s[j] = 0.3; c[j] = 0.9; qd[j] = 0.5; }
    NullOut out;
    g_flops = 0;
    dynamics_body<Cnt, ConstParams>(s, c, Cnt(0.3), Cnt(0.9), qd, Cnt(1.0), want_M, want_C, want_g, want_J,
                                    ConstParams(), out);
    return g_flops;
}

// FP64 operations of one table-driven sin / cos evaluation (node selection + reduction + polynomials + rotation).
extern "C" int64_t host_sincos_flops(void) {
    g_flops = 0;
    Cnt x(0.7), s, c;
    const Cnt kt = fma(x, Cnt(162.97466172610082), Cnt(6755399441055744.0));
    sincos_from_node<Cnt>(x, kt - Cnt(6755399441055744.0), Cnt(0.6), Cnt(0.8), s, c);
    return g_flops;
}
