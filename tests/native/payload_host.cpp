// tests/native/payload_host.cpp -- TEST HARNESS: compiles K11/K12's per-state code (csrc/payload_core.cuh, the same
// source payload_kernels.cu instantiates, table-driven sincos included) for the HOST, so the affine torque terms a, b
// and the payload-mass intervals can be checked against the oracle on a CPU-only box, and counts the FP64 operations
// of the algorithm with an instrumented scalar type.  Never linked into libtcmp.so; not a fallback path.
#include <cmath>
#include <cstdint>

#include "../../torque_constrained_motion_planning_b200/csrc/payload_core.cuh"

using namespace tcmp;

static const SinCos kTable[kSinCosTableSize] = {
#include "../../torque_constrained_motion_planning_b200/csrc/sincos_table.inc"
};

template <bool DYN, bool TOOL, typename P>
static void run(int64_t n, const double *q, const double *qd, const double *qdd, double *a_out, double *b_out,
                double *lo, double *hi, uint8_t *ok, const P &p) {
    for (int64_t i = 0; i < n; ++i) {
        double qs[7], vs[7] = {0}, as[7] = {0}, a[7], b[7];
        for (int j = 0; j < 7; ++j) {
            qs[j] = q[j * n + i];
            if (DYN) { vs[j] = qd[j * n + i]; as[j] = qdd[j * n + i]; }
        }
        const MassInterval<double> r = payload_state<DYN, TOOL, P>(qs, vs, as, p, kTable, a, b);
        for (int j = 0; j < 7; ++j) {
            if (a_out) a_out[j * n + i] = a[j];
            if (b_out) b_out[j * n + i] = b[j];
        }
        if (lo) lo[i] = r.lo;
        if (hi) hi[i] = r.hi;
        if (ok) ok[i] = (uint8_t)r.ok;
    }
}

template <typename P>
static void dispatch(int mode, int64_t n, const double *q, const double *qd, const double *qdd, double *a, double *b,
                     double *lo, double *hi, uint8_t *ok, const P &p) {
    const bool dynamic = mode != TCMP_MODE_NOV && qd && qdd, tool = mode == TCMP_MODE_DYN;
    if (dynamic) {
        if (tool) run<true, true>(n, q, qd, qdd, a, b, lo, hi, ok, p);
        else run<true, false>(n, q, qd, qdd, a, b, lo, hi, ok, p);
    } else {
        if (tool) run<false, true>(n, q, qd, qdd, a, b, lo, hi, ok, p);
        else run<false, false>(n, q, qd, qdd, a, b, lo, hi, ok, p);
    }
}

// tcmp_payload_interval_batch on the host, plus a [7][n] and b [7][n] (each output may be NULL; mode != BASE).
// model == NULL: the compiled-in Panda (ConstParams), else the record folded and regrouped at run time.
extern "C" void host_payload_batch(const tcmp_model *model, int mode, int64_t n, const double *q, const double *qd,
                                   const double *qdd, double *a, double *b, double *lo, double *hi, uint8_t *ok) {
    if (model) dispatch(mode, n, q, qd, qdd, a, b, lo, hi, ok, params_from_desc<double>(*model));
    else dispatch(mode, n, q, qd, qdd, a, b, lo, hi, ok, ConstParams());
}

// ---- operation count -------------------------------------------------------------------------------------------------
// A double that counts the FP64 operations applied to it: add / sub / mul / div = 1, fma = 2; negation, compares and
// constants free.
static int64_t g_flops = 0;
struct Cnt {
    double v;
    Cnt() : v(0) {}
    Cnt(double x) : v(x) {}
};
static inline Cnt operator+(Cnt a, Cnt b) { ++g_flops; return Cnt(a.v + b.v); }
static inline Cnt operator-(Cnt a, Cnt b) { ++g_flops; return Cnt(a.v - b.v); }
static inline Cnt operator*(Cnt a, Cnt b) { ++g_flops; return Cnt(a.v * b.v); }
static inline Cnt operator/(Cnt a, Cnt b) { ++g_flops; return Cnt(a.v / b.v); }
static inline Cnt operator-(Cnt a) { return Cnt(-a.v); }
static inline Cnt &operator+=(Cnt &a, Cnt b) { return a = a + b; }
static inline Cnt &operator-=(Cnt &a, Cnt b) { return a = a - b; }
static inline bool operator<(Cnt a, Cnt b) { return a.v < b.v; }
static inline bool operator>(Cnt a, Cnt b) { return a.v > b.v; }
static inline bool operator>=(Cnt a, Cnt b) { return a.v >= b.v; }
static inline bool operator==(Cnt a, Cnt b) { return a.v == b.v; }
static inline bool operator!=(Cnt a, Cnt b) { return a.v != b.v; }
static inline Cnt fabs(Cnt a) { return Cnt(std::fabs(a.v)); }
static inline Cnt fma(Cnt a, Cnt b, Cnt c) { g_flops += 2; return Cnt(a.v * b.v + c.v); }

// FP64 operations per state of the compiled-in Panda (a, b and the interval; sincos excluded -- six angles of
// host_sincos_flops in tests/native/dynamics_host.cpp).
extern "C" int64_t host_payload_flops(int mode, int dynamic) {
    Cnt s[7], c[7], qd[7], qdd[7], a[7], b[7];
    for (int j = 0; j < 7; ++j) { s[j] = 0.3; c[j] = 0.9; qd[j] = 0.5; qdd[j] = 1.5; }
    g_flops = 0;
    const bool tool = mode == TCMP_MODE_DYN;
    const ConstParams p;
    if (dynamic) {
        if (tool) payload_terms<Cnt, true, true>(s, c, qd, qdd, Cnt(kGravity), p, a, b);
        else payload_terms<Cnt, true, false>(s, c, qd, qdd, Cnt(kGravity), p, a, b);
    } else {
        if (tool) payload_terms<Cnt, false, true>(s, c, qd, qdd, Cnt(kGravity), p, a, b);
        else payload_terms<Cnt, false, false>(s, c, qd, qdd, Cnt(kGravity), p, a, b);
    }
    payload_interval<Cnt>(a, b, p);
    return g_flops;
}
