// select_core.cuh -- K7's per-candidate logic: the joint-limit filter, the cost in both norms and the (cost, key)
// ordering that the per-lane scan and the warp arg-min both use.  The same source builds for the host
// (tests/native/select_host.cpp), which runs one pose's whole selection serially for the CPU tests.
#pragma once
#include "panda_model.cuh"

namespace tcmp {

struct JointLimits {
    double lo[7], hi[7];
};

// One IK solution s[7] against the limits and the reference: copies it to q, returns whether every joint lies in
// [lo, hi] (violates_limits; a NaN limit bounds nothing, as !(q < NaN) holds) and accumulates the squared L2
// distance c2 and the max-norm distance cmax.  cmax keeps a NaN distance, as np.linalg.norm(..., ord=inf) does
// (fmax would drop it).
TCMP_FN bool scan_candidate(const double *s, const double (&ref)[7], const JointLimits &lim, double (&q)[7],
                            double &c2, double &cmax) {
    bool keep = true;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
        q[j] = s[j];
        keep = keep && !(q[j] < lim.lo[j]) && !(q[j] > lim.hi[j]);
        const double d = fabs(q[j] - ref[j]);
        c2 += d * d;
        cmax = d > cmax || d != d ? d : cmax;
    }
    return keep;
}

TCMP_FN double candidate_cost(double c2, double cmax, int use_max_norm) { return use_max_norm ? cmax : sqrt(c2); }

constexpr int kNoKey = 0x7fffffff;   // the key of "nothing selected yet" (its cost is +inf)

// (cost, key) ranks before (best_cost, best_key); key = f * 8 + s orders candidates by (free value, solver order).
// Costs rank in numeric order, a NaN cost after every number (+inf included), equal costs by the smaller key.  Any
// candidate ranks before the empty state best_key == kNoKey, so a NaN cost can still be selected; the empty state
// ranks before nothing.
TCMP_FN bool better(double cost, int key, double best_cost, int best_key) {
    return key != kNoKey && (best_key == kNoKey || cost < best_cost || (cost == best_cost && key < best_key) ||
                             (best_cost != best_cost && (cost == cost || key < best_key)));
}

}  // namespace tcmp
