// tests/native/collision_host.cpp -- TEST HARNESS: compiles K8/K9's per-configuration and per-edge code
// (csrc/collision_core.cuh, the same source collision_kernels.cu instantiates) for the HOST, so the collision
// predicate, the step count and the extend steps can be checked against a long-double reference on a CPU-only box.
// Never linked into libtcmp.so; not a fallback path.
#include <cstdint>

#include "../../torque_constrained_motion_planning_b200/csrc/collision_core.cuh"

using namespace tcmp;

// collision_kernel: q [7][n] -> hit [n]
extern "C" void host_collision_batch(int64_t n, const double *q, int n_obs, const tcmp_obstacle *obs,
                                     const double *q_lo, const double *q_hi, double payload_radius, uint8_t *hit) {
    Scene S;
    fill_scene(n_obs, obs, q_lo, q_hi, payload_radius, &S);
    for (int64_t i = 0; i < n; ++i) {
        double qs[7];
        for (int j = 0; j < 7; ++j) qs[j] = q[j * n + i];
        hit[i] = (uint8_t)config_collides(S, qs);
    }
}

// extend_prefix_kernel in BASE mode (no torque test): q1, q2 [7][n_edges] -> n_steps, prefix [n_edges]
extern "C" void host_extend_prefix(int64_t n_edges, const double *q1, const double *q2, const double *res_in,
                                   int n_obs, const tcmp_obstacle *obs, const double *q_lo, const double *q_hi,
                                   double payload_radius, int32_t *n_steps, int32_t *prefix) {
    Scene S;
    fill_scene(n_obs, obs, q_lo, q_hi, payload_radius, &S);
    double res[7];
    for (int j = 0; j < 7; ++j) res[j] = res_in[j];
    for (int64_t e = 0; e < n_edges; ++e) {
        double a[7], b[7], nrm2 = 0.0;
        for (int j = 0; j < 7; ++j) {
            a[j] = q1[j * n_edges + e];
            b[j] = q2[j * n_edges + e];
            nrm2 = extend_norm2_add(nrm2, a[j], b[j], res[j]);
        }
        const int N = extend_num_configs(nrm2);
        int k = 0;
        for (; k < N; ++k) {
            double q[7];
            extend_config(a, b, N, k, q);
            if (config_collides(S, q)) break;
        }
        n_steps[e] = N;
        prefix[e] = k;
    }
}

// Configuration k of the N-configuration edge a -> b (a, b, q_out [7]).
extern "C" void host_extend_config(const double *a_in, const double *b_in, int N, int k, double *q_out) {
    double a[7], b[7], q[7];
    for (int j = 0; j < 7; ++j) { a[j] = a_in[j]; b[j] = b_in[j]; }
    extend_config(a, b, N, k, q);
    for (int j = 0; j < 7; ++j) q_out[j] = q[j];
}
