// tests/native/ik_host.cpp -- TEST HARNESS: compiles the product's IK solver core (csrc/ik_core.cuh,
// the same source the CUDA kernel uses) for the HOST so the decision tree can be exercised against the
// compiled reference on a CPU-only box.  Never linked into libtcmp.so; not a fallback path.
#define _GNU_SOURCE 1
#include <cmath>
#include <cstdint>
#include "../../torque_constrained_motion_planning_b200/csrc/ik_core.cuh"

extern "C" void host_ik_batch(int64_t n, const double *rot9, const double *trans3, const double *free_vals,
                              int n_free, int free_broadcast, double *sols_out, int32_t *count_out,
                              uint8_t *status_out) {
    using namespace tcmp::ik;
#pragma omp parallel for schedule(static)
    for (int64_t p = 0; p < n; ++p)
        for (int f = 0; f < n_free; ++f) {
            double R[9];
            for (int i = 0; i < 9; ++i) R[i] = rot9[i * n + p];
            Pose P;
            prepare_pose(R, trans3[p], trans3[n + p], trans3[2 * n + p],
                         free_broadcast ? free_vals[f] : free_vals[(int64_t)f * n + p], P);
            const int64_t o = p * n_free + f;
            Emit out;
            out.sols = sols_out ? sols_out + o * 56 : nullptr;
            out.count = 0;
            out.status = 0;
            solve_one(P, out);
            if (out.sols)
                for (int k = (out.count < 8 ? out.count : 8) * 7; k < 56; ++k) out.sols[k] = 0.0;
            count_out[o] = out.count;
            if (status_out) status_out[o] = (uint8_t)out.status;
        }
}

// Panda flange pose (the reference's ComputeFk convention: panda_link8 in panda_link0), q SoA [7][n] ->
// trans3 [3][n], rot9 [9][n] row-major.  The modified-DH chain of ik_kernels.cu fk_kernel, with glibc's sin / cos
// and no FMA contraction, so the poses the tests feed to both solvers are the same bits on every x86-64 host.
extern "C" void host_fk_batch(int64_t n, const double *q, double *trans3, double *rot9) {
    static const double A[7] = {0, 0, 0, 0.0825, -0.0825, 0, 0.088};
    static const double D[7] = {0.333, 0, 0.316, 0, 0.384, 0, 0};
    static const int AL[7] = {0, -1, 1, 1, -1, 1, 1};
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; ++i) {
        double X[3] = {1, 0, 0}, Y[3] = {0, 1, 0}, Z[3] = {0, 0, 1}, p[3] = {0, 0, 0};
        for (int k = 0; k < 7; ++k) {
            const double s = std::sin(q[k * n + i]), c = std::cos(q[k * n + i]);
            for (int r = 0; r < 3; ++r) {
                const double y = AL[k] == 0 ? Y[r] : (AL[k] > 0 ? Z[r] : -Z[r]);
                const double z = AL[k] == 0 ? Z[r] : (AL[k] > 0 ? -Y[r] : Y[r]);
                p[r] += A[k] * X[r] + D[k] * z;
                const double x = X[r];
                X[r] = c * x + s * y;
                Y[r] = c * y - s * x;
                Z[r] = z;
            }
        }
        for (int r = 0; r < 3; ++r) {
            trans3[r * n + i] = p[r] + 0.107 * Z[r];
            rot9[(r * 3 + 0) * n + i] = X[r];
            rot9[(r * 3 + 1) * n + i] = Y[r];
            rot9[(r * 3 + 2) * n + i] = Z[r];
        }
    }
}
