#!/usr/bin/env python
"""bench_tracking.py -- closed-loop tracking rollouts (tcmp_track_batch, K15) in rollout-steps/s on one B200, against
the composition a user has without it: per control step one K1 launch for the controller torque (threshold 0), a torch
clamp, one K14 step (tcmp_rollout_batch, n_steps = 1) and the reference as torch element-wise ops.

    python bench_tracking.py [--steps K] [--warmup W]

Workloads (fp64, rne, kp = 100, kd = 20 on every joint, dt = 1 ms, payloads from bench.sample_states):
  throughput   1 M rollouts x 32 steps, one min-jerk edge reference per rollout ([1][7][6][n], 336 MB a set):
               final state, first_saturation and max_err.  Inputs rotate over 4 distinct sets so no step finds
               them in the 126 MB L2.
  montecarlo   65 536 rollouts x 1000 steps tracking one shared min-jerk trajectory, each rollout with its own plant
               mass and initial offset, the controller's mass fixed at 1 kg: first_saturation and max_err.  Its
               inputs (8 MB) fit in L2 by nature; the workload is FP64-bound.
Protocol as bench_rollout.py: W warm-up steps, ~1 s hold of the same step (sustained clocks), then K steps captured
in one CUDA graph and timed with CUDA events; nvidia-smi clocks sampled throughout; card name and power limit read in
the same run.  The composition is graph-captured too, with the same inputs, and its outputs are compared with K15's.

FLOP per rollout-step is the instrumented count of the host builds (tests/native/track_host.cpp, compiled here into a
temporary directory): K14's step (4 x K13's qdd + the RK4 combination) plus the controller's rne_body with its sincos,
the reference with a_cmd, and the reference and error after the step.  Saturation and the running maximum are
compares and count nothing.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402
from bench_dynamics import card_info  # noqa: E402

N_SETS = bench.N_SETS
LIMIT = [87.0, 87.0, 87.0, 87.0, 12.0, 12.0, 12.0]
DT, KP, KD = 1e-3, 100.0, 20.0
WORKLOADS = {"throughput": (bench.N_STATES, 32, False), "montecarlo": (65536, 1000, True)}


def op_counts():
    """FP64 operations per rollout-step from the instrumented host build."""
    tmp = tempfile.mkdtemp(prefix="tcmp_track_count_")
    so = os.path.join(tmp, "libtrack_count.so")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                           "-Wno-unknown-pragmas", "-o", so, os.path.join(ROOT, "tests", "native", "track_host.cpp")])
    L = ctypes.CDLL(so)
    for f in ("host_fd_flops", "host_sincos_flops", "host_rollout_combination_flops", "host_track_flops"):
        getattr(L, f).restype = ctypes.c_int64
    sincos = 6 * int(L.host_sincos_flops())
    qdd = int(L.host_fd_flops(0)) + int(L.host_fd_flops(1)) + sincos
    k14 = 4 * qdd + int(L.host_rollout_combination_flops())
    control = int(L.host_track_flops(0)) + sincos
    ref = int(L.host_track_flops(1)) + int(L.host_track_flops(2))
    return {"k14_step": k14, "controller": control, "reference_and_error": ref, "per_step": k14 + control + ref}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--hold-s", type=float, default=1.0)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")

    import numpy as np
    import torch
    from torque_constrained_motion_planning_b200 import _lib, engine
    from torque_constrained_motion_planning_b200.engine import _ptr

    if not torch.cuda.is_available():
        raise SystemExit("bench_tracking.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    flops = op_counts()
    f64 = dict(dtype=torch.float64, device=dev)
    RNE = _lib.MODE["rne"]
    kp, kd = np.full(7, KP), np.full(7, KD)
    L7 = torch.tensor(LIMIT, **f64)[:, None]

    def edge_coeffs(n, seed):
        qa, qb = bench.sample_states(n, seed)[0], bench.sample_states(n, seed + 1)[0]
        return engine.edge_coefficients(qa, qa + 0.3 * (qb - qa))        # [1][7][6][n]

    def make_sets(name, n):
        sets = []
        shared = np.ascontiguousarray(edge_coeffs(1, 3000)[..., 0])     # [1][7][6]
        for s in range(N_SETS):
            q, qd, _, mass = bench.sample_states(n, seed=1000 + s)
            if name == "throughput":
                c = edge_coeffs(n, 2000 + 2 * s)
                x0 = c[0, :, 0]
            else:
                c = shared
                x0 = np.broadcast_to(shared[0, :, 0][:, None], (7, n))
            q0 = x0 + 0.01 * np.tanh(q)
            qd0 = 0.05 * np.tanh(qd)
            sets.append(tuple(torch.as_tensor(np.ascontiguousarray(a), device=dev) for a in (c, q0, qd0, mass)))
        return sets

    def k15(sets, n, T, out):
        def step(i):
            c, q0, qd0, mass = sets[i % N_SETS]
            _lib.check(lib.tcmp_track_batch(None, RNE, n, T, DT, 1, _ptr(c), int(c.dim() == 3), _ptr(q0), _ptr(qd0),
                                            kp.ctypes.data, kd.ctypes.data, _ptr(mass), 0.0, None, 1.0, None, None,
                                            None, _ptr(out["q"]), _ptr(out["qd"]), None, None, None, None,
                                            _ptr(out["fs"]), _ptr(out["err"]), engine._stream_ptr()))
        return step

    def composed(sets, n, T, out):
        tau = torch.empty((7, n), **f64)
        ctrl = torch.full((n,), 1.0, **f64)

        def step(i):
            c, q, qd, mass = sets[i % N_SETS]
            cc = [(c[0, :, k] if c.dim() == 4 else c[0, :, k][:, None]) for k in range(6)]
            fs = torch.full((n,), T, dtype=torch.int32, device=dev)
            err = torch.zeros((n,), **f64)
            s = engine._stream_ptr()
            for k in range(T):
                u = k * DT
                x = cc[0] + u * (cc[1] + u * (cc[2] + u * (cc[3] + u * (cc[4] + u * cc[5]))))
                v = cc[1] + u * (2.0 * cc[2] + u * (3.0 * cc[3] + u * (4.0 * cc[4] + u * (5.0 * cc[5]))))
                a = 2.0 * cc[2] + u * (6.0 * cc[3] + u * (12.0 * cc[4] + u * (20.0 * cc[5])))
                acmd = (a + KP * (x - q)) + KD * (v - qd)
                _lib.check(lib.tcmp_rne_batch(RNE, 0, n, _ptr(q), _ptr(qd), _ptr(acmd), _ptr(ctrl), 0.0, 0.0,
                                              _ptr(tau), None, s))
                over = tau.abs() > L7
                fs = torch.where(over.any(0) & (fs == T), torch.full_like(fs, k), fs)
                t = torch.where(over, torch.copysign(L7.expand_as(tau), tau), tau)
                qn, vn = torch.empty_like(q), torch.empty_like(qd)
                _lib.check(lib.tcmp_rollout_batch(None, RNE, n, 1, DT, _ptr(q), _ptr(qd), _ptr(t), 0, _ptr(mass), 0.0,
                                                  None, None, None, _ptr(qn), _ptr(vn), None, None, None, s))
                q, qd = qn, vn
                un = (k + 1) * DT
                xn = cc[0] + un * (cc[1] + un * (cc[2] + un * (cc[3] + un * (cc[4] + un * cc[5]))))
                err = torch.maximum(err, (q - xn).abs().amax(0))
            out["q"].copy_(q)
            out["qd"].copy_(qd)
            out["fs"].copy_(fs)
            out["err"].copy_(err)
        return step

    class Graph:
        def __init__(self, fn, k):
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for i in range(2):
                    fn(i)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self.g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.g, stream=side):
                for i in range(k):
                    fn(i)

        def run(self):
            self.g.replay()

    def timed(graph, reps=1):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        graph.run()                  # untimed pre-roll: the timed replay is enqueued while it runs
        e0.record()
        for _ in range(reps):
            graph.run()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def measure(fn, units, steps):
        for i in range(args.warmup):
            fn(i)
        torch.cuda.synchronize()
        g = Graph(fn, steps)
        probe = timed(g)
        timed(g, max(1, int(args.hold_s / max(probe * 1e-3, 1e-6))))     # ~1 s hold: sustained clocks
        ms = timed(g)
        del g
        return units * steps / (ms * 1e-3), ms / steps

    sampler = bench.ClockSampler(0)
    sampler.start()
    card = card_info()
    fp64_peak = max(engine.fp64_peak(2048) for _ in range(3))
    results = {}
    for name, (n, T, _) in WORKLOADS.items():
        sets = make_sets(name, n)
        mk = lambda: {"q": torch.empty((7, n), **f64), "qd": torch.empty((7, n), **f64),
                      "fs": torch.empty((n,), dtype=torch.int32, device=dev), "err": torch.empty((n,), **f64)}
        out_k, out_c = mk(), mk()
        rate, ms = measure(k15(sets, n, T, out_k), n * T, args.steps)
        # the composition of the 1000-step workload is one graph of ~20 000 nodes a call: one call per graph
        crate, cms = measure(composed(sets, n, T, out_c), n * T, args.steps if T <= 64 else 1)
        k15(sets, n, T, out_k)(N_SETS - 1)
        composed(sets, n, T, out_c)(N_SETS - 1)
        torch.cuda.synchronize()
        diff = {k: float(((out_k[k] - out_c[k]).abs() / (1.0 + out_c[k].abs())).nan_to_num(0.0).max())
                for k in ("q", "qd", "err")}
        results[name] = {
            "rollouts": n, "n_steps": T, "dt": DT, "kp": KP, "kd": KD, "shared_reference": name == "montecarlo",
            "rollout_steps_per_s": rate, "ms_per_call": ms,
            "achieved_tflops": rate * flops["per_step"] / 1e12, "frac_fp64_peak": rate * flops["per_step"] / fp64_peak,
            "composed_rollout_steps_per_s": crate, "composed_ms_per_call": cms, "k15_speedup": rate / crate,
            "composed_cuda_graph": True, "max_rel_diff_vs_composed": diff,
            "first_saturation_mismatches": int((out_k["fs"] != out_c["fs"]).sum()),
            "saturating_rollouts": int((out_k["fs"] < T).sum()),
            "nonfinite_rollouts": int((~torch.isfinite(out_k["q"]).all(0)).sum()),
            "max_err_median": float(out_k["err"].nan_to_num(0.0).median())}
        del sets, out_k, out_c
        torch.cuda.empty_cache()
    clocks = sampler.stop()
    line = {"metric": "closed-loop tracking rollout-steps/s (tcmp_track_batch, computed torque + saturation + RK4, "
                      "Panda 7-DOF, rne, fp64)",
            "unit": "rollout-steps/s", "input_sets": N_SETS, "steps": args.steps, "warmup": args.warmup,
            "card": card, "clocks": clocks, "fp64_peak_tflops_measured": fp64_peak / 1e12,
            "flop_per_rollout_step": flops["per_step"], "flop_k14_step": flops["k14_step"],
            "flop_controller": flops["controller"], "flop_reference_and_error": flops["reference_and_error"],
            "flop_source": "instrumented host build of csrc/track_core.cuh (tests/native/track_host.cpp)",
            "workloads": results}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
