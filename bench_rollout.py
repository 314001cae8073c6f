#!/usr/bin/env python
"""bench_rollout.py -- forward-dynamics rollouts (tcmp_rollout_batch, K14) in rollout-steps/s on one B200, against the
composition a user has without it: 4 T K13 launches, the RK4 updates as torch element-wise ops and the limit check.

    python bench_rollout.py [--steps K] [--warmup W]

Workloads (fp64, rne, SoA [7][n], held torque tau ~ U(-limit, +limit), payloads from bench.sample_states):
  throughput  1 M rollouts x 32 steps of 1 ms: final state and first_violation against the stock joint and velocity
              limits.
  planner     16 384 rollouts x 256 steps of 1 ms: final state, first_violation and the whole trajectory.
Inputs rotate over 4 distinct sets so no step finds them in the 126 MB L2 (the planner's trajectory output alone is
470 MB a step).  Protocol as bench_forward_dynamics.py: W warm-up steps, ~1 s hold of the same step (sustained
clocks), then K steps captured in one CUDA graph and timed with CUDA events; nvidia-smi clocks sampled throughout;
card name and power limit read in the same run.  The composition is graph-captured too, with the same inputs, and its
outputs are compared with K14's at the timed sizes.

FLOP per rollout-step is the instrumented count (tests/native/rollout_host.cpp, compiled here into a temporary
directory): 4 x K13's qdd count (M and its factor, h and the solve, sincos of joints 2..7) plus the RK4 combination.
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
DT = 1e-3
WORKLOADS = {"throughput": (bench.N_STATES, 32, False), "planner": (16384, 256, True)}


def op_counts():
    """FP64 operations per rollout-step from the instrumented host build."""
    tmp = tempfile.mkdtemp(prefix="tcmp_rollout_count_")
    so = os.path.join(tmp, "librollout_count.so")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                           "-Wno-unknown-pragmas", "-o", so, os.path.join(ROOT, "tests", "native", "rollout_host.cpp")])
    L = ctypes.CDLL(so)
    for f in ("host_fd_flops", "host_sincos_flops", "host_rollout_combination_flops"):
        getattr(L, f).restype = ctypes.c_int64
    qdd = int(L.host_fd_flops(0)) + int(L.host_fd_flops(1)) + 6 * int(L.host_sincos_flops())
    comb = int(L.host_rollout_combination_flops())
    return {"qdd": qdd, "rk4_combination": comb, "per_step": 4 * qdd + comb}


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
        raise SystemExit("bench_rollout.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    flops = op_counts()
    lo, hi, vmax = (np.ascontiguousarray(a) for a in (bench.Q_LO, bench.Q_HI, bench.V_LIM))
    f64 = dict(dtype=torch.float64, device=dev)
    RNE = _lib.MODE["rne"]

    def make_sets(n):
        sets = []
        lim = np.array(LIMIT)[:, None]
        for s in range(N_SETS):
            q, qd, _, mass = bench.sample_states(n, seed=1000 + s)
            tau = np.random.default_rng(2000 + s).uniform(-lim, lim, size=q.shape)
            sets.append(tuple(torch.as_tensor(a, device=dev) for a in (q, qd, tau, mass)))
        return sets

    def k14(sets, n, T, traj, out):
        def step(i):
            q, qd, tau, mass = sets[i % N_SETS]
            _lib.check(lib.tcmp_rollout_batch(None, RNE, n, T, DT, _ptr(q), _ptr(qd), _ptr(tau), 0, _ptr(mass), 0.0,
                                              lo.ctypes.data, hi.ctypes.data, vmax.ctypes.data, _ptr(out["q"]),
                                              _ptr(out["qd"]), _ptr(out["q_traj"]) if traj else None,
                                              _ptr(out["qd_traj"]) if traj else None, _ptr(out["fv"]),
                                              engine._stream_ptr()))
        return step

    lo_t, hi_t, vm_t = (torch.as_tensor(a, device=dev)[:, None] for a in (lo, hi, vmax))

    def composed(sets, n, T, traj, out):
        qdd = [torch.empty((7, n), **f64) for _ in range(4)]
        h2, h6 = 0.5 * DT, DT / 6.0

        def step(i):
            q, qd, tau, mass = sets[i % N_SETS]
            s = engine._stream_ptr()

            def f(k, a, b):
                _lib.check(lib.tcmp_forward_dynamics_batch(None, RNE, n, _ptr(a), _ptr(b), _ptr(tau), _ptr(mass), 0.0,
                                                           _ptr(qdd[k]), None, s))
                return qdd[k]
            fv = torch.full((n,), T, dtype=torch.int32, device=dev)
            for k in range(T):
                a1 = f(0, q, qd)
                q2, v2 = q + h2 * qd, qd + h2 * a1
                a2 = f(1, q2, v2)
                q3, v3 = q + h2 * v2, qd + h2 * a2
                a3 = f(2, q3, v3)
                q4, v4 = q + DT * v3, qd + DT * a3
                a4 = f(3, q4, v4)
                q, qd = q + h6 * (((qd + 2 * v2) + 2 * v3) + v4), qd + h6 * (((a1 + 2 * a2) + 2 * a3) + a4)
                if traj:
                    out["q_traj"][k].copy_(q)
                    out["qd_traj"][k].copy_(qd)
                ok = ((q >= lo_t) & (q <= hi_t) & (qd.abs() <= vm_t)).all(dim=0)
                fv = torch.where((fv == T) & ~ok, torch.full_like(fv, k), fv)
            out["q"].copy_(q)
            out["qd"].copy_(qd)
            out["fv"].copy_(fv)
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

    def measure(fn, units):
        for i in range(args.warmup):
            fn(i)
        torch.cuda.synchronize()
        g = Graph(fn, args.steps)
        probe = timed(g)
        timed(g, max(1, int(args.hold_s / max(probe * 1e-3, 1e-6))))     # ~1 s hold: sustained clocks
        ms = timed(g)
        del g
        return units * args.steps / (ms * 1e-3), ms / args.steps

    sampler = bench.ClockSampler(0)
    sampler.start()
    card = card_info()
    fp64_peak = max(engine.fp64_peak(2048) for _ in range(3))
    results = {}
    for name, (n, T, traj) in WORKLOADS.items():
        sets = make_sets(n)
        mk = lambda: {"q": torch.empty((7, n), **f64), "qd": torch.empty((7, n), **f64),
                      "q_traj": torch.empty((T, 7, n), **f64) if traj else None,
                      "qd_traj": torch.empty((T, 7, n), **f64) if traj else None,
                      "fv": torch.empty((n,), dtype=torch.int32, device=dev)}
        out_k, out_c = mk(), mk()
        rate, ms = measure(k14(sets, n, T, traj, out_k), n * T)
        crate, cms = measure(composed(sets, n, T, traj, out_c), n * T)
        # outputs of the last input set, both ways
        k14(sets, n, T, traj, out_k)(N_SETS - 1)
        composed(sets, n, T, traj, out_c)(N_SETS - 1)
        torch.cuda.synchronize()
        diff = {k: float(((out_k[k] - out_c[k]).abs() / (1.0 + out_c[k].abs())).max())
                for k in ("q", "qd", "q_traj", "qd_traj") if out_k[k] is not None}
        results[name] = {
            "rollouts": n, "n_steps": T, "dt": DT, "trajectory": traj,
            "rollout_steps_per_s": rate, "ms_per_call": ms,
            "achieved_tflops": rate * flops["per_step"] / 1e12, "frac_fp64_peak": rate * flops["per_step"] / fp64_peak,
            "composed_rollout_steps_per_s": crate, "composed_ms_per_call": cms, "k14_speedup": rate / crate,
            "composed_cuda_graph": True, "max_rel_diff_vs_composed": diff,
            "first_violation_mismatches": int((out_k["fv"] != out_c["fv"]).sum()),
            "first_violation_histogram_head": torch.bincount(out_k["fv"].long(), minlength=T + 1)[[0, 1, T]].tolist()}
        del sets, out_k, out_c
        torch.cuda.empty_cache()
    clocks = sampler.stop()
    line = {"metric": "forward-dynamics rollout-steps/s (tcmp_rollout_batch, RK4, Panda 7-DOF, rne, fp64)",
            "unit": "rollout-steps/s", "input_sets": N_SETS, "steps": args.steps, "warmup": args.warmup,
            "card": card, "clocks": clocks, "fp64_peak_tflops_measured": fp64_peak / 1e12,
            "flop_per_rollout_step": flops["per_step"], "flop_qdd": flops["qdd"],
            "flop_rk4_combination": flops["rk4_combination"],
            "flop_source": "instrumented host build of csrc/rollout_core.cuh (tests/native/rollout_host.cpp)",
            "workloads": results}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
