#!/usr/bin/env python
"""bench_forward_dynamics.py -- forward dynamics (tcmp_forward_dynamics_batch, K13) in states/s on one B200, against
the composition a user has without it: K10's M, K1's h and a batched Cholesky solve from torch.linalg.

    python bench_forward_dynamics.py [--steps K] [--warmup W]

Workload: 1 M config-2 states (bench.sample_states: q, qd, payload mass in {0, 1, 3, 5} kg) with torques
tau ~ U(-limit, +limit), fp64, SoA [7][n], rne mode.  Inputs rotate over 4 distinct sets so no step finds them in the
126 MB L2.  Output sets: {qdd} and {qdd, M^-1}.  Protocol as bench_dynamics.py: W warm-up steps, ~1 s hold of the same
step (sustained clocks), then K steps captured in one CUDA graph (launched eagerly if a torch.linalg call of the baseline
cannot be captured; the line says which) and timed with CUDA events; nvidia-smi clocks sampled
throughout; card name and power limit read in the same run.

Composed baseline (same run, same inputs, outputs preallocated):
  tcmp_dynamics_batch {M} + tcmp_rne_batch h = rne(q, qd, 0) (threshold 0) + torch.linalg.cholesky_ex on M viewed as
  [n][7][7] + torch.cholesky_solve of (tau - h).  Its qdd is compared with K13's at the timed size.

FLOP/state is the instrumented count of the algorithm (tests/native/fd_host.cpp: every FP64 add, mul, div = 1, fma = 2
of csrc/fd_core.cuh, sincos included), compiled here into a temporary directory.  Bytes/state are the compulsory HBM
bytes: q, qd, tau and the mass read once (232 B with qdd written), M^-1 written once (+392 B).
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

N = bench.N_STATES
N_SETS = bench.N_SETS
LIMIT = [87.0, 87.0, 87.0, 87.0, 12.0, 12.0, 12.0]


def op_counts():
    """{"qdd": flops, "qdd_minv": flops} per state from the instrumented host build, sincos of joints 2..7 included."""
    tmp = tempfile.mkdtemp(prefix="tcmp_fd_count_")
    so = os.path.join(tmp, "libfd_count.so")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                           "-Wno-unknown-pragmas", "-o", so, os.path.join(ROOT, "tests", "native", "fd_host.cpp")])
    L = ctypes.CDLL(so)
    L.host_fd_flops.restype = ctypes.c_int64
    L.host_sincos_flops.restype = ctypes.c_int64
    m, solve, inv = (int(L.host_fd_flops(i)) for i in range(3))
    base = m + 6 * int(L.host_sincos_flops())
    return {"qdd": base + solve, "qdd_minv": base + solve + inv}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--hold-s", type=float, default=1.0)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")

    import numpy as np
    import torch
    from torque_constrained_motion_planning_b200 import _lib, engine
    from torque_constrained_motion_planning_b200.engine import _ptr

    if not torch.cuda.is_available():
        raise SystemExit("bench_forward_dynamics.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    flops = op_counts()

    sets = []
    lim = np.array(LIMIT)[:, None]
    for s in range(N_SETS):
        q, qd, _, mass = bench.sample_states(N, seed=1000 + s)
        tau = np.random.default_rng(2000 + s).uniform(-lim, lim, size=q.shape)
        sets.append(tuple(torch.as_tensor(a, device=dev) for a in (q, qd, tau, mass)))
    f64 = dict(dtype=torch.float64, device=dev)
    qdd = torch.empty((7, N), **f64)
    minv = torch.empty((7, 7, N), **f64)
    RNE = _lib.MODE["rne"]

    def k13(want_minv):
        def step(i):
            q, qd, tau, mass = sets[i % N_SETS]
            _lib.check(lib.tcmp_forward_dynamics_batch(None, RNE, N, _ptr(q), _ptr(qd), _ptr(tau), _ptr(mass), 0.0,
                                                       _ptr(qdd), _ptr(minv) if want_minv else None,
                                                       engine._stream_ptr()))
        return step

    # composed baseline: preallocated M and h; torch allocates the right-hand side and its own workspaces
    M = torch.empty((7, 7, N), **f64)
    h = torch.empty((7, N), **f64)
    zero = torch.zeros((7, N), **f64)
    comp = {}

    def composed(i):
        q, qd, tau, mass = sets[i % N_SETS]
        _lib.check(lib.tcmp_dynamics_batch(None, N, _ptr(q), None, _ptr(mass), 0.0, _ptr(M), None, None, None,
                                           engine._stream_ptr()))
        _lib.check(lib.tcmp_rne_batch(RNE, 0, N, _ptr(q), _ptr(qd), _ptr(zero), _ptr(mass), 0.0, 0.0, _ptr(h), None,
                                      engine._stream_ptr()))
        Lc, _ = torch.linalg.cholesky_ex(M.permute(2, 0, 1))
        comp["qdd"] = torch.cholesky_solve((tau - h).T.unsqueeze(-1), Lc)

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

    class Eager:
        def __init__(self, fn, k):
            self.fn, self.k = fn, k

        def run(self):
            for i in range(self.k):
                self.fn(i)

    def measure(fn):
        for i in range(args.warmup):
            fn(i)
        torch.cuda.synchronize()
        try:
            g = Graph(fn, args.steps)
        except RuntimeError as e:    # a library call that cannot be captured: the same steps, launched eagerly
            torch.cuda.synchronize()
            print("graph capture failed (%s); timing eagerly" % str(e).splitlines()[0], file=sys.stderr)
            g = Eager(fn, args.steps)
        probe = timed(g)
        timed(g, max(1, int(args.hold_s / max(probe * 1e-3, 1e-6))))     # ~1 s hold: sustained clocks
        ms = timed(g)
        return N * args.steps / (ms * 1e-3), ms, isinstance(g, Graph)

    sampler = bench.ClockSampler(0)
    sampler.start()
    card = card_info()
    fp64_peak = max(engine.fp64_peak(2048) for _ in range(3))
    peaks, peak_src = bench.measured_peaks()
    hbm = float(peaks.get("hbm_gbs", 6650.0)) * 1e9
    results = {}
    for name, want_minv in (("qdd", False), ("qdd_minv", True)):
        rate, ms, _ = measure(k13(want_minv))
        b = 232 + (392 if want_minv else 0)
        f = flops[name]
        t_fp, t_mem = f / fp64_peak, b / hbm
        results[name] = {"states_per_s": rate, "ms_per_step": ms / args.steps, "flop_per_state": f,
                         "achieved_tflops": rate * f / 1e12, "frac_fp64_peak": rate * f / fp64_peak,
                         "bytes_per_state": b, "achieved_gbs": rate * b / 1e9, "frac_hbm": rate * b / hbm,
                         "bound": "fp64" if t_fp > t_mem else "hbm", "frac_of_bound": rate * max(t_fp, t_mem)}
    rate, ms, graphed = measure(composed)
    baseline = {"states_per_s": rate, "ms_per_step": ms / args.steps, "cuda_graph": graphed,
                "k13_qdd_speedup": results["qdd"]["states_per_s"] / rate}
    clocks = sampler.stop()

    # outputs at the timed size: K13's qdd against the composition's, on the last input set
    last = N_SETS - 1
    k13(False)(last)
    composed(last)
    torch.cuda.synchronize()
    ref = comp["qdd"].view(N, 7).T
    diff = (qdd - ref).abs()
    baseline["max_abs_diff_qdd"] = float(diff.max())
    baseline["max_rel_diff_qdd"] = float((diff / (1.0 + ref.abs())).max())

    line = {"metric": "forward dynamics states/s (tcmp_forward_dynamics_batch, Panda 7-DOF, rne, fp64)",
            "unit": "states/s", "states": N, "input_sets": N_SETS, "steps": args.steps, "warmup": args.warmup,
            "card": card, "clocks": clocks, "fp64_peak_tflops_measured": fp64_peak / 1e12,
            "hbm_peak_gbs": hbm / 1e9, "hbm_peak_source": peak_src,
            "flop_source": "instrumented host build of csrc/fd_core.cuh (tests/native/fd_host.cpp)",
            "outputs": results, "composed_k10_k1_cholesky_baseline": baseline}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
