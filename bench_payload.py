#!/usr/bin/env python
"""bench_payload.py -- payload-mass intervals (K11 tcmp_payload_interval_batch, K12 tcmp_edge_payload_interval) on one
B200, against what a user has without them: bisecting the mass with the torque test.

    python bench_payload.py [--steps K] [--warmup W]

Workloads (fp64, SoA [7][n]):
  K11  1 M config-2 states (bench.sample_states) per mode rne / nov / dyn, inputs rotating over 4 distinct sets so no
       step finds them in the 126 MB L2; measured in the same process, on the same states, as tcmp_rne_batch at one
       mass (5 kg, threshold 0.01, verdict only -- the call a bisection step makes).
  K12  100 k configs[3] edges (bench.sample_edges) x 64 min-jerk waypoints, rne, against tcmp_edge_feasibility on the
       same edges at 0 kg (no payload attached).  Some configs[3] edges fail at every mass, and K4 stops at an edge's
       first failing round, so the edges are the first 100 k of the configs[3] stream that K4 judges feasible at 0 kg:
       on them K4 visits every waypoint, as K12 does on every edge.
Bisection baseline: pinning max_payload to 1e-6 kg over [0, 64] kg takes ceil(log2(64 / 1e-6)) = 26 torque-test
launches per query, each at the measured rate of the torque kernel above.
Protocol as bench_dynamics.py: W warm-up steps, ~1 s hold of the same step (sustained clocks), then K steps captured
in one CUDA graph and timed with CUDA events; card name and power limit read in the same run.
FLOP/state is the instrumented count of the algorithm (tests/native/payload_host.cpp: every FP64 add, mul, div = 1,
fma = 2 of csrc/payload_core.cuh, plus six table sincos of tests/native/dynamics_host.cpp), compiled into a temporary
directory.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
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
N_EDGES = 100_000
W = 64
BISECT_STEPS = math.ceil(math.log2(64.0 / 1e-6))     # 26


def op_counts():
    """FLOP per state of K11 for (mode, dynamic) from the instrumented host builds, sincos included."""
    tmp = tempfile.mkdtemp(prefix="tcmp_payload_count_")
    libs = {}
    for name in ("payload_host", "dynamics_host"):
        so = os.path.join(tmp, "lib%s_count.so" % name)
        subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                               "-Wno-unknown-pragmas", "-o", so, os.path.join(ROOT, "tests", "native", name + ".cpp")])
        libs[name] = ctypes.CDLL(so)
    libs["payload_host"].host_payload_flops.restype = ctypes.c_int64
    libs["dynamics_host"].host_sincos_flops.restype = ctypes.c_int64
    per_angle = int(libs["dynamics_host"].host_sincos_flops())
    count = lambda mode, dyn: int(libs["payload_host"].host_payload_flops(mode, dyn)) + 6 * per_angle
    return {"rne": count(0, 1), "nov": count(1, 0), "dyn": count(2, 1)}


def feasible_edges(torch, lib, dev, ptr):
    """The first N_EDGES configs[3] edges (bench.sample_edges, seed 3 and up) that tcmp_edge_feasibility (rne, 0 kg,
    W waypoints) judges feasible -> (qa, qb [7][N_EDGES] on the device, number of edges drawn)."""
    from torque_constrained_motion_planning_b200 import _lib
    keep_a, keep_b, kept, drawn, seed = [], [], 0, 0, 3
    while kept < N_EDGES:
        a, b = (torch.as_tensor(x, device=dev) for x in bench.sample_edges(2 * N_EDGES, seed=seed))
        ff = torch.empty(a.shape[1], dtype=torch.int32, device=dev)
        _lib.check(lib.tcmp_edge_feasibility(0, 0, a.shape[1], W, ptr(a), ptr(b), 0.0, 0.01, 0, ptr(ff), None))
        sel = (ff == W).nonzero().flatten()
        keep_a.append(a[:, sel])
        keep_b.append(b[:, sel])
        kept += int(sel.numel())
        drawn += a.shape[1]
        seed += 1
    qa = torch.cat(keep_a, 1)[:, :N_EDGES].contiguous()
    qb = torch.cat(keep_b, 1)[:, :N_EDGES].contiguous()
    return qa, qb, drawn


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--hold-s", type=float, default=1.0)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")

    import torch
    from torque_constrained_motion_planning_b200 import _lib, engine
    from torque_constrained_motion_planning_b200.engine import _ptr

    if not torch.cuda.is_available():
        raise SystemExit("bench_payload.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    flops = op_counts()

    sets = []
    for s in range(N_SETS):
        q, qd, qdd, _ = bench.sample_states(N, seed=1000 + s)
        sets.append(tuple(torch.as_tensor(a, device=dev) for a in (q, qd, qdd)))
    f64 = dict(dtype=torch.float64, device=dev)
    lo, hi = torch.empty(N, **f64), torch.empty(N, **f64)
    ok, mask = torch.empty(N, dtype=torch.uint8, device=dev), torch.empty(N, dtype=torch.uint8, device=dev)
    qa, qb, drawn = feasible_edges(torch, lib, dev, _ptr)
    elo, ehi = torch.empty(N_EDGES, **f64), torch.empty(N_EDGES, **f64)
    eok, ff = torch.empty(N_EDGES, dtype=torch.uint8, device=dev), torch.empty(N_EDGES, dtype=torch.int32, device=dev)

    def k11(mode):
        m = _lib.MODE[mode]

        def step(i):
            q, qd, qdd = sets[i % N_SETS]
            _lib.check(lib.tcmp_payload_interval_batch(None, m, N, _ptr(q), _ptr(qd), _ptr(qdd), _ptr(lo), _ptr(hi),
                                                       _ptr(ok), engine._stream_ptr()))
        return step

    def k1(mode):
        m = _lib.MODE[mode]

        def step(i):
            q, qd, qdd = sets[i % N_SETS]
            _lib.check(lib.tcmp_rne_batch(m, 0, N, _ptr(q), _ptr(qd), _ptr(qdd), None, 5.0, 0.01, None, _ptr(mask),
                                          engine._stream_ptr()))
        return step

    def k12(i):
        _lib.check(lib.tcmp_edge_payload_interval(None, 0, N_EDGES, W, _ptr(qa), _ptr(qb), 0, _ptr(elo), _ptr(ehi),
                                                  _ptr(eok), engine._stream_ptr()))

    def k4(i):
        _lib.check(lib.tcmp_edge_feasibility(0, 0, N_EDGES, W, _ptr(qa), _ptr(qb), 0.0, 0.01, 0, _ptr(ff),
                                             engine._stream_ptr()))

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

    def timed(graph, reps=1):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        graph.g.replay()
        e0.record()
        for _ in range(reps):
            graph.g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def measure(fn, units):
        for i in range(args.warmup):
            fn(i)
        torch.cuda.synchronize()
        g = Graph(fn, args.steps)
        probe = timed(g)
        timed(g, max(1, int(args.hold_s / max(probe * 1e-3, 1e-6))))
        ms = timed(g)
        return units * args.steps / (ms * 1e-3), ms / args.steps

    sampler = bench.ClockSampler(0)
    sampler.start()
    card = card_info()
    fp64_peak = max(engine.fp64_peak(2048) for _ in range(3))
    states = {}
    for mode in ("rne", "nov", "dyn"):
        # alternate the two kernels twice so drift in clocks shows up in both
        r11, r1 = [], []
        for _ in range(2):
            r11.append(measure(k11(mode), N))
            r1.append(measure(k1(mode), N))
        rate11 = max(r for r, _ in r11)
        rate1 = max(r for r, _ in r1)
        states[mode] = {"k11_states_per_s": rate11, "k11_runs": [r for r, _ in r11],
                        "k1_one_mass_states_per_s": rate1, "k1_runs": [r for r, _ in r1],
                        "k11_over_k1": rate11 / rate1,
                        "bisection_states_per_s": rate1 / BISECT_STEPS,
                        "k11_over_bisection": rate11 / (rate1 / BISECT_STEPS),
                        "k11_flop_per_state": flops[mode],
                        "k11_achieved_tflops": rate11 * flops[mode] / 1e12,
                        "k11_frac_fp64_peak": rate11 * flops[mode] / fp64_peak}
    r12, r4 = [], []
    for _ in range(2):
        r12.append(measure(k12, N_EDGES))
        r4.append(measure(k4, N_EDGES))
    rate12, rate4 = max(r for r, _ in r12), max(r for r, _ in r4)
    edges = {"mode": "rne", "edges": N_EDGES, "waypoints": W, "k12_edges_per_s": rate12,
             "k12_runs": [r for r, _ in r12], "k4_feasible_edges_per_s": rate4, "k4_runs": [r for r, _ in r4],
             "k4_mass_kg": 0.0, "k4_all_feasible": bool((ff == W).all()),
             "edges_drawn_for_feasible_set": drawn, "k12_over_k4": rate12 / rate4,
             "bisection_edges_per_s": rate4 / BISECT_STEPS, "k12_over_bisection": rate12 / (rate4 / BISECT_STEPS)}
    clocks = sampler.stop()
    line = {"metric": "payload-mass intervals (tcmp_payload_interval_batch K11, tcmp_edge_payload_interval K12), fp64",
            "unit": "states/s, edges/s", "states": N, "input_sets": N_SETS, "steps": args.steps,
            "warmup": args.warmup, "card": card, "clocks": clocks, "fp64_peak_tflops_measured": fp64_peak / 1e12,
            "bisection_launches_per_query": BISECT_STEPS,
            "flop_source": "instrumented host build of csrc/payload_core.cuh (tests/native/payload_host.cpp)",
            "states_k11": states, "edges_k12": edges}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
