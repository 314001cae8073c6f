#!/usr/bin/env python
"""bench_dynamics.py -- joint-space dynamics terms (tcmp_dynamics_batch, K10) in states/s on one B200, against the
composition a user has without it: tcmp_rne_batch launches combined on the device.

    python bench_dynamics.py [--steps K] [--warmup W]

Workload: 1 M config-2 states (bench.sample_states: q, qd, payload mass in {0, 1, 3, 5} kg), fp64, SoA [7][n].
Inputs rotate over 4 distinct sets so no step finds them in the 126 MB L2.  Output sets: {g}, {M}, {M, g},
{M, C, g}, {J}, {all}.  Protocol as bench.py: W warm-up steps, ~1 s hold of the same step (sustained clocks), then K
steps captured in one CUDA graph and timed with CUDA events; nvidia-smi clocks sampled throughout; card name and
power limit read in the same run.

Composed baseline (same run, same inputs, outputs preallocated, inputs qd +- e_j prepared outside the timed region):
  {M, g}     8 tcmp_rne_batch launches, g = rne(q, 0, 0), M[:, j] = rne(q, 0, e_j) - g on the device;
  {M, C, g}  + 14 launches, C[:, j] = (rne(q, qd + e_j, 0) - rne(q, qd - e_j, 0)) / 4.

FLOP/state is the instrumented count of the algorithm (tests/native/dynamics_host.cpp: every FP64 add, mul = 1,
fma = 2 of csrc/dynamics_core.cuh, sincos included), compiled here into a temporary directory.  Bytes/state are the
compulsory HBM bytes: inputs read once, outputs written once.
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

N = bench.N_STATES
N_SETS = bench.N_SETS
SUBSETS = {"g": "g", "M": "M", "Mg": "Mg", "MCg": "MCg", "J": "J", "all": "MCgJ"}
OUT_BYTES = {"M": 392, "C": 392, "g": 56, "J": 336}


def op_counts():
    """(flops per subset, sincos flops per angle) from the instrumented host build."""
    tmp = tempfile.mkdtemp(prefix="tcmp_dyn_count_")
    so = os.path.join(tmp, "libdynamics_count.so")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                           "-Wno-unknown-pragmas", "-o", so, os.path.join(ROOT, "tests", "native", "dynamics_host.cpp")])
    L = ctypes.CDLL(so)
    L.host_dynamics_flops.restype = ctypes.c_int64
    L.host_sincos_flops.restype = ctypes.c_int64
    per_angle = int(L.host_sincos_flops())
    out = {}
    for name, terms in SUBSETS.items():
        rec = int(L.host_dynamics_flops(*(int(t in terms) for t in "MCgJ")))
        angles = 6 + ("J" in terms)     # joints 2..7 always; joint 1 only for J
        out[name] = rec + angles * per_angle
    return out, per_angle


def card_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20)
        name, plim, smax = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit_w": float(plim), "sm_max_mhz": float(smax)}
    except Exception as e:   # pragma: no cover
        return {"name": None, "power_limit_w": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--hold-s", type=float, default=1.0)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")

    import torch
    from torque_constrained_motion_planning_b200 import _lib, engine
    from torque_constrained_motion_planning_b200.engine import _ptr

    if not torch.cuda.is_available():
        raise SystemExit("bench_dynamics.py needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    flops, per_angle = op_counts()

    sets = []
    for s in range(N_SETS):
        q, qd, _, mass = bench.sample_states(N, seed=1000 + s)
        sets.append(tuple(torch.as_tensor(a, device=dev) for a in (q, qd, mass)))
    f64 = dict(dtype=torch.float64, device=dev)
    outs = {"M": torch.empty((7, 7, N), **f64), "C": torch.empty((7, 7, N), **f64), "g": torch.empty((7, N), **f64),
            "J": torch.empty((6, 7, N), **f64)}

    def k10(terms):
        def step(i):
            q, qd, mass = sets[i % N_SETS]
            o = [outs[t] if t in terms else None for t in "MCgJ"]
            _lib.check(lib.tcmp_dynamics_batch(None, N, _ptr(q), _ptr(qd), _ptr(mass), 0.0, *(_ptr(x) for x in o),
                                               engine._stream_ptr()))
        return step

    # composed baseline: preallocated unit accelerations / shifted velocities and torque buffers
    zero = torch.zeros((7, N), **f64)
    unit = []
    for j in range(7):
        e = torch.zeros((7, N), **f64)
        e[j] = 1.0
        unit.append(e)
    shifted = [[(qd + unit[j], qd - unit[j]) for j in range(7)] for _, qd, _ in sets]
    tau = [torch.empty((7, N), **f64) for _ in range(3)]
    RNE = _lib.MODE["rne"]

    def rne(q, qd, qdd, mass, out):
        _lib.check(lib.tcmp_rne_batch(RNE, 0, N, _ptr(q), _ptr(qd), _ptr(qdd), _ptr(mass), 0.0, 0.0, _ptr(out), None,
                                      engine._stream_ptr()))

    def composed(with_c):
        def step(i):
            q, qd, mass = sets[i % N_SETS]
            rne(q, None, None, mass, outs["g"])      # static call: no velocity rows read
            for j in range(7):
                rne(q, zero, unit[j], mass, tau[0])
                torch.sub(tau[0], outs["g"], out=outs["M"][:, j])
            if with_c:
                for j in range(7):
                    vp, vm = shifted[i % N_SETS][j]
                    rne(q, vp, zero, mass, tau[1])
                    rne(q, vm, zero, mass, tau[2])
                    torch.sub(tau[1], tau[2], out=outs["C"][:, j])
                    outs["C"][:, j].mul_(0.25)
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

    def measure(fn):
        for i in range(args.warmup):
            fn(i)
        torch.cuda.synchronize()
        g = Graph(fn, args.steps)
        probe = timed(g)
        timed(g, max(1, int(args.hold_s / max(probe * 1e-3, 1e-6))))     # ~1 s hold: sustained clocks
        ms = timed(g)
        return N * args.steps / (ms * 1e-3), ms

    sampler = bench.ClockSampler(0)
    sampler.start()
    card = card_info()
    fp64_peak = max(engine.fp64_peak(2048) for _ in range(3))
    peaks, peak_src = bench.measured_peaks()
    hbm = float(peaks.get("hbm_gbs", 6650.0)) * 1e9
    results = {}
    for name, terms in SUBSETS.items():
        rate, ms = measure(k10(terms))
        b = 56 + 8 + (56 if "C" in terms else 0) + sum(OUT_BYTES[t] for t in terms)
        f = flops[name]
        t_fp, t_mem = f / fp64_peak, b / hbm
        results[name] = {"states_per_s": rate, "ms_per_step": ms / args.steps, "flop_per_state": f,
                         "achieved_tflops": rate * f / 1e12, "frac_fp64_peak": rate * f / fp64_peak,
                         "bytes_per_state": b, "achieved_gbs": rate * b / 1e9, "frac_hbm": rate * b / hbm,
                         "bound": "fp64" if t_fp > t_mem else "hbm",
                         "frac_of_bound": rate * max(t_fp, t_mem)}
    baseline = {}
    for name, with_c in (("Mg", False), ("MCg", True)):
        rate, ms = measure(composed(with_c))
        baseline[name] = {"states_per_s": rate, "ms_per_step": ms / args.steps,
                          "launches_per_step": 8 + (14 if with_c else 0),
                          "k10_speedup": results[name]["states_per_s"] / rate}
    clocks = sampler.stop()
    line = {"metric": "joint-space dynamics terms states/s (tcmp_dynamics_batch, Panda 7-DOF, fp64)",
            "unit": "states/s", "states": N, "input_sets": N_SETS, "steps": args.steps, "warmup": args.warmup,
            "card": card, "clocks": clocks, "fp64_peak_tflops_measured": fp64_peak / 1e12,
            "hbm_peak_gbs": hbm / 1e9, "hbm_peak_source": peak_src, "sincos_flop_per_angle": per_angle,
            "flop_source": "instrumented host build of csrc/dynamics_core.cuh (tests/native/dynamics_host.cpp)",
            "subsets": results, "composed_rne_baseline": baseline}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
