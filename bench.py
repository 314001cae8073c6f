#!/usr/bin/env python
"""bench.py -- torque-feasibility states/s (Panda 7-DOF RNE) on N B200s, with the roofline of the
dominant kernel, an end-to-end number through the host-buffer C-ABI call, and the CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): 1 M synthetic Panda states (q, qd, qdd, payload mass in
{0,1,3,5} kg) per GPU, fp64, structure-of-arrays [7][n].  A step = one `rne`-mode pass of the
torque test over the batch (tcmp_rne_batch: joint torques [7][n] + feasibility mask [n]); the `nov`
and `dyn` modes are timed the same way and reported under "modes".  Inputs rotate over 4 distinct
1 M-state sets (4 x 176 MB) so no step finds its inputs in the 126 MB L2.  For N > 1 the states shard
across ranks with no data-path collective (weak scaling: 1 M states per GPU); the per-step all-gather of
the 1 MB feasibility masks IS inside the timed region: fused into the kernel as NVLink peer stores with
device-side completion flags (tcmp_peer_signal / tcmp_peer_wait on a side stream, under the next step's kernel);
the timed region ends when the last step's masks are complete on every rank.

Timing (same at every N): W warm-up steps, then the step is held for ~1 s so every GPU is in its sustained
(power-capped) clock regime, then EXACTLY K steps -- captured once into one CUDA graph per rank, so the timed
region is K back-to-back kernels, not K Python launches -- between a barrier + synchronize on both sides,
CUDA events on the launching stream, max over ranks.

--dump-outputs DIR (N = 1) writes what the last timed step returned, so two builds can be compared output for
output on the same seeded inputs: DIR/tau.npy (float64 [7][1M] joint torques) and DIR/feasible.npy (the uint8
mask [1M] as float32), 60 MB in all.

--impl reference times the CPU implementation of the same path on the host cores: the reference's
rne.py is pure Python/NumPy and cannot travel to the GPU box, so this arm runs the C oracle port of
it (oracle/rne_oracle.c, validated <= 2e-13 N.m against rne.py) on all host threads, on the same
1 M-state workload per step, inputs generated once outside the timed loop.
"""
from __future__ import annotations

import argparse
import csv
import glob
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_STATES = 1_000_000
N_SETS = 4
FLOPS_PER_STATE = 1654.0       # BASELINE.md section 4 (rne, payload > 0)
BYTES_PER_STATE = 233.0        # 168 q/qd/qdd + 8 mass in; 56 tau + 1 mask out
METRIC = "torque-feasibility states/sec (Panda 7-DOF RNE)"
UNIT = "states/s"

Q_LO = np.array([-2.8973, -1.7628, -2.8973, -3.0718, -2.8973, -0.0175, -2.8973])
Q_HI = np.array([2.8973, 1.7628, 2.8973, -0.0698, 2.8973, 3.7525, 2.8973])
V_LIM = np.array([2.175, 2.175, 2.175, 2.175, 2.61, 2.61, 2.61])


def sample_states(n, seed):
    rng = np.random.default_rng(seed)
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
    qd = rng.uniform(-V_LIM[:, None], V_LIM[:, None], size=(7, n))
    qdd = rng.uniform(-10.0, 10.0, size=(7, n))
    mass = rng.choice(np.array([0.0, 1.0, 3.0, 5.0]), size=n)
    return q, qd, qdd, mass


def workload_config(n_gpus):
    return {
        "workload": "configs[1]: batched RNE sweep, 1M synthetic Panda states (q, qd, qdd, payload) per GPU, "
                    "fp64, mode rne (tau + mask); nov/dyn under 'modes'",
        "states_per_gpu": N_STATES,
        "layout": "SoA [7][n] fp64",
        "l2": "inputs rotate over %d distinct 1M-state sets (%d MB) > 126 MB L2; no explicit flush"
              % (N_SETS, N_SETS * 176),
        "sharding": "states sharded across %d rank(s), no data-path collective; the all-gather of the feasibility "
                    "masks is inside every timed step when N > 1: peer stores fused into the kernel "
                    "(tcmp_rne_batch_scatter), completion flags on a side stream (tcmp_peer_signal / tcmp_peer_wait), "
                    "checked against NCCL all_gather; --gather nccl = NCCL all_gather_into_tensor on a side stream" % n_gpus,
        "timing": "W warm-up steps, ~1 s hold of the same step (sustained clocks at every N), then K steps replayed "
                  "from one CUDA graph per rank between barrier + synchronize, CUDA events on the launching stream "
                  "(the start event sits behind one untimed pre-roll replay of the same steps), max over ranks",
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe's clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smmax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smmax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smmax) if smmax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "MEASURED_PEAKS.json"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md: 6.65 TB/s)"


_CPU_INPUTS = {}


def cpu_baseline_run(n_sample, reps, nthreads=0):
    """C oracle port of rne.py + the limit compare, OpenMP over states.  Inputs are generated once (cached) and the
    thread pool / pages are warmed OUTSIDE the timed region, which holds nothing but `reps` oracle passes.
    nthreads = 0 -> every core this process may run on (torchrun exports OMP_NUM_THREADS=1; ignore it)."""
    import oracle
    if nthreads == 0:
        nthreads = len(os.sched_getaffinity(0))
    if n_sample not in _CPU_INPUTS:
        _CPU_INPUTS[n_sample] = sample_states(n_sample, seed=2)
    q, qd, qdd, mass = _CPU_INPUTS[n_sample]
    for _ in range(2):      # thread pool, page tables and clocks warm, like the reference arm's warm-up steps
        oracle.torque_test_batch("rne", q, qd, qdd, mass, nthreads=nthreads)
    t0 = time.perf_counter()
    for _ in range(reps):
        oracle.torque_test_batch("rne", q, qd, qdd, mass, nthreads=nthreads)
    dt = time.perf_counter() - t0
    return n_sample * reps / dt, nthreads, dt


# What K1 EXECUTES per state on the FP64 pipe: 317 DFMA + 162 DMUL + 70 DADD + 7 DSETP thread instructions, from the
# source page of the committed ncu capture (profiles/r02/k1_executed_instruction_mix.txt).  Round 1 quoted 669, the
# STATIC count of the kernel text, which includes the never-taken libm sincos fallback.
FP64_INSTR_PER_STATE = 556.0
EXEC_FLOPS_PER_STATE = 2 * 317.0 + 162.0 + 70.0


def sample_edges(n, seed):
    """configs[3] distribution (SURVEY.md 8d): q_a uniform in the joint limits, q_b = clip(q_a + N(0, 0.5^2))."""
    rng = np.random.default_rng(seed)
    qa = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
    qb = np.clip(qa + rng.normal(0.0, 0.5, size=(7, n)), Q_LO[:, None], Q_HI[:, None])
    return qa, qb


def cpu_baseline_extras(nthreads=0):
    """CPU arms of the two other workloads, on bounded samples: the UNMODIFIED reference IKFast (oracle/_ref, compiled
    from the reference's own ikfast_panda_arm.cpp) on 40k poses x 25 free values of configs[2], and the C oracle's
    edge check on 4k edges x 64 waypoints of configs[3]; OpenMP over every host thread."""
    import oracle
    if nthreads == 0:
        nthreads = len(os.sched_getaffinity(0))
    out = {}
    if oracle.have_ref():
        rng = np.random.default_rng(3)
        n, n_free = 40_000, 25
        q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
        free = np.empty((n_free, n))
        free[0] = q[6]
        free[1:] = rng.uniform(-2.8973, 2.8973, size=(n_free - 1, n))
        trans, rot = oracle.ref_fk_batch(q)
        oracle.ref_ik_batch(rot, trans, free, nthreads=nthreads, want_sols=False)      # warm: threads, pages
        t0 = time.perf_counter()
        oracle.ref_ik_batch(rot, trans, free, nthreads=nthreads, want_sols=False)
        dt = time.perf_counter() - t0
        out["ik"] = {"value": n * n_free / dt, "unit": "solves/s", "cores": nthreads, "kind": "reference",
                     "sample": "40k poses x 25 free values (1M solves) of configs[2], ComputeIk of the unmodified "
                               "ikfast_panda_arm.cpp compiled as oracle/_ref, solution counts kept"}
    qa, qb = sample_edges(4_000, 4)
    oracle.edge_feasibility("rne", qa[:, :64], qb[:, :64], 64, 5.0, nthreads=nthreads)
    t0 = time.perf_counter()
    oracle.edge_feasibility("rne", qa, qb, 64, 5.0, nthreads=nthreads)
    dt = time.perf_counter() - t0
    out["edges"] = {"value": 4_000 / dt, "unit": "edges/s", "cores": nthreads, "kind": "port",
                    "sample": "4k edges x 64 min-jerk waypoints of configs[3], rne, 5 kg, C oracle"}
    return out


def python_port_rate(n=300):
    """States/s of ONE core running the NumPy restatement that keeps rne.py's per-call structure (np.block 6x6
    algebra, np.linalg.inv per link): what the reference's own torque test costs on this host."""
    from oracle import rne_numpy_port as P
    q, qd, qdd, mass = sample_states(n, seed=2)
    P.torque_test(q[:, 0], qd[:, 0], qdd[:, 0], mass[0])
    t0 = time.perf_counter()
    for i in range(n):
        P.torque_test(q[:, i], qd[:, i], qdd[:, i], mass[i])
    return n / (time.perf_counter() - t0)


def run_extras(engine, dev, K):
    """IK solves/s (config 3: 1M reachable poses x 25 free values) and RRT* edge checks/s (config 4: 100k edges
    x 64 min-jerk waypoints, rne, 5 kg), device-resident, CUDA-event timed."""
    import torch
    out = {}
    rng = np.random.default_rng(3)
    n, n_free = 1_000_000, 25
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
    free = np.empty((n_free, n))
    free[0] = q[6]
    free[1:] = rng.uniform(-2.8973, 2.8973, size=(n_free - 1, n))
    qd_, fd = torch.as_tensor(q, device=dev), torch.as_tensor(free, device=dev)

    def timeit(fn, reps):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / reps

    t_fk = timeit(lambda: engine.fk_batch(qd_), 5)
    trans, rot = engine.fk_batch(qd_)
    t_cnt = timeit(lambda: engine.ik_batch(rot, trans, fd, want_sols=False, want_status=False), 3)
    ns = 200_000   # with the [8][7] solution sets written (448 B/solve): 5M solves = 2.2 GB of output
    t_sol = timeit(lambda: engine.ik_batch(rot[:, :ns].contiguous(), trans[:, :ns].contiguous(),
                                           fd[:, :ns].contiguous(), want_status=False), 3)
    _, counts, _ = engine.ik_batch(rot, trans, fd, want_sols=False, want_status=False)
    hist = torch.bincount(counts.flatten().long(), minlength=9).tolist()
    out["ik"] = {"workload": "configs[2]: 1M reachable poses x 25 free-joint values", "solves": n * n_free,
                 "solves_per_s_counts_only": n * n_free / t_cnt, "solves_per_s_with_solutions": ns * n_free / t_sol,
                 "fk_poses_per_s": n / t_fk, "count_histogram": hist}
    E, W = 100_000, 64
    rng = np.random.default_rng(4)
    qa = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, E))
    qb = np.clip(qa + rng.normal(0.0, 0.5, size=(7, E)), Q_LO[:, None], Q_HI[:, None])
    a, b = torch.as_tensor(qa, device=dev), torch.as_tensor(qb, device=dev)
    t_e = timeit(lambda: engine.edge_feasibility(a, b, W, 5.0, mode="rne"), max(K, 5))
    ff = engine.edge_feasibility(a, b, W, 5.0, mode="rne")
    evaluated = int(torch.clamp(((ff + 32) // 32) * 32, max=W).sum().item())   # waypoints actually evaluated (32/round)
    out["edges"] = {"workload": "configs[3]: 100k edges x 64 min-jerk waypoints, rne, 5 kg", "edges_per_s": E / t_e,
                    "waypoint_states_per_s_nominal": E * W / t_e, "waypoint_states_evaluated": evaluated,
                    "feasible_fraction": float((ff == W).float().mean().item()), "ms": t_e * 1e3}
    return out


def run_reference(args):
    """CPU arm: the C oracle port of rne.py on every host thread, the SAME 1 M-state workload per step as the GPU arm,
    inputs generated once before the timed loop (round 1 timed its own NumPy input generation: VERDICT r01 weak #2)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    nthreads = len(os.sched_getaffinity(0))
    q, qd, qdd, mass = sample_states(N_STATES, seed=2)
    for _ in range(max(args.warmup, 1)):
        oracle.torque_test_batch("rne", q, qd, qdd, mass, nthreads=nthreads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle.torque_test_batch("rne", q, qd, qdd, mass, nthreads=nthreads)
    dt = time.perf_counter() - t0
    value = N_STATES * args.steps / dt
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nthreads, "kind": "port",
                         "sample": "%d passes over the full 1M-state workload (tau + mask), inputs pre-generated, C "
                                   "oracle port of rne.py with OpenMP" % args.steps,
                         "python_port_states_per_s_per_core": python_port_rate(),
                         "python_port_note": "oracle/rne_numpy_port.py: NumPy restatement at rne.py's own per-call "
                                             "granularity, 300 states on one core"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the newest committed `ncu --set full`
    capture (profiles/r*/ncu_full_rne_batch_kernel*_raw.csv: header row, unit row, one row per captured launch)."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*", "ncu_full_rne_batch_kernel*_raw.csv")),
                   key=lambda f: (os.path.basename(os.path.dirname(f)), os.path.getmtime(f)))
    for path in reversed(files):
        try:
            rows = list(csv.reader(open(path)))
            head, units = rows[0], rows[1]
            ir, iw, ik = head.index("dram__bytes_read.sum"), head.index("dram__bytes_write.sum"), head.index("Kernel Name")
            vals = [float(r[ir]) * unit[units[ir]] + float(r[iw]) * unit[units[iw]] for r in rows[2:]
                    if "rne_batch_kernel<double" in r[ik]]
            if vals:
                return float(np.mean(vals)), os.path.relpath(path, ROOT), len(vals)
        except Exception:
            continue
    return None, None, 0


def bind_rank_to_cores(local, world):
    """Per-rank CPU affinity BEFORE any pinned allocation (first-touch places the pages): the cores of the GPU's NUMA
    node when sysfs reports one, split evenly between the ranks that share it; else an even split of the allowed set."""
    allowed = sorted(os.sched_getaffinity(0))
    info = {"allowed": len(allowed), "numa_node": None}
    if world <= 1:
        return allowed, info
    cpus = allowed
    peers_on_node, my_slot = world, local
    try:
        import torch
        bus = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (bus.pci_domain_id, bus.pci_bus_id, bus.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        info["numa_node"] = node
        if node >= 0:
            txt = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
            node_cpus = []
            for part in txt.split(","):
                lo, _, hi = part.partition("-")
                node_cpus += list(range(int(lo), int(hi or lo) + 1))
            node_cpus = [c for c in node_cpus if c in allowed]
            if len(node_cpus) >= world:
                cpus = node_cpus
    except Exception:
        pass
    per = max(1, len(cpus) // peers_on_node)
    mine = cpus[my_slot * per:(my_slot + 1) * per] or cpus
    try:
        os.sched_setaffinity(0, mine)
    except Exception:
        mine = allowed
    info["cores"] = len(mine)
    return allowed, info


def planner_extras():
    """End-to-end planner_fn_force_aware wall time on BASELINE.json configs[0] / configs[4] (the synthetic-scene stand-ins
    of collision.py), next to the MEASURED reference loop: profiles/r02/reference_planner_cpu.json is the reference's
    own rrt_star_force_aware + rne.rne + min_jerk_v2 + IKFast with the Python collision twin, run once in the CPU
    container by scripts/reference_planner_cpu.py with the same seed, scene, start and target."""
    import random
    import torch
    from torque_constrained_motion_planning_b200 import collision, ikfast_panda_arm as ik, ik_utils
    from torque_constrained_motion_planning_b200 import panda_primitives as pp, utils
    q_home = [0, -math.pi / 4, 0.0, -3 * math.pi / 4, 0, math.pi / 2, math.pi / 4]
    goal_q = [0.7, 0.3, 0.2, -1.9, 0.1, 2.2, 1.0]
    try:
        ref = {r["scene"]: r for r in json.load(open(os.path.join(ROOT, "profiles", "r02",
                                                                  "reference_planner_cpu.json")))["results"]}
    except Exception:
        ref = {}
    pos8, rot8 = ik.get_fk(goal_q)
    c, s_ = math.cos(-math.pi / 4), math.sin(-math.pi / 4)
    Rt = np.array(rot8) @ np.array([[c, -s_, 0], [s_, c, 0], [0, 0, 1.0]])
    pose = (tuple(np.array(pos8) + Rt @ np.array([0, 0, 0.105])), tuple(ik_utils.quat_from_matrix(Rt)))
    out = []
    for name, scene, mass in [("configs[0]: demo scene, rne, 1 kg, T=5 s", collision.hiro_scene(), 1.0),
                              ("configs[4]: cluttered scene, rne, 5 kg, T=5 s", collision.cluttered_scene(), 5.0)]:
        problem = lambda: utils.Problem(robot=None, fixed=scene, payload="coke", payload_mass=mass, execution_time=5,
                                        torque_test="rne")

        def timed(fn, reps=3):
            best, res = None, None
            for _ in range(reps):
                random.seed(3)
                np.random.seed(3)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = fn()
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            return best, res

        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):      # the planner prints like the reference does
            pp.planner_fn_force_aware(tuple(q_home), pose, problem())         # warm-up
            t_strict, traj = timed(lambda: pp.planner_fn_force_aware(tuple(q_home), pose, problem()))
            t_batched, traj_b = timed(lambda: pp.planner_fn_force_aware(tuple(q_home), pose, problem(), batch=32))
            t_arrays, _ = timed(lambda: pp.planner_fn_force_aware(tuple(q_home), pose, problem(), batch=32,
                                                                  as_arrays=True))
        r = ref.get(name)
        same = None
        if r is not None and traj is not None:
            qs = np.array([c_.values for c_ in traj.path])
            want = np.array(r["sample_q_every_200"])
            same = bool(len(qs) == r["samples"] and qs[::200].shape == want.shape and
                        np.abs(qs[::200] - want).max() < 1e-9)
        out.append({
            "scene": name, "samples": None if traj is None else len(traj.path),
            "gpu_strict_s": t_strict, "gpu_batched_s": t_batched, "gpu_batched_arrays_s": t_arrays,
            "gpu_batched_samples": None if traj_b is None else len(traj_b.path),
            "reference_measured_s": None if r is None else r["reference_measured_s"],
            "reference_rne_calls": None if r is None else r["rne_calls"],
            "reference_source": "profiles/r02/reference_planner_cpu.json (scripts/reference_planner_cpu.py: reference "
                                "rrt_star_force_aware + rne.rne + min_jerk_v2 + IKFast, NumPy collision twin, 1 core of "
                                "the CPU container; not re-run on the GPU box, /root/reference does not travel)",
            "gpu_strict_trajectory_equals_reference": same,
            "speedup_strict_vs_reference": None if r is None else r["reference_measured_s"] / t_strict,
            "speedup_batched_vs_reference": None if r is None else r["reference_measured_s"] / t_batched,
        })
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the IK / edge / planner workloads (N = 1 extras)")
    ap.add_argument("--eager", action="store_true", help="time K Python launches instead of one captured CUDA graph")
    ap.add_argument("--settle-s", type=float, default=1.0,
                    help="seconds the step is held before the timed region (same sustained clock regime at every N)")
    ap.add_argument("--multicast", action="store_true",
                    help="p2p gather through NVSwitch multicast stores (tcmp_rne_batch_scatter_mc, torch symmetric memory) "
                         "instead of unicast peer stores; measured within 1 %% of each other at N = 8")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: how the feasibility masks are all-gathered each step: p2p = peer stores fused into the "
                         "torque kernel (tcmp_rne_batch_scatter) + completion flags (tcmp_peer_signal / tcmp_peer_wait) on "
                         "a side stream; nccl = all_gather_into_tensor on a side stream")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs as DIR/tau.npy and DIR/feasible.npy (N = 1 only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the GPU path, not --impl reference")
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from torque_constrained_motion_planning_b200 import engine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback")
    all_cores, affinity = bind_rank_to_cores(local, world)
    torch.cuda.set_device(local)
    if world > 1 and args.dump_outputs:
        raise SystemExit("--dump-outputs needs a single-GPU run")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    W = max(args.warmup, 3)
    K = args.steps

    # ---- synthetic inputs, resident in HBM before the timed region -------------------------------
    sets = []
    for s in range(N_SETS):
        q, qd, qdd, mass = sample_states(N_STATES, seed=2 + 1000 * rank + s)
        sets.append(tuple(torch.as_tensor(a, device=dev) for a in (q, qd, qdd, mass)))
    host0 = sample_states(N_STATES, seed=2 + 1000 * rank)
    from torque_constrained_motion_planning_b200.distributed import OverlappedGather, PeerMaskBuffer
    gather = None
    peer = None
    if world > 1 and args.gather == "nccl":
        gather = OverlappedGather((N_STATES,), torch.uint8, dev)
    elif world > 1:
        try:
            # gathered [3][world][N_STATES] mask buffer, written by every rank's kernel
            peer = PeerMaskBuffer(N_STATES, multicast=args.multicast)
            ok_flag = torch.ones(1, device=dev)
        except Exception as e:                # CUDA IPC unavailable in this container: every rank must agree
            print("rank %d: peer-store gather unavailable (%s)" % (rank, e), file=sys.stderr)
            ok_flag = torch.zeros(1, device=dev)
        dist.all_reduce(ok_flag, op=dist.ReduceOp.MIN)
        if ok_flag.item() < 1:
            if peer is not None:
                peer.close()
            peer = None
            args.gather = "nccl (p2p unavailable)"
            gather = OverlappedGather((N_STATES,), torch.uint8, dev)

    # outputs are preallocated once: a step is the kernel, not the caching allocator
    out_tau = torch.empty((7, N_STATES), dtype=torch.float64, device=dev)
    out_mask = torch.empty((N_STATES,), dtype=torch.uint8, device=dev)

    def step(i, mode="rne"):
        q, qd, qdd, mass = sets[i % N_SETS]
        if peer is not None:
            # fused compute + all-gather: the kernel stores each mask byte into every rank's gathered buffer; a side
            # stream publishes the step's completion to every rank and waits for every rank's (tcmp_peer_signal /
            # tcmp_peer_wait) under the next step's kernel, like the NCCL path overlaps its collective; the timed
            # region ends (Runner.run -> peer.join) when the last step's gather is complete on this rank
            return peer.torque_test(q, qd, qdd, mass, mode=mode, out_tau=out_tau, overlap_gather=True), None
        tau, ok = engine.torque_test_batch(q, qd, qdd, mass, mode=mode, out_tau=out_tau, out_mask=out_mask)
        if gather is not None:
            gather.submit(ok)      # NCCL all-gather of this step's mask on a side stream (overlaps step i+1)
        return tau, ok

    def kernel_only(i):
        engine.torque_test_batch(*sets[i % N_SETS], mode="rne", out_tau=out_tau, out_mask=out_mask)

    use_graph = not args.eager and gather is None     # NCCL on a side stream is left to eager launches

    class Runner:
        """k calls of fn(i), i = 0..k-1: captured once into a CUDA graph (one launch = k back-to-back kernels, no
        Python or launch jitter inside the timed region) or, with --eager / NCCL, issued one by one."""

        def __init__(self, fn, k):
            self.fn, self.k, self.graph = fn, k, None
            if use_graph:
                try:
                    side = torch.cuda.Stream(device=dev)
                    side.wait_stream(torch.cuda.current_stream())
                    with torch.cuda.stream(side):
                        for i in range(2):
                            fn(i)
                    torch.cuda.current_stream().wait_stream(side)
                    torch.cuda.synchronize()
                    if peer is not None:
                        peer.reset()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=side):
                        for i in range(k):
                            fn(i)
                        if peer is not None:
                            peer.join()
                    if peer is not None:
                        peer.reset()
                    self.graph = g
                except Exception as e:      # pragma: no cover -- reported in the JSON line as launch = "eager"
                    print("rank %d: CUDA graph capture failed (%s); timing eager launches" % (rank, e), file=sys.stderr)
                    torch.cuda.synchronize()
                    self.graph = None

        def run(self):
            if self.graph is not None:
                self.graph.replay()
            else:
                for i in range(self.k):
                    self.fn(i)
                if peer is not None:
                    peer.join()

    def gate(runner):
        """Untimed pre-roll enqueued AFTER the barrier + synchronize and BEFORE the start event: one more replay of the
        same K steps.  The host enqueues the timed replay while it runs, so the first timed launch pays no launch
        latency, and (N > 1) the completion flags inside the steps have pulled the ranks into lock-step -- the start
        events of the ranks then differ by an NVLink round trip, not by a host barrier's exit skew (tens of us, several
        per cent of a 1 ms region)."""
        runner.run()

    def timed(runner, reps=1):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gate(runner)
        e0.record()
        for _ in range(reps):
            runner.run()
        if gather is not None:
            gather.join()          # the timed region ends when the last mask all-gather has landed
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def hold(runner, seconds):
        """Run `runner` back to back for about `seconds` (device-timed); the repetition count is agreed between the
        ranks (with completion flags in the step no rank may run more steps than another).  Returns (reps, ms)."""
        probe = timed(runner)                              # max over ranks: identical everywhere
        reps = max(1, int(seconds / max(probe * 1e-3, 1e-6)))
        return reps, timed(runner, reps)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()              # covers warm-up, the timed region and the sustained hold below
    for i in range(W):               # the contract's W warm-up steps
        step(i)
    torch.cuda.synchronize()
    main_run = Runner(step, K)
    hold200 = Runner(step, 200)
    kern200 = Runner(kernel_only, 200)
    # same clock regime at every N: the timed K steps follow ~settle_s of the same step, so they run at the
    # sustained (power-capped) clocks whatever N is, not at the boost clocks of a cold 1 ms burst
    timed(main_run)                  # first replay of a graph uploads it (~0.1 ms): not part of a step
    settle_reps, _ = hold(hold200, args.settle_s)
    ms_total = timed(main_run)       # the contract's number: exactly K timed steps
    # the outputs of timed step K - 1, copied before the runs below overwrite the buffers
    dumped = (out_tau.clone(), out_mask.clone()) if args.dump_outputs else None
    # sustained rate over >= 1.5 s, and the kernel alone (no gather epilogue, no wait) over the same >= 200 launches
    # at every N for the roofline of the dominant kernel
    sus_reps, sus_ms = hold(hold200, 1.5)
    sustained = world * N_STATES * 200 * sus_reps / (sus_ms * 1e-3)
    k_reps, k_ms = hold(kern200, 0.5)
    kernel_s = k_ms * 1e-3 / (200 * k_reps)
    clocks = sampler.stop() if rank == 0 else None
    value = world * N_STATES * K / (ms_total * 1e-3)

    modes = {}
    for mode in ("nov", "dyn"):
        r = Runner(lambda i, m=mode: step(i, m), K)
        timed(r)
        modes[mode] = world * N_STATES * K / (timed(r) * 1e-3)
    modes["rne"] = value
    if world == 1:   # the optional fp32 path (1e-4 relative), same launch geometry
        f32 = [tuple(t.float() for t in s_) for s_ in sets[:2]]
        for i in range(3):
            engine.torque_test_batch(*f32[i % 2], mode="rne", dtype="f32")
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            engine.torque_test_batch(*f32[i % 2], mode="rne", dtype="f32")
        e1.record()
        torch.cuda.synchronize()
        modes["rne_f32"] = N_STATES * K / (e0.elapsed_time(e1) * 1e-3)
        del f32
    # mask-only rne (the planner's actual need: 177 B/state)
    r = Runner(lambda i: engine.torque_test_batch(*sets[i % N_SETS], mode="rne", want_tau=False, out_mask=out_mask), K)
    timed(r)
    modes["rne_mask_only"] = world * N_STATES * K / (timed(r) * 1e-3)
    gather_check = None
    if peer is not None:
        # correctness of the fused gather + completion flags: after step + wait, WITHOUT any host barrier, this rank
        # must hold every rank's mask of that step
        last = (K - 1) % N_SETS
        torch.cuda.synchronize()
        peer.reset()
        step(last)
        with torch.cuda.stream(peer.side):    # enqueued behind this step's wait kernel: no host barrier in between
            got = peer.gathered.clone()
        peer.join()
        mine = engine.torque_test_batch(*sets[last], mode="rne", want_tau=False)[1]
        refm = torch.empty((world, N_STATES), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(refm, mine)
        assert torch.equal(refm, got), "peer-store gather != NCCL all-gather"
        peer.check()              # no tcmp_peer_wait of this run gave up on a rank
        gather_check = "peer-store gather + device-side wait == NCCL all_gather_into_tensor"

    # ---- the other hot-path workloads (BASELINE.json configs[0], [2], [3], [4]); single-GPU runs only -------
    extras = {}
    if world == 1 and not args.no_extras:
        extras = run_extras(engine, dev, K)
        try:
            extras["planner"] = planner_extras()
        except Exception as e:      # pragma: no cover
            extras["planner"] = {"error": repr(e)}

    # ---- end to end through the host-buffer C-ABI call (pinned host arrays, H2D + D2H inside) -------
    pin = lambda a: torch.as_tensor(np.ascontiguousarray(a)).pin_memory()
    hq, hqd, hqdd, hm = (pin(a) for a in host0)
    htau = torch.empty((7, N_STATES), dtype=torch.float64).pin_memory()
    hok = torch.empty((N_STATES,), dtype=torch.uint8).pin_memory()
    ws = engine.Workspace()
    nq, nqd, nqdd, nm, ntau, nok = (t.numpy() for t in (hq, hqd, hqdd, hm, htau, hok))

    def e2e_step(_i=0):
        engine.torque_test_batch_host_into(ws, "rne", "f64", nq, nqd, nqdd, nm, 0.0, 0.01, ntau, nok)

    def timed_host(fn, reps):
        """Wall clock around `reps` host calls, every rank starting together, max over ranks."""
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t_ = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t_) / reps
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt

    e2e_s = timed_host(e2e_step, K)
    e2e_value = world * N_STATES / e2e_s

    # the same K batches through the asynchronous form of the call (tcmp_rne_batch_host_async + one
    # tcmp_workspace_sync): batch i + 1's host->device copies run under batch i's last chunk and read-back, which is how
    # a caller streaming batches would use the library; every batch's 176 MB in / 57 MB out still moves inside the region
    def e2e_pipelined():
        for _ in range(K):
            engine.torque_test_batch_host_async(ws, "rne", "f64", nq, nqd, nqdd, nm, 0.0, 0.01, ntau, nok)
        engine.workspace_sync(ws)
    e2e_pipe_s = timed_host(e2e_pipelined, 1) / K

    # sanity: the host path and the device path agree bit for bit on the same inputs
    tau_d, ok_d = engine.torque_test_batch(*sets[0], mode="rne")
    assert torch.equal(tau_d.cpu(), htau) and torch.equal(ok_d.cpu(), hok)

    # what bounds it: the same byte volumes as the call (176 MB host->device, 57 MB device->host) moved by plain pinned
    # cudaMemcpyAsync on two streams, EVERY RANK AT ONCE (barriered) -- the concurrent ceiling of this box's host
    # links at this N -- and the call without the torque read-back (the planner's predicate needs the mask only)
    mask_only_s = timed_host(lambda: engine.torque_test_batch_host_into(ws, "rne", "f64", nq, nqd, nqdd, nm, 0.0, 0.01,
                                                                       None, nok), max(3, K // 2))
    d_in = [torch.empty((7, N_STATES), dtype=torch.float64, device=dev) for _ in range(3)]
    d_m = torch.empty((N_STATES,), dtype=torch.float64, device=dev)
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def plain_both():
        with torch.cuda.stream(s_in):
            for d_, h_ in zip(d_in, (hq, hqd, hqdd)):
                d_.copy_(h_, non_blocking=True)
            d_m.copy_(hm, non_blocking=True)
        with torch.cuda.stream(s_out):
            htau.copy_(d_in[0], non_blocking=True)
            hok.copy_(out_mask, non_blocking=True)

    def plain_h2d():
        with torch.cuda.stream(s_in):
            for d_, h_ in zip(d_in, (hq, hqd, hqdd)):
                d_.copy_(h_, non_blocking=True)
            d_m.copy_(hm, non_blocking=True)

    def plain_d2h():
        with torch.cuda.stream(s_out):
            htau.copy_(d_in[0], non_blocking=True)
            hok.copy_(out_mask, non_blocking=True)

    def plain_sequential():       # the same bytes, one direction at a time (what wins on a half-duplex-like host link)
        with torch.cuda.stream(s_in):
            for d_, h_ in zip(d_in, (hq, hqd, hqdd)):
                d_.copy_(h_, non_blocking=True)
            d_m.copy_(hm, non_blocking=True)
            htau.copy_(d_in[0], non_blocking=True)
            hok.copy_(out_mask, non_blocking=True)

    both_s = timed_host(plain_both, 10)
    seq_s = timed_host(plain_sequential, 10)
    h2d_s = timed_host(plain_h2d, 10)
    d2h_s = timed_host(plain_d2h, 10)
    ceiling_s = min(both_s, seq_s)
    link = {"h2d_gbs_in_call": N_STATES * 176 / e2e_s / 1e9,
            "h2d_gbs_in_call_mask_only": N_STATES * 176 / mask_only_s / 1e9,
            "ms_in_call": e2e_s * 1e3,
            "ms_plain_overlapped": both_s * 1e3, "ms_plain_sequential": seq_s * 1e3,
            "h2d_gbs_plain_h2d_only": N_STATES * 176 / h2d_s / 1e9,
            "d2h_gbs_plain_d2h_only": N_STATES * 57 / d2h_s / 1e9,
            "ceiling": "overlapped" if both_s <= seq_s else "sequential",
            "in_call_share_of_ceiling": ceiling_s / e2e_s,
            "mask_only_states_per_s": world * N_STATES / mask_only_s,
            "affinity": affinity,
            "note": "per rank, slowest rank, ALL RANKS COPYING AT ONCE (barriered).  Ceiling = the faster of two plain "
                    "pinned cudaMemcpyAsync schedules moving the call's own bytes (176 MB in, 57 MB out): both "
                    "directions overlapped on two streams, or one after the other.  The GPU boxes of this pool are "
                    "KVM guests with one virtual NUMA node (no NUMA placement possible from inside); their host "
                    "link is full duplex for one or two GPUs (overlapped wins) and behaves like a shared half-duplex "
                    "pipe of ~190 GB/s aggregate at 8 (sequential wins): the end-to-end number is bounded by it."}
    if world > 1:
        try:
            os.sched_setaffinity(0, all_cores)      # the CPU baseline leg uses every host thread again
        except Exception:
            pass

    if rank == 0:
        peaks, peak_src = measured_peaks()
        fp64_peak = max(engine.fp64_peak(2048) for _ in range(3))
        # the same DFMA loop held for ~1 s: what the pipe sustains at this box's power cap (pure DFMA draws the most)
        t_end = time.perf_counter() + 1.0
        sus_peak = []
        while time.perf_counter() < t_end:
            sus_peak.append(engine.fp64_peak(2048))
        fp64_peak_sustained = float(np.median(sus_peak[len(sus_peak) // 2:]))
        achieved_tf = FLOPS_PER_STATE * N_STATES / kernel_s / 1e12
        achieved_gbs = BYTES_PER_STATE * N_STATES / kernel_s / 1e9
        traffic, traffic_src, traffic_n = ncu_traffic()
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(world),
            "launch": ("one CUDA graph of K steps per rank" if main_run.graph is not None else "K eager launches"),
            "settle": {"seconds": args.settle_s, "steps": 200 * settle_reps,
                       "note": "the same step held before the timed region at every N: the timed steps run in the "
                               "sustained (power-capped) clock regime"},
            "roofline": {
                "bound": "fp64", "achieved": achieved_tf, "peak": fp64_peak / 1e12, "unit": "TFLOP/s",
                "frac": achieved_tf / (fp64_peak / 1e12),
                "peak_sustained": fp64_peak_sustained / 1e12,
                "frac_of_sustained_peak": achieved_tf / (fp64_peak_sustained / 1e12),
                # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel at this size, read from the
                # committed ncu --set full capture (<= 233 MB algorithmic: the dirty output lines still in the 126 MB
                # L2 at kernel end are not counted by the DRAM counters)
                "traffic": traffic, "traffic_source": traffic_src, "traffic_launches_averaged": traffic_n,
                "peak_source": "tcmp_fp64_peak DFMA microbenchmark measured in this run (MEASURED_PEAKS.json "
                               "carries no FP64 entry; datasheet 37.2 TFLOP/s)",
                "flops_per_state": FLOPS_PER_STATE, "kernel": "rne_batch_kernel<double,DYN,!TOOL,tau,mask>",
                # what the kernel EXECUTES per state (static SASS count of the loop body, scripts/sass_mix.sh);
                # pipe_frac = FP64 instructions issued / the DFMA rate behind `peak`
                "note": "achieved / frac use SURVEY 8d's ALGORITHMIC 1654 FLOP per state; the kernel executes fewer "
                        "(customised recursion, regrouped parameters, table-driven sincos), so frac can reach 1 "
                        "while the FP64 pipe is at executed.pipe_frac; kernel_ms is the sustained-clock figure",
                "executed": {"fp64_instr_per_state": FP64_INSTR_PER_STATE, "flops_per_state": EXEC_FLOPS_PER_STATE,
                             "achieved": EXEC_FLOPS_PER_STATE * N_STATES / kernel_s / 1e12,
                             "pipe_frac": FP64_INSTR_PER_STATE * N_STATES / kernel_s / (fp64_peak / 2.0)},
                "kernel_ms": kernel_s * 1e3, "kernel_launches_averaged": 200 * k_reps,
                "hbm": {"achieved": achieved_gbs, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                        "frac": achieved_gbs / peaks.get("hbm_gbs"), "bytes_per_state": BYTES_PER_STATE,
                        "peak_source": peak_src},
            },
            "modes": modes,
            "gather": "none (N = 1)" if world == 1 else
                      (("p2p/NVLS: NVSwitch multicast stores (multimem.st) fused into the torque kernel"
                        if peer.mc_ptr else "p2p: peer stores fused into the torque kernel") +
                       "; tcmp_peer_signal + tcmp_peer_wait per step on a side stream, joined inside the timed region"
                       if peer is not None else args.gather),
            "gather_check": gather_check,
            "extras": extras,
            "sustained": {"value": sustained, "unit": UNIT, "steps": 200 * sus_reps, "ms_per_step": sus_ms / (200 * sus_reps),
                          "note": "same step (gather and wait included) held back to back for >= 1.5 s, device-timed, "
                                  "max over ranks; clocks sampled over it"},
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": int(N_STATES * 176), "d2h_bytes_per_step": int(N_STATES * 57),
                    "api": "tcmp_rne_batch_host (pinned host SoA arrays, 3-stage chunked H2D/kernel/D2H pipeline), one "
                           "synchronous call per step",
                    "pipelined": {"value": world * N_STATES / e2e_pipe_s, "unit": UNIT,
                                  "api": "tcmp_rne_batch_host_async x K + tcmp_workspace_sync: the K batches pipeline "
                                         "across calls; same bytes per step"},
                    "link": link},
            "gpu_launches": K * (3 if peer is not None else 1),
            "clocks": clocks,
        }
        if not args.no_cpu_baseline:
            v, cores, dt = cpu_baseline_run(N_STATES, 10)
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                   "sample": "10 passes over the same 1M-state workload after 2 warm passes (%.1f s "
                                             "wall), C oracle port of rne.py with OpenMP, inputs pre-generated" % dt,
                                   "python_port_states_per_s_per_core": python_port_rate(),
                                   "python_port_note": "oracle/rne_numpy_port.py: NumPy restatement at rne.py's own "
                                                       "per-call granularity (np.block / np.linalg.inv per link), "
                                                       "300 states on one core"}
            if world == 1 and not args.no_extras:
                out["cpu_baseline"]["other_workloads"] = cpu_baseline_extras()
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "tau.npy"), dumped[0].cpu().numpy())
            np.save(os.path.join(args.dump_outputs, "feasible.npy"), dumped[1].cpu().numpy().astype(np.float32))
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
