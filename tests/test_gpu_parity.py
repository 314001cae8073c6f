"""GPU parity tests proper: the CUDA path, called through the C-ABI (libtcmp.so), against
(a) golden vectors produced by the unmodified reference and (b) the C oracle on seeded inputs.

Tolerances (BASELINE.json north_star): torques <= 1e-9 N.m on the fp64 path, 1e-4 relative on the
fp32 path; feasibility masks, first-failure indices and IK solution counts bit-exact.
"""
import math

import numpy as np
import pytest

import ik_reference as ref
import oracle
from conftest import load_golden, sample_edges, sample_states

pytestmark = pytest.mark.gpu

TOL64 = 1e-9
LIMITS = np.array([87.0, 87, 87, 87, 12, 12])


@pytest.fixture(scope="module")
def eng():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from torque_constrained_motion_planning_b200 import engine
    assert engine.device_count() >= 1
    return engine


def dev(x):
    import torch
    return torch.as_tensor(np.ascontiguousarray(x), device="cuda")


def test_kats_from_reference(eng):
    g = load_golden("kat_rne.npz")
    tau, ok = eng.torque_test_batch(dev(g["q"]), dev(g["qd"]), dev(g["qdd"]), dev(g["mass"]), mode="rne")
    assert np.abs(tau.cpu().numpy() - g["tau"]).max() < TOL64
    assert (ok.cpu().numpy() == g["feasible"]).all()
    # raw rne.add_payload rule (threshold 0)
    tau, _ = eng.torque_test_batch(dev(g["q"]), dev(g["qd"]), dev(g["qdd"]), dev(g["mass"]), mode="rne",
                                   payload_threshold=0.0)
    assert np.abs(tau.cpu().numpy() - g["tau_raw"]).max() < TOL64


@pytest.mark.parametrize("mode", ["rne", "nov"])
def test_states_cfg2_vs_reference(eng, mode):
    g = load_golden("states_cfg2.npz")
    tau, ok = eng.torque_test_batch(dev(g["q"]), dev(g["qd"]), dev(g["qdd"]), dev(g["mass"]), mode=mode)
    err = np.abs(tau.cpu().numpy() - g["tau_" + mode]).max()
    assert err < TOL64, err
    assert (ok.cpu().numpy() == g["feasible_" + mode]).all()


@pytest.mark.parametrize("mode", ["rne", "nov", "dyn"])
def test_200k_states_vs_oracle(eng, mode):
    n = 200_000
    q, qd, qdd, mass = sample_states(n, seed=2)
    tau_o, ok_o = oracle.torque_test_batch(mode, q, qd, qdd, mass)
    tau, ok = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode=mode)
    tau = tau.cpu().numpy()
    err = np.abs(tau - tau_o).max()
    assert err < TOL64, err
    assert (ok.cpu().numpy() == ok_o).all()
    # no state sits within the tolerance of a limit, so the masks cannot depend on rounding
    margin = np.abs(LIMITS[:, None] - np.abs(tau_o[:6])).min()
    assert margin > TOL64, margin
    # mask-only and tau-only launches agree with the combined one
    _, ok2 = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode=mode, want_tau=False)
    tau3, _ = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode=mode, want_mask=False)
    assert (ok2.cpu().numpy() == ok_o).all()
    assert np.array_equal(tau3.cpu().numpy(), tau)


def test_static_call_without_velocities(eng):
    """torque(q) as tree growth calls it (rrt_star.py:95): qd = qdd = None -> zeros (panda_primitives.py:175-177)."""
    q, qd, qdd, mass = sample_states(5000, seed=7)
    for mode in ["rne", "dyn"]:
        tau_o, ok_o = oracle.torque_test_batch(mode, q, None, None, mass)
        tau, ok = eng.torque_test_batch(dev(q), None, None, dev(mass), mode=mode)
        assert np.abs(tau.cpu().numpy() - tau_o).max() < TOL64
        assert (ok.cpu().numpy() == ok_o).all()
        z = np.zeros_like(q)
        tau_z, _ = eng.torque_test_batch(dev(q), dev(z), dev(z), dev(mass), mode=mode)
        assert np.abs(tau_z.cpu().numpy() - tau_o).max() < TOL64


def test_scalar_payload_and_base_mode(eng):
    q, qd, qdd, _ = sample_states(3000, seed=8)
    tau_o, ok_o = oracle.torque_test_batch("rne", q, qd, qdd, 3.0)
    tau, ok = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), 3.0, mode="rne")
    assert np.abs(tau.cpu().numpy() - tau_o).max() < TOL64
    assert (ok.cpu().numpy() == ok_o).all()
    tau, ok = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), 3.0, mode="base")
    assert ok.cpu().numpy().all() and (tau.cpu().numpy() == 0).all()


@pytest.mark.parametrize("n", [1, 31, 33, 127, 129, 4097])
def test_ragged_sizes(eng, n):
    q, qd, qdd, mass = sample_states(n, seed=100 + n)
    tau_o, ok_o = oracle.torque_test_batch("rne", q, qd, qdd, mass)
    tau, ok = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode="rne")
    assert np.abs(tau.cpu().numpy() - tau_o).max() < TOL64
    assert (ok.cpu().numpy() == ok_o).all()


def test_large_and_nonfinite_angles_take_the_exact_path(eng):
    """The hot loop's branch-free sincos covers |q| < 1e5 rad; anything larger is redone with CUDA's
    sincos() (exact argument reduction), so parity with libm holds for absurd angles too, and NaN/inf
    propagate like the reference (NaN torque -> the `>=` compare is False -> feasible)."""
    q, qd, qdd, mass = sample_states(4096, seed=9)
    rng = np.random.default_rng(9)
    big = rng.choice(4096, size=300, replace=False)
    q[rng.integers(1, 7, size=300), big] = rng.uniform(-1, 1, size=300) * 10.0 ** rng.uniform(5, 15, size=300)
    q[3, 17] = 99999.99999   # just inside the fast range
    q[3, 18] = 100000.0      # first value outside
    tau_o, ok_o = oracle.torque_test_batch("rne", q, qd, qdd, mass)
    tau, ok = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode="rne")
    assert np.abs(tau.cpu().numpy() - tau_o).max() < TOL64
    assert (ok.cpu().numpy() == ok_o).all()
    q[2, 5] = np.nan
    q[4, 6] = np.inf
    tau, ok = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode="rne")
    t = tau.cpu().numpy()
    assert np.isnan(t[:, 5]).any() and np.isnan(t[:, 6]).any()
    good = np.ones(4096, bool); good[[5, 6]] = False
    assert np.abs(t[:, good] - tau_o[:, good]).max() < TOL64
    tau_o2, ok_o2 = oracle.torque_test_batch("rne", q, qd, qdd, mass)
    assert (ok.cpu().numpy() == ok_o2).all()


def test_empty_batch(eng):
    import torch
    z = torch.empty((7, 0), dtype=torch.float64, device="cuda")
    tau, ok = eng.torque_test_batch(z, z, z, 0.0)
    assert tau.shape == (7, 0) and ok.shape == (0,)


def test_fp32_path(eng):
    q, qd, qdd, mass = sample_states(50_000, seed=3)
    tau_o, ok_o = oracle.torque_test_batch("rne", q, qd, qdd, mass)
    tau, ok = eng.torque_test_batch(dev(q.astype(np.float32)), dev(qd.astype(np.float32)),
                                    dev(qdd.astype(np.float32)), dev(mass.astype(np.float32)), mode="rne", dtype="f32")
    tau = tau.cpu().numpy().astype(np.float64)
    scale = np.maximum(np.abs(tau_o).max(axis=0, keepdims=True), 1.0)  # relative to the state's torque scale
    rel = (np.abs(tau - tau_o) / scale).max()
    assert rel < 1e-4, rel
    # masks may differ only where a torque is within fp32 resolution of a limit
    diff = ok.cpu().numpy() != ok_o
    margin = np.abs(LIMITS[:, None] - np.abs(tau_o[:6])).min(axis=0)
    assert (margin[diff] < 1e-2).all()


def test_host_path_matches_device_path(eng):
    q, qd, qdd, mass = sample_states(300_001, seed=4)
    tau_d, ok_d = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode="rne")
    ws = eng.Workspace(chunk_states=1 << 16)  # forces several pipeline stages + a ragged tail
    tau_h, ok_h = eng.torque_test_batch(q, qd, qdd, mass, mode="rne", workspace=ws)
    assert np.array_equal(tau_h, tau_d.cpu().numpy())
    assert np.array_equal(ok_h, ok_d.cpu().numpy())
    _, ok_h2 = eng.torque_test_batch(q, None, None, 1.0, mode="nov", want_tau=False, workspace=ws)
    _, ok_o = oracle.torque_test_batch("nov", q, None, None, 1.0)
    assert np.array_equal(ok_h2, ok_o)
    ws.close()


def test_async_host_batches_pipeline_and_match(eng):
    """tcmp_rne_batch_host_async: three batches enqueued back to back on one workspace (pinned arrays, distinct
    outputs), one tcmp_workspace_sync -- every batch equals the synchronous call bit for bit."""
    import torch
    ws = eng.Workspace(chunk_states=1 << 15)
    pin = lambda a: torch.as_tensor(np.ascontiguousarray(a)).pin_memory().numpy()
    batches, outs = [], []
    for b in range(3):
        q, qd, qdd, mass = (pin(a) for a in sample_states(100_003 + 17 * b, seed=40 + b))
        tau = pin(np.empty_like(q))
        ok = pin(np.empty(q.shape[1], dtype=np.uint8))
        eng.torque_test_batch_host_async(ws, "rne", "f64", q, qd, qdd, mass, 0.0, 0.01, tau, ok)
        batches.append((q, qd, qdd, mass))
        outs.append((tau, ok))
    eng.workspace_sync(ws)
    for (q, qd, qdd, mass), (tau, ok) in zip(batches, outs):
        tau_s, ok_s = eng.torque_test_batch(q, qd, qdd, mass, mode="rne", workspace=ws)
        assert np.array_equal(tau, tau_s) and np.array_equal(ok, ok_s)
    ws.close()


def test_payload_affinity_property_1m(eng):
    """Size-independent property at the BASELINE size (1M states): the torque is affine in the payload
    mass (the payload link's inertia is linear in m, rne.py:85-100), so tau(5) - tau(0) == 5 (tau(1) - tau(0));
    and the mask is exactly the |tau| < limit predicate of the returned torques."""
    n = 1_000_000
    q, qd, qdd, _ = sample_states(n, seed=2)
    Q, V, A = dev(q), dev(qd), dev(qdd)
    t0, _ = eng.torque_test_batch(Q, V, A, 0.0)
    t1, _ = eng.torque_test_batch(Q, V, A, 1.0)
    t5, ok5 = eng.torque_test_batch(Q, V, A, 5.0)
    lin = ((t5 - t0) - 5.0 * (t1 - t0)).abs().max().item()
    assert lin < 1e-9, lin
    import torch
    lim = torch.as_tensor(LIMITS, device="cuda")[:, None]
    pred = (t5[:6].abs() < lim).all(dim=0)
    assert torch.equal(pred, ok5.bool())


# ---- edges / trajectories -------------------------------------------------------------------------
def test_edges_vs_reference(eng):
    e = load_golden("edges_cfg4.npz")
    ff = eng.edge_feasibility(dev(e["qa"]), dev(e["qb"]), int(e["W"]), float(e["mass"]), mode="rne")
    assert (ff.cpu().numpy() == e["first_fail"]).all()


@pytest.mark.parametrize("W", [64, 1, 7, 100])
def test_edges_vs_oracle(eng, W):
    qa, qb = sample_edges(20_000 if W == 64 else 2_000, seed=4)
    for mode, static in [("rne", False), ("rne", True), ("nov", False), ("dyn", False)]:
        ff_o = oracle.edge_feasibility(mode, qa, qb, W, 5.0) if not static else None
        if static:  # tree-growth semantics: every waypoint tested as (q, 0, 0) == nov arithmetic on the same waypoints
            ff_o = oracle.edge_feasibility("nov", qa, qb, W, 5.0)
        ff = eng.edge_feasibility(dev(qa), dev(qb), W, 5.0, mode=mode, static_only=static)
        assert (ff.cpu().numpy() == ff_o).all(), (mode, static, W)
    ff_h = eng.edge_feasibility(qa, qb, W, 5.0, mode="rne")
    assert (ff_h == oracle.edge_feasibility("rne", qa, qb, W, 5.0)).all()


def test_edges_round_trip_property_100k(eng):
    """BASELINE size (100k edges x 64): an edge's first failure equals the first zero of the per-state mask
    of its 64 explicitly generated waypoints run through the state kernel."""
    import torch
    E, W = 100_000, 64
    qa, qb = sample_edges(E, seed=4)
    ff = eng.edge_feasibility(dev(qa), dev(qb), W, 5.0, mode="rne")
    t = torch.as_tensor(np.linspace(1.0 / W, 1.0, W), device="cuda")
    px = t ** 3 * (10 - 15 * t + 6 * t * t)
    pv = t ** 2 * (30 - 60 * t + 30 * t * t)
    pa = t * (60 - 180 * t + 120 * t * t)
    A = dev(qb - qa)
    q = (dev(qa)[:, :, None] + A[:, :, None] * px).reshape(7, -1).contiguous()
    qd = (A[:, :, None] * pv).reshape(7, -1).contiguous()
    qdd = (A[:, :, None] * pa).reshape(7, -1).contiguous()
    _, ok = eng.torque_test_batch(q, qd, qdd, 5.0, want_tau=False)
    bad = (ok.reshape(E, W) == 0)
    first = torch.where(bad.any(dim=1), bad.float().argmax(dim=1), torch.full((E,), W, device="cuda")).int()
    assert torch.equal(first, ff)


def test_traj_vs_reference(eng):
    t = load_golden("traj.npz")
    coeffs = oracle.minjerk_coefficients(t["points"])
    out = eng.traj_feasibility(coeffs, int(t["n_int"]), float(t["mass"]), mode="rne")
    assert np.abs(out["q"].cpu().numpy().T - t["x"]).max() < 1e-12
    assert np.abs(out["qd"].cpu().numpy().T - t["v"]).max() < 1e-11
    assert np.abs(out["qdd"].cpu().numpy().T - t["a"]).max() < 1e-10
    assert np.abs(out["tau"].cpu().numpy().T - t["tau"]).max() < TOL64
    assert (out["feasible"].cpu().numpy() == t["feasible"]).all()
    bad = np.nonzero(t["feasible"] == 0)[0]
    assert out["first_fail"] == (bad[0] if len(bad) else len(t["feasible"]))
    out0 = eng.traj_feasibility(coeffs, int(t["n_int"]), 0.0, mode="rne")
    assert np.abs(out0["tau"].cpu().numpy().T - t["tau_nopayload"]).max() < TOL64


# ---- IK / FK ---------------------------------------------------------------------------------------
def _match_solutions(sols, ref, count):
    """max over reference solutions of the distance to the nearest returned solution."""
    worst = 0.0
    for i in range(count):
        d = np.abs(sols[:count] - ref[i]).max(axis=1).min()
        worst = max(worst, d)
    return worst


def test_fk_vs_reference(eng):
    g = load_golden("ik_cfg3.npz")
    trans, rot = eng.fk_batch(dev(g["q"]))
    assert np.abs(trans.cpu().numpy() - g["trans"]).max() < 1e-14
    assert np.abs(rot.cpu().numpy() - g["rot"]).max() < 1e-14


def test_ik_vs_reference_golden(eng):
    g = load_golden("ik_cfg3.npz")
    sols, counts, status = eng.ik_batch(dev(g["rot"]), dev(g["trans"]), dev(g["free"]))
    sols, counts, status = sols.cpu().numpy(), counts.cpu().numpy(), status.cpu().numpy()
    assert (counts == g["counts"]).all()                 # bit-exact solution counts
    assert (status == 0).all()                           # random poses never touch a degenerate branch
    worst = max(_match_solutions(sols[i], g["sols"][i], counts[i]) for i in range(len(counts)))
    assert worst < 1e-9, worst
    # host path (pose-chunked pipeline) gives the same bits
    ws = eng.Workspace(chunk_states=1000)
    s2, c2, _ = eng.ik_batch(g["rot"], g["trans"], g["free"], workspace=ws)
    assert np.array_equal(c2, counts) and np.array_equal(s2, sols)


def test_ik_round_trip_100k(eng):
    """FK(IK(pose)) == pose for every returned solution (the reference's own self-check idea,
    ikfast.py:93-102, tolerance 1e-6), and counts match the reference on 100k x 3 solves."""
    import torch
    rng = np.random.default_rng(33)
    n = 100_000
    from conftest import Q_HI, Q_LO
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
    trans_h, rot_h = ref.fk_batch(q)
    trans, rot = dev(trans_h), dev(rot_h)
    free = np.stack([q[6], rng.uniform(-2.8973, 2.8973, n), rng.uniform(-2.8973, 2.8973, n)])
    sols, counts, status = eng.ik_batch(rot, trans, dev(free))
    cnt = counts.cpu().numpy()
    ref.check("round_trip_100k", cnt, sols.cpu().numpy(), inputs=(rot_h, trans_h, free), tol=1e-9)
    assert (cnt.reshape(n, 3)[:, 0] >= 1).all()          # the pose's own j7 always yields a solution
    # round trip on the valid slots
    valid = (torch.arange(8, device="cuda")[None, :] < counts[:, None])
    qs = sols[valid].T.contiguous()                      # [7][m]
    t2, r2 = eng.fk_batch(qs)
    idx = torch.nonzero(valid)[:, 0] // 3                # pose index of each solution
    assert (t2 - trans[:, idx]).abs().max().item() < 1e-6
    assert (r2 - rot[:, idx]).abs().max().item() < 1e-6


# ---- fused peer-store gather (single process: the only destination is this rank's own buffer) -----------
def test_scatter_kernel_single_rank(eng):
    import torch
    from torque_constrained_motion_planning_b200.distributed import PeerMaskBuffer
    n = 100_003
    q, qd, qdd, mass = sample_states(n, seed=21)
    buf = PeerMaskBuffer(n)
    assert buf.world == 1 and buf.gathered.shape == (1, n)
    seen = []
    for mode in ["rne", "nov", "dyn", "base"]:
        buf._slots.zero_()
        tau = buf.torque_test(dev(q), dev(qd), dev(qdd), dev(mass), mode=mode)
        buf.barrier()
        seen.append(buf.gathered.data_ptr())
        tau_o, ok_o = oracle.torque_test_batch(mode, q, qd, qdd, mass)
        assert np.array_equal(buf.gathered[0].cpu().numpy(), ok_o)
        if mode != "base":
            assert np.abs(tau.cpu().numpy() - tau_o).max() < TOL64
    # completion-flag form: signal + wait ride on the side stream, the copies cycle 0, 1, 2; no host synchronisation
    # between the step and the read (the read is enqueued on the side stream behind the wait); an empty shard
    # publishes its epoch too
    for mode in ["rne", "base", "nov"]:
        buf._slots.zero_()
        buf.torque_test(dev(q), dev(qd), dev(qdd), dev(mass), mode=mode, want_tau=False, overlap_gather=True)
        with torch.cuda.stream(buf.side):
            got = buf.gathered[0].clone()
        buf.join()
        _, ok_o = oracle.torque_test_batch(mode, q, qd, qdd, mass)
        assert np.array_equal(got.cpu().numpy(), ok_o)
    buf.torque_test(dev(q[:, :0]), dev(qd[:, :0]), dev(qdd[:, :0]), dev(mass[:0]), want_tau=False, overlap_gather=True)
    buf.join()
    buf.check()              # synchronises; raises if a wait kernel had timed out
    seen = seen[:4]
    # consecutive steps cycle through the three copies of the gathered buffer (read -> next-write ordering)
    assert len(set(seen[:3])) == 3 and seen[0] == seen[3]
    buf.close()


def test_ik_select_vs_composed_reference(eng):
    """tcmp_ik_select == reference IK -> joint-limit filter (ikfast.py:167) -> static torque test
    (oracle) -> nearest to the current configuration (max norm, ikfast.py:172-188), composed on the CPU."""
    from conftest import Q_HI, Q_LO
    rng = np.random.default_rng(44)
    n, nf = 3000, 6
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
    trans, rot = ref.fk_batch(q)
    free = np.vstack([q[6:7], rng.uniform(Q_LO[6], Q_HI[6], size=(nf - 1, n))])
    q_ref = np.clip(q + rng.normal(0, 0.4, size=q.shape), Q_LO[:, None], Q_HI[:, None])
    sols, counts = ref.ik_batch("select_composed", rot, trans, free)
    for mode, mass, norm in [("rne", 5.0, "inf"), ("nov", 3.0, "l2"), ("base", 0.0, "inf"), ("dyn", 4.0, "inf")]:
        best, cost, nv = eng.ik_select(rot, trans, free, q_ref, mass, mode=mode, norm=norm)
        exp_cost = np.full(n, np.inf)
        exp_best = np.zeros((7, n))
        exp_nv = np.zeros(n, dtype=np.int32)
        # flatten all candidate solutions, test them in one oracle call
        cand, owner = [], []
        for p in range(n):
            for f in range(nf):
                s = p * nf + f
                for k in range(counts[s]):
                    c = sols[s, k]
                    if np.all(c >= Q_LO) and np.all(c <= Q_HI):
                        cand.append(c); owner.append(p)
        cand = np.array(cand); owner = np.array(owner)
        _, ok = oracle.torque_test_batch(mode, np.ascontiguousarray(cand.T), None, None, mass)
        for c, p, o in zip(cand, owner, ok):
            if not o:
                continue
            exp_nv[p] += 1
            d = np.abs(c - q_ref[:, p])
            cst = d.max() if norm == "inf" else np.sqrt((d * d).sum())
            if cst < exp_cost[p]:
                exp_cost[p], exp_best[:, p] = cst, c
        assert np.array_equal(nv, exp_nv), mode
        fin = np.isfinite(exp_cost)
        assert np.array_equal(np.isfinite(cost), fin)
        assert np.abs(cost[fin] - exp_cost[fin]).max() < 1e-9
        assert np.abs(best[:, fin] - exp_best[:, fin]).max() < 1e-9
        assert fin.mean() > 0.3


# ---- collision stand-in + fused tree-growth edge check (SURVEY 8f-1/8f-2) ---------------------------
def test_collision_kernel_matches_numpy_stand_in(eng):
    from conftest import Q_HI, Q_LO
    from torque_constrained_motion_planning_b200 import collision
    rng = np.random.default_rng(50)
    qs = rng.uniform(Q_LO - 0.05, Q_HI + 0.05, size=(20_000, 7))       # a few outside the joint limits
    for scene, pr in [(collision.hiro_scene(), 0.0), (collision.cluttered_scene(), 0.04), ([], 0.0)]:
        ref = collision.get_collision_fn(obstacles=scene, payload_radius=pr).batch(qs)
        hit = eng.collision_batch(np.ascontiguousarray(qs.T), scene, payload_radius=pr)
        assert np.array_equal(hit.astype(bool), ref)
        assert 0.02 < ref.mean() < 0.98


def test_extend_prefix_matches_serial_safe_path(eng):
    """One launch over many candidate edges == safe_path_force_aware(extend(q1, q2), collision, torque)
    (rrt_star.py:90-98) edge by edge with the NumPy collision stand-in and the CPU oracle torque test."""
    from conftest import Q_HI, Q_LO
    from torque_constrained_motion_planning_b200 import collision, rrt_star, utils
    rng = np.random.default_rng(51)
    E = 400
    q1 = rng.uniform(Q_LO, Q_HI, size=(E, 7))
    q2 = np.clip(q1 + rng.normal(0, 0.8, size=(E, 7)), Q_LO - 0.02, Q_HI + 0.02)
    q2[:20] = q1[:20]                                                    # zero-length edges: 1 configuration
    res = 0.1 * np.ones(7)
    scene = collision.cluttered_scene()
    col = collision.get_collision_fn(obstacles=scene)
    ext = utils.get_extend_fn(None, list(range(7)), resolutions=res)
    for mode, mass in [("rne", 5.0), ("nov", 1.0), ("base", 0.0)]:
        def tq(q, _mode=mode, _mass=mass):
            _, ok = oracle.torque_test_batch(_mode, np.asarray(q, dtype=float).reshape(7, 1), None, None, _mass)
            return bool(ok[0])
        ns, pre = eng.extend_prefix(np.ascontiguousarray(q1.T), np.ascontiguousarray(q2.T), res, scene, mass, mode=mode)
        for e in range(E):
            seq = list(ext(tuple(q1[e]), tuple(q2[e])))
            safe = rrt_star.safe_path_force_aware(seq, lambda q: col(q), tq)
            assert ns[e] == len(seq), (e, ns[e], len(seq))
            assert pre[e] == len(safe), (mode, e, pre[e], len(safe))
        assert (pre < ns).mean() > 0.1 and (pre == ns).mean() > 0.1


def test_forty_million_states_int64_offsets(eng):
    """Maximum-size property: 40 M states (each joint row 320 MB, arrays 2.2 GB, offsets beyond 2^31 bytes).
    The input is a 1 M-state pattern tiled 40 times, so the mask must tile identically and equal the oracle's
    mask of the pattern."""
    import torch
    base = 1_000_000
    reps = 40
    q, qd, qdd, mass = sample_states(base, seed=2)
    _, ok_o = oracle.torque_test_batch("rne", q[:, :50_000], qd[:, :50_000], qdd[:, :50_000], mass[:50_000])
    tile = lambda a: dev(a).repeat(*([1] * (a.ndim - 1) + [reps])).contiguous()
    Q, V, A, M = tile(q), tile(qd), tile(qdd), tile(mass)
    assert Q.shape == (7, base * reps)
    _, ok = eng.torque_test_batch(Q, V, A, M, mode="rne", want_tau=False)
    ok = ok.view(reps, base)
    assert bool((ok == ok[0:1]).all())
    assert np.array_equal(ok[reps - 1, :50_000].cpu().numpy(), ok_o)
    del Q, V, A, M
    torch.cuda.empty_cache()


def test_ik_select_sweep_longer_than_a_warp(eng):
    """n_free = 40 > 32: the select kernel walks the sweep in two rounds and must keep the best across rounds."""
    from conftest import Q_HI, Q_LO
    rng = np.random.default_rng(45)
    n, nf = 600, 40
    q = rng.uniform(Q_LO[:, None] + 1e-6, Q_HI[:, None] - 1e-6, size=(7, n))
    q[5] = np.minimum(q[5], 3.1)      # the solver returns angles wrapped to (-pi, pi]: joint 6 above pi would come back
    trans, rot = ref.fk_batch(q)          # as q - 2 pi, outside its limits, and be filtered like the reference does
    free = np.vstack([rng.uniform(Q_LO[6], Q_HI[6], size=(nf - 1, n)), q[6:7]])     # the exact j7 comes LAST
    best, cost, nv = eng.ik_select(rot, trans, free, q, 0.0, mode="base", norm="inf")
    # the pose's own configuration is reachable with cost ~ 0 and lives in the second round
    assert (cost < 1e-9).all() and np.abs(best - q).max() < 1e-9 and (nv >= 1).all()
    sols, counts = ref.ik_batch("select_sweep_40", rot, trans, free)
    inside = ((sols >= Q_LO) & (sols <= Q_HI)).all(axis=2) & (np.arange(8)[None, :] < counts[:, None])
    assert np.array_equal(nv, inside.reshape(n, nf, 8).sum(axis=(1, 2)).astype(np.int32))


@pytest.mark.parametrize("mode", ["nov", "dyn"])
def test_traj_kernel_other_modes(eng, mode):
    t = load_golden("traj.npz")
    coeffs = oracle.minjerk_coefficients(t["points"])
    out = eng.traj_feasibility(coeffs, int(t["n_int"]), float(t["mass"]), mode=mode)
    tau_o, mask_o, ff_o = oracle.traj_feasibility(mode, t["points"], int(t["n_int"]), float(t["mass"]))
    assert np.abs(out["tau"].cpu().numpy().T - tau_o).max() < TOL64
    assert np.array_equal(out["feasible"].cpu().numpy(), mask_o) and out["first_fail"] == ff_o


def test_traj_kernel_base_mode_writes_samples_and_log_torques(eng):
    """TCMP_MODE_BASE (constant-true test): mask all 1, first_fail = n, and q / qd / qdd / tau are the same samples and
    rne torques the rne mode writes (the planner returns them as the trajectory; ADVICE r01, edge_kernels.cu)."""
    t = load_golden("traj.npz")
    coeffs = oracle.minjerk_coefficients(t["points"])
    base = eng.traj_feasibility(coeffs, int(t["n_int"]), float(t["mass"]), mode="base")
    rne = eng.traj_feasibility(coeffs, int(t["n_int"]), float(t["mass"]), mode="rne")
    n = base["feasible"].shape[0]
    assert bool(base["feasible"].all()) and base["first_fail"] == n
    for k in ("q", "qd", "qdd", "tau"):
        assert np.array_equal(base[k].cpu().numpy(), rne[k].cpu().numpy()), k


def test_edge_kernel_fp32_path(eng):
    qa, qb = sample_edges(5000, seed=14)
    ff_o = oracle.edge_feasibility("rne", qa, qb, 64, 5.0)
    ff = eng.edge_feasibility(dev(qa.astype(np.float32)), dev(qb.astype(np.float32)), 64, 5.0, mode="rne", dtype="f32")
    ff = ff.cpu().numpy()
    # fp32 may move a first failure only where a torque sits within fp32 resolution of a limit
    assert (ff == ff_o).mean() > 0.995
    assert ((ff >= 0) & (ff <= 64)).all()


@pytest.mark.parametrize("mode", ["rne", "nov", "dyn"])
def test_model_override_vs_oracle(eng, mode):
    """tcmp_rne_batch_model with another inertial set: 200k states against the model-parametrised oracle (itself
    pinned to rne.py with overwritten tables, tests/golden/model_override.npz)."""
    g = load_golden("model_override.npz")
    model = eng.InertialModel(g["model"])
    q, qd, qdd, mass = sample_states(200_000, seed=41)
    tau, ok = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode=mode, model=model)
    tau_o, ok_o = oracle.torque_test_batch(mode, q, qd, qdd, mass, model=g["model"])
    assert np.abs(tau.cpu().numpy() - tau_o).max() < 1e-9
    assert np.array_equal(ok.cpu().numpy(), ok_o)
    # outputs are independently optional, host arrays are staged
    _, ok_only = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode=mode, model=model, want_tau=False)
    assert np.array_equal(ok_only.cpu().numpy(), ok_o)
    tau_h, ok_h = eng.torque_test_batch(q[:, :999], qd[:, :999], qdd[:, :999], mass[:999], mode=mode, model=model)
    assert np.abs(tau_h - tau_o[:, :999]).max() < 1e-9 and np.array_equal(ok_h, ok_o[:999])


def test_model_override_vs_reference_golden(eng):
    g = load_golden("model_override.npz")
    model = eng.InertialModel(g["model"])
    tau, ok = eng.torque_test_batch(dev(g["q"]), dev(g["qd"]), dev(g["qdd"]), dev(g["mass"]), model=model)
    assert np.abs(tau.cpu().numpy() - g["tau_rne"]).max() < 1e-9 and np.array_equal(ok.cpu().numpy(), g["feasible_rne"])
    tau, ok = eng.torque_test_batch(dev(g["q"]), None, None, dev(g["mass"]), mode="nov", model=model)
    assert np.abs(tau.cpu().numpy() - g["tau_nov"]).max() < 1e-9 and np.array_equal(ok.cpu().numpy(), g["feasible_nov"])


def test_default_model_record_equals_compiled_in_kernels(eng):
    """The run-time folded default record and the compile-time constants are the same robot; fp32 too."""
    q, qd, qdd, mass = sample_states(100_000, seed=42)
    d = eng.InertialModel.default()
    for mode in ("rne", "nov", "dyn"):
        a, oa = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode=mode)
        b, ob = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode=mode, model=d)
        assert (a - b).abs().max().item() < 1e-11 and bool((oa == ob).all())
    a, _ = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), dtype="f32")
    b, _ = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), dtype="f32", model=d)
    assert (a - b).abs().max().item() < 2e-3     # both fp32: rounding of two evaluation orders
    _, ok = eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), mode="base", model=d)
    assert bool(ok.all())
    bad = eng.InertialModel.default()
    bad.mass[0] = float("inf")
    with pytest.raises(eng.TcmpError, match="mass"):
        eng.torque_test_batch(dev(q), dev(qd), dev(qdd), dev(mass), model=bad)


# ---- caller-supplied inertial set on the planner-side entry points ---------------------------------------------
def _other_robot(eng):
    g = load_golden("model_override.npz")
    return eng.InertialModel(g["model"]), g["model"]


def test_model_edges_and_trajectory_vs_oracle(eng):
    """tcmp_edge_feasibility_model / tcmp_traj_feasibility_model against the model-parametrised oracle."""
    model, rec = _other_robot(eng)
    qa, qb = sample_edges(5_000, seed=71)
    for mode, W in [("rne", 64), ("nov", 64), ("dyn", 40)]:
        ff = eng.edge_feasibility(dev(qa), dev(qb), W, 3.0, mode=mode, model=model)
        ff_o = oracle.edge_feasibility(mode, qa, qb, W, 3.0, model=rec)
        assert (ff.cpu().numpy() == ff_o).all(), mode
        assert 0.05 < (ff_o < W).mean() < 0.95
        assert (ff_o != oracle.edge_feasibility(mode, qa, qb, W, 3.0)).any()       # and it is another robot
    assert (eng.edge_feasibility(qa[:, :300], qb[:, :300], 64, 3.0, model=model)
            == oracle.edge_feasibility("rne", qa[:, :300], qb[:, :300], 64, 3.0, model=rec)).all()   # host arrays
    t = load_golden("traj.npz")
    coeffs = oracle.minjerk_coefficients(t["points"])
    for mode in ("rne", "nov", "dyn"):
        out = eng.traj_feasibility(coeffs, int(t["n_int"]), 2.0, mode=mode, model=model)
        tau_o, mask_o, ff_o = oracle.traj_feasibility(mode, t["points"], int(t["n_int"]), 2.0, model=rec)
        assert np.abs(out["tau"].cpu().numpy().T - tau_o).max() < TOL64
        assert (out["feasible"].cpu().numpy() == mask_o).all() and out["first_fail"] == ff_o


def test_model_ik_select_and_extend_prefix(eng):
    """tcmp_ik_select_model / tcmp_extend_prefix_model: the static torque test inside both uses the caller's robot."""
    from conftest import Q_HI, Q_LO
    from torque_constrained_motion_planning_b200 import collision, rrt_star, utils
    model, rec = _other_robot(eng)
    rng = np.random.default_rng(72)
    n, nf = 1500, 5
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
    trans, rot = ref.fk_batch(q)
    free = np.vstack([q[6:7], rng.uniform(Q_LO[6], Q_HI[6], size=(nf - 1, n))])
    q_ref = np.clip(q + rng.normal(0, 0.4, size=q.shape), Q_LO[:, None], Q_HI[:, None])
    sols, counts = ref.ik_batch("select_model", rot, trans, free)
    best, cost, nv = eng.ik_select(rot, trans, free, q_ref, 3.0, mode="rne", model=model)
    exp_cost, exp_nv = np.full(n, np.inf), np.zeros(n, dtype=np.int32)
    cand, owner = [], []
    for p in range(n):
        for s in range(p * nf, (p + 1) * nf):
            for k in range(counts[s]):
                if np.all(sols[s, k] >= Q_LO) and np.all(sols[s, k] <= Q_HI):
                    cand.append(sols[s, k]); owner.append(p)
    cand = np.array(cand)
    _, ok = oracle.torque_test_batch("rne", np.ascontiguousarray(cand.T), None, None, 3.0, model=rec)
    _, ok_stock = oracle.torque_test_batch("rne", np.ascontiguousarray(cand.T), None, None, 3.0)
    assert (ok != ok_stock).any()
    for c, p, o in zip(cand, owner, ok):
        if o:
            exp_nv[p] += 1
            exp_cost[p] = min(exp_cost[p], np.abs(c - q_ref[:, p]).max())
    assert np.array_equal(nv, exp_nv)
    fin = np.isfinite(exp_cost)
    assert np.array_equal(np.isfinite(cost), fin) and np.abs(cost[fin] - exp_cost[fin]).max() < 1e-9
    # extend prefix
    E = 200
    q1 = rng.uniform(Q_LO, Q_HI, size=(E, 7))
    q2 = np.clip(q1 + rng.normal(0, 0.8, size=(E, 7)), Q_LO, Q_HI)
    res = 0.1 * np.ones(7)
    scene = collision.hiro_scene()
    col = collision.get_collision_fn(obstacles=scene)
    ext = utils.get_extend_fn(None, list(range(7)), resolutions=res)

    def tq(qc):
        return bool(oracle.torque_test_batch("rne", np.asarray(qc, dtype=float).reshape(7, 1), None, None, 3.0,
                                             model=rec)[1][0])
    ns, pre = eng.extend_prefix(np.ascontiguousarray(q1.T), np.ascontiguousarray(q2.T), res, scene, 3.0, mode="rne",
                                model=model)
    for e in range(E):
        seq = list(ext(tuple(q1[e]), tuple(q2[e])))
        assert ns[e] == len(seq) and pre[e] == len(rrt_star.safe_path_force_aware(seq, lambda c: col(c), tq))
