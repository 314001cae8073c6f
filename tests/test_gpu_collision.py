"""GPU: K8 (collision_kernel, tcmp_collision_batch) and K9 (extend_prefix_kernel, tcmp_extend_prefix[_model]) against
the long-double reference of tests/collision_reference.py, with the same case generators the host-build tests use:
contact and joint-limit boundaries, the obstacle table, the extend steps bit for bit, the step count, the extend
prefix with the torque test against the CPU oracle, own guard bands and the grid-stride loop."""
import ctypes

import numpy as np
import pytest

import collision_reference as ref
import oracle
from conftest import Q_HI, Q_LO, load_golden, sample_edges

pytestmark = pytest.mark.gpu

TORQUE_BAND = 1e-9      # N.m: the kernels' torques agree with the oracle to well inside this (the torque contract)


@pytest.fixture(scope="module")
def eng():
    from torque_constrained_motion_planning_b200 import engine
    return engine


@pytest.fixture(scope="module")
def gpu(eng):
    def collide(qs, obstacles, q_lo, q_hi, payload_radius):
        q = np.ascontiguousarray(np.atleast_2d(qs).T, dtype=np.float64)
        return eng.collision_batch(q, obstacles, q_lo, q_hi, payload_radius).astype(bool)

    def extend(q1, q2, res, obstacles, q_lo, q_hi, payload_radius):
        a = np.ascontiguousarray(np.atleast_2d(q1).T, dtype=np.float64)
        b = np.ascontiguousarray(np.atleast_2d(q2).T, dtype=np.float64)
        return eng.extend_prefix(a, b, res, obstacles, 0.0, mode="base", q_lo=q_lo, q_hi=q_hi,
                                 payload_radius=payload_radius)

    collide.extend = extend
    return collide


def test_contact_boundaries(gpu):
    band, pinned = ref.check_contacts(gpu)
    print("contact cases in the band: %d; pinned per sphere: %s" % (band, pinned))
    assert band == 0


def test_obstacle_table(gpu):
    band = ref.check_obstacle_table(gpu)
    print("obstacle-table configurations in the band: %d" % band)
    assert band == 0


def test_joint_limits_and_non_finite_joints(gpu, eng):
    ref.check_joint_limits(gpu)

    def packed(qs, obstacles, q_lo, q_hi, payload_radius):   # limits marshalled once, as the planner does
        sc = eng.PackedScene(obstacles, q_lo, q_hi, payload_radius)
        return eng.collision_batch(np.ascontiguousarray(np.atleast_2d(qs).T), sc).astype(bool)
    ref.check_joint_limits(packed)


def test_extend_steps_bit_for_bit(gpu):
    """Configuration k of the kernel's extend sequence equals the host's ExtendSequence exactly, for every joint and
    k in {0, 31, 32, 33, 63, 64, N - 1} (the ballot rounds' edges), one launch per case."""
    print("launches: %d" % ref.check_extend_steps(gpu.extend))


def test_step_count(gpu):
    differ = ref.check_step_count(gpu.extend)
    print("edges whose np.linalg.norm count differs from the sequentially rounded one: %d" % differ)


CASES = [  # mode, payload mass, payload radius, scene, inertial set
    ("dyn", 5.0, 0.0, "hiro", "stock"),
    ("dyn", 0.01, ref.PAYLOAD_R, "cluttered", "override"),  # at the threshold: dyn applies it
    ("rne", 0.01, ref.PAYLOAD_R, "cluttered", "override"),  # at the threshold: rne attaches nothing
    ("rne", 3.0, ref.PAYLOAD_R, "cluttered", "override"),
    ("dyn", 3.0, 0.0, "cluttered", "override"),
    ("nov", 5.0, ref.PAYLOAD_R, "hiro", "override"),
]


@pytest.mark.parametrize("mode,mass,pr,scene_name,model_name", CASES)
def test_extend_prefix_with_torque(eng, mode, mass, pr, scene_name, model_name):
    """The safe prefix of every edge equals safe_path_force_aware's on the host: the stand-in's collisions, then the
    oracle's static torque test on collision-free configurations.  Edges whose decision rests on an oracle torque
    within 1e-9 N.m of its limit, or on a clearance within the reference's band, are excluded and counted."""
    from torque_constrained_motion_planning_b200 import collision
    rec = None if model_name == "stock" else load_golden("model_override.npz")["model"]
    model = None if rec is None else eng.InertialModel(rec)
    limit = (eng.get_limits()["torque"] if rec is None else oracle.model_fields(rec.copy())["torque_limit"])[:, None]
    scene = collision.hiro_scene() if scene_name == "hiro" else collision.cluttered_scene()
    rng = np.random.default_rng(80)
    E = 300
    q1 = rng.uniform(Q_LO, Q_HI, size=(E, 7))
    q2 = np.clip(q1 + rng.normal(0, 0.8, size=(E, 7)), Q_LO - 0.02, Q_HI + 0.02)
    q2[:10] = q1[:10]
    res = np.full(7, 0.1)
    ns, pre = eng.extend_prefix(np.ascontiguousarray(q1.T), np.ascontiguousarray(q2.T), res, scene, mass, mode=mode,
                                payload_radius=pr, model=model)
    seqs = [ref.extend_sequence(a, b, res) for a, b in zip(q1, q2)]
    X = np.vstack(seqs)
    col = collision.get_collision_fn(obstacles=scene, payload_radius=pr).batch(X)
    _, band = ref.verdict(X, scene, payload_radius=pr)
    z = np.zeros((7, len(X)))
    tau, ok = oracle.torque_test_batch(mode, np.ascontiguousarray(X.T), z, z, mass, model=rec)
    close = (np.abs(np.abs(tau) - limit) < TORQUE_BAND).any(axis=0) & ~col
    bad = col | ~ok.astype(bool)
    excluded, at = 0, 0
    for e, s in enumerate(seqs):
        sl = slice(at, at + len(s))
        at += len(s)
        want = int(np.argmax(bad[sl])) if bad[sl].any() else len(s)
        decisive = slice(sl.start, sl.start + min(want + 1, len(s)))
        assert ns[e] == len(s), (e, ns[e], len(s))
        if close[decisive].any() or band[decisive].any():
            excluded += 1
            continue
        assert pre[e] == want, (mode, e, pre[e], want)
    print("edges excluded (torque within %g N.m of a limit or clearance in the band): %d of %d"
          % (TORQUE_BAND, excluded, E))
    assert excluded <= 2
    assert (pre < ns).mean() > 0.05 and (pre == ns).mean() > 0.05     # both truncated and whole edges occur


GUARD = 4096


def _guarded(torch, n, dtype, sentinel):
    big = torch.full((n + 2 * GUARD,), sentinel, dtype=dtype, device="cuda")
    return big, big[GUARD:GUARD + n]


def _intact(big, n, sentinel):
    return bool((big[:GUARD] == sentinel).all()) and bool((big[GUARD + n:] == sentinel).all())


@pytest.mark.parametrize("n", [1, 31, 33, 129, 20011])
def test_output_guard_bands(eng, n):
    """Own bounds check: hit_out, n_steps_out and prefix_out are carved out of sentinel-filled allocations; the bands
    on both sides stay untouched, every element is written, and the values equal the host's."""
    import torch
    from torque_constrained_motion_planning_b200 import collision
    lib = eng.load()
    st = int(torch.cuda.current_stream().cuda_stream)
    scene = collision.cluttered_scene()
    sc = eng.PackedScene(scene, None, None, ref.PAYLOAD_R)
    rng = np.random.default_rng(n)
    qs = rng.uniform(Q_LO - 0.05, Q_HI + 0.05, size=(n, 7))
    q = torch.as_tensor(np.ascontiguousarray(qs.T), device="cuda")
    bh, hit = _guarded(torch, n, torch.uint8, 0xA5)
    eng.check(lib.tcmp_collision_batch(n, q.data_ptr(), sc.n, ctypes.addressof(sc.obs), sc.lo.ctypes.data,
                                       sc.hi.ctypes.data, sc.payload_radius, hit.data_ptr(), st))
    torch.cuda.synchronize()
    assert _intact(bh, n, 0xA5)
    want = collision.get_collision_fn(obstacles=scene, payload_radius=ref.PAYLOAD_R).batch(qs)
    assert np.array_equal(hit.cpu().numpy(), want.astype(np.uint8))
    qa, qb = sample_edges(n, seed=n)
    a, b = (torch.as_tensor(np.ascontiguousarray(x), device="cuda") for x in (qa, qb))
    res = np.full(7, 0.1)
    want_ns = np.array([ref.sequential_num_configs(qa[:, e], qb[:, e], res) for e in range(n)])
    for mode in range(4):
        bs, ns = _guarded(torch, n, torch.int32, -1234567)
        bp, pre = _guarded(torch, n, torch.int32, -1234567)
        eng.check(lib.tcmp_extend_prefix(mode, n, a.data_ptr(), b.data_ptr(), res.ctypes.data, sc.n,
                                         ctypes.addressof(sc.obs), sc.lo.ctypes.data, sc.hi.ctypes.data,
                                         sc.payload_radius, 3.0, 0.01, ns.data_ptr(), pre.data_ptr(), st))
        torch.cuda.synchronize()
        assert _intact(bs, n, -1234567) and _intact(bp, n, -1234567)
        ns, pre = ns.cpu().numpy(), pre.cpu().numpy()
        assert np.array_equal(ns, want_ns) and ((pre >= 0) & (pre <= ns)).all()


def test_collision_batch_larger_than_the_grid(eng):
    """4 M configurations, far more threads than the launch grid has, so every thread runs the grid-stride loop many
    times.  The input is a 50 k pattern tiled 80 times: the hits must tile identically and equal the reference's
    verdicts on the pattern."""
    import torch
    from torque_constrained_motion_planning_b200 import collision
    base, reps = 50_000, 80
    qs = np.random.default_rng(81).uniform(Q_LO - 0.05, Q_HI + 0.05, size=(base, 7))
    scene = collision.cluttered_scene()
    q = torch.as_tensor(np.ascontiguousarray(qs.T), device="cuda").repeat(1, reps).contiguous()
    hit = eng.collision_batch(q, scene, payload_radius=ref.PAYLOAD_R)
    torch.cuda.synchronize()
    h = hit.view(reps, base)
    assert bool((h == h[0]).all())
    band = ref.assert_verdicts(h[0].cpu().numpy(), qs, scene, payload_radius=ref.PAYLOAD_R, what="tiled")
    print("tiled pattern configurations in the band: %d" % band)
    assert band == 0
