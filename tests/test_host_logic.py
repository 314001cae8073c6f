"""CPU: host-side logic of the drop-in layer (no GPU): min-jerk coefficients vs the reference's golden
vectors, extend/refine/distance helpers, batched vs serial safe_path, RRT* against the reference's own
rrt_star_force_aware (imported read-only from $TCMP_REFERENCE_SRC, the original's src/ directory, when set), pose algebra, collision stand-in.
The torque predicate in these tests is the CPU oracle -- the thing being tested is the host logic."""
import math
import os
import random
import sys

import numpy as np
import pytest

import oracle
from conftest import Q_HI, Q_LO, load_golden

from torque_constrained_motion_planning_b200 import collision, ik_utils, min_jerk_v2, panda_model, rrt_star, utils

REF_SRC = os.environ.get("TCMP_REFERENCE_SRC", "")
HAVE_REF = os.path.exists(os.path.join(REF_SRC, "rrt_star.py"))


def oracle_torque_fn(mass, mode="rne"):
    def test(q, ptotalMass=None, velocities=None, accelerations=None):
        col = lambda v: None if v is None else np.asarray(v, dtype=float)[:7].reshape(7, 1)
        _, ok = oracle.torque_test_batch(mode, col(q), col(velocities), col(accelerations), mass)
        return bool(ok[0])

    def batch(confs, ptotalMass=None, velocities=None, accelerations=None):
        soa = lambda v: None if v is None else np.ascontiguousarray(np.asarray(v, dtype=float)[:, :7].T)
        _, ok = oracle.torque_test_batch(mode, soa(confs), soa(velocities), soa(accelerations), mass)
        return ok.astype(bool)
    test.batch = batch
    return test


def test_minjerk_coefficients_match_reference_golden():
    m = load_golden("minjerk.npz")
    for name in ["p2", "p5", "p20", "p3_1"]:
        c = min_jerk_v2.minjerk_coefficients(m[name + "_points"])
        assert c.shape == (7, m[name + "_points"].shape[0] - 1, 7)
        k = min_jerk_v2.coefficients_for_kernel(c)
        assert np.abs(k - m[name + "_coeffs"]).max() < 1e-12
        traj = min_jerk_v2.minjerk_trajectory(c, int(m[name + "_n"]))
        x = np.array([p[0] for p in traj]); v = np.array([p[1] for p in traj]); a = np.array([p[2] for p in traj])
        assert np.abs(x - m[name + "_x"]).max() < 1e-12
        assert np.abs(v - m[name + "_v"]).max() < 1e-12
        assert np.abs(a - m[name + "_a"]).max() < 1e-11


def test_minjerk_rejects_non_unit_durations_for_kernel():
    pts = np.random.default_rng(0).uniform(Q_LO, Q_HI, size=(4, 7))
    c = min_jerk_v2.minjerk_coefficients(pts, duration_array=[1.0, 2.0, 1.0])
    with pytest.raises(ValueError):
        min_jerk_v2.coefficients_for_kernel(c)


def test_extend_and_refine_semantics():
    """utils.py:3031-3041,3068-3077: floor(||dq/res||_2) + 1 configurations, last one == q2, q1 excluded."""
    ext = utils.get_extend_fn(None, list(range(7)), resolutions=0.1 * np.ones(7))
    q1 = np.zeros(7); q2 = np.array([0.35, 0, 0, 0, 0, 0, 0.0])
    seq = list(ext(tuple(q1), tuple(q2)))
    assert len(seq) == int(np.linalg.norm((q2 - q1) / 0.1)) + 1 == 4
    assert np.allclose(seq[-1], q2) and not np.allclose(seq[0], q1)
    assert np.allclose(np.diff(np.array(seq)[:, 0]), 0.35 / 4)
    d = utils.get_distance_fn(None, list(range(7)), weights=10 * np.ones(7))
    assert abs(d(q1, q2) - math.sqrt(10 * 0.35 ** 2)) < 1e-15


def test_safe_path_batch_equals_serial():
    rng = np.random.default_rng(1)
    tq = oracle_torque_fn(5.0)
    col = collision.get_collision_fn(obstacles=collision.hiro_scene())
    ext = utils.get_extend_fn(None, list(range(7)), resolutions=0.1 * np.ones(7))
    n_cut = 0
    for _ in range(60):
        a = tuple(rng.uniform(Q_LO, Q_HI)); b = tuple(rng.uniform(Q_LO, Q_HI))
        serial_col = lambda q: col(q)
        serial_tq = lambda q: tq(q)          # plain callables: no .batch -> reference loop
        p_serial = rrt_star.safe_path_force_aware(ext(a, b), serial_col, serial_tq)
        p_batch = rrt_star.safe_path_force_aware(ext(a, b), col, tq)
        assert p_serial == p_batch
        n_cut += len(p_batch) < len(list(ext(a, b)))
    assert n_cut > 5   # the scene and the 5 kg payload really cut some edges


@pytest.mark.skipif(not HAVE_REF, reason="reference tree not present")
@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_rrt_star_matches_reference_tree_growth(seed):
    """Same seeds, same predicates -> the batched RRT* returns exactly what the reference's
    rrt_star_force_aware returns (strict_reference mode)."""
    sys.dont_write_bytecode = True
    if REF_SRC not in sys.path:
        sys.path.insert(0, REF_SRC)
    import importlib
    ref = importlib.import_module("rrt_star")
    assert ref.__file__.startswith(REF_SRC)

    joints = list(range(7))
    res = 0.1 * np.ones(7)
    tq = oracle_torque_fn(3.0)
    col = collision.get_collision_fn(obstacles=collision.hiro_scene())
    dist = utils.get_distance_fn(None, joints, weights=np.reciprocal(res))
    ext = utils.get_extend_fn(None, joints, resolutions=res)
    start = tuple(panda_model.TOP_HOLDING_LEFT_ARM)
    goal = (0.6, -0.2, 0.3, -1.9, 0.1, 1.8, 0.9)
    assert not col(start) and not col(goal) and tq(start) and tq(goal)

    def dynam_fn(path, n=None):   # cheap stand-in: linear samples, zero velocity
        q = [list(p) for p in path]
        z = [[0.0] * 7 for _ in path]
        return q, [0.0] * len(path), z, z

    def run(fn, **kw):
        random.seed(seed)
        samp = utils.get_sample_fn(None, joints, rng=np.random.RandomState(seed))
        return fn(start, goal, dist, samp, ext, col, tq, dynam_fn, radius=[0.01], max_time=50, max_iterations=50, **kw)

    out_ref = run(ref.rrt_star_force_aware)
    out_new = run(rrt_star.rrt_star_force_aware)
    assert (out_ref[0] is None) == (out_new[0] is None)
    if out_ref[0] is not None:
        assert np.array_equal(np.array(out_ref[0]), np.array(out_new[0]))
        assert len(out_new[0]) > 2


def test_plain_rrt_star_and_safe_path():
    """The torque-blind planner (rrt_star.py:99-149) and safe_path (:82-88): batched prefix == serial prefix, and
    the returned path is collision-free, starts at start and ends at the goal."""
    joints = list(range(7))
    res = 0.1 * np.ones(7)
    col = collision.get_collision_fn(obstacles=collision.hiro_scene())
    serial = lambda q: col(q)                     # plain callable: no .batch -> the reference's loop
    dist = utils.get_distance_fn(None, joints, weights=np.reciprocal(res))
    ext = utils.get_extend_fn(None, joints, resolutions=res)
    start = tuple(panda_model.TOP_HOLDING_LEFT_ARM)
    goal = (0.6, -0.2, 0.3, -1.9, 0.1, 1.8, 0.9)
    into_table = (0.0, 1.7, 0.0, -0.8, 0.0, 3.0, 0.0)          # hand below the table top
    for a, b in ((start, goal), (start, into_table)):
        assert rrt_star.safe_path(ext(a, b), col) == rrt_star.safe_path(ext(a, b), serial)
    assert len(rrt_star.safe_path(ext(start, into_table), col)) < len(list(ext(start, into_table)))
    random.seed(4)
    samp = utils.get_sample_fn(None, joints, rng=np.random.RandomState(4))
    path = rrt_star.rrt_star(start, goal, dist, samp, ext, col, radius=0.5, max_iterations=60)
    assert path is not None and np.allclose(path[0], start) and np.allclose(path[-1], goal)
    assert not np.asarray(col.batch(path)).any()
    assert rrt_star.rrt_star(into_table, goal, dist, samp, ext, col, radius=0.5, max_iterations=5) is None
    assert rrt_star.elapsed_time(0.0) > 0


def test_small_boundary_helpers():
    from torque_constrained_motion_planning_b200 import franka_ik_fast, ikfast
    assert franka_ik_fast.get_joint_distances([0] * 7, [1] * 7) == pytest.approx(1.0)
    assert franka_ik_fast.get_tool_from_ik(None, "right") == ((0.0, 0.0, 0.0), (0.0, 0.0, 0.0, 1.0))
    assert ik_utils.get_ik_limits(None, 6) == (-2.8973, 2.8973)
    assert ik_utils.get_ik_limits(None, 6, limits=ik_utils.USE_CURRENT, current_conf=[0, 0, 0, 0, 0, 0, 0.3]) == (0.3, 0.3)
    assert ik_utils.get_ik_limits(None, 6, limits=(-1, 1)) == (-1, 1)
    assert ikfast.get_ik_joints() == list(range(7)) and ikfast.get_module_name() == "ikfast_panda_arm"


def test_pose_algebra_round_trip():
    rng = np.random.default_rng(2)
    for _ in range(50):
        q = rng.normal(size=4); q /= np.linalg.norm(q)
        R = ik_utils.matrix_from_quat(q)
        assert np.allclose(R @ R.T, np.eye(3), atol=1e-14) and abs(np.linalg.det(R) - 1) < 1e-14
        q2 = ik_utils.quat_from_matrix(R)
        assert min(np.abs(q2 - q).max(), np.abs(q2 + q).max()) < 1e-12


def test_collision_stand_in():
    col = collision.get_collision_fn(obstacles=collision.hiro_scene())
    assert not col(panda_model.TOP_HOLDING_LEFT_ARM)
    over = list(panda_model.TOP_HOLDING_LEFT_ARM); over[3] = 0.5           # joint-limit violation == collision
    assert col(over)
    down = [0, 1.7, 0, -0.8, 0, 3.0, 0]                                    # hand below the table top
    assert col(down)
    qs = np.random.default_rng(3).uniform(Q_LO, Q_HI, size=(200, 7))
    assert np.array_equal(col.batch(qs), np.array([col(q) for q in qs]))
    # link frames agree with the reference FK (ikfast ComputeFk, golden poses) at the flange
    g = load_golden("ik_cfg3.npz")
    o = collision.link_frames(np.ascontiguousarray(g["q"].T))
    assert np.abs(o[:, 7].T - g["trans"]).max() < 1e-12


def test_problem_and_panda_model_surface():
    p = utils.Problem(robot=None, fixed=[], payload=None, payload_mass=1.0, execution_time=5, torque_test="rne")
    assert (p.payload_mass, p.execution_time, p.torque_test) == (1.0, 5, "rne")
    assert utils.Problem(None, [], None, 0, 1).torque_test == "arne"      # the reference's (broken) default
    r = panda_model.Panda()
    assert r.qdlim.shape == (9,) and r.qz.shape == (7,) and abs(r.qr[6] - math.pi / 4) < 1e-15
    assert panda_model.TAU_MAX.tolist() == [87, 87, 87, 87, 12, 12, 12]
