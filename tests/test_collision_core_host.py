"""CPU: K8/K9's per-configuration and per-edge code (csrc/collision_core.cuh -- the same source collision_kernels.cu
instantiates) built for the host by tests/native/collision_host.cpp, and the NumPy stand-in (collision.py), both
against the long-double reference of tests/collision_reference.py at contact and joint-limit boundaries; the extend
steps and step count against utils.ExtendSequence bit for bit; and the argument checks of tcmp_collision_batch /
tcmp_extend_prefix, which return before any CUDA call."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import collision_reference as ref
from conftest import ROOT

NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "csrc")
_dp = ctypes.POINTER(ctypes.c_double)
_i32p = ctypes.POINTER(ctypes.c_int32)


def _load_host():
    so = os.path.join(NATIVE, "libcollision_host.so")
    src = os.path.join(NATIVE, "collision_host.cpp")
    deps = [src, os.path.join(CSRC, "collision_core.cuh"), os.path.join(ROOT, "include", "tcmp.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        # Inline functions hidden: libtcmp.so, loaded into the same process, exports a host stub of the device
        # function tcmp::config_collides, and the harness must not bind to it.
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                               "-fvisibility-inlines-hidden", "-Wno-unknown-pragmas", "-o", so, src])
    return ctypes.CDLL(so)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


@pytest.fixture(scope="module")
def host():
    from torque_constrained_motion_planning_b200 import engine
    L = _load_host()
    p = lambda a: a.ctypes.data_as(_dp)

    def collide(qs, obstacles, q_lo, q_hi, payload_radius):
        q = _f64(np.atleast_2d(qs).T)
        n = q.shape[1]
        hit = np.empty(n, dtype=np.uint8)
        lo, hi = _f64(q_lo), _f64(q_hi)
        L.host_collision_batch(ctypes.c_int64(n), p(q), len(obstacles), engine.pack_obstacles(obstacles), p(lo), p(hi),
                               ctypes.c_double(payload_radius), hit.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
        return hit.astype(bool)

    def extend(q1, q2, res, obstacles, q_lo, q_hi, payload_radius):
        a, b = _f64(np.atleast_2d(q1).T), _f64(np.atleast_2d(q2).T)
        n = a.shape[1]
        ns, pre = np.empty(n, dtype=np.int32), np.empty(n, dtype=np.int32)
        r, lo, hi = _f64(res), _f64(q_lo), _f64(q_hi)
        L.host_extend_prefix(ctypes.c_int64(n), p(a), p(b), p(r), len(obstacles), engine.pack_obstacles(obstacles),
                             p(lo), p(hi), ctypes.c_double(payload_radius), ns.ctypes.data_as(_i32p),
                             pre.ctypes.data_as(_i32p))
        return ns, pre

    def config(q1, q2, N, k):
        out = np.empty(7)
        L.host_extend_config(p(_f64(q1)), p(_f64(q2)), N, k, p(out))
        return out

    collide.extend, collide.config = extend, config
    return collide


def stand_in(qs, obstacles, q_lo, q_hi, payload_radius):
    from torque_constrained_motion_planning_b200 import collision
    limits = {j: (q_lo[j], q_hi[j]) for j in range(7)}
    return collision.get_collision_fn(obstacles=obstacles, custom_limits=limits, payload_radius=payload_radius).batch(qs)


@pytest.mark.parametrize("impl", ["host", "stand_in"])
def test_contact_boundaries(host, impl):
    """An obstacle 1e-6 / 1e-9 m inside or outside each link sphere and the payload sphere, through sphere, box
    face, edge and corner, zero-radius sphere and zero-size box: every verdict equals the reference's."""
    band, pinned = ref.check_contacts(host if impl == "host" else stand_in)
    print("contact cases in the band: %d; pinned per sphere: %s" % (band, pinned))
    assert band == 0


@pytest.mark.parametrize("impl", ["host", "stand_in"])
def test_obstacle_table(host, impl):
    band = ref.check_obstacle_table(host if impl == "host" else stand_in)
    print("obstacle-table configurations in the band: %d" % band)
    assert band == 0


@pytest.mark.parametrize("impl", ["host", "stand_in"])
def test_joint_limits_and_non_finite_joints(host, impl):
    ref.check_joint_limits(host if impl == "host" else stand_in)


def test_extend_configurations_bit_for_bit(host):
    """Every configuration of the host build's extend recurrence equals ExtendSequence's, on monotone edges and on
    random ones, and the limit-pinning check the GPU test runs passes on the host build."""
    q1s, q2s, res = ref.monotone_edges(14)
    rng = np.random.default_rng(16)
    a = rng.uniform(-2.5, 2.5, size=(20, 7))
    q1s, q2s = np.vstack([q1s, a]), np.vstack([q2s, a + rng.normal(0, 0.5, size=a.shape)])
    for q1, q2 in zip(q1s, q2s):
        X = ref.extend_sequence(q1, q2, res)
        for k in range(len(X)):
            assert np.array_equal(host.config(q1, q2, len(X), k), X[k]), k
    assert ref.check_extend_steps(host.extend) > 0


def test_step_count(host):
    differ = ref.check_step_count(host.extend)
    print("edges whose np.linalg.norm count differs from the sequentially rounded one: %d" % differ)


def test_host_extend_prefix_matches_stand_in(host):
    """The collision-only safe prefix of the host build equals the first collision of the stand-in along the host's
    extend sequence, in the cluttered scene with a payload sphere."""
    from torque_constrained_motion_planning_b200 import collision
    from conftest import Q_HI, Q_LO, sample_edges
    qa, qb = sample_edges(300, seed=17)
    q1, q2, res = qa.T, qb.T, np.full(7, 0.1)
    scene = collision.cluttered_scene()
    col = collision.get_collision_fn(obstacles=scene, payload_radius=ref.PAYLOAD_R)
    ns, pre = host.extend(q1, q2, res, scene, Q_LO, Q_HI, ref.PAYLOAD_R)
    for e in range(len(q1)):
        X = ref.extend_sequence(q1[e], q2[e], res)
        hit = col.batch(X)
        assert ns[e] == len(X) and pre[e] == (int(np.argmax(hit)) if hit.any() else len(X))
    assert (pre < ns).mean() > 0.1 and (pre == ns).mean() > 0.1


def test_argument_checks_without_gpu():
    """More than TCMP_MAX_OBSTACLES obstacles is TCMP_ERR_UNSUPPORTED even for an empty batch; a resolution <= 0 or
    NaN is TCMP_ERR_INVALID_ARG.  Both are rejected before any CUDA call."""
    from torque_constrained_motion_planning_b200 import _lib, engine
    lib = _lib.load()
    obs = engine.pack_obstacles([engine_box() for _ in range(33)])
    lo, hi = _f64(ref.Q_LO), _f64(ref.Q_HI)
    buf = np.zeros(7)
    ib = np.zeros(1, dtype=np.int32)
    P = lambda a: a.ctypes.data
    for n in (0, 1):
        assert lib.tcmp_collision_batch(n, P(buf), 33, ctypes.addressof(obs), P(lo), P(hi), 0.0, P(ib), None) == -4
        assert lib.tcmp_extend_prefix(3, n, P(buf), P(buf), P(_f64(np.ones(7))), 33, ctypes.addressof(obs), P(lo), P(hi),
                                      0.0, 0.0, 0.01, P(ib), P(ib), None) == -4
    assert b"obstacles" in lib.tcmp_last_error()
    for bad in (0.0, -0.1, np.nan):
        res = np.full(7, 0.1)
        res[3] = bad
        res = _f64(res)
        assert lib.tcmp_extend_prefix(3, 1, P(buf), P(buf), P(res), 0, None, P(lo), P(hi), 0.0, 0.0, 0.01, P(ib),
                                      P(ib), None) == -1
        assert b"resolution[3]" in lib.tcmp_last_error()


def engine_box():
    from torque_constrained_motion_planning_b200.collision import Box
    return Box([1.0, 0.0, 0.0], [0.1, 0.1, 0.1])
