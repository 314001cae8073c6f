"""CPU: the product's IK decision tree (csrc/ik_core.cuh -- the same source the CUDA kernel compiles)
built for the host by tests/native/ik_host.cpp and compared with the reference solver (the golden vectors of the
compiled, unmodified reference, and the pinned reference data of tests/ik_reference.py): solution counts bit-exact
on random reachable poses AND on poses built from special joint values (0, +-pi/2, +-pi/4, pi ...) that drive the
solver into its singular branches."""
import math

import numpy as np
import pytest

import ik_reference as ref
import oracle
from conftest import Q_HI, Q_LO, load_golden


@pytest.fixture(scope="module")
def host_ik():
    return ref.wrap_host_ik(ref.build_host_ik("libik_host.so"))


@pytest.fixture(scope="module")
def host_ik_table():
    """The same source with TCMP_IK_TABLE_SINCOS=1 (table-driven sin / cos of the solved joints; default off)."""
    return ref.wrap_host_ik(ref.build_host_ik("libik_host_table.so", ["TCMP_IK_TABLE_SINCOS=1"]))


def test_pose_builder_matches_the_reference_fk():
    """ik_reference.fk_batch, which builds the poses of the IK tests, against the reference's ComputeFk (golden)."""
    g = load_golden("ik_cfg3.npz")
    trans, rot = ref.fk_batch(g["q"])
    assert np.abs(trans - g["trans"]).max() < 1e-15 and np.abs(rot - g["rot"]).max() < 1e-15


def angular_match(sols, ref, count):
    worst = 0.0
    for a in range(count):
        d = np.abs((sols[:count] - ref[a] + np.pi) % (2 * np.pi) - np.pi).max(axis=1).min()
        worst = max(worst, d)
    return worst


def test_golden_random_poses(host_ik):
    g = load_golden("ik_cfg3.npz")
    s, c, st = host_ik(g["rot"], g["trans"], g["free"])
    assert (c == g["counts"]).all() and (st == 0).all()
    assert max(angular_match(s[i], g["sols"][i], c[i]) for i in range(0, len(c), 4)) < 1e-9


def test_golden_special_poses(host_ik):
    g = load_golden("ik_cfg3.npz")
    s, c, st = host_ik(g["special_rot"], g["special_trans"], g["special_free"])
    assert c.tolist() == g["special_counts"].tolist() == [8, 4, 7, 4, 7, 2]
    assert (st & 2 == 0).all() and (st & 1).any()     # singular branches entered and resolved


def test_special_value_sweep_counts_bit_exact(host_ik):
    vals = np.array([0, math.pi / 2, -math.pi / 2, math.pi / 4, -math.pi / 4, 0.3, -1.2, 2.0, math.pi, 1.0, -2.5])
    rng = np.random.default_rng(5)
    n = 30_000
    q = rng.choice(vals, size=(7, n))
    q[:, : n // 2] = np.clip(q[:, : n // 2], Q_LO[:, None], Q_HI[:, None])   # half inside the joint limits
    trans, rot = ref.fk_batch(q)
    free = np.stack([q[6], rng.choice(vals, size=n), rng.uniform(-3, 3, size=n)])
    s, c, st = host_ik(rot, trans, free)
    # values on the stored sample: well-conditioned solves to 1e-9; singular neighbourhoods only to the solver's ~1e-6
    ref.check("host_special_value_sweep", c, s, inputs=(rot, trans, free), tol=1e-6)
    assert (st & 2 == 0).all()
    assert sorted(set(c.tolist())) == list(range(9))           # every count 0..8 occurs in this sweep
    assert (st & 1).sum() > 100                                # and the singular family is exercised


def test_structured_singular_families_counts_bit_exact(host_ik):
    """Every joint at 0, +-pi/2, +-pi/4, +-3pi/4, +-pi and its limits, joint 4 at +-2.63084142381503 (the elbow
    singularity the generated solver special-cases, ikfast_panda_arm.cpp:2774-2835) and at 0 (:2436-2598), singly, in
    pairs, mixed and perturbed by 1e-5 .. 1e-9: the solution COUNT equals the reference's on every solve and
    no solve reports an unimplemented branch.  VERDICT r01 repro included."""
    from ik_families import structured_families, wrist_axis_family
    total = 0
    for name, (q, free) in structured_families(n_per=1500, seed=11).items():
        trans, rot = ref.fk_batch(q)
        s, c, st = host_ik(rot, trans, free)
        ref.check("host_structured_" + name, c, inputs=(rot, trans, free))
        assert (st & 2 == 0).all(), name
        total += len(c)
        if name in ("j4_sing_p", "j4_sing_p_special"):
            assert (st & 1).sum() >= q.shape[1]            # the elbow branch is entered on every own-j7 solve
            # every returned solution -- including the member of the one-parameter family the solver picks at the
            # elbow singularity -- reproduces the pose
            idx = np.nonzero(c > 0)[0][:400]
            for i in idx:
                p = i // free.shape[0]
                t2, r2 = ref.fk_batch(np.ascontiguousarray(s[i, :c[i]].T))
                assert np.abs(t2 - trans[:, p:p + 1]).max() < 2e-5 and np.abs(r2 - rot[:, p:p + 1]).max() < 2e-5
    assert total > 200_000
    rot, trans, free = wrist_axis_family(4000)
    _, c, st = host_ik(rot, trans, free)
    ref.check("host_wrist_axis", c, inputs=(rot, trans, free))
    assert (c == 0).all() and (st & 2 == 0).all() and (st & 1).sum() > 1000
    # VERDICT r01 "what's weak" #1
    q = np.array([[0.3, -0.5, 0.7, 2.63084142381503, 0.4, 1.9, -0.6]]).T
    trans, rot = ref.fk_batch(q)
    _, c, st = host_ik(rot, trans, np.array([[-0.6]]))
    ref.check("host_elbow_repro", c, inputs=(rot, trans, np.array([[-0.6]])))
    assert c[0] == 6 and st[0] & 3 == 1


def test_host_build_returns_the_reference_solutions_bit_for_bit(host_ik):
    """The count-critical chain of csrc/ik_core.cuh is written in the reference's own association order without FMA
    contraction (xmul / xadd), and this harness links the same glibc: on the singular families -- where the elbow angle
    is a quotient of rounding residues and roots sit 1e-6 apart -- the returned SOLUTIONS equal the compiled
    reference's to the last bit, in the same order.  (On the GPU only CUDA's libm stands between the two.)"""
    from ik_families import structured_families
    fams = structured_families(n_per=2000, seed=5)
    checked = 0
    for name in ("j4_sing_p", "j4_sing_p_special", "j4_zero_pm1e-06", "pin_j2", "pin_j2_j4", "mixed_p6", "grid_unlimited",
                 "near_special_1e-06", "j4_sing_pm3e-07"):
        q, free = fams[name]
        trans, rot = ref.fk_batch(q)
        s, c, st = host_ik(rot, trans, free)
        ref.check("host_bit_for_bit_" + name, c, s, inputs=(rot, trans, free), tol=0.0, bitwise=True)
        checked += int(c.sum())
    assert checked > 100_000


@pytest.mark.skipif(not oracle.have_ref(), reason="oracle/_ref not built")
def test_non_rigid_inputs_flag_every_dropped_branch(host_ik):
    """Inputs that are not rigid transforms (rotation off orthonormal by 1e-8 .. 1e-5) can reach special cases of the
    generated solver that are not built (its polynomial-root fall-backs, :3335-9540): the count may then be lower
    than the reference's, and status bit 1 must say so on EVERY such solve."""
    from ik_families import structured_families
    rng = np.random.default_rng(0)
    mism = total = 0
    for name, (q, free) in structured_families(n_per=600, seed=21).items():
        trans, rot = oracle.ref_fk_batch(q)
        for eps in (1e-8, 1e-6, 1e-5):
            r2 = rot + rng.normal(0, eps, size=rot.shape)
            t2 = trans + rng.normal(0, eps, size=trans.shape)
            _, cr = oracle.ref_ik_batch(r2, t2, free)
            _, c, st = host_ik(r2, t2, free)
            bad = c != cr
            assert not (bad & ((st & 2) == 0)).any(), name
            mism += int(bad.sum())
            total += len(c)
    assert mism < 2e-3 * total


def test_table_sincos_variant_keeps_every_solution_count(host_ik_table):
    """TCMP_IK_TABLE_SINCOS=1: the solver's decisions hang on residuals compared with 1e-5 .. 1e-7, the table's sin /
    cos differ from libm's by <= 2.3e-16 -- 1.5 M solves over random reachable poses and the special-value poses of
    the golden set must give the reference's counts exactly and its solutions to 1e-9."""
    g = load_golden("ik_cfg3.npz")
    s, c, st = host_ik_table(g["special_rot"], g["special_trans"], g["special_free"])
    assert (c == g["special_counts"]).all()
    rng = np.random.default_rng(81)
    n, nf = 60_000, 25
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
    trans, rot = ref.fk_batch(q)
    free = np.vstack([q[6:7], rng.uniform(Q_LO[6], Q_HI[6], size=(nf - 1, n))])
    sols_r, counts_r = ref.ik_batch("host_table_sincos_60k", rot, trans, free)
    sols, counts, status = host_ik_table(rot, trans, free)
    assert np.array_equal(counts, counts_r) and (status == 0).all()
    idx = np.nonzero(counts_r)[0][::97]
    assert max(angular_match(sols[i], sols_r[i], counts_r[i]) for i in idx) < 1e-9
