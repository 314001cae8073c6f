"""CPU: goal-IK selection (K7) built for the host from its own sources (tests/native/select_host.cpp: csrc/ik_core.cuh,
csrc/select_core.cuh and the static torque test of csrc/panda_model.cuh) against the composed reference of
tests/select_reference.py, on the designed boundary cases and on random poses; and the generated cases themselves
against the oracle and the host IK."""
import numpy as np
import pytest

import select_reference as sr
from conftest import Q_HI, Q_LO
from ik_reference import fk_batch, host_ik


@pytest.fixture(scope="module")
def fams():
    return sr.all_cases()


@pytest.fixture(scope="module")
def torque_fams():
    return sr.torque_families()


def _run(case):
    got = sr.host_of(case)
    want = sr.reference_of(case)
    skipped = sr.check_select(got[:3], want, case["norm"])
    assert skipped == 0, (case["family"], case["label"])
    return got, want


# ---- the cases are what they claim --------------------------------------------------------------------------------
def test_every_family_is_non_empty(fams, torque_fams):
    for name in ("j7_limit", "tie", "solver_tie", "full_list", "sweep_round", "threshold", "nonfinite_ref",
                 "nan_limit"):
        assert fams.get(name), name
    assert {c["label"] for c in fams["j7_limit"]} == {s + d for s in ("lo", "hi") for d in ("-1", "+0", "+1")}
    for key, cases in torque_fams.items():
        for d in sr.DELTAS:
            for side in ("pass", "fail"):
                assert any(c["label"].endswith("_d%g_%s" % (d, side)) for c in cases), (key, d, side)


def test_joint7_of_every_solution_is_the_free_value():
    rng = np.random.default_rng(20)
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, 500))
    trans, rot = fk_batch(q)
    free = np.vstack([q[6:7], rng.uniform(Q_LO[6], Q_HI[6], size=(3, 500))])
    s, c, _ = host_ik(rot, trans, free)
    live = np.arange(8)[None] < np.minimum(c, 8)[:, None]
    j7 = s[:, :, 6]
    want = np.broadcast_to(free.T.reshape(-1)[:, None], j7.shape)
    assert live.sum() > 1000 and np.array_equal(j7[live], want[live])


def test_joint7_limit_cases_sit_on_the_limit(fams):
    for c in fams["j7_limit"]:
        v = c["limit_value"]
        assert (c["free"][0] == v).all()
        lim = Q_HI[6] if c["label"].startswith("hi") else Q_LO[6]
        step = int(c["label"][2:])
        outward = 1.0 if c["label"].startswith("hi") else -1.0
        assert v == {0: lim, -1: np.nextafter(lim, -outward * np.inf), 1: np.nextafter(lim, outward * np.inf)}[step]
        want = sr.reference_of(c)
        assert (want["key"] == c["want_key"])[c["want_key"] >= 0].all()
        if step == 1:      # one ulp outside: nothing of the first free value survives
            assert (want["key"] // 8 != 0).all()


def test_tie_cases_are_exact(fams):
    for c in fams["tie"] + fams["solver_tie"]:
        want = sr.reference_of(c)
        assert np.array_equal(want["key"], c["want_key"]), c["label"]
        s, cnt, _ = sr.ik_of(c)
        nf = c["free"].shape[0]
        for p in range(c["rot"].shape[1]):
            q, _, key = sr.candidates(s.reshape(-1, nf, 8, 7)[p], cnt.reshape(-1, nf)[p], 1, nf)
            d = np.abs(q - c["q_ref"][:, p])
            cost = d.max(1)
            near = cost < cost.min() + 1e-6
            assert near.sum() >= 2 or c["label"].endswith("flip"), c["label"]
            assert (d[near, 6] >= d[near, :6].max(1) + sr.J7_MARGIN).all(), c["label"]
        if c["family"] == "tie":
            f = c["free"][:, 0]
            i1, i2 = (int(x) for x in c["label"].split("_")[1:3])
            r7 = c["q_ref"][6, 0]
            if c["label"].endswith("tie"):
                assert abs(f[i1] - r7) == abs(f[i2] - r7)
            else:
                late = max(i1, i2)
                assert abs(f[late] - r7) < abs(f[min(i1, i2)] - r7)


def test_full_list_case_fills_the_candidate_list(fams):
    (c,) = fams["full_list"]
    want = sr.reference_of(c)
    assert (want["nv"] == 256).all() and (want["key"] == 5).all() and (want["cost"] == 0).all()


def test_torque_cases_keep_out_of_the_band(torque_fams):
    for key, cases in torque_fams.items():
        for c in cases:
            want = sr.reference_of(c)
            assert not want["band"].any(), (key, c["label"])
            d = float(c["label"].split("_d")[1].split("_")[0])
            assert abs(abs(c["margin"]) - d) <= 1e-3 * d + 1e-11 and (c["margin"] > 0) == c["label"].endswith("fail")


def test_threshold_model_gap_is_millinewton_metres(fams):
    for c in fams["threshold"]:
        assert c["limit_gap"] > 1e-3, c["label"]
        assert not sr.reference_of(c)["band"].any()
    at = {c["label"]: sr.reference_of(c) for c in fams["threshold"]}
    for mode in ("rne", "nov"):     # the two masses straddle the limit: the verdicts differ
        assert at[mode + "_at"]["nv"][0] != at[mode + "_above"]["nv"][0], mode


# ---- the host build equals the reference ----------------------------------------------------------------------------
@pytest.mark.parametrize("family", ["j7_limit", "tie", "solver_tie", "full_list", "sweep_round", "threshold",
                                    "nan_limit"])
def test_host_matches_reference_on_designed_cases(fams, family):
    for c in fams[family]:
        got, want = _run(c)
        if "want_key" in c:
            k = c["want_key"] >= 0
            assert np.array_equal(want["key"][k], c["want_key"][k]), c["label"]
        if "winner_index" in c:
            assert (got[1] < 1e-9).all() and (want["key"] // 8 == c["winner_index"]).all(), c["label"]


def test_host_matches_reference_on_torque_boundaries(torque_fams):
    for key, cases in torque_fams.items():
        for c in cases:
            _run(c)


@pytest.mark.parametrize("model_name", list(sr.MODELS))
@pytest.mark.parametrize("mode", ["rne", "nov", "dyn", "base"])
def test_host_matches_reference_on_random_poses(mode, model_name):
    rng = np.random.default_rng(21)
    n, nf = 2000, 4
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
    trans, rot = fk_batch(q)
    free = np.vstack([q[6:7], rng.uniform(Q_LO[6], Q_HI[6], size=(nf - 1, n))])
    q_ref = np.clip(q + rng.normal(0, 0.4, size=q.shape), Q_LO[:, None], Q_HI[:, None])
    model = sr.model_record(model_name)
    s, c, _ = host_ik(rot, trans, free)
    for norm in ("inf", "l2"):
        got = sr.host_select(rot, trans, free, q_ref, mode=mode, mass=5.0, norm=norm, model=model)
        want = sr.reference_select(s, c, nf, q_ref, mode=mode, mass=5.0, norm=norm, model=model)
        sr.check_select(got[:3], want, norm)
        assert (want["nv"] > 0).mean() > 0.3


# ---- non-finite q_ref and limits ---------------------------------------------------------------------------------
def test_nan_reference_selects_the_first_survivor(fams):
    """A NaN in q_ref: every cost is NaN, the first surviving solution in (free value, solver order) is returned with
    best_cost = NaN, and n_valid is that of a finite q_ref (fails with fmax in the max norm or the plain (cost, key)
    compare: the NaN joint is dropped, or nothing is selected)."""
    for c in fams["nonfinite_ref"]:
        if not c["label"].startswith("nan"):
            continue
        got, want = _run(c)
        best, cost, nv, _ = got
        live = want["nv"] > 0
        assert live.any() and np.isnan(cost[live]).all(), c["label"]
        s, cnt, _ = sr.ik_of(c)
        finite = sr.reference_select(s, cnt, c["free"].shape[0], np.nan_to_num(c["q_ref"]), norm=c["norm"])
        assert np.array_equal(nv, finite["nv"]), c["label"]
        q, pose, key = sr.candidates(s, cnt, c["rot"].shape[1], c["free"].shape[0])
        inl = ((q >= Q_LO) & (q <= Q_HI)).all(1)
        first = {}
        for i in np.flatnonzero(inl):
            first.setdefault(pose[i], q[i])
        for p, qq in first.items():
            assert np.array_equal(best[:, p], qq), (c["label"], p)
        assert np.array_equal(cost[~live], np.full((~live).sum(), np.inf)) and (best[:, ~live] == 0).all()


def test_infinite_reference_selects_the_first_survivor(fams):
    """+-inf in q_ref: every cost is +inf and the smaller key wins."""
    for c in fams["nonfinite_ref"]:
        if c["label"].startswith("nan"):
            continue
        got, want = _run(c)
        live = want["nv"] > 0
        assert live.any() and (got[1][live] == np.inf).all()
        s, cnt, _ = sr.ik_of(c)
        q, pose, key = sr.candidates(s, cnt, c["rot"].shape[1], c["free"].shape[0])
        inl = ((q >= Q_LO) & (q <= Q_HI)).all(1)
        firstkey = {}
        for i in np.flatnonzero(inl):
            firstkey.setdefault(pose[i], key[i])
        assert all(want["key"][p] == k for p, k in firstkey.items())


def test_nan_limit_bounds_nothing(fams):
    for c in fams["nan_limit"]:
        j = int(c["label"][2:])
        opened = dict(c)
        opened["lo"], opened["hi"] = c["lo"].copy(), c["hi"].copy()
        side = c["label"][:2]
        (opened["lo"] if side == "lo" else opened["hi"])[j] = -np.inf if side == "lo" else np.inf
        got = sr.host_of(c)
        ref = sr.host_of(opened)
        for a, b in zip(got, ref):
            assert np.array_equal(a, b, equal_nan=True), c["label"]


def test_inverted_limits_leave_no_survivor():
    rng = np.random.default_rng(22)
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, 64))
    trans, rot = fk_batch(q)
    lo, hi = Q_LO.copy(), Q_HI.copy()
    lo[2], hi[2] = 0.1, -0.1
    best, cost, nv, _ = sr.host_select(rot, trans, q[6:7], q, lo, hi)
    assert (nv == 0).all() and (cost == np.inf).all() and (best == 0).all()


def test_redo_path_is_reached_by_the_singular_families():
    """The elbow-singular redo path (solve_one_t<true> after solve_one_t<false> bails out) is reached by the j4
    singular families, and the host selection there equals the reference built on the complete solver."""
    from ik_families import structured_families
    fams = structured_families(n_per=300)
    total = 0
    for name, (q, free) in fams.items():
        if not (name.startswith("j4_sing_") or any(name.startswith("j4_%s_pm" % k) for k in ("sing", "zero", "msing"))):
            continue
        trans, rot = fk_batch(q)
        lo, hi = np.full(7, -np.inf), np.full(7, np.inf)
        got = sr.host_select(rot, trans, free, q, lo, hi)
        s, cnt, _ = host_ik(rot, trans, free)
        want = sr.reference_select(s, cnt, free.shape[0], q, lo, hi)
        sr.check_select(got[:3], want, "inf")
        total += int(got[3].sum())
    assert total > 0
