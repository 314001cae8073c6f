"""GPU: goal-IK selection (K7, tcmp_ik_select[_model] / engine.ik_select) against the composed reference of
tests/select_reference.py built on the kernel's own IK (K5, tcmp_ik_batch), on the designed boundary cases of the
same generators the CPU tests use: joint limits, exact ties, sweep rounds, a full candidate list, torque and payload
threshold boundaries, non-finite inputs; plus K7's IK against K5's, shapes, forms, guard bands and n = 0."""
import numpy as np
import pytest

import select_reference as sr
from conftest import Q_HI, Q_LO
from ik_reference import fk_batch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from torque_constrained_motion_planning_b200 import engine
    return torch, engine


@pytest.fixture(scope="module")
def fams():
    return sr.all_cases()


def _model(engine, rec):
    return None if rec is None else engine.InertialModel(rec)


def gpu_select(env, case, model=None, free=None, q_ref=None):
    torch, engine = env
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    m = model if model is not None else _model(engine, case["model"])
    out = engine.ik_select(d(case["rot"]), d(case["trans"]), d(case["free"] if free is None else free),
                           d(case["q_ref"] if q_ref is None else q_ref), case["mass"], mode=case["mode"],
                           q_lo=case["lo"], q_hi=case["hi"], payload_threshold=case["threshold"], norm=case["norm"],
                           model=m)
    return [t.cpu().numpy() for t in out]


def k5(env, rot, trans, free):
    torch, engine = env
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    s, c, st = engine.ik_batch(d(rot), d(trans), d(free))
    return s.cpu().numpy(), c.cpu().numpy(), st.cpu().numpy()


def reference_k5(env, case):
    s, c, _ = k5(env, case["rot"], case["trans"], case["free"])
    return sr.reference_of(case, s, c)


def _check_case(env, case, model=None):
    got = gpu_select(env, case, model)
    want = reference_k5(env, case)
    assert sr.check_select(got, want, case["norm"]) == 0, (case["family"], case["label"])
    return got, want


# ---- 1. K7's IK is K5's ---------------------------------------------------------------------------------------------
def _singular_families():
    from ik_families import structured_families
    return {k: v for k, v in structured_families(n_per=1000).items()
            if k.startswith("j4_sing_") or any(k.startswith("j4_%s_pm" % s) for s in ("sing", "zero", "msing"))}


def test_k7_solutions_are_k5s(env):
    rng = np.random.default_rng(30)
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, 3000))
    sets = {"random": (q, np.vstack([q[6:7], rng.uniform(Q_LO[6], Q_HI[6], size=(7, 3000))]))}
    sets.update(_singular_families())
    flagged_mismatch, redo = 0, 0
    for name, (qq, free) in sets.items():
        trans, rot = fk_batch(qq)
        n, nf = qq.shape[1], free.shape[0]
        s, c, st = k5(env, rot, trans, free)
        redo += int(sr.host_select(rot, trans, free, qq, -sr.INF7, sr.INF7)[3].sum())
        case = sr._case(rot, trans, free, qq, lo=-sr.INF7, hi=sr.INF7)
        best, cost, nv = gpu_select(env, case)
        want = np.minimum(c, 8).reshape(n, nf).sum(1)
        clean = ~((st.reshape(n, nf) & 8) != 0).any(1)
        assert np.array_equal(nv[clean], want[clean]), name
        flagged_mismatch += int((nv[~clean] != want[~clean]).sum())
        # q_ref = the first K5 solution of each pose: selected at cost 0.0, bit for bit
        first = np.argmax(c.reshape(n, nf) > 0, axis=1)
        has = c.reshape(n, nf).max(1) > 0
        ref = s.reshape(n, nf, 8, 7)[np.arange(n), first, 0].T.copy()
        best, cost, nv = gpu_select(env, case, q_ref=ref)
        assert (cost[has] == 0.0).all() and np.array_equal(best[:, has], ref[:, has]), name
    print("K7 vs K5: %d flagged poses with a count mismatch; %d host solves took the redo path" % (flagged_mismatch,
                                                                                                    redo))
    assert redo > 0


# ---- 2-4. limits, ties, rounds, the full list ------------------------------------------------------------------------
@pytest.mark.parametrize("family", ["j7_limit", "tie", "solver_tie", "full_list", "sweep_round", "nan_limit"])
def test_designed_cases(env, fams, family):
    for c in fams[family]:
        got, want = _check_case(env, c)
        if "want_key" in c:
            k = c["want_key"] >= 0
            assert np.array_equal(want["key"][k], c["want_key"][k]), c["label"]
        if "winner_index" in c:
            assert (want["key"] // 8 == c["winner_index"]).all() and (got[1] < 1e-9).all(), c["label"]
        if family == "full_list":
            assert (got[2] == 256).all()
        if family == "nan_limit":
            opened = dict(c, lo=np.where(np.isnan(c["lo"]), -np.inf, c["lo"]),
                          hi=np.where(np.isnan(c["hi"]), np.inf, c["hi"]))
            for a, b in zip(got, gpu_select(env, opened)):
                assert np.array_equal(a, b, equal_nan=True), c["label"]


def test_joint_limits_at_a_candidates_bits(env):
    """Caller limits on joints 1-6 at a K7 candidate's own bits and one ulp either side, the other joints boxed
    +-1e-3 around it: the candidate survives iff lo <= q <= hi."""
    rng = np.random.default_rng(31)
    q = rng.uniform(Q_LO[:, None] + 0.05, Q_HI[:, None] - 0.05, size=(7, 6))
    trans, rot = fk_batch(q)
    base = sr._case(rot, trans, q[6:7], q, lo=-sr.INF7, hi=sr.INF7)
    b, cost, nv = gpu_select(env, base)
    assert (nv > 0).all()
    for p in range(q.shape[1]):
        cand = b[:, p]
        one = dict(base, rot=rot[:, p:p + 1], trans=trans[:, p:p + 1], free=q[6:7, p:p + 1],
                   q_ref=cand[:, None].copy())
        for j in range(6):
            for side in ("lo", "hi"):
                for step in (-1, 0, 1):
                    lo, hi = cand - 1e-3, cand + 1e-3
                    v = cand[j] if step == 0 else np.nextafter(cand[j], step * np.inf)
                    (lo if side == "lo" else hi)[j] = v
                    got = gpu_select(env, dict(one, lo=lo, hi=hi))
                    inside = (side == "lo" and step <= 0) or (side == "hi" and step >= 0)
                    assert (got[1][0] == 0.0) == inside and (np.array_equal(got[0][:, 0], cand) or not inside), \
                        (p, j, side, step)
                    want = reference_k5(env, dict(one, lo=lo, hi=hi))
                    sr.check_select(got, want, "inf")


def test_inverted_limits_leave_no_survivor(env):
    rng = np.random.default_rng(32)
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, 256))
    trans, rot = fk_batch(q)
    lo, hi = Q_LO.copy(), Q_HI.copy()
    lo[4], hi[4] = 0.1, -0.1
    best, cost, nv = gpu_select(env, sr._case(rot, trans, q[6:7], q, lo=lo, hi=hi))
    assert (nv == 0).all() and (cost == np.inf).all() and (best == 0).all()


# ---- 5. torque and payload threshold boundaries --------------------------------------------------------------------
@pytest.mark.parametrize("norm", ["inf", "l2"])
@pytest.mark.parametrize("model_name", list(sr.MODELS))
@pytest.mark.parametrize("mode", ["rne", "nov", "dyn"])
def test_torque_boundaries(env, mode, model_name, norm):
    torch, engine = env
    cases = sr.torque_cases(mode, sr.model_record(model_name), norm)
    assert cases
    for c in cases:
        _check_case(env, c)
        if model_name == "stock":
            _check_case(env, c, model=engine.InertialModel.default())
    c = dict(cases[0], mode="base")
    _check_case(env, c)


def test_payload_threshold(env, fams):
    got = {}
    for c in fams["threshold"]:
        got[c["label"]] = _check_case(env, c)[0]
    for mode in ("rne", "nov"):
        assert got[mode + "_at"][2][0] != got[mode + "_above"][2][0], mode


# ---- 6. shapes and forms -------------------------------------------------------------------------------------------
def _random_case(n, seed, nf=5, norm="inf", mode="rne"):
    rng = np.random.default_rng(seed)
    q = rng.uniform(Q_LO[:, None], Q_HI[:, None], size=(7, n))
    trans, rot = fk_batch(q)
    free = np.vstack([q[6:7], rng.uniform(Q_LO[6], Q_HI[6], size=(nf - 1, n))])
    q_ref = np.clip(q + rng.normal(0, 0.4, size=q.shape), Q_LO[:, None], Q_HI[:, None])
    return sr._case(rot, trans, free, q_ref, mode=mode, mass=5.0, norm=norm)


def test_broadcast_and_per_pose_forms_agree(env):
    c = _random_case(300, 33)
    fb = c["free"][:, 0].copy()
    rb = c["q_ref"][:, 0].copy()
    a = gpu_select(env, c, free=fb, q_ref=rb)
    b = gpu_select(env, c, free=np.repeat(fb[:, None], 300, 1), q_ref=np.repeat(rb[:, None], 300, 1))
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("n", [1, 7, 8, 9, 255, 257])
def test_batch_sizes(env, n):
    for norm in ("inf", "l2"):
        _check_case(env, _random_case(n, 34 + n, norm=norm))


def test_grid_stride_tiling(env):
    """50 000 poses, past the ~18 944-warp grid: the loop strides and the idle warps repeat pose n - 1."""
    pat = _random_case(500, 35)
    ref = gpu_select(env, pat)
    sr.check_select(ref, reference_k5(env, pat), "inf")
    k = 100
    big = dict(pat, rot=np.tile(pat["rot"], k), trans=np.tile(pat["trans"], k), free=np.tile(pat["free"], k),
               q_ref=np.tile(pat["q_ref"], k))
    got = gpu_select(env, big)
    for x, y in zip(got, ref):
        assert np.array_equal(x, np.tile(y, k) if y.ndim == 1 else np.tile(y, (1, k)))


def test_outputs_touch_nothing_outside_their_views(env):
    torch, engine = env
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr
    lib = _lib.load()
    c = _random_case(333, 36)
    n, nf = 333, c["free"].shape[0]
    want = gpu_select(env, c)
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    rot, trans, free, ref = d(c["rot"]), d(c["trans"]), d(c["free"]), d(c["q_ref"])
    lo, hi = np.ascontiguousarray(Q_LO), np.ascontiguousarray(Q_HI)
    for count in (n, 0):
        bq = torch.full((37 + 7 * n + 41,), float("nan"), dtype=torch.float64, device="cuda")
        bc = torch.full((37 + n + 41,), float("nan"), dtype=torch.float64, device="cuda")
        bn = torch.full((37 + n + 41,), -12345, dtype=torch.int32, device="cuda")
        vq, vc, vn = bq[37:37 + 7 * n], bc[37:37 + n], bn[37:37 + n]
        rc = lib.tcmp_ik_select(count, _ptr(rot), _ptr(trans), _ptr(free), nf, 0, _ptr(ref), 0,
                                lo.ctypes.data, hi.ctypes.data, 0, 5.0, 0.01, 1, _ptr(vq), _ptr(vc), _ptr(vn),
                                engine._stream_ptr())
        assert rc == 0
        torch.cuda.synchronize()
        if count:
            assert np.array_equal(vq.cpu().numpy().reshape(7, n), want[0])
            assert np.array_equal(vc.cpu().numpy(), want[1]) and np.array_equal(vn.cpu().numpy(), want[2])
            for buf, fill in ((bq, None), (bc, None), (bn, -12345)):
                rest = torch.cat([buf[:37], buf[-41:]])
                assert rest.isnan().all() if fill is None else (rest == fill).all()
        else:   # n = 0: OK, nothing written
            assert bq.isnan().all() and bc.isnan().all() and (bn == -12345).all()


# ---- 7. non-finite inputs --------------------------------------------------------------------------------------------
def test_nonfinite_reference(env, fams):
    for c in fams["nonfinite_ref"]:
        best, cost, nv = _check_case(env, c)[0]
        live = nv > 0
        assert live.any()
        if c["label"].startswith("nan"):
            assert np.isnan(cost[live]).all(), c["label"]
        else:
            assert (cost[live] == np.inf).all(), c["label"]


def test_nonfinite_free_values_and_poses(env):
    c = _random_case(200, 37, nf=3, mode="base")
    plain = gpu_select(env, c)
    for bad in (np.nan, np.inf, -np.inf):
        free = np.insert(c["free"], 1, bad, axis=0)     # 0 solutions for that value, the others unaffected
        got = gpu_select(env, c, free=free)
        for x, y in zip(got, plain):
            assert np.array_equal(x, y, equal_nan=True)
    rot = c["rot"].copy()
    rot[4, ::3] = np.nan                                # NaN poses: no solution at all
    best, cost, nv = gpu_select(env, dict(c, rot=rot))
    assert (nv[::3] == 0).all() and (cost[::3] == np.inf).all() and (best[:, ::3] == 0).all()
