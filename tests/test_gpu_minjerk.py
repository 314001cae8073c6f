"""GPU: K4 (edge_kernel: tcmp_edge_feasibility[_model|_host|_scatter]; traj_kernel: tcmp_traj_feasibility[_model])
against the long-double min-jerk reference of tests/minjerk_reference.py, with the boundary cases the CPU tests check
against the oracle: a first failure at every lane and round edge of the warp reduction, a torque delta = 1e-8, 1e-5
or 1 N.m above or below its limit, the payload threshold, the scatter form, the grid-stride loop, fp32 first
failures justified by the fp32 contract, the trajectory's sample times bit for bit and its atomicMin first failure,
the exact `>=` limit compare, and a non-finite joint-1 angle through the torque and edge kernels.  (An extend edge
with a non-finite end point has no steps, so K9's torque test never sees one.)"""
import ctypes

import numpy as np
import pytest

import minjerk_reference as R
import oracle
from conftest import sample_edges, sample_states

pytestmark = pytest.mark.gpu

EDGE_MODES = [("rne", False), ("nov", False), ("dyn", False), ("rne", True)]   # (mode, static_only)


@pytest.fixture(scope="module")
def eng():
    from torque_constrained_motion_planning_b200 import engine
    return engine


def dev(a, dtype=None):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a if dtype is None else np.asarray(a, dtype)), device="cuda")


def _family(mode, static, model_name=None):
    return R.edge_family("nov" if static else mode, model_name)


def _runner(eng, path, mode, static):
    if path == "device":
        return lambda qa, qb, W, m: eng.edge_feasibility(dev(qa), dev(qb), W, m, mode=mode,
                                                          static_only=static).cpu().numpy()
    if path == "model":
        model = eng.InertialModel.default()
        return lambda qa, qb, W, m: eng.edge_feasibility(dev(qa), dev(qb), W, m, mode=mode, static_only=static,
                                                          model=model).cpu().numpy()
    ws = eng.Workspace(chunk_states=2)     # 3 copies of each edge straddle two chunks
    return lambda qa, qb, W, m: eng.edge_feasibility(qa, qb, W, m, mode=mode, static_only=static, workspace=ws)


@pytest.mark.parametrize("path", ["device", "model", "host"])
@pytest.mark.parametrize("mode,static", EDGE_MODES)
def test_edge_first_failure_at_boundaries(eng, mode, static, path):
    cases = _family(mode, static)
    R.check_edge_cases(cases, _runner(eng, path, mode, static))
    print("%s static=%d %s: %d cases, 0 in band" % (mode, static, path, len(cases)))


@pytest.mark.parametrize("mode,static", EDGE_MODES)
def test_edge_first_failure_at_boundaries_other_robot(eng, mode, static):
    rec = R.override_model()
    model = eng.InertialModel(rec)
    cases = _family(mode, static, "override")
    R.check_edge_cases(cases, lambda qa, qb, W, m: eng.edge_feasibility(
        dev(qa), dev(qb), W, m, mode=mode, static_only=static, model=model).cpu().numpy())


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_edge_payload_threshold(eng, mode):
    qa, qb, (m_lo, f_lo), (m_hi, f_hi) = R.threshold_edge(mode)
    for m, f in ((m_lo, f_lo), (m_hi, f_hi)):
        for model in (None, eng.InertialModel.default()):
            ff = eng.edge_feasibility(dev(qa[:, None]), dev(qb[:, None]), 64, m, mode=mode, model=model)
            assert int(ff.item()) == f, (mode, m, model)
    # payload_threshold = 0: mass 0 carries no payload, 5e-324 does (a torque change far below any margin)
    qa, qb = sample_edges(512, 60)
    for m in (0.0, 5e-324):
        ff = eng.edge_feasibility(dev(qa), dev(qb), 64, m, mode=mode, payload_threshold=0.0).cpu().numpy()
        assert np.array_equal(ff, oracle.edge_feasibility(mode, qa, qb, 64, m, 0.0))


def test_edge_scatter_two_buffers(eng):
    import torch
    from torque_constrained_motion_planning_b200 import _lib
    lib = _lib.load()
    cases = [c for c in _family("rne", False) if c.W == 64]
    n, G, off = len(cases), 64, 37
    qa = np.stack([c.qa for c in cases], 1)
    qb = np.stack([c.qb for c in cases], 1)
    # one mass for the whole launch: the local form at that mass is the reference of the scatter form
    m = cases[0].mass
    want = eng.edge_feasibility(dev(qa), dev(qb), 64, m, mode="rne").cpu().numpy()
    assert np.array_equal(want, oracle.edge_feasibility("rne", qa, qb, 64, m))
    st = torch.cuda.current_stream().cuda_stream
    a, b = dev(qa), dev(qb)
    for mode, expect in ((0, want), (3, np.full(n, 64))):
        bufs = [torch.full((off + n + 2 * G,), -1234567, dtype=torch.int32, device="cuda") for _ in range(2)]
        ptrs = (ctypes.c_void_p * 2)(*[b_.data_ptr() + 4 * G for b_ in bufs])
        _lib.check(lib.tcmp_edge_feasibility_scatter(mode, n, 64, a.data_ptr(), b.data_ptr(), m, 0.01, 0, 2, ptrs,
                                                     off, st))
        torch.cuda.synchronize()
        for b in bufs:
            h = b.cpu().numpy()
            assert (h[:G + off] == -1234567).all() and (h[G + off + n:] == -1234567).all()
            assert np.array_equal(h[G + off:G + off + n], expect)


def test_edge_grid_stride_tiles(eng):
    """The W = 33 case pattern tiled to >= 1 M edges: many passes of the edge kernel's grid."""
    cases = [c for c in _family("rne", False) if c.W == 33]
    qa = np.stack([c.qa for c in cases], 1)
    qb = np.stack([c.qb for c in cases], 1)
    # one launch has one mass: take the case mass that gives the most distinct first failures, none in the band
    best = None
    for m in sorted({c.mass for c in cases}):
        mg, _ = R.edge_reference("rne", qa, qb, 33, m)
        ff, _ = R.first_fail_from_margins(mg)
        clear = min(np.abs(mg[e, :min(f, 32) + 1]).min() for e, f in enumerate(ff))
        if clear > R.BAND and (best is None or len(set(ff.tolist())) > best[0]):
            best = (len(set(ff.tolist())), m, ff)
    _, m, want = best
    assert np.array_equal(want, oracle.edge_feasibility("rne", qa, qb, 33, m)) and best[0] >= 3
    reps = -(-(1 << 20) // len(cases))
    ff = eng.edge_feasibility(dev(np.tile(qa, reps)), dev(np.tile(qb, reps)), 33, m, mode="rne").cpu().numpy()
    assert np.array_equal(ff.reshape(reps, -1), np.broadcast_to(want, (reps, len(cases))))


@pytest.mark.parametrize("mode", ["rne", "nov", "dyn"])
def test_edge_fp32_first_failures_are_justified(eng, mode):
    """f32 edges: each first failure f has every earlier margin > -eps and (f == W or) a margin at f > +eps, eps =
    1e-4 max(|tau|, 1) on the reference of the f32-rounded endpoints; the delta = 1 N.m cases match exactly."""
    differ = 0
    for c in _family(mode, False):
        qa = c.qa.astype(np.float32)[:, None]
        qb = c.qb.astype(np.float32)[:, None]
        f = int(eng.edge_feasibility(dev(qa), dev(qb), c.W, c.mass, mode=mode, dtype="f32").item())
        mg, tau = R.edge_reference(mode, qa.astype(np.float64), qb.astype(np.float64), c.W, c.mass)
        mg, eps = mg[0], 1e-4 * np.maximum(np.abs(tau[0, :, :6]), 1.0)
        assert (mg[:f] < eps[:f]).all(), (c.W, c.first, f)
        assert f == c.W or (mg[f] > -eps[f]).any(), (c.W, c.first, f)
        if c.delta == 1.0:
            assert f == c.first
        differ += f != c.first
    print("%s: %d fp32 first failures differ from the f64 design, each justified" % (mode, differ))


# ---- trajectories ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2, 3, 6, 7, 31, 32, 33, 63, 64, 100, 1000, 4096])
def test_traj_sample_times_bit_for_bit(eng, S):
    c = np.zeros((3, 7, 6))
    c[:, :, 1] = 1.0
    for dtype, npt in (("f64", np.float64), ("f32", np.float32)):
        out = eng.traj_feasibility(c, S, 0.0, mode="rne", dtype=dtype)
        R.check_times(S, out["q"].cpu().numpy(), npt)


@pytest.mark.parametrize("mode", ["rne", "nov", "dyn"])
def test_traj_samples_within_the_long_double_bound(eng, mode):
    rng = np.random.default_rng(61)
    pts = rng.uniform(-2.5, 2.5, size=(40, 7))
    c = oracle.minjerk_coefficients(pts)
    c[::3] += rng.normal(0, 1, size=c[::3].shape)           # arbitrary caller coefficients too
    for S in (7, 64, 100):
        ref = R.traj_reference(mode, c, S, 3.0)
        out = eng.traj_feasibility(c, S, 3.0, mode=mode)
        R.check_samples(ref, *(out[k].cpu().numpy() for k in ("q", "qd", "qdd")))
        R.check_traj(ref, out["feasible"].cpu().numpy(), out["first_fail"])


def _traj_layouts(S, n_seg):
    # (designed local first failure or S for a feasible segment, segment it sits in)
    return [(0, 0), (S - 1, 0), (0, 1), (30, n_seg - 1), (S - 1, n_seg - 1), (S, n_seg // 2)]


@pytest.mark.parametrize("S,n_seg", [(64, 200), (100, 5000)])
@pytest.mark.parametrize("mode,model_name", [("rne", None), ("nov", None), ("dyn", None), ("rne", "override"),
                                             ("dyn", "override")])
def test_traj_first_failure(eng, mode, model_name, S, n_seg):
    rec = None if model_name is None else R.override_model()
    model = None if rec is None else eng.InertialModel(rec)
    by_key = {(c.W, c.first, c.delta): c for c in R.edge_family(mode, model_name) if c.W == S}
    for first_local, at_seg in _traj_layouts(S, n_seg):
        case = by_key[(S, first_local, R.DELTAS[0])]
        coeffs = R.traj_with_failure(case, S, n_seg, at_seg)
        ref = R.traj_reference(mode, coeffs, S, case.mass, model=rec)
        want = n_seg * S if first_local == S else at_seg * S + first_local
        assert ref["first_fail"] == want
        out = eng.traj_feasibility(coeffs, S, case.mass, mode=mode, want_samples=False, model=model)
        R.check_traj(ref, out["feasible"].cpu().numpy(), out["first_fail"])


def test_traj_exact_limit_compare(eng):
    """The kernel's own |tau_j(s)| as joint j's limit makes sample s infeasible; one ulp above it, feasible."""
    rng = np.random.default_rng(62)
    c = oracle.minjerk_coefficients(rng.uniform(-1.0, 1.0, size=(6, 7)) * 0.3)
    S = 50
    model = eng.InertialModel.default()
    out = eng.traj_feasibility(c, S, 2.0, mode="rne", model=model)
    tau = out["tau"].cpu().numpy()
    assert out["feasible"].cpu().numpy().all()
    for s, j in ((0, 1), (77, 3), (249, 5)):
        v = abs(float(tau[j, s]))
        for lim, ok in ((v, 0), (float(np.nextafter(v, np.inf)), 1)):
            m = eng.InertialModel.default()
            m.torque_limit[j] = lim
            o = eng.traj_feasibility(c, S, 2.0, mode="rne", model=m)
            assert int(o["feasible"][s].item()) == ok, (s, j, lim)


# ---- non-finite joint 1 -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("v", [np.nan, np.inf, -np.inf])
def test_nonfinite_joint1_gives_nan_torques_everywhere(eng, v):
    q, qd, qdd, mass = sample_states(1000, seed=63)
    q[0, ::2] = v
    bad = np.zeros(1000, bool)
    bad[::2] = True
    ws = eng.Workspace(chunk_states=300)
    for mode in ("rne", "nov", "dyn"):
        tau_o, ok_o = oracle.torque_test_batch(mode, q, qd, qdd, mass)
        assert np.isnan(tau_o[:, bad]).all() and ok_o[bad].all()
        for dtype, npt in (("f64", np.float64), ("f32", np.float32)):
            runs = [eng.torque_test_batch(dev(q, npt), dev(qd, npt), dev(qdd, npt), dev(mass, npt), mode=mode,
                                          dtype=dtype),
                    eng.torque_test_batch(dev(q, npt), dev(qd, npt), dev(qdd, npt), dev(mass, npt), mode=mode,
                                          dtype=dtype, model=eng.InertialModel.default()),
                    eng.torque_test_batch(q.astype(npt), qd.astype(npt), qdd.astype(npt), mass.astype(npt),
                                          mode=mode, dtype=dtype, workspace=ws)]
            for tau, ok in runs:
                tau = tau.cpu().numpy() if hasattr(tau, "cpu") else tau
                ok = ok.cpu().numpy() if hasattr(ok, "cpu") else ok
                assert np.isnan(tau[:, bad]).all() and ok[bad].all(), (mode, dtype)
    # edges: a non-finite joint 1 at either end makes every waypoint's torque NaN -> feasible (first failure W)
    qa, qb = sample_edges(256, 64)
    qa[0, ::3] = v
    qb[0, 1::3] = v
    for mode, static in EDGE_MODES:
        want = oracle.edge_feasibility("nov" if static else mode, qa, qb, 64, 5.0)
        ff = eng.edge_feasibility(dev(qa), dev(qb), 64, 5.0, mode=mode, static_only=static).cpu().numpy()
        assert np.array_equal(ff, want) and (ff[(np.arange(256) % 3) < 2] == 64).all(), (mode, static)
