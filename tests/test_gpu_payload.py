"""GPU: the payload-mass intervals -- K11 (tcmp_payload_interval_batch) against the host build of the same source and
against the torque kernel's verdict at probe masses; K12 (tcmp_edge_payload_interval) against the boundary edges of
tests/minjerk_reference.py and against tcmp_edge_feasibility; engine.traj_payload_interval against
tcmp_traj_feasibility; guard bands, empty batches, graph capture and a tiling of more than 1 M edges."""
import numpy as np
import pytest

import minjerk_reference as R
from conftest import load_golden, sample_edges, sample_states
from test_payload_host import BAND, CASES, PROBES, THRESHOLD, host_payload

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from torque_constrained_motion_planning_b200 import engine
    return torch, engine, torch.device("cuda", 0)


def _models(engine):
    rec = np.ascontiguousarray(load_golden("model_override.npz")["model"], np.float64)
    return {"stock": (None, None), "override": (rec, engine.InertialModel(rec))}


def _limits(rec):
    return R.limits(rec)


def _binding_tolerance(lo, hi, a, b, lim):
    """Per-state tolerances of lo / hi: 1e-12 relative, or 1e-11 N.m through |b| of the joint that sets the end."""
    with np.errstate(divide="ignore", invalid="ignore"):
        u, v = (-lim[:, None] - a[:6]) / b[:6], (lim[:, None] - a[:6]) / b[:6]
        jlo, jhi = np.where(b[:6] > 0, u, v), np.where(b[:6] > 0, v, u)
    out = []
    for e, ends in ((lo, jlo), (hi, jhi)):
        j = np.argmin(np.abs(ends - e[None]), axis=0)
        bj = np.abs(b[:6][j, np.arange(len(e))])
        with np.errstate(divide="ignore"):
            out.append(np.maximum(1e-12 * np.abs(e), 1e-11 / bj))
    return out


@pytest.mark.parametrize("model_name", ["stock", "override"])
@pytest.mark.parametrize("mode,dynamic", CASES)
def test_k11_matches_the_host_build(env, mode, dynamic, model_name):
    torch, engine, dev = env
    rec, model = _models(engine)[model_name]
    q, qd, qdd, _ = sample_states(1_000_000, seed=91)
    qd, qdd = (qd, qdd) if dynamic else (None, None)
    t = lambda a: None if a is None else torch.as_tensor(a, device=dev)
    lo, hi, ok = (x.cpu().numpy() for x in engine.payload_interval_batch(t(q), t(qd), t(qdd), mode, model))
    ref = host_payload(q, qd, qdd, mode, rec)
    lim = _limits(rec)
    for got, want in ((lo, ref["lo"]), (hi, ref["hi"])):
        inf = ~np.isfinite(want)
        assert np.array_equal(got[inf], want[inf])
    tlo, thi = _binding_tolerance(ref["lo"], ref["hi"], ref["a"], ref["b"], lim)
    fin = np.isfinite(ref["lo"])
    assert (np.abs(lo - ref["lo"])[fin] <= tlo[fin]).all()
    fin = np.isfinite(ref["hi"])
    assert (np.abs(hi - ref["hi"])[fin] <= thi[fin]).all()
    band = (np.abs(np.abs(ref["a"][:6]) - lim[:, None]) < BAND).any(0)
    assert np.array_equal(ok[~band], ref["ok"][~band])
    print("%s dynamic=%d %s: %d states in the band" % (mode, dynamic, model_name, int(band.sum())))


@pytest.mark.parametrize("model_name", ["stock", "override"])
@pytest.mark.parametrize("mode,dynamic", CASES)
def test_k11_predicts_the_torque_kernel_at_probe_masses(env, mode, dynamic, model_name):
    """tcmp_rne_batch[_model] at every probe mass (threshold 0.01) gives the verdict payload_passes predicts."""
    torch, engine, dev = env
    rec, model = _models(engine)[model_name]
    q, qd, qdd, _ = (torch.as_tensor(a, device=dev) for a in sample_states(1_000_000, seed=92))
    qd, qdd = (qd, qdd) if dynamic else (None, None)
    lo, hi, ok = engine.payload_interval_batch(q, qd, qdd, mode, model)
    lim = torch.as_tensor(_limits(rec), device=dev)
    probes = list(PROBES)
    for e in (lo, hi):
        for f in (1 - 1e-6, 1 + 1e-6):
            probes.append(torch.where(torch.isfinite(e), e * f, torch.ones_like(e)))
    skipped = 0
    for m in probes:
        tau, got = engine.torque_test_batch(q, qd, qdd, m, mode=mode, payload_threshold=THRESHOLD, model=model)
        band = ((tau[:6].abs() - lim[:, None]).abs() < BAND).any(0)
        want = engine.payload_passes(lo, hi, ok, m, mode, THRESHOLD)
        assert torch.equal(got.bool()[~band], want[~band]), (mode, m if np.ndim(m) == 0 else "endpoint")
        skipped += int(band.sum())
    print("%s dynamic=%d %s: %d of %d probes in the band" % (mode, dynamic, model_name, skipped, 15 * q.shape[1]))


def test_k11_numpy_in_numpy_out_and_base(env):
    torch, engine, dev = env
    q, qd, qdd, _ = sample_states(1000, seed=93)
    lo, hi, ok = engine.payload_interval_batch(q, qd, qdd, "rne")
    assert isinstance(lo, np.ndarray) and ok.dtype == np.uint8
    ref = host_payload(q, qd, qdd, "rne")
    assert np.abs(lo - ref["lo"]).max() <= 1e-9 and np.array_equal(ok, ref["ok"])
    blo, bhi, bok = engine.payload_interval_batch(q, mode="base")
    assert (blo == -np.inf).all() and (bhi == np.inf).all() and (bok == 1).all()
    elo, ehi, eok = engine.edge_payload_interval(q, q, 8, mode="base")
    assert (elo == -np.inf).all() and (ehi == np.inf).all() and (eok == 1).all()
    assert (engine.max_payload(blo, bhi, bok, "base") == np.inf).all()


# ---- K12 -------------------------------------------------------------------------------------------------------------
EDGE_MODES = [("rne", False), ("nov", False), ("dyn", False), ("rne", True)]


def _check_cases(engine, torch, cases, mode, static, model=None):
    for case in cases:
        t = lambda a: torch.as_tensor(np.repeat(a[:, None], 3, 1), device="cuda")
        lo, hi, ok = (x.cpu().numpy() for x in engine.edge_payload_interval(t(case.qa), t(case.qb), case.W, mode,
                                                                            static, model))
        passes = engine.payload_passes(lo, hi, ok, case.mass, mode, THRESHOLD)
        assert (passes == (case.first == case.W)).all(), (mode, static, case.W, case.first, case.delta, case.mass,
                                                          lo, hi)


@pytest.mark.parametrize("mode,static", EDGE_MODES)
def test_k12_against_the_boundary_edges(env, mode, static):
    torch, engine, _ = env
    cases = R.edge_family("nov" if static else mode)
    _check_cases(engine, torch, cases, mode, static)
    print("%s static=%d: %d cases" % (mode, static, len(cases)))


@pytest.mark.parametrize("mode,static", EDGE_MODES)
def test_k12_against_the_boundary_edges_other_robot(env, mode, static):
    torch, engine, _ = env
    model = engine.InertialModel(R.override_model())
    _check_cases(engine, torch, R.edge_family("nov" if static else mode, "override"), mode, static, model)


def _edge_samples(engine, qa, qb, W, static):
    """The edges' min-jerk samples [7][n W] (traj kernel on the edges' coefficients)."""
    s = engine.traj_feasibility(R.edge_coeffs(qa, qb), W, mode="base", want_tau=False)
    return s["q"], (None if static else s["qd"]), (None if static else s["qdd"])


@pytest.mark.parametrize("model_name", ["stock", "override"])
@pytest.mark.parametrize("mode,static", EDGE_MODES)
def test_k12_predicts_the_edge_kernel(env, mode, static, model_name):
    """On 10 k random edges x the probe masses: tcmp_edge_feasibility(..., m) == W iff payload_passes, outside the
    band (the band from the torques of the same samples)."""
    torch, engine, dev = env
    rec, model = _models(engine)[model_name]
    W, n = 64, 10_000
    qa, qb = sample_edges(n, seed=94)
    a, b = torch.as_tensor(qa, device=dev), torch.as_tensor(qb, device=dev)
    lo, hi, ok = engine.edge_payload_interval(a, b, W, mode, static, model)
    sq, sv, sa = _edge_samples(engine, qa, qb, W, static)
    lim = torch.as_tensor(_limits(rec), device=dev)
    skipped = 0
    for m in PROBES:
        ff = engine.edge_feasibility(a, b, W, m, mode=mode, payload_threshold=THRESHOLD, static_only=static,
                                     model=model)
        tau, _ = engine.torque_test_batch(sq, sv, sa, m, mode="nov" if mode == "rne" and static else mode,
                                          payload_threshold=THRESHOLD, want_mask=False, model=model)
        band = ((tau[:6].abs() - lim[:, None]).abs() < BAND).any(0).reshape(n, W).any(1)
        want = engine.payload_passes(lo, hi, ok, m, mode, THRESHOLD)
        assert torch.equal((ff == W)[~band], want[~band]), (mode, static, m)
        skipped += int(band.sum())
    print("%s static=%d %s: %d of %d edge probes in the band" % (mode, static, model_name, skipped, n * len(PROBES)))


@pytest.mark.parametrize("mode", ["rne", "nov", "dyn"])
def test_traj_payload_interval_predicts_the_trajectory_kernel(env, mode):
    torch, engine, dev = env
    S, n_seg = 33, 40
    qa, qb = sample_edges(n_seg, seed=95)
    coeffs = R.edge_coeffs(qa, qb)
    lo, hi, ok = engine.traj_payload_interval(coeffs, S, mode)
    assert isinstance(lo, float) and isinstance(ok, int)
    lim = torch.as_tensor(R.limits(), device=dev)
    checked = 0
    for m in list(PROBES) + [x * f for x in (lo, hi) if np.isfinite(x) for f in (1 - 1e-6, 1 + 1e-6)]:
        r = engine.traj_feasibility(coeffs, S, m, mode=mode, payload_threshold=THRESHOLD, want_samples=False)
        if ((r["tau"][:6].abs() - lim[:, None]).abs() < BAND).any():
            continue
        want = bool(engine.payload_passes(np.array([lo]), np.array([hi]), np.array([ok]), m, mode, THRESHOLD)[0])
        assert (r["first_fail"] == n_seg * S) == want, (mode, m, lo, hi, ok)
        checked += 1
    assert checked >= len(PROBES)


# ---- guards and stress -----------------------------------------------------------------------------------------------
def _guarded(torch, n, dtype, off=37, tail=41):
    buf = torch.full((off + n + tail,), float("nan") if dtype == torch.float64 else 0xAB, dtype=dtype, device="cuda")
    return buf, buf[off:off + n]


def test_outputs_touch_nothing_outside_their_views(env):
    torch, engine, dev = env
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr
    lib = _lib.load()
    n = 1000
    q, qd, qdd, _ = (torch.as_tensor(a, device=dev) for a in sample_states(n, seed=96))
    ref = engine.payload_interval_batch(q, qd, qdd, "dyn")
    eref = engine.edge_payload_interval(q, qd, 33, "rne")
    for call, want in ((lambda o: lib.tcmp_payload_interval_batch(None, 2, n, _ptr(q), _ptr(qd), _ptr(qdd), *o,
                                                                   engine._stream_ptr()), ref),
                       (lambda o: lib.tcmp_edge_payload_interval(None, 0, n, 33, _ptr(q), _ptr(qd), 0, *o,
                                                                  engine._stream_ptr()), eref)):
        (blo, vlo), (bhi, vhi), (bok, vok) = (_guarded(torch, n, torch.float64), _guarded(torch, n, torch.float64),
                                              _guarded(torch, n, torch.uint8))
        _lib.check(call([_ptr(vlo), _ptr(vhi), _ptr(vok)]))
        torch.cuda.synchronize()
        for buf, view, w in ((blo, vlo, want[0]), (bhi, vhi, want[1]), (bok, vok, want[2])):
            assert torch.equal(view, w)
            rest = torch.cat([buf[:37], buf[37 + n:]])
            assert (rest.isnan().all() if buf.dtype == torch.float64 else (rest == 0xAB).all())
        # one output at a time: the others stay untouched
        for k in range(3):
            bufs = [_guarded(torch, n, torch.float64), _guarded(torch, n, torch.float64), _guarded(torch, n, torch.uint8)]
            _lib.check(call([_ptr(bufs[i][1]) if i == k else None for i in range(3)]))
            torch.cuda.synchronize()
            for i, (buf, view) in enumerate(bufs):
                if i == k:
                    assert torch.equal(view, want[i])
                else:
                    assert (buf.isnan().all() if buf.dtype == torch.float64 else (buf == 0xAB).all())


def test_empty_batches_with_null_buffers(env):
    torch, engine, _ = env
    from torque_constrained_motion_planning_b200 import _lib
    lib = _lib.load()
    for mode in range(4):
        assert lib.tcmp_payload_interval_batch(None, mode, 0, None, None, None, None, None, None, None) == 0
        assert lib.tcmp_edge_payload_interval(None, mode, 0, 64, None, None, 0, None, None, None, None) == 0
    empty = torch.empty((7, 0), dtype=torch.float64, device="cuda")
    lo, hi, ok = engine.payload_interval_batch(empty)
    assert lo.numel() == hi.numel() == ok.numel() == 0
    assert engine.edge_payload_interval(empty, empty)[0].numel() == 0


def test_graph_capture_and_replay(env):
    torch, engine, dev = env
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr
    lib = _lib.load()
    n = 100_000
    q, qd, qdd, _ = (torch.as_tensor(a, device=dev) for a in sample_states(n, seed=97))
    model = engine.InertialModel(R.override_model())
    outs = [torch.empty((n,), dtype=torch.float64, device=dev) for _ in range(4)] + \
        [torch.empty((n,), dtype=torch.uint8, device=dev) for _ in range(2)]
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        _lib.check(lib.tcmp_payload_interval_batch(model.record.ctypes.data, 0, n, _ptr(q), _ptr(qd), _ptr(qdd),
                                                   _ptr(outs[0]), _ptr(outs[1]), _ptr(outs[4]), int(side.cuda_stream)))
        _lib.check(lib.tcmp_edge_payload_interval(None, 2, n, 64, _ptr(q), _ptr(qd), 0, _ptr(outs[2]), _ptr(outs[3]),
                                                  _ptr(outs[5]), int(side.cuda_stream)))
    for o in outs:
        o.fill_(0)
    g.replay()
    torch.cuda.synchronize()
    r1 = engine.payload_interval_batch(q, qd, qdd, "rne", model)
    r2 = engine.edge_payload_interval(q, qd, 64, "dyn")
    for o, w in zip(outs, (r1[0], r1[1], r2[0], r2[1], r1[2], r2[2])):
        assert torch.equal(o, w)


def test_tiling_beyond_one_million_edges(env):
    """>= 1 M edges at W = 33 (the grid-stride loop over edges runs many times): every copy equals its original."""
    torch, engine, dev = env
    base, copies = 1000, 1001
    qa, qb = sample_edges(base, seed=98)
    a, b = torch.as_tensor(qa, device=dev), torch.as_tensor(qb, device=dev)
    want = engine.edge_payload_interval(a, b, 33, "rne")
    got = engine.edge_payload_interval(a.repeat(1, copies), b.repeat(1, copies), 33, "rne")
    assert got[0].numel() == base * copies >= 1_000_000
    for g, w in zip(got, want):
        assert torch.equal(g.reshape(copies, base), w.expand(copies, base))
