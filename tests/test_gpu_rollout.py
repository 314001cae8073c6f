"""GPU: K14 (tcmp_rollout_batch, engine.rollout_batch) against its host build (tests/native/rollout_host.cpp) and
against the composition of K13 launches with torch RK4 updates; output subsets, per-step torque, the limit compare at
its exact boundary on K14's own trajectory, guard bands, the empty batch, CUDA-graph capture and the 64-bit offset
path."""
import numpy as np
import pytest

from conftest import Q_HI, Q_LO, V_LIM, sample_states
from test_rollout_host import (MODELS, check_limit_boundaries, first_violation, host_rollout, load_rollout_host,
                               model_record, rollout_inputs)

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

N_BIG, T_BIG, DT = 1 << 20, 16, 1e-3
HOST_STRIDE = 128          # the host build checks every 128th of the 1 M rollouts


@pytest.fixture(scope="module")
def eng():
    from torque_constrained_motion_planning_b200 import engine
    return engine


@pytest.fixture(scope="module")
def L():
    return load_rollout_host()


def cuda(*arrs):
    return [None if a is None else (torch.as_tensor(a, device="cuda") if np.ndim(a) else a) for a in arrs]


def _model(eng, name):
    rec = model_record(name)
    return None if rec is None else eng.InertialModel(rec)


def composed(eng, q, qd, tau, mass, mode, model, dt, T):
    """4 T K13 launches and the RK4 updates as torch element-wise ops, in include/tcmp.h's order."""
    f = lambda a, b: eng.forward_dynamics_batch(a, b, tau, mass, mode, model=model)["qdd"]
    h2, h6 = 0.5 * dt, dt / 6.0
    for _ in range(T):
        a1 = f(q, qd)
        q2, v2 = q + h2 * qd, qd + h2 * a1
        a2 = f(q2, v2)
        q3, v3 = q + h2 * v2, qd + h2 * a2
        a3 = f(q3, v3)
        q4, v4 = q + dt * v3, qd + dt * a3
        a4 = f(q4, v4)
        q, qd = q + h6 * (((qd + 2 * v2) + 2 * v3) + v4), qd + h6 * (((a1 + 2 * a2) + 2 * a3) + a4)
    return q, qd


def rel(a, b):
    return float(((a - b).abs() / (1.0 + b.abs())).max())


@pytest.mark.parametrize("mode", ["rne", "dyn"])
@pytest.mark.parametrize("model_name", list(MODELS))
def test_k14_matches_host_and_composition_on_1m_rollouts(eng, L, mode, model_name):
    model = _model(eng, model_name)
    q, qd, tau, mass = rollout_inputs(N_BIG, 400, model_record(model_name))
    qg, qdg, taug, mg = cuda(q, qd, tau, mass)
    out = eng.rollout_batch(qg, qdg, taug, DT, T_BIG, mg, mode, q_lo=Q_LO, q_hi=Q_HI, qd_max=V_LIM,
                            trajectory=True, model=model)
    torch.cuda.synchronize()
    sub = slice(0, None, HOST_STRIDE)
    host = host_rollout(L, q[:, sub], qd[:, sub], tau[:, sub], DT, T_BIG, mass[sub], mode, False, Q_LO, Q_HI, V_LIM,
                        model_record(model_name))
    err = 0.0
    for key in ("q_traj", "qd_traj"):
        g = out[key][:, :, sub].cpu().numpy()
        err = max(err, float((np.abs(g - host[key]) / (1.0 + np.abs(host[key]))).max()))
    print("K14 vs host %s %s: max rel %.3e" % (mode, model_name, err))
    assert err <= 1e-9
    # first_violation against K14's own trajectory
    fv = first_violation(out["q_traj"].cpu().numpy(), out["qd_traj"].cpu().numpy(), Q_LO, Q_HI, V_LIM)
    assert np.array_equal(out["first_violation"].cpu().numpy(), fv)
    cq, cv = composed(eng, qg, qdg, taug, mg, mode, model, DT, T_BIG)
    d = max(rel(out["q"], cq), rel(out["qd"], cv))
    print("K14 vs composed K13 RK4 %s %s: max rel %.3e" % (mode, model_name, d))
    assert d <= 1e-9
    # the last trajectory slice is the final state, bit for bit
    assert torch.equal(out["q_traj"][-1], out["q"]) and torch.equal(out["qd_traj"][-1], out["qd"])


def test_output_subsets_and_per_step_torque(eng):
    n, T = 50_000, 9
    q, qd, tau, mass = cuda(*rollout_inputs(n, 410))
    full = eng.rollout_batch(q, qd, tau, DT, T, mass, q_lo=Q_LO, q_hi=Q_HI, qd_max=V_LIM, trajectory=True)
    only_final = eng.rollout_batch(q, qd, tau, DT, T, mass)
    assert only_final["q_traj"] is None and only_final["first_violation"] is None
    assert torch.equal(only_final["q"], full["q"]) and torch.equal(only_final["qd"], full["qd"])
    per_step = eng.rollout_batch(q, qd, tau.unsqueeze(0).expand(T, 7, n).contiguous(), DT, T, mass,
                                 tau_per_step=True, q_lo=Q_LO, q_hi=Q_HI, qd_max=V_LIM, trajectory=True)
    for k in full:
        assert torch.equal(per_step[k], full[k]), k
    # one output alone, through the C ABI
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr, _stream_ptr
    lib = _lib.load()
    lim = [np.ascontiguousarray(a) for a in (Q_LO, Q_HI, V_LIM)]
    fv = torch.empty(n, dtype=torch.int32, device="cuda")
    qt = torch.empty((T, 7, n), dtype=torch.float64, device="cuda")
    _lib.check(lib.tcmp_rollout_batch(None, 0, n, T, DT, _ptr(q), _ptr(qd), _ptr(tau), 0, _ptr(mass), 0.0,
                                      *(a.ctypes.data for a in lim), None, None, None, None, _ptr(fv), _stream_ptr()))
    _lib.check(lib.tcmp_rollout_batch(None, 0, n, T, DT, _ptr(q), _ptr(qd), _ptr(tau), 0, _ptr(mass), 0.0,
                                      None, None, None, None, None, _ptr(qt), None, None, _stream_ptr()))
    assert torch.equal(fv, full["first_violation"]) and torch.equal(qt, full["q_traj"])


def test_limit_compare_at_its_exact_boundary_on_k14(eng):
    T = 8

    def run(q, qd, tau, m):
        o = eng.rollout_batch(*cuda(q, qd, tau), DT, T, torch.as_tensor(m, device="cuda"), trajectory=True)
        return o["q_traj"].cpu().numpy(), o["qd_traj"].cpu().numpy()

    def run_fv(x, lo, hi, vm):
        if lo is None and vm is None:
            return np.full(x[0].shape[1], T)       # engine returns None: nothing checked
        o = eng.rollout_batch(*cuda(*x[:3]), DT, T, torch.as_tensor(x[3], device="cuda"), q_lo=lo, q_hi=hi,
                              qd_max=vm)
        return o["first_violation"].cpu().numpy()

    check_limit_boundaries(run, run_fv, T, 340)
    # through the C ABI: first_violation requested with every limit pointer NULL (no check) is n_steps; with limits
    # that cannot fail it is n_steps too
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr, _stream_ptr
    lib = _lib.load()
    q, qd, tau, mass = cuda(*rollout_inputs(64, 420))
    fv = torch.full((64,), -1, dtype=torch.int32, device="cuda")
    _lib.check(lib.tcmp_rollout_batch(None, 0, 64, T, DT, _ptr(q), _ptr(qd), _ptr(tau), 0, _ptr(mass), 0.0, None,
                                      None, None, None, None, None, None, _ptr(fv), _stream_ptr()))
    assert (fv.cpu().numpy() == T).all()
    o = eng.rollout_batch(q, qd, tau, DT, T, mass, q_lo=np.full(7, -np.inf), q_hi=np.full(7, np.inf))
    assert (o["first_violation"].cpu().numpy() == T).all()


def test_nan_states_violate_on_k14(eng):
    q, qd, tau, mass = rollout_inputs(8, 350, n_steps=6, per_step=True)
    tau[3, 2, 5] = np.nan
    inf = np.full(7, np.inf)
    q, qd, tau, mass = cuda(q, qd, tau, mass)
    o = eng.rollout_batch(q, qd, tau, DT, 6, mass, tau_per_step=True, q_lo=-inf, q_hi=inf,
                          trajectory=True)
    fv = o["first_violation"].cpu().numpy()
    assert fv[5] == 3 and (np.delete(fv, 5) == 6).all()
    assert torch.isnan(o["q_traj"][3:, :, 5]).all() and torch.isfinite(o["q_traj"][:3, :, 5]).all()


def test_guard_bands_around_offset_views(eng):
    n, T, pad = 3000, 5, 37
    q, qd, tau, mass = cuda(*rollout_inputs(n, 430))
    ref = eng.rollout_batch(q, qd, tau, DT, T, mass, q_lo=Q_LO, q_hi=Q_HI, qd_max=V_LIM, trajectory=True)
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr, _stream_ptr
    lib = _lib.load()
    bufs = {k: torch.full((v.numel() + 2 * pad,), -7, dtype=v.dtype, device="cuda") for k, v in ref.items()}
    views = {k: bufs[k][pad:pad + ref[k].numel()] for k in ref}
    lim = [np.ascontiguousarray(a) for a in (Q_LO, Q_HI, V_LIM)]
    _lib.check(lib.tcmp_rollout_batch(None, 0, n, T, DT, _ptr(q), _ptr(qd), _ptr(tau), 0, _ptr(mass), 0.0,
                                      *(a.ctypes.data for a in lim), _ptr(views["q"]), _ptr(views["qd"]),
                                      _ptr(views["q_traj"]), _ptr(views["qd_traj"]), _ptr(views["first_violation"]),
                                      _stream_ptr()))
    for k in ref:
        assert torch.equal(views[k].view(ref[k].shape), ref[k]), k
        assert (bufs[k][:pad] == -7).all() and (bufs[k][-pad:] == -7).all(), k


def test_empty_batch_and_graph_capture(eng):
    e = eng.rollout_batch(torch.empty((7, 0), dtype=torch.float64, device="cuda"), n_steps=3, q_lo=Q_LO, q_hi=Q_HI,
                          trajectory=True)
    assert e["q"].shape == (7, 0) and e["q_traj"].shape == (3, 7, 0) and e["first_violation"].shape == (0,)
    n, T = 20_000, 6
    q, qd, tau, mass = cuda(*rollout_inputs(n, 440))
    ref = eng.rollout_batch(q, qd, tau, DT, T, mass, q_lo=Q_LO, q_hi=Q_HI, trajectory=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eng.rollout_batch(q, qd, tau, DT, T, mass, q_lo=Q_LO, q_hi=Q_HI, trajectory=True)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = eng.rollout_batch(q, qd, tau, DT, T, mass, q_lo=Q_LO, q_hi=Q_HI, trajectory=True)
    g.replay()
    torch.cuda.synchronize()
    for k in ref:
        if ref[k] is not None:
            assert torch.equal(out[k], ref[k]), k


def test_64bit_offset_path(eng):
    """80 k rollouts x 4000 steps of trajectory: 7 n T > 2^31, so the kernel runs on 64-bit offsets; a slice of the
    same rollouts on its own (32-bit offsets) gives the same trajectory bit for bit."""
    n, T = 80_000, 4000
    assert 7 * n * T > 2 ** 31
    q, qd, _, mass = sample_states(n, seed=450)
    z = np.zeros_like(q)
    import oracle
    tau, _ = oracle.torque_test_batch("rne", q, z, z, mass, payload_threshold=0.0)   # gravity held: slow motion
    q, qd, tau, mass = cuda(q, 0.1 * qd, tau, mass)
    big = eng.rollout_batch(q, qd, tau, DT, T, mass, q_lo=Q_LO, q_hi=Q_HI, trajectory=True)
    cols = torch.arange(n - 512, n, device="cuda")
    small = eng.rollout_batch(q[:, cols].contiguous(), qd[:, cols].contiguous(), tau[:, cols].contiguous(), DT, T,
                              mass[cols].contiguous(), q_lo=Q_LO, q_hi=Q_HI, trajectory=True)
    for k in ("q", "qd", "first_violation"):
        assert torch.equal(big[k][..., cols], small[k]), k
    for k, final in (("q_traj", "q"), ("qd_traj", "qd")):
        assert torch.equal(big[k][:, :, cols], small[k]), k
        assert torch.equal(big[k][-1], big[final]), k
