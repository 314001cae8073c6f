"""GPU: K15 (tcmp_track_batch, engine.track_batch) against its host build (tests/native/track_host.cpp) on 1 M
rollouts and against the composition on the device (K1 torque test + torch clamp + K14 one step at a time); output
subsets, tiled per-rollout coefficients against shared ones, the empty batch, CUDA-graph capture, the 64-bit offset
path and the torque test's designed edge cases."""
import numpy as np
import pytest

from conftest import Q_HI, Q_LO, V_LIM, sample_states
from test_rollout_host import MODELS, limits, model_record
from test_tracking_host import KD, KP, check_edge_saturation, edge_chain, host_track, load_track_host, reference

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

N_BIG, T_BIG, DT = 1 << 20, 16, 1e-3
HOST_STRIDE = 128
BAND = 1e-6                # N.m: a commanded torque this close to its limit may saturate on one side and not the other


@pytest.fixture(scope="module")
def eng():
    from torque_constrained_motion_planning_b200 import engine
    return engine


@pytest.fixture(scope="module")
def L():
    return load_track_host()


def cuda(*arrs):
    return [None if a is None else (torch.as_tensor(a, device="cuda") if np.ndim(a) else a) for a in arrs]


def _model(eng, name):
    rec = model_record(name)
    return None if rec is None else eng.InertialModel(rec)


def track_inputs(n, seed):
    coeffs = edge_chain(n, seed, n_seg=1)
    x0, v0, _ = reference(coeffs, 0.0, n)
    q, qd, _, mass = sample_states(n, seed + 7)
    return coeffs, x0 + 0.02 * np.tanh(q), v0 + 0.05 * np.tanh(qd), mass


def near_limit(tau, lim):
    """[T][7][n] applied torques -> [n]: some joint of some step within BAND of its limit (saturated or not)."""
    return (np.abs(np.abs(tau) - np.asarray(lim)[None, :, None]) < BAND).any(axis=(0, 1))


@pytest.mark.parametrize("mode", ["rne", "dyn"])
@pytest.mark.parametrize("model_name", list(MODELS))
def test_k15_matches_host_on_1m_rollouts(eng, L, mode, model_name):
    rec = model_record(model_name)
    coeffs, q0, qd0, mass = track_inputs(N_BIG, 600)
    ctrl = np.where(mass > 0, mass - 0.5, 0.0)
    cg, q0g, qd0g, mg, cmg = cuda(coeffs, q0, qd0, mass, ctrl)
    out = eng.track_batch(cg, DT, T_BIG, KP, KD, q0g, qd0g, mg, cmg, mode, Q_LO, Q_HI, V_LIM, trajectory=True,
                          model=_model(eng, model_name))
    torch.cuda.synchronize()
    sub = slice(0, None, HOST_STRIDE)
    host = host_track(L, np.ascontiguousarray(coeffs[..., sub]), DT, T_BIG, KP, KD, q0[:, sub], qd0[:, sub],
                      mass[sub], ctrl[sub], mode, Q_LO, Q_HI, V_LIM, rec)
    g = {k: v[..., sub].cpu().numpy() for k, v in out.items()}
    # a rollout may saturate on one side and not the other only where its commanded torque lies within BAND of a limit
    # at the first step that differs: there one side's applied torque is +-L, the other's unsaturated and within BAND
    lim = np.asarray(limits(rec))
    split = (g["first_saturation"] != host["first_saturation"]) | (g["first_violation"] != host["first_violation"])
    for i in np.nonzero(split)[0]:
        k = min(g["first_saturation"][i], host["first_saturation"][i])
        assert k < T_BIG, ("first_violation differs without a saturation", i)
        near = np.abs(np.abs(host["tau_traj"][k, :, i]) - lim) < BAND
        assert near.any(), (i, k, host["tau_traj"][k, :, i], g["tau_traj"][k, :, i])
    keep = ~split
    err = 0.0
    for key in ("q_traj", "qd_traj", "tau_traj", "max_err"):
        a, b = g[key][..., keep], host[key][..., keep]
        err = max(err, float((np.abs(a - b) / (1.0 + np.abs(b))).max()))
    sat = host["first_saturation"] < T_BIG
    print("K15 vs host %s %s: max rel %.3e over %d rollouts, %d of them saturating; %d split at a limit (within %.0e "
          "N.m) set aside" % (mode, model_name, err, keep.sum(), (sat & keep).sum(), split.sum(), BAND))
    assert err <= 1e-9
    assert torch.equal(out["q_traj"][-1], out["q"]) and torch.equal(out["qd_traj"][-1], out["qd"])


def composed(eng, coeffs, q, qd, mass, ctrl, mode, model, lim, T):
    """K1 (threshold 0) for the controller torque, a torch clamp, K14 one step at a time."""
    n = q.shape[1]
    L7 = torch.as_tensor(lim, device="cuda")[:, None]
    kp, kd = (torch.as_tensor(g, device="cuda")[:, None] for g in (KP, KD))
    c = [coeffs[0, :, k] for k in range(6)]
    fs = torch.full((n,), T, dtype=torch.int32, device="cuda")
    for k in range(T):
        u = k * DT
        x = c[0] + u * (c[1] + u * (c[2] + u * (c[3] + u * (c[4] + u * c[5]))))
        v = c[1] + u * (2.0 * c[2] + u * (3.0 * c[3] + u * (4.0 * c[4] + u * (5.0 * c[5]))))
        a = 2.0 * c[2] + u * (6.0 * c[3] + u * (12.0 * c[4] + u * (20.0 * c[5])))
        acmd = (a + kp * (x - q)) + kd * (v - qd)
        tau, _ = eng.torque_test_batch(q, qd, acmd, ctrl, mode, payload_threshold=0.0, model=model)
        over = tau.abs() > L7
        fs = torch.where(over.any(0) & (fs == T), torch.full_like(fs, k), fs)
        tau = torch.where(over, torch.copysign(L7.expand_as(tau), tau), tau)
        o = eng.rollout_batch(q, qd, tau, DT, 1, mass, mode, model=model)
        q, qd = o["q"], o["qd"]
    return q, qd, fs


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_k15_matches_the_composition_on_the_device(eng, mode):
    n, T = 65536, 16
    coeffs, q0, qd0, mass = track_inputs(n, 610)
    cg, q0g, qd0g, mg = cuda(coeffs, q0, qd0, mass)
    out = eng.track_batch(cg, DT, T, KP, KD, q0g, qd0g, mg, 1.0, mode, trajectory=True)
    cq, cv, cfs = composed(eng, cg, q0g, qd0g, mg, torch.full((n,), 1.0, dtype=torch.float64, device="cuda"), mode,
                           None, limits(None), T)
    band = torch.as_tensor(near_limit(out["tau_traj"].cpu().numpy(), limits(None)), device="cuda")
    keep = ~band
    rel = lambda a, b: float(((a - b).abs() / (1.0 + b.abs()))[:, keep].max())
    d = max(rel(out["q"], cq), rel(out["qd"], cv))
    print("K15 vs composed K1 + clamp + K14 %s: max rel %.3e; first_saturation differs on %d of %d (within %.0e N.m "
          "of a limit: %d)" % (mode, d, int((out["first_saturation"] != cfs).sum()), n, BAND, int(band.sum())))
    assert d <= 1e-9
    assert not ((out["first_saturation"] != cfs) & keep).any()


def test_output_subsets_and_tiled_coefficients(eng):
    n, T = 40_000, 12
    coeffs, q0, qd0, mass = track_inputs(n, 620)
    cg, q0g, qd0g, mg = cuda(coeffs, q0, qd0, mass)
    full = eng.track_batch(cg, DT, T, KP, KD, q0g, qd0g, mg, 0.5, q_lo=Q_LO, q_hi=Q_HI, qd_max=V_LIM, trajectory=True)
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr, _stream_ptr
    lib = _lib.load()
    kp, kd = np.ascontiguousarray(KP), np.ascontiguousarray(KD)
    for want in ("max_err", "first_saturation", "tau_traj", "q"):
        o = torch.empty_like(full[want])
        outs = {k: None for k in ("q", "qd", "q_traj", "qd_traj", "tau_traj", "first_violation", "first_saturation",
                                  "max_err")}
        outs[want] = o
        _lib.check(lib.tcmp_track_batch(None, 0, n, T, DT, 1, _ptr(cg), 0, _ptr(q0g), _ptr(qd0g), kp.ctypes.data,
                                        kd.ctypes.data, _ptr(mg), 0.0, None, 0.5, None, None, None,
                                        *(_ptr(outs[k]) for k in outs), _stream_ptr()))
        assert torch.equal(o, full[want]), want
    # one shared trajectory: tiled per-rollout coefficients give the same result bit for bit
    one = np.ascontiguousarray(coeffs[..., 5])
    tiled = torch.as_tensor(np.ascontiguousarray(np.broadcast_to(one[..., None], one.shape + (n,))), device="cuda")
    shared = eng.track_batch(torch.as_tensor(one, device="cuda"), DT, T, KP, KD, None, qd0g, mg, 0.5, trajectory=True)
    per = eng.track_batch(tiled, DT, T, KP, KD, None, qd0g, mg, 0.5, trajectory=True)
    for k in shared:
        if shared[k] is not None:
            assert torch.equal(shared[k], per[k]), k


def test_empty_batch_and_graph_capture(eng):
    c = torch.zeros((1, 7, 6), dtype=torch.float64, device="cuda")
    e = eng.track_batch(c, DT, 3, KP, KD, n=0, q_lo=Q_LO, q_hi=Q_HI, trajectory=True)
    assert e["q"].shape == (7, 0) and e["tau_traj"].shape == (3, 7, 0) and e["max_err"].shape == (0,)
    n, T = 20_000, 6
    coeffs, q0, qd0, mass = track_inputs(n, 630)
    cg, q0g, qd0g, mg = cuda(coeffs, q0, qd0, mass)
    ref = eng.track_batch(cg, DT, T, KP, KD, q0g, qd0g, mg, 2.0, q_lo=Q_LO, q_hi=Q_HI, trajectory=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eng.track_batch(cg, DT, T, KP, KD, q0g, qd0g, mg, 2.0, q_lo=Q_LO, q_hi=Q_HI, trajectory=True)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = eng.track_batch(cg, DT, T, KP, KD, q0g, qd0g, mg, 2.0, q_lo=Q_LO, q_hi=Q_HI, trajectory=True)
    g.replay()
    torch.cuda.synchronize()
    for k in ref:
        if ref[k] is not None:
            assert torch.equal(out[k], ref[k]), k


def test_64bit_offset_path(eng):
    """80 k rollouts x 4000 steps of trajectory: 7 n T > 2^31, so the kernel runs on 64-bit offsets; a slice of the
    same rollouts on its own (32-bit offsets) gives the same results bit for bit."""
    n, T = 80_000, 4000
    assert 7 * n * T > 2 ** 31
    coeffs, q0, qd0, mass = track_inputs(n, 640)
    cg, q0g, qd0g, mg = cuda(coeffs, q0, qd0, mass)
    big = eng.track_batch(cg, DT, T, KP, KD, q0g, qd0g, mg, trajectory=True)
    cols = torch.arange(n - 512, n, device="cuda")
    small = eng.track_batch(cg[..., cols].contiguous(), DT, T, KP, KD, q0g[:, cols].contiguous(),
                            qd0g[:, cols].contiguous(), mg[cols].contiguous(), trajectory=True)
    for k in small:
        if small[k] is not None:
            assert torch.equal(big[k][..., cols], small[k]), k


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_saturation_against_the_torque_tests_edge_cases_on_k15(eng, mode):
    """CPU check 5 on the device: each designed edge as a one-segment reference, dt = 1/W, W + 1 steps, kp = kd = 0."""
    def run(c, dt, T, mass, model):
        o = eng.track_batch(torch.as_tensor(c, device="cuda"), dt, T, 0.0, 0.0, payload_mass=mass, mode=mode,
                            trajectory=True, model=None if model is None else eng.InertialModel(model))
        return o["tau_traj"][:, :, 0].cpu().numpy(), int(o["first_saturation"][0])
    used, excluded = check_edge_saturation(run, mode)
    print("%s on K15: %d designed edge cases checked, %d excluded by the preconditions" % (mode, used, excluded))
    assert used >= 10
