"""GPU: K13 (tcmp_forward_dynamics_batch) against the host build of the same source, as the inverse of the pinned
torque kernels (K1 / K3, K1m for a caller record, at threshold 0), M^-1 against K10's M, output subsets, batch sizes
with guard bands, graph capture, the 64-bit offset path, the non-finite and singular-record rules and the
panda_dynamics_model drop-in."""
import ctypes

import numpy as np
import pytest

from conftest import load_golden, sample_states
from test_forward_dynamics_host import (STOCK_LIMIT, check_nonfinite_rules, host_fd, limits, load_fd_host,
                                        nonfinite_cases, tail_record)

pytestmark = pytest.mark.gpu
MODE = {"rne": 0, "dyn": 2}


@pytest.fixture(scope="module")
def env():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from torque_constrained_motion_planning_b200 import engine
    return torch, engine, torch.device("cuda", 0)


@pytest.fixture(scope="module")
def L():
    return load_fd_host()


def _close(a, b, rel):
    """|a - b| <= rel * (1 + |b|) elementwise (NumPy)."""
    return bool((np.abs(a - b) <= rel * (1.0 + np.abs(b))).all())


def _minv_close(a, b):
    """M^-1 entries against a reference, relative to the largest entry of the state's M^-1."""
    scale = np.abs(b).max(axis=(0, 1))[None, None, :]
    return bool((np.abs(a - b) <= 1e-10 * (1.0 + scale)).all())


@pytest.mark.parametrize("mode", ["rne", "dyn"])
@pytest.mark.parametrize("model_name", ["stock", "override"])
def test_gpu_matches_host_build_and_inverts_the_torque_kernels(env, L, mode, model_name):
    """1 M config-2 states, tau ~ U(+-limit): qdd and M^-1 equal the host build; the torque kernel at
    (q, qd, qdd) reproduces tau within 1e-9 N.m; the qdd-only and M^-1-only calls equal the full call bit for bit;
    M^-1 M = I with K10's M."""
    torch, engine, dev = env
    rec = None if model_name == "stock" else load_golden("model_override.npz")["model"]
    model = None if rec is None else engine.InertialModel(rec)
    n = 1_000_000
    q, qd, _, mass = sample_states(n, seed=101)
    lim = limits(rec)
    tau = np.random.default_rng(102).uniform(-lim[:, None], lim[:, None], size=q.shape)
    t = lambda a: torch.as_tensor(a, device=dev)
    tq, tqd, ttau, tm = t(q), t(qd), t(tau), t(mass)
    full = engine.forward_dynamics_batch(tq, tqd, ttau, tm, mode=mode, qdd=True, minv=True, model=model)
    only_qdd = engine.forward_dynamics_batch(tq, tqd, ttau, tm, mode=mode, model=model)
    only_minv = engine.forward_dynamics_batch(tq, tqd, ttau, tm, mode=mode, qdd=False, minv=True, model=model)
    assert only_qdd["Minv"] is None and only_minv["qdd"] is None
    assert torch.equal(only_qdd["qdd"], full["qdd"])
    assert torch.equal(only_minv["Minv"], full["Minv"])
    Mi = full["Minv"]
    assert torch.equal(Mi, Mi.transpose(0, 1))
    tau_k, _ = engine.torque_test_batch(tq, tqd, full["qdd"], tm, mode=mode, payload_threshold=0.0, want_mask=False,
                                        model=model)
    res = float((tau_k - ttau).abs().max())
    print("max residual %s %s: %.3e N.m" % (mode, model_name, res))
    assert res <= 1e-9
    M = engine.dynamics_batch(tq, None, tm if mode == "rne" else 0.0, gravity=False, model=model)["M"]
    eye = torch.einsum("ijn,jkn->ikn", Mi, M) - torch.eye(7, dtype=torch.float64, device=dev)[:, :, None]
    assert float(eye.abs().max()) <= 1e-9
    del M, eye
    s = slice(0, 200_000)
    ref = host_fd(L, q[:, s], qd[:, s], tau[:, s], mass[s], mode, rec)
    assert _close(full["qdd"][:, s].cpu().numpy(), ref["qdd"], 1e-10)
    assert _minv_close(Mi[:, :, s].cpu().numpy(), ref["Minv"])


def _guarded(torch, dev, count, guard=4099):
    buf = torch.full((guard + count + guard,), 1234.5, dtype=torch.float64, device=dev)
    return buf, buf[guard:guard + count]


@pytest.mark.parametrize("n", [1, 127, 128, 129, 100_003])
def test_batch_sizes_and_guard_bands(env, L, n):
    torch, engine, dev = env
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr, _stream_ptr
    lib = _lib.load()
    q, qd, _, mass = sample_states(n, seed=103)
    tau = np.random.default_rng(104).uniform(-STOCK_LIMIT[:, None], STOCK_LIMIT[:, None], size=q.shape)
    # the device inputs stay bound until the kernel has run: a freed temporary's memory may back the next one
    tq, tqd, ttau, tm = (torch.as_tensor(np.ascontiguousarray(a), device=dev) for a in (q, qd, tau, mass))
    for mode in ("rne", "dyn"):
        qb, qv = _guarded(torch, dev, 7 * n)
        mb, mv = _guarded(torch, dev, 49 * n)
        _lib.check(lib.tcmp_forward_dynamics_batch(None, MODE[mode], n, _ptr(tq), _ptr(tqd), _ptr(ttau), _ptr(tm), 0.0,
                                                   _ptr(qv), _ptr(mv), _stream_ptr()))
        torch.cuda.synchronize()
        for buf, view in ((qb, qv), (mb, mv)):
            g = (buf.numel() - view.numel()) // 2
            assert bool((buf[:g] == 1234.5).all()) and bool((buf[g + view.numel():] == 1234.5).all())
        ref = host_fd(L, q, qd, tau, mass, mode)
        assert _close(qv.view(7, n).cpu().numpy(), ref["qdd"], 1e-10)
        assert _minv_close(mv.view(7, 7, n).cpu().numpy(), ref["Minv"])


def test_empty_batch(env):
    torch, engine, dev = env
    z = torch.empty((7, 0), dtype=torch.float64, device=dev)
    out = engine.forward_dynamics_batch(z, z, z, minv=True)
    assert tuple(out["qdd"].shape) == (7, 0) and tuple(out["Minv"].shape) == (7, 7, 0)


def test_graph_capture_and_replay(env):
    torch, engine, dev = env
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr
    lib = _lib.load()
    n = 100_000
    q, qd, qdd, mass = (torch.as_tensor(a, device=dev) for a in sample_states(n, seed=105))
    tau = qdd * 3.0
    qo = torch.empty((7, n), dtype=torch.float64, device=dev)
    mo = torch.empty((7, 7, n), dtype=torch.float64, device=dev)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        _lib.check(lib.tcmp_forward_dynamics_batch(None, 2, n, _ptr(q), _ptr(qd), _ptr(tau), _ptr(mass), 0.0,
                                                   _ptr(qo), _ptr(mo), int(side.cuda_stream)))
    qo.fill_(float("nan"))
    mo.fill_(float("nan"))
    g.replay()
    torch.cuda.synchronize()
    ref = engine.forward_dynamics_batch(q, qd, tau, mass, mode="dyn", minv=True)
    assert torch.equal(qo, ref["qdd"]) and torch.equal(mo, ref["Minv"])


def test_beyond_32_bit_offsets(env, L):
    """49 n > 2^31 elements: the 64-bit offset path, checked on a strided sample of states."""
    torch, engine, dev = env
    n = 44_000_000
    free, _ = torch.cuda.mem_get_info(dev)
    if free < 30 * 2**30:
        pytest.skip("needs 30 GB of free device memory")
    lo = torch.tensor([-2.8973, -1.7628, -2.8973, -3.0718, -2.8973, -0.0175, -2.8973], dtype=torch.float64, device=dev)
    hi = torch.tensor([2.8973, 1.7628, 2.8973, -0.0698, 2.8973, 3.7525, 2.8973], dtype=torch.float64, device=dev)
    gen = torch.Generator(device=dev).manual_seed(106)
    q = lo[:, None] + (hi - lo)[:, None] * torch.rand((7, n), dtype=torch.float64, device=dev, generator=gen)
    tau = 20.0 * torch.rand((7, n), dtype=torch.float64, device=dev, generator=gen) - 10.0
    out = engine.forward_dynamics_batch(q, None, tau, 1.0, minv=True)
    assert 49 * n > 2**31
    idx = torch.cat([torch.arange(0, n, 4099, device=dev), torch.tensor([n - 1], device=dev)])
    qs, ts = q[:, idx].cpu().numpy(), tau[:, idx].cpu().numpy()
    qdd, Mi = out["qdd"][:, idx].cpu().numpy(), out["Minv"][:, :, idx].cpu().numpy()
    del out, q, tau
    ref = host_fd(L, qs, None, ts, 1.0)
    assert _close(qdd, ref["qdd"], 1e-10)
    assert _minv_close(Mi, ref["Minv"])


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_nonfinite_inputs(env, mode):
    torch, engine, dev = env
    q, qd, _, mass = sample_states(9, seed=87)
    tau = np.random.default_rng(88).uniform(-10, 10, size=q.shape)
    run = lambda a, b, c, m: engine.forward_dynamics_batch(a, b, c, m, mode=mode, minv=True)
    base = run(q, qd, tau, mass)
    assert np.isfinite(base["qdd"]).all() and np.isfinite(base["Minv"]).all()
    k = 4
    for what, j, v in nonfinite_cases():
        arrs = {"q": q.copy(), "qd": qd.copy(), "tau": tau.copy(), "mass": mass.copy()}
        if what == "mass":
            arrs["mass"][k] = v
        else:
            arrs[what][j, k] = v
        check_nonfinite_rules(mode, base, run(arrs["q"], arrs["qd"], arrs["tau"], arrs["mass"]), what, k)


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_singular_record_and_tiny_tail_inertia(env, mode):
    torch, engine, dev = env
    q, qd, _, mass = sample_states(2000, seed=89)
    tau = np.random.default_rng(90).uniform(-STOCK_LIMIT[:, None], STOCK_LIMIT[:, None], size=q.shape)
    out = engine.forward_dynamics_batch(q, qd, tau, mass, mode=mode, minv=True,
                                        model=engine.InertialModel(tail_record(0.0)))
    assert np.isnan(out["qdd"]).all() and np.isnan(out["Minv"]).all()
    model = engine.InertialModel(tail_record(1e-4))
    out = engine.forward_dynamics_batch(q, qd, tau, mass, mode=mode, minv=True, model=model)
    assert np.isfinite(out["qdd"]).all() and np.isfinite(out["Minv"]).all()
    tau_k, _ = engine.torque_test_batch(q, qd, out["qdd"], mass, mode=mode, payload_threshold=0.0, want_mask=False,
                                        model=model)
    assert np.abs(tau_k - tau).max() <= 1e-9


def test_drop_in_module_equals_the_batch_path(env):
    torch, engine, dev = env
    from torque_constrained_motion_planning_b200 import panda_dynamics_model as pdm
    q, qd, _, _ = sample_states(5, seed=107)
    tau = np.random.default_rng(108).uniform(-10, 10, size=q.shape)
    out = engine.forward_dynamics_batch(q, qd, tau, 0.0, minv=True)
    for i in range(5):
        qi, qdi, ti = list(q[:, i]) + [0.0, 0.0], list(qd[:, i]), list(tau[:, i])   # extra entries are ignored
        assert np.array_equal(pdm.get_forward_dynamics(qi, qdi, ti), out["qdd"][:, i])
        assert np.array_equal(pdm.get_inverse_mass_matrix(qi), out["Minv"][:, :, i])
    assert np.array_equal(pdm.get_forward_dynamics_batch(q, qd, tau), out["qdd"])
    assert np.array_equal(pdm.get_inverse_mass_matrix_batch(q), out["Minv"])
    # the arm alone: M^-1 inverts get_mass_matrix_batch
    M = pdm.get_mass_matrix_batch(q)
    assert np.abs(np.einsum("ijn,jkn->ikn", out["Minv"], M) - np.eye(7)[:, :, None]).max() <= 1e-9
    m = engine.InertialModel(load_golden("model_override.npz")["model"])
    mi = engine.forward_dynamics_batch(q, minv=True, qdd=False, model=m)["Minv"]
    assert np.array_equal(pdm.get_inverse_mass_matrix_batch(q, model=m), mi) and not np.array_equal(mi, out["Minv"])
