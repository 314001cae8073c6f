"""GPU: K10 (tcmp_dynamics_batch) against the host build of the same source, the oracle, the pinned torque kernels
(M qdd + C qd + g == rne, and the dyn decomposition), finite differences of the FK kernel, graph capture, the
64-bit offset path and the panda_dynamics_model drop-in."""
import numpy as np
import pytest

import oracle
from conftest import load_golden, sample_states
from test_dynamics_host import _load_host, oracle_mass_matrix

pytestmark = pytest.mark.gpu
G = 9.81


@pytest.fixture(scope="module")
def env():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from torque_constrained_motion_planning_b200 import engine
    return torch, engine, torch.device("cuda", 0)


@pytest.fixture(scope="module")
def host():
    import ctypes
    L = _load_host()
    dp = ctypes.POINTER(ctypes.c_double)

    def fn(q, qd, mass, model=None):
        n = q.shape[1]
        arr = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        q, qd = arr(q), arr(qd)
        pm = None if np.ndim(mass) == 0 else arr(mass)
        out = {"M": np.empty((7, 7, n)), "C": np.empty((7, 7, n)), "g": np.empty((7, n)), "J": np.empty((6, 7, n))}
        p = lambda a: None if a is None else a.ctypes.data_as(dp)
        L.host_dynamics_batch(p(None if model is None else arr(model)), ctypes.c_int64(n), p(q), p(qd), p(pm),
                              ctypes.c_double(0.0 if pm is not None else float(mass)), p(out["M"]), p(out["C"]),
                              p(out["g"]), p(out["J"]))
        return out
    return fn


def _all(engine, q, qd, mass, model=None):
    return engine.dynamics_batch(q, qd, mass, mass_matrix=True, coriolis=True, gravity=True, jacobian=True,
                                 model=model)


@pytest.mark.parametrize("model_name", ["stock", "override"])
@pytest.mark.parametrize("payload", ["scalar", "per_state"])
def test_gpu_matches_host_build_and_oracle(env, host, model_name, payload):
    torch, engine, dev = env
    rec = None if model_name == "stock" else load_golden("model_override.npz")["model"]
    model = None if rec is None else engine.InertialModel(rec)
    q, qd, _, mass = sample_states(200_000, seed=71)
    m = 3.0 if payload == "scalar" else mass
    t = lambda a: torch.as_tensor(a, device=dev)
    out = _all(engine, t(q), t(qd), m if np.ndim(m) == 0 else t(m), model)
    ref = host(q, qd, m, rec)
    for k in ("M", "C", "g", "J"):
        assert np.abs(out[k].cpu().numpy() - ref[k]).max() <= 1e-11, k
    M = out["M"].cpu().numpy()
    assert np.array_equal(M, M.transpose(1, 0, 2))
    s = slice(0, 20_000)
    ms = m if np.ndim(m) == 0 else m[s]
    assert np.abs(M[:, :, s] - oracle_mass_matrix(q[:, s], ms, rec)).max() <= 1e-11
    tau, _ = oracle.torque_test_batch("nov", q[:, s], None, None, ms, payload_threshold=0.0, model=rec)
    assert np.abs(out["g"].cpu().numpy()[:, s] - tau).max() <= 1e-11


def test_output_subsets_equal_the_full_call(env):
    torch, engine, dev = env
    q, qd, _, mass = sample_states(50_000, seed=72)
    q, qd, mass = (torch.as_tensor(a, device=dev) for a in (q, qd, mass))
    full = _all(engine, q, qd, mass)
    names = {"M": "mass_matrix", "C": "coriolis", "g": "gravity", "J": "jacobian"}
    subsets = [("M",), ("C",), ("g",), ("J",), ("M", "g"), ("M", "C", "g"), ("C", "J")]
    for sub in subsets:
        flags = {names[k]: k in sub for k in names}
        out = engine.dynamics_batch(q, qd, mass, **flags)
        for k in names:
            assert (out[k] is None) == (k not in sub)
            if k in sub:
                assert torch.equal(out[k], full[k]), (sub, k)


@pytest.mark.parametrize("n", [0, 1, 31, 129, 1_000_007])
def test_batch_sizes(env, host, n):
    torch, engine, dev = env
    q, qd, _, mass = sample_states(max(n, 1), seed=73)
    q, qd, mass = q[:, :n], qd[:, :n], mass[:n]
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev)
    out = _all(engine, t(q), t(qd), t(mass))
    assert tuple(out["M"].shape) == (7, 7, n) and tuple(out["J"].shape) == (6, 7, n)
    if n:
        idx = np.unique(np.linspace(0, n - 1, min(n, 20_000)).astype(np.int64))
        ref = host(q[:, idx], qd[:, idx], mass[idx])
        for k in ("M", "C", "g", "J"):
            assert np.abs(out[k].cpu().numpy()[..., idx] - ref[k]).max() <= 1e-11, k


def test_terms_recompose_the_torque_kernels(env):
    """On 1 M states: M qdd + C qd + g(m) == tcmp_rne_batch(RNE, threshold 0) and
    M qdd + C qd + g(0) + J[0:3]^T (0, 0, m g) == tcmp_rne_batch(DYN)."""
    torch, engine, dev = env
    q, qd, qdd, mass = (torch.as_tensor(a, device=dev) for a in sample_states(1_000_000, seed=74))
    t = _all(engine, q, qd, mass)
    rec = torch.einsum("ijn,jn->in", t["M"], qdd) + torch.einsum("ijn,jn->in", t["C"], qd) + t["g"]
    tau, _ = engine.torque_test_batch(q, qd, qdd, mass, mode="rne", payload_threshold=0.0, want_mask=False)
    assert float((rec - tau).abs().max()) <= 1e-10
    t0 = _all(engine, q, qd, 0.0)
    rec0 = torch.einsum("ijn,jn->in", t0["M"], qdd) + torch.einsum("ijn,jn->in", t0["C"], qd) + t0["g"]
    dyn, _ = engine.torque_test_batch(q, qd, qdd, mass, mode="dyn", want_mask=False)
    assert float((rec0 + t0["J"][2] * (mass * G) - dyn).abs().max()) <= 1e-10


def test_jacobian_against_differences_of_the_fk_kernel(env):
    """Linear rows = d(tool point)/dq with the tool point = fk_batch's flange origin + tool_z * its z axis."""
    torch, engine, dev = env
    q, _, _, _ = sample_states(100_000, seed=75)
    J = engine.dynamics_batch(torch.as_tensor(q, device=dev), mass_matrix=False, gravity=False,
                              jacobian=True)["J"].cpu().numpy()

    def tool(qq):
        tr, rot = engine.fk_batch(torch.as_tensor(qq, device=dev))
        tr, rot = tr.cpu().numpy(), rot.cpu().numpy()
        return tr + 0.105 * rot[[2, 5, 8]]
    h = 1e-6
    for j in range(7):
        e = np.zeros_like(q)
        e[j] = h
        fd = (tool(q + e) - tool(q - e)) / (2 * h)
        assert np.abs(J[0:3, j] - fd).max() <= 1e-8, j


def test_graph_capture_and_replay(env):
    torch, engine, dev = env
    from torque_constrained_motion_planning_b200 import _lib
    from torque_constrained_motion_planning_b200.engine import _ptr
    lib = _lib.load()
    n = 100_000
    q, qd, _, mass = (torch.as_tensor(a, device=dev) for a in sample_states(n, seed=76))
    outs = [torch.empty((7, 7, n), dtype=torch.float64, device=dev), torch.empty((7, 7, n), dtype=torch.float64, device=dev),
            torch.empty((7, n), dtype=torch.float64, device=dev), torch.empty((6, 7, n), dtype=torch.float64, device=dev)]
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        _lib.check(lib.tcmp_dynamics_batch(None, n, _ptr(q), _ptr(qd), _ptr(mass), 0.0, *(_ptr(o) for o in outs),
                                           int(side.cuda_stream)))
    for o in outs:
        o.fill_(float("nan"))
    g.replay()
    torch.cuda.synchronize()
    ref = _all(engine, q, qd, mass)
    for o, k in zip(outs, ("M", "C", "g", "J")):
        assert torch.equal(o, ref[k]), k


def test_mass_matrix_beyond_32_bit_offsets(env, host):
    """49 n > 2^31 elements: the 64-bit offset path, checked on a strided sample of states."""
    torch, engine, dev = env
    n = 44_000_000
    free, _ = torch.cuda.mem_get_info(dev)
    if free < 22 * 2**30:
        pytest.skip("needs 22 GB of free device memory")
    lo = torch.tensor([-2.8973, -1.7628, -2.8973, -3.0718, -2.8973, -0.0175, -2.8973], dtype=torch.float64, device=dev)
    hi = torch.tensor([2.8973, 1.7628, 2.8973, -0.0698, 2.8973, 3.7525, 2.8973], dtype=torch.float64, device=dev)
    gen = torch.Generator(device=dev).manual_seed(77)
    q = lo[:, None] + (hi - lo)[:, None] * torch.rand((7, n), dtype=torch.float64, device=dev, generator=gen)
    M = engine.dynamics_batch(q, gravity=False, payload_mass=1.0)["M"]
    assert 49 * n > 2**31
    idx = torch.arange(0, n, 4099, device=dev)
    idx = torch.cat([idx, torch.tensor([n - 1], device=dev)])
    Ms = M[:, :, idx].cpu().numpy()
    qs = q[:, idx].cpu().numpy()
    del M, q
    ref = host(qs, np.zeros_like(qs), 1.0)
    assert np.abs(Ms - ref["M"]).max() <= 1e-11


def test_drop_in_module_equals_the_batch_path(env):
    torch, engine, dev = env
    from torque_constrained_motion_planning_b200 import panda_dynamics_model as pdm
    q, qd, _, _ = sample_states(5, seed=78)
    out = engine.dynamics_batch(q, qd, 0.0, coriolis=True)
    for i in range(5):
        qi, qdi = list(q[:, i]) + [0.0, 0.0], list(qd[:, i])   # extra entries are ignored, as by rne.rne
        assert np.array_equal(pdm.get_mass_matrix(qi), out["M"][:, :, i])
        assert np.array_equal(pdm.get_coriolis_matrix(qi, qdi), out["C"][:, :, i])
        assert np.array_equal(pdm.get_gravity_vector(qi), out["g"][:, i])
    assert np.array_equal(pdm.get_mass_matrix_batch(q), out["M"])
    assert np.array_equal(pdm.get_coriolis_matrix_batch(q, qd), out["C"])
    assert np.array_equal(pdm.get_gravity_vector_batch(q), out["g"])
    m = engine.InertialModel(load_golden("model_override.npz")["model"])
    mm = engine.dynamics_batch(q, model=m)["M"]
    assert np.array_equal(pdm.get_mass_matrix_batch(q, model=m), mm) and not np.array_equal(mm, out["M"])
