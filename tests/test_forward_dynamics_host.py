"""CPU: K13's forward dynamics (csrc/fd_core.cuh -- the same per-state source fd_kernels.cu instantiates) built for the
host by tests/native/fd_host.cpp and checked as the exact inverse of the pinned oracle's torque test: no new oracle.
Also M^-1 against K10's M (host build of dynamics_core.cuh), payload edges, the non-finite-input and singular-model
rules, the argument validation of tcmp_forward_dynamics_batch and the sm_100a code of the kernel."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from conftest import ROOT, load_golden, sample_states

NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "csrc")
_dp = ctypes.POINTER(ctypes.c_double)
MODE = {"rne": 0, "dyn": 2}
STOCK_LIMIT = np.array([87.0, 87.0, 87.0, 87.0, 12.0, 12.0, 12.0])
MODELS = {"stock": None, "override": "model_override.npz"}


def load_fd_host():
    so = os.path.join(NATIVE, "libfd_host.so")
    src = os.path.join(NATIVE, "fd_host.cpp")
    deps = [src, os.path.join(NATIVE, "dynamics_host.cpp"), os.path.join(CSRC, "fd_core.cuh"),
            os.path.join(CSRC, "dynamics_core.cuh"), os.path.join(CSRC, "panda_model.cuh"),
            os.path.join(CSRC, "sincos_table.inc"), os.path.join(ROOT, "include", "tcmp.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                               "-Wno-unknown-pragmas", "-o", so, src])
    L = ctypes.CDLL(so)
    L.host_fd_flops.restype = ctypes.c_int64
    return L


def _arr(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return None if a is None else a.ctypes.data_as(_dp)


def host_fd(L, q, qd=None, tau=None, mass=0.0, mode="rne", model=None, qdd=True, minv=True):
    """-> {"qdd": [7][n] or None, "Minv": [7][7][n] or None} from the host build."""
    q, qd, tau = _arr(q), _arr(qd), _arr(tau)
    n = q.shape[1]
    pm = None if np.ndim(mass) == 0 else _arr(mass)
    out = {"qdd": np.empty((7, n)) if qdd else None, "Minv": np.empty((7, 7, n)) if minv else None}
    L.host_forward_dynamics_batch(_p(_arr(model)), MODE[mode], ctypes.c_int64(n), _p(q), _p(qd), _p(tau), _p(pm),
                                  ctypes.c_double(0.0 if pm is not None else float(mass)), _p(out["qdd"]),
                                  _p(out["Minv"]))
    return out


def host_mass_matrix(L, q, mass=0.0, model=None):
    """K10's M from the same library (dynamics_host.cpp): a rigid payload iff m > 0."""
    q = _arr(q)
    n = q.shape[1]
    pm = None if np.ndim(mass) == 0 else _arr(mass)
    M = np.empty((7, 7, n))
    L.host_dynamics_batch(_p(_arr(model)), ctypes.c_int64(n), _p(q), None, _p(pm),
                          ctypes.c_double(0.0 if pm is not None else float(mass)), _p(M), None, None, None)
    return M


def torque(mode, q, qd, qdd, mass, model):
    """The pinned oracle's torques with the raw payload rule (rne: attached iff m > 0; dyn: every m)."""
    tau, _ = oracle.torque_test_batch(mode, q, qd, qdd, mass, payload_threshold=0.0, model=model)
    return tau


def model_record(name):
    return None if MODELS[name] is None else load_golden(MODELS[name])["model"]


def limits(model):
    return STOCK_LIMIT if model is None else oracle.model_fields(np.ascontiguousarray(model))["torque_limit"].copy()


@pytest.fixture(scope="module")
def L():
    return load_fd_host()


CASES = [(mode, name, payload, static) for mode in ("rne", "dyn") for name in MODELS
         for payload in ("scalar", "per_state") for static in (False, True)]


def _case(name, payload, static, seed):
    q, qd, qdd, mass = sample_states(20000, seed=seed)
    return q, None if static else qd, qdd, (3.0 if payload == "scalar" else mass)


@pytest.mark.parametrize("mode,model_name,payload,static", CASES)
def test_round_trip_recovers_the_accelerations(L, mode, model_name, payload, static):
    """tau = oracle(q, qd, qdd), then FD(q, qd, tau) = qdd within 1e-9 (1 + |qdd|)."""
    model = model_record(model_name)
    q, qd, qdd, mass = _case(model_name, payload, static, 81)
    tau = torque(mode, q, qd, qdd, mass, model)
    out = host_fd(L, q, qd, tau, mass, mode, model, minv=False)
    err = np.abs(out["qdd"] - qdd) / (1.0 + np.abs(qdd))
    assert err.max() <= 1e-9, err.max()


@pytest.mark.parametrize("mode,model_name,payload,static", CASES)
def test_residual_of_sampled_torques(L, mode, model_name, payload, static):
    """tau ~ U(-limit, +limit): oracle(q, qd, FD(q, qd, tau)) - tau <= 1e-9 N.m on all 7 joints."""
    model = model_record(model_name)
    q, qd, _, mass = _case(model_name, payload, static, 82)
    lim = limits(model)
    tau = np.random.default_rng(83).uniform(-lim[:, None], lim[:, None], size=q.shape)
    qdd = host_fd(L, q, qd, tau, mass, mode, model, minv=False)["qdd"]
    res = np.abs(torque(mode, q, qd, qdd, mass, model) - tau).max()
    print("max residual %s %s %s static=%s: %.3e N.m" % (mode, model_name, payload, static, res))
    assert res <= 1e-9


@pytest.mark.parametrize("mode", ["rne", "dyn"])
@pytest.mark.parametrize("model_name", list(MODELS))
def test_inverse_mass_matrix(L, mode, model_name):
    """M^-1 bitwise symmetric, M^-1 M - I <= 1e-9 per entry with K10's M, and M^-1 (tau - h) = qdd."""
    model = model_record(model_name)
    q, qd, _, mass = sample_states(20000, seed=84)
    lim = limits(model)
    tau = np.random.default_rng(85).uniform(-lim[:, None], lim[:, None], size=q.shape)
    out = host_fd(L, q, qd, tau, mass, mode, model)
    Mi = out["Minv"]
    assert np.array_equal(Mi, Mi.transpose(1, 0, 2))
    M = host_mass_matrix(L, q, mass if mode == "rne" else 0.0, model)
    eye = np.einsum("ijn,jkn->ikn", Mi, M) - np.eye(7)[:, :, None]
    assert np.abs(eye).max() <= 1e-9, np.abs(eye).max()
    h = torque(mode, q, qd, np.zeros_like(q), mass, model)
    qdd = np.einsum("ijn,jn->in", Mi, tau - h)
    assert (np.abs(qdd - out["qdd"]) <= 1e-9 * (1.0 + np.abs(out["qdd"]))).all()
    # the qdd-only call gives the same qdd, and the Minv-only call the same M^-1
    assert np.array_equal(host_fd(L, q, qd, tau, mass, mode, model, minv=False)["qdd"], out["qdd"])
    assert np.array_equal(host_fd(L, q, qd, tau, mass, mode, model, qdd=False)["Minv"], Mi)


@pytest.mark.parametrize("mode", ["rne", "dyn"])
@pytest.mark.parametrize("model_name", list(MODELS))
@pytest.mark.parametrize("m", [0.0, 5e-324, 0.01, -1.0])
def test_payload_edges(L, mode, model_name, m):
    """rne: m <= 0 is the arm alone, 5e-324 attaches; dyn: every m is a tool-point force (negative too).  Each case is
    the inverse of the oracle at threshold 0."""
    model = model_record(model_name)
    q, qd, qdd, _ = sample_states(5000, seed=86)
    tau = torque(mode, q, qd, qdd, m, model)
    out = host_fd(L, q, qd, tau, m, mode, model)
    assert (np.abs(out["qdd"] - qdd) <= 1e-9 * (1.0 + np.abs(qdd))).all()
    M = host_mass_matrix(L, q, m if mode == "rne" else 0.0, model)
    assert np.abs(np.einsum("ijn,jkn->ikn", out["Minv"], M) - np.eye(7)[:, :, None]).max() <= 1e-9
    per_state = host_fd(L, q, qd, tau, np.full(q.shape[1], m), mode, model)
    assert np.array_equal(per_state["qdd"], out["qdd"]) and np.array_equal(per_state["Minv"], out["Minv"])
    if mode == "rne" and m <= 0.0:
        arm = host_fd(L, q, qd, tau, 0.0, mode, model)
        assert np.array_equal(arm["qdd"], out["qdd"]) and np.array_equal(arm["Minv"], out["Minv"])


def nonfinite_cases():
    """(input, joint, value): every q[j] (joint 1 included), qd[j], tau[j] and the mass, NaN / +inf / -inf."""
    for what in ("q", "qd", "tau"):
        for j in range(7):
            for v in (np.nan, np.inf, -np.inf):
                yield what, j, v
    for v in (np.nan, np.inf, -np.inf):
        yield "mass", 0, v


def check_nonfinite_rules(mode, base, poisoned, what, k):
    """Outputs of state k follow include/tcmp.h's rules; every other state equals the unpoisoned run bit for bit."""
    others = np.arange(base["qdd"].shape[1]) != k
    assert np.array_equal(poisoned["qdd"][:, others], base["qdd"][:, others])
    assert np.array_equal(poisoned["Minv"][:, :, others], base["Minv"][:, :, others])
    assert np.isnan(poisoned["qdd"][:, k]).all(), (mode, what)
    if what in ("q", "mass"):
        assert np.isnan(poisoned["Minv"][:, :, k]).all(), (mode, what)
    else:
        assert np.array_equal(poisoned["Minv"][:, :, k], base["Minv"][:, :, k]), (mode, what)


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_nonfinite_inputs(L, mode):
    q, qd, _, mass = sample_states(9, seed=87)
    tau = np.random.default_rng(88).uniform(-10, 10, size=q.shape)
    base = host_fd(L, q, qd, tau, mass, mode)
    assert np.isfinite(base["qdd"]).all() and np.isfinite(base["Minv"]).all()
    k = 4
    for what, j, v in nonfinite_cases():
        arrs = {"q": q.copy(), "qd": qd.copy(), "tau": tau.copy(), "mass": mass.copy()}
        if what == "mass":
            arrs["mass"][k] = v
        else:
            arrs[what][j, k] = v
        out = host_fd(L, arrs["q"], arrs["qd"], arrs["tau"], arrs["mass"], mode)
        check_nonfinite_rules(mode, base, out, what, k)


def tail_record(inertia):
    """The stock record with link 7, link8 and the hand massless and with isotropic inertia `inertia` (0 = none)."""
    rec = oracle.default_model()
    f = oracle.model_fields(rec)
    f["mass"][6:9] = 0.0
    f["inertia"][6:9] = 0.0
    f["inertia"][6:9, [0, 3, 5]] = inertia
    return rec


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_singular_model_gives_nan_and_a_tiny_tail_inertia_does_not(L, mode):
    q, qd, _, mass = sample_states(2000, seed=89)
    tau = np.random.default_rng(90).uniform(-STOCK_LIMIT[:, None], STOCK_LIMIT[:, None], size=q.shape)
    out = host_fd(L, q, qd, tau, mass, mode, tail_record(0.0))
    assert np.isnan(out["qdd"]).all() and np.isnan(out["Minv"]).all()
    rec = tail_record(1e-4)
    out = host_fd(L, q, qd, tau, mass, mode, rec)
    assert np.isfinite(out["qdd"]).all() and np.isfinite(out["Minv"]).all()
    assert np.abs(torque(mode, q, qd, out["qdd"], mass, rec) - tau).max() <= 1e-9


def test_large_angles_follow_libm(L):
    """Angles of 4096 rad and beyond leave the table sincos for libm's: still the inverse of the oracle."""
    q, qd, qdd, mass = sample_states(512, seed=91)
    q[3, ::7] += 2e5
    q[0, ::5] += 5000.0
    q[2, ::13] = 4096.0
    tau = torque("rne", q, qd, qdd, mass, None)
    out = host_fd(L, q, qd, tau, mass)
    assert (np.abs(out["qdd"] - qdd) <= 1e-9 * (1.0 + np.abs(qdd))).all()


def test_null_tau_and_qd_are_zeros(L):
    q, qd, _, mass = sample_states(1000, seed=92)
    z = np.zeros_like(q)
    for mode in ("rne", "dyn"):
        a = host_fd(L, q, None, None, mass, mode)
        b = host_fd(L, q, z, z, mass, mode)
        assert np.array_equal(a["qdd"], b["qdd"]) and np.array_equal(a["Minv"], b["Minv"])


def test_operation_counts():
    """What bench_forward_dynamics.py reports: M and its factor, h and the solve, M^-1."""
    L = load_fd_host()
    parts = [L.host_fd_flops(i) for i in range(3)]
    assert all(p > 0 for p in parts)
    assert parts[0] > L.host_dynamics_flops(1, 0, 0, 0)       # M's column passes plus the factorisation


# ---- the C ABI, without a GPU -------------------------------------------------------------------------------------
def test_argument_validation_without_gpu():
    from torque_constrained_motion_planning_b200 import _lib, engine
    lib = _lib.load()
    f = lib.tcmp_forward_dynamics_batch
    p = ctypes.c_void_p(0x1000)      # never dereferenced: every call below is rejected or empty
    for mode in (1, 3, 4, -1):       # nov, base and bad modes, even for an empty batch
        for n in (4, 0):
            assert f(None, mode, n, p, p, p, None, 0.0, p, p, None) == -1
            assert b"mode" in lib.tcmp_last_error()
    assert f(None, 0, -1, p, p, p, None, 0.0, p, None, None) == -1
    assert b"negative" in lib.tcmp_last_error()
    assert f(None, 2, 4, None, p, p, None, 0.0, p, None, None) == -1
    assert b"q is NULL" in lib.tcmp_last_error()
    assert f(None, 0, 4, p, p, p, None, 0.0, None, None, None) == -1
    assert b"outputs" in lib.tcmp_last_error()
    bad = engine.InertialModel.default()
    bad.mass[2] = -1.0
    assert f(bad.record.ctypes.data, 0, 4, p, None, None, None, 0.0, p, None, None) == -1
    assert b"mass" in lib.tcmp_last_error()
    for mode in (0, 2):
        assert f(None, mode, 0, None, None, None, None, 0.0, None, None, None) == 0
        assert f(engine.InertialModel.default().record.ctypes.data, mode, 0, None, None, None, None, 0.0, p, None,
                 None) == 0
    with pytest.raises(ValueError):
        engine.forward_dynamics_batch(np.zeros((7, 1)), qdd=False, minv=False)


def test_library_carries_the_forward_dynamics_kernel_as_sm_100a_code():
    from torque_constrained_motion_planning_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    usage = subprocess.run([cuobjdump, "-res-usage", _lib.LIB_PATH], capture_output=True, text=True).stdout
    blocks = re.findall(r"Function (\S*forward_dynamics_kernel\S*):\s*\n\s*(REG:\d+ STACK:\d+ SHARED:\d+ LOCAL:\d+)",
                        usage)
    assert len(blocks) == 8, usage[:2000]      # {int, int64 offsets} x {rne, dyn} x {compiled-in, record}
    for name, res in blocks:
        assert "LOCAL:0" in res, (name, res)
    log = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "build", "fd_kernels.cu.ptxas.log")
    if os.path.exists(log):
        props = re.findall(r"Function properties for (\S*forward_dynamics_kernel\S*)\n\s*(\d+) bytes stack frame, "
                           r"(\d+) bytes spill stores, (\d+) bytes spill loads", open(log).read())
        assert len(props) == 8 and all(st == "0" and ld == "0" for _, _, st, ld in props), props


def test_drop_in_additions_exist():
    from torque_constrained_motion_planning_b200 import panda_dynamics_model as pdm
    for name in ("get_forward_dynamics", "get_inverse_mass_matrix", "get_forward_dynamics_batch",
                 "get_inverse_mass_matrix_batch"):
        assert callable(getattr(pdm, name)), name
