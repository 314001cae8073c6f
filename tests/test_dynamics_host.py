"""CPU: K10's joint-space dynamics terms (csrc/dynamics_core.cuh -- the same per-state source dynamics_kernels.cu
instantiates) built for the host by tests/native/dynamics_host.cpp and checked against the oracle: M and C composed
from the pinned rne, g against nov, J against a dense DH chain, finite differences and the oracle's dyn.  Also the
argument validation of tcmp_dynamics_batch, the sm_100a code of the kernel, and the drop-in module's imports."""
import ctypes
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

import oracle
from conftest import ROOT, load_golden, sample_states

NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "csrc")
_dp = ctypes.POINTER(ctypes.c_double)
G = 9.81


def _load_host():
    so = os.path.join(NATIVE, "libdynamics_host.so")
    src = os.path.join(NATIVE, "dynamics_host.cpp")
    deps = [src, os.path.join(CSRC, "dynamics_core.cuh"), os.path.join(CSRC, "panda_model.cuh"),
            os.path.join(CSRC, "sincos_table.inc"), os.path.join(ROOT, "include", "tcmp.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                               "-Wno-unknown-pragmas", "-o", so, src])
    L = ctypes.CDLL(so)
    L.host_dynamics_flops.restype = ctypes.c_int64
    L.host_sincos_flops.restype = ctypes.c_int64
    return L


@pytest.fixture(scope="module")
def host_dyn():
    L = _load_host()

    def fn(q, qd=None, mass=0.0, model=None, M=True, C=True, g=True, J=True):
        arr = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
        q, qd = arr(q), arr(qd)
        n = q.shape[1]
        pm = None if np.ndim(mass) == 0 else arr(mass)
        out = {"M": np.empty((7, 7, n)) if M else None, "C": np.empty((7, 7, n)) if C else None,
               "g": np.empty((7, n)) if g else None, "J": np.empty((6, 7, n)) if J else None}
        p = lambda a: None if a is None else a.ctypes.data_as(_dp)
        L.host_dynamics_batch(p(arr(model)), ctypes.c_int64(n), p(q), p(qd), p(pm),
                              ctypes.c_double(0.0 if pm is not None else float(mass)),
                              p(out["M"]), p(out["C"]), p(out["g"]), p(out["J"]))
        return out
    return fn


def _rne(q, qd, qdd, mass, model):
    """The pinned oracle rne with the raw payload rule (attached iff m > 0)."""
    z = np.zeros_like(q)
    tau, _ = oracle.torque_test_batch("rne", q, z if qd is None else qd, z if qdd is None else qdd, mass,
                                      payload_threshold=0.0, model=model)
    return tau


def oracle_mass_matrix(q, mass, model):
    g = _rne(q, None, None, mass, model)
    M = np.empty((7, 7, q.shape[1]))
    for j in range(7):
        e = np.zeros_like(q)
        e[j] = 1.0
        M[:, j] = _rne(q, None, e, mass, model) - g
    return M


def oracle_coriolis_matrix(q, qd, mass, model):
    """Columns (c(qd + e_j) - c(qd - e_j)) / 4 with c(v) = rne(q, v, 0) - g: exact for the quadratic c."""
    g = _rne(q, None, None, mass, model)
    C = np.empty((7, 7, q.shape[1]))
    for j in range(7):
        e = np.zeros_like(q)
        e[j] = 1.0
        C[:, j] = ((_rne(q, qd + e, None, mass, model) - g) - (_rne(q, qd - e, None, mass, model) - g)) / 4.0
    return C


# The unmodified DH chain of oracle/rne_oracle.c (dh_matrix, dyn_with), dense 4x4 products, vectorised over states.
DH_A = [0, 0, 0, 0.0825, -0.0825, 0, 0.088, 0]
DH_D = [0.333, 0, 0.316, 0, 0.384, 0, 0.0, 0.107]
DH_ALPHA = [0, -np.pi / 2, np.pi / 2, np.pi / 2, -np.pi / 2, np.pi / 2, np.pi / 2, 0]


def dh_frames(q):
    """-> z [7][3][n], origins [7][3][n] of the joint frames, flange frame T [4][4][n]."""
    n = q.shape[1]
    T = np.broadcast_to(np.eye(4)[:, :, None], (4, 4, n)).copy()
    z, o = np.empty((7, 3, n)), np.empty((7, 3, n))
    for k in range(8):
        th = q[k] if k < 7 else np.zeros(n)
        ca, sa = np.cos(DH_ALPHA[k]), np.sin(DH_ALPHA[k])
        cq, sq = np.cos(th), np.sin(th)
        D = np.zeros((4, 4, n))
        D[0, 0], D[0, 1], D[0, 3] = cq, -sq, DH_A[k]
        D[1, 0], D[1, 1], D[1, 2], D[1, 3] = sq * ca, cq * ca, -sa, -sa * DH_D[k]
        D[2, 0], D[2, 1], D[2, 2], D[2, 3] = sq * sa, cq * sa, ca, ca * DH_D[k]
        D[3, 3] = 1.0
        T = np.einsum("ikn,kjn->ijn", T, D)
        if k < 7:
            z[k], o[k] = T[:3, 2], T[:3, 3]
    return z, o, T


def tool_point(q, tool_z):
    _, _, T = dh_frames(q)
    return T[:3, 3] + T[:3, 2] * tool_z


def dense_jacobian(q, tool_z):
    z, o, _ = dh_frames(q)
    pt = tool_point(q, tool_z)
    J = np.empty((6, 7, q.shape[1]))
    for j in range(7):
        J[0:3, j] = np.cross(z[j], pt - o[j], axis=0)
        J[3:6, j] = z[j]
    return J


MODELS = {"stock": None, "override": "model_override.npz"}


def _model(name):
    return None if MODELS[name] is None else load_golden(MODELS[name])["model"]


def _tool_z(model):
    return 0.105 if model is None else float(oracle.model_fields(np.ascontiguousarray(model))["tool_z"][0])


@pytest.mark.parametrize("model_name", list(MODELS))
def test_mass_matrix_and_coriolis_match_oracle_composition(host_dyn, model_name):
    """20 k config-2 states, payloads {0, 1, 3, 5} kg: M bitwise symmetric and positive definite, M and C equal the
    compositions of the pinned oracle rne, C qd = rne(q, qd, 0) - g."""
    model = _model(model_name)
    q, qd, _, mass = sample_states(20000, seed=61)
    out = host_dyn(q, qd, mass, model)
    M, C = out["M"], out["C"]
    assert np.array_equal(M, M.transpose(1, 0, 2))
    np.linalg.cholesky(M.transpose(2, 0, 1))      # raises unless every state's M is positive definite
    assert np.abs(M - oracle_mass_matrix(q, mass, model)).max() <= 1e-11
    assert np.abs(C - oracle_coriolis_matrix(q, qd, mass, model)).max() <= 1e-11
    cqd = np.einsum("ijn,jn->in", C, qd)
    assert np.abs(cqd - (_rne(q, qd, None, mass, model) - _rne(q, None, None, mass, model))).max() <= 1e-11


@pytest.mark.parametrize("model_name", list(MODELS))
def test_coriolis_is_christoffel_consistent(host_dyn, model_name):
    """Mdot = C + C^T (so Mdot - 2C is skew), against a central difference of M along qd (h = 1e-5)."""
    model = _model(model_name)
    q, qd, _, mass = sample_states(20000, seed=62)
    h = 1e-5
    C = host_dyn(q, qd, mass, model, M=False, g=False, J=False)["C"]
    Mp = host_dyn(q + h * qd, None, mass, model, C=False, g=False, J=False)["M"]
    Mm = host_dyn(q - h * qd, None, mass, model, C=False, g=False, J=False)["M"]
    Mdot = (Mp - Mm) / (2 * h)
    err = np.abs(Mdot - (C + C.transpose(1, 0, 2)))
    assert (err <= 1e-7 * np.maximum(1.0, np.abs(Mdot))).all(), err.max()


@pytest.mark.parametrize("model_name", list(MODELS))
def test_gravity_matches_oracle_nov(host_dyn, model_name):
    model = _model(model_name)
    q, _, _, mass = sample_states(20000, seed=63)
    g = host_dyn(q, None, mass, model, M=False, C=False, J=False)["g"]
    tau, _ = oracle.torque_test_batch("nov", q, None, None, mass, payload_threshold=0.0, model=model)
    assert np.abs(g - tau).max() <= 1e-11


@pytest.mark.parametrize("model_name", list(MODELS))
def test_jacobian_matches_dense_chain_differences_and_dyn(host_dyn, model_name):
    model = _model(model_name)
    q, qd, qdd, mass = sample_states(20000, seed=64)
    tz = _tool_z(model)
    J = host_dyn(q, None, mass, model, M=False, C=False, g=False)["J"]
    assert np.abs(J - dense_jacobian(q, tz)).max() <= 1e-12
    h = 1e-6
    for j in range(7):
        e = np.zeros_like(q)
        e[j] = h
        fd = (tool_point(q + e, tz) - tool_point(q - e, tz)) / (2 * h)
        assert np.abs(J[0:3, j] - fd).max() <= 1e-8, j
    # the dyn closure's tool term: J[0:3]^T (0, 0, m g) = oracle dyn - oracle rne without payload
    dyn, _ = oracle.torque_test_batch("dyn", q, qd, qdd, mass, model=model)
    rne0, _ = oracle.torque_test_batch("rne", q, qd, qdd, 0.0, model=model)
    assert np.abs(J[2] * (mass * G) - (dyn - rne0)).max() <= 1e-11


@pytest.mark.parametrize("model_name", list(MODELS))
def test_terms_recompose_rne_and_dyn(host_dyn, model_name):
    """M qdd + C qd + g(m) = rne(q, qd, qdd, m) and M qdd + C qd + g(0) + J[0:3]^T (0, 0, m g) = dyn."""
    model = _model(model_name)
    q, qd, qdd, mass = sample_states(20000, seed=65)
    t = host_dyn(q, qd, mass, model)
    rec = np.einsum("ijn,jn->in", t["M"], qdd) + np.einsum("ijn,jn->in", t["C"], qd) + t["g"]
    assert np.abs(rec - _rne(q, qd, qdd, mass, model)).max() <= 1e-10
    t0 = host_dyn(q, qd, 0.0, model)
    dyn, _ = oracle.torque_test_batch("dyn", q, qd, qdd, mass, model=model)
    rec0 = np.einsum("ijn,jn->in", t0["M"], qdd) + np.einsum("ijn,jn->in", t0["C"], qd) + t0["g"]
    assert np.abs(rec0 + t0["J"][2] * (mass * G) - dyn).max() <= 1e-10


def test_output_subsets_match_the_full_call(host_dyn):
    q, qd, _, mass = sample_states(3000, seed=66)
    full = host_dyn(q, qd, mass)
    for key in ("M", "C", "g", "J"):
        flags = {k: k == key for k in ("M", "C", "g", "J")}
        one = host_dyn(q, qd, mass, **flags)
        assert np.array_equal(one[key], full[key]), key
        assert all(one[k] is None for k in flags if k != key)


def test_large_and_nonfinite_angles_follow_libm(host_dyn):
    """Angles of 4096 rad and beyond (or non-finite) leave the table sincos for libm's: still the oracle's result."""
    q, qd, _, mass = sample_states(512, seed=67)
    q[3, ::7] += 2e5
    q[5, ::11] = 1e300
    q[0, ::5] += 5000.0
    q[2, ::13] = 4096.0
    out = host_dyn(q, qd, mass)
    assert np.abs(out["M"] - oracle_mass_matrix(q, mass, None)).max() <= 1e-9
    assert np.abs(out["C"] - oracle_coriolis_matrix(q, qd, mass, None)).max() <= 1e-9
    tau, _ = oracle.torque_test_batch("nov", q, None, None, mass, payload_threshold=0.0)
    assert np.abs(out["g"] - tau).max() <= 1e-9
    assert np.abs(out["J"] - dense_jacobian(q, 0.105)).max() <= 1e-9
    q[2, 0] = np.nan
    out = host_dyn(q, qd, mass)
    assert np.isnan(out["M"][:, :, 0]).any() and np.isnan(out["g"][:, 0]).any()


def test_operation_counts_are_positive_and_additive():
    """The instrumented count bench_dynamics.py reports: each term costs something, and the full call is the sum."""
    L = _load_host()
    parts = [L.host_dynamics_flops(*(int(i == k) for i in range(4))) for k in range(4)]
    assert all(p > 0 for p in parts)
    assert L.host_dynamics_flops(1, 1, 1, 1) == sum(parts)
    assert 10 < L.host_sincos_flops() < 40


# ---- the C ABI, without a GPU -------------------------------------------------------------------------------------
def test_argument_validation_without_gpu():
    from torque_constrained_motion_planning_b200 import _lib, engine
    lib = _lib.load()
    f = lib.tcmp_dynamics_batch
    p = ctypes.c_void_p(0x1000)      # never dereferenced: every call below is rejected or empty
    assert f(None, -1, p, p, None, 0.0, p, None, None, None, None) == -1
    assert f(None, 4, None, None, None, 0.0, p, None, None, None, None) == -1          # q NULL
    assert b"q" in lib.tcmp_last_error()
    assert f(None, 4, p, None, None, 0.0, None, p, None, None, None) == -1             # C without qd
    assert b"qd" in lib.tcmp_last_error()
    assert f(None, 4, p, p, None, 0.0, None, None, None, None, None) == -1             # nothing requested
    bad = engine.InertialModel.default()
    bad.mass[2] = -1.0
    assert f(bad.record.ctypes.data, 4, p, None, None, 0.0, p, None, None, None, None) == -1
    assert b"mass" in lib.tcmp_last_error()
    assert f(bad.record.ctypes.data, 0, None, None, None, 0.0, None, None, None, None, None) == -1   # record first
    assert f(None, 0, None, None, None, 0.0, p, None, None, None, None) == 0
    # an empty batch is a no-op whatever the buffers: empty tensors / arrays may have NULL data pointers
    assert f(None, 0, None, None, None, 0.0, None, None, None, None, None) == 0
    assert f(None, 0, None, None, None, 0.0, None, p, None, None, None) == 0
    assert f(engine.InertialModel.default().record.ctypes.data, 0, None, None, None, 0.0, None, None, p, None,
             None) == 0


def test_library_carries_the_dynamics_kernel_as_sm_100a_code():
    from torque_constrained_motion_planning_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    usage = subprocess.run([cuobjdump, "-res-usage", _lib.LIB_PATH], capture_output=True, text=True).stdout
    blocks = re.findall(r"Function (\S*dynamics_kernel\S*):\s*\n\s*(REG:\d+ STACK:\d+ SHARED:\d+ LOCAL:\d+)", usage)
    assert len(blocks) >= 2, usage[:2000]               # compiled-in Panda and caller-supplied record
    for name, res in blocks:
        assert "LOCAL:0" in res, (name, res)       # (STACK holds the libm slow path's frame, as in K1)
    log = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "build", "dynamics_kernels.cu.ptxas.log")
    if os.path.exists(log):
        props = re.findall(r"Function properties for (\S*dynamics_kernel\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill "
                           r"stores, (\d+) bytes spill loads", open(log).read())
        assert len(props) >= 2 and all(st == "0" and ld == "0" for _, _, st, ld in props), props
    elfs = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert {arch for _, arch in re.findall(r"(\w+)\.(sm_\w+)\.cubin", elfs)} == {"sm_100a"}


def test_drop_in_module_does_not_import_the_oracle():
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from torque_constrained_motion_planning_b200 import panda_dynamics_model as pdm\n"
            "assert callable(pdm.get_mass_matrix) and callable(pdm.get_coriolis_matrix)\n"
            "assert callable(pdm.get_gravity_vector)\n"
            "assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules), 'oracle imported'\n" % ROOT)
    subprocess.check_call([sys.executable, "-c", code])
