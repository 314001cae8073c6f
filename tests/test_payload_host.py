"""CPU: the payload-mass intervals of K11/K12 (csrc/payload_core.cuh -- the same per-state source payload_kernels.cu
instantiates) built for the host by tests/native/payload_host.cpp and checked against the pinned oracle: the affine
terms a and b, membership of probe masses, tightness of the endpoints and non-finite angles.  Also the argument
validation of tcmp_payload_interval_batch / tcmp_edge_payload_interval, engine.max_payload / engine.payload_passes
on hand-made intervals, and the sm_100a code of the kernels."""
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
MODE = {"rne": 0, "nov": 1, "dyn": 2, "base": 3}
BAND = 1e-9
THRESHOLD = 0.01
PROBES = (0.0, 0.01, float(np.nextafter(0.01, 1.0)), 0.5, 1.0, 2.0, 5.0, 10.0, 20.0, 40.0, 100.0)
# (mode, dynamic): the torque test's four specialisations
CASES = [("rne", True), ("nov", False), ("dyn", True), ("dyn", False)]
MODELS = {"stock": None, "override": "model_override.npz"}


def _load_host():
    so = os.path.join(NATIVE, "libpayload_host.so")
    src = os.path.join(NATIVE, "payload_host.cpp")
    deps = [src, os.path.join(CSRC, "payload_core.cuh"), os.path.join(CSRC, "panda_model.cuh"),
            os.path.join(CSRC, "sincos_table.inc"), os.path.join(ROOT, "include", "tcmp.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                               "-Wno-unknown-pragmas", "-o", so, src])
    L = ctypes.CDLL(so)
    L.host_payload_flops.restype = ctypes.c_int64
    return L


def host_payload(q, qd=None, qdd=None, mode="rne", model=None):
    """-> dict(a, b [7][n], lo, hi [n], ok uint8 [n]) from the host build."""
    L = _load_host()
    arr = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    q, qd, qdd, model = arr(q), arr(qd), arr(qdd), arr(model)
    n = q.shape[1]
    out = {"a": np.empty((7, n)), "b": np.empty((7, n)), "lo": np.empty(n), "hi": np.empty(n),
           "ok": np.empty(n, np.uint8)}
    p = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)
    L.host_payload_batch(p(model), ctypes.c_int(MODE[mode]), ctypes.c_int64(n), p(q), p(qd), p(qdd), p(out["a"]),
                         p(out["b"]), p(out["lo"]), p(out["hi"]), p(out["ok"]))
    return out


def _model(name):
    return None if MODELS[name] is None else np.ascontiguousarray(load_golden(MODELS[name])["model"], np.float64)


def _limits(model):
    if model is None:
        return np.array([87.0, 87.0, 87.0, 87.0, 12.0, 12.0])
    return np.array(oracle.model_fields(model)["torque_limit"][:6])


def oracle_tau(mode, q, qd, qdd, mass, model, threshold=THRESHOLD):
    tau, ok = oracle.torque_test_batch(mode, q, qd, qdd, mass, threshold, model=model)
    return tau, ok.astype(bool)


def oracle_affine(mode, q, qd, qdd, model):
    """a, b [7][n] from the oracle at two masses with threshold 0 (every positive mass attached)."""
    t1, _ = oracle_tau(mode, q, qd, qdd, 2.0, model, 0.0)
    t2, _ = oracle_tau(mode, q, qd, qdd, 6.0, model, 0.0)
    b = (t2 - t1) / 4.0
    return t1 - 2.0 * b, b


def probe_masses(lo, hi):
    """The fixed grid plus every finite endpoint x (1 +- 1e-6) -> list of scalar or per-state masses."""
    out = list(PROBES)
    for e in (lo, hi):
        fin = np.isfinite(e)
        for f in (1 - 1e-6, 1 + 1e-6):
            out.append(np.where(fin, e * f, 1.0))
    return out


def check_membership(mode, q, qd, qdd, model, iv):
    """The oracle's verdict at every probe mass equals engine.payload_passes outside the band -> states skipped."""
    from torque_constrained_motion_planning_b200 import engine
    lim = _limits(model)
    skipped = 0
    for m in probe_masses(iv["lo"], iv["hi"]):
        tau, ok = oracle_tau(mode, q, qd, qdd, m, model)
        band = (np.abs(np.abs(tau[:6]) - lim[:, None]) < BAND).any(0)
        want = engine.payload_passes(iv["lo"], iv["hi"], iv["ok"], m, mode, THRESHOLD)
        assert np.array_equal(ok[~band], want[~band]), (mode, m if np.ndim(m) == 0 else "endpoint")
        skipped += int(band.sum())
    return skipped


@pytest.mark.parametrize("model_name", list(MODELS))
@pytest.mark.parametrize("mode,dynamic", CASES)
def test_affine_terms_match_the_oracle(mode, dynamic, model_name):
    model = _model(model_name)
    q, qd, qdd, _ = sample_states(20000, seed=81)
    qd, qdd = (qd, qdd) if dynamic else (None, None)
    out = host_payload(q, qd, qdd, mode, model)
    a, b = oracle_affine(mode, q, qd, qdd, model)
    assert np.abs(out["a"] - a).max() <= 1e-11
    assert np.abs(out["b"] - b).max() <= 1e-11
    t0, _ = oracle_tau(mode, q, qd, qdd, 0.0, model)
    assert np.abs(out["a"] - t0).max() <= 1e-11      # a is the arm alone


@pytest.mark.parametrize("model_name", list(MODELS))
@pytest.mark.parametrize("mode,dynamic", CASES)
def test_probe_masses_get_the_oracle_verdict(mode, dynamic, model_name):
    model = _model(model_name)
    q, qd, qdd, _ = sample_states(20000, seed=82)
    qd, qdd = (qd, qdd) if dynamic else (None, None)
    iv = host_payload(q, qd, qdd, mode, model)
    skipped = check_membership(mode, q, qd, qdd, model, iv)
    print("%s dynamic=%d %s: %d of %d probes in the band" % (mode, dynamic, model_name, skipped,
                                                            len(probe_masses(iv["lo"], iv["hi"])) * q.shape[1]))


@pytest.mark.parametrize("model_name", list(MODELS))
@pytest.mark.parametrize("mode,dynamic", CASES)
def test_endpoints_are_tight(mode, dynamic, model_name):
    """At every finite endpoint above 0.01 kg of a non-empty interval, the largest oracle margin |tau_j| - L_j is 0."""
    model = _model(model_name)
    q, qd, qdd, _ = sample_states(20000, seed=83)
    qd, qdd = (qd, qdd) if dynamic else (None, None)
    iv = host_payload(q, qd, qdd, mode, model)
    lim = _limits(model)
    nonempty = iv["lo"] < iv["hi"]
    checked = 0
    for e in (iv["lo"], iv["hi"]):
        sel = nonempty & np.isfinite(e) & (e > THRESHOLD)
        if not sel.any():
            continue
        s = np.nonzero(sel)[0]
        tau, _ = oracle_tau(mode, q[:, s], None if qd is None else qd[:, s], None if qdd is None else qdd[:, s],
                            e[s], model, 0.0)
        margin = (np.abs(tau[:6]) - lim[:, None]).max(0)
        assert np.abs(margin).max() <= BAND, float(np.abs(margin).max())
        checked += len(s)
    assert checked > 1000


@pytest.mark.parametrize("joint", [0, 3])
@pytest.mark.parametrize("value", [np.nan, np.inf, -np.inf])
@pytest.mark.parametrize("mode,dynamic", CASES)
def test_nonfinite_angles_allow_every_mass(mode, dynamic, joint, value):
    """A non-finite angle (joint 1's too) makes every torque NaN: (-inf, +inf) and unloaded_ok, as the torque test
    judges such a state feasible at every mass."""
    q, qd, qdd, _ = sample_states(64, seed=84)
    q[joint, ::2] = value
    qd, qdd = (qd, qdd) if dynamic else (None, None)
    iv = host_payload(q, qd, qdd, mode)
    assert np.isnan(iv["a"][:6, ::2]).all() and np.isnan(iv["b"][:6, ::2]).all()    # the six tested joints
    assert (iv["lo"][::2] == -np.inf).all() and (iv["hi"][::2] == np.inf).all() and (iv["ok"][::2] == 1).all()
    assert np.isfinite(iv["lo"][1::2]).any()
    _, ok = oracle_tau(mode, q, qd, qdd, 5.0, None)
    assert ok[::2].all()


def test_operation_counts():
    """The instrumented count bench_payload.py reports: the dynamic pass costs more than the static one."""
    L = _load_host()
    static, dynamic = L.host_payload_flops(0, 0), L.host_payload_flops(0, 1)
    assert 0 < static < dynamic < 2000
    assert L.host_payload_flops(1, 0) == static


# ---- engine helpers on hand-made intervals --------------------------------------------------------------------------
def test_max_payload_and_payload_passes_on_hand_made_intervals():
    from torque_constrained_motion_planning_b200 import engine
    inf = np.inf
    #                ordinary  empty   lo > thr  hi < 0  unloaded fails  everything
    lo = np.array([-3.0,      5.0,    2.0,      -9.0,   -3.0,           -inf])
    hi = np.array([7.5,       1.0,    9.0,      -1.0,   7.5,            inf])
    ok = np.array([1,         1,      1,        1,      0,              1], np.uint8)
    np.testing.assert_array_equal(engine.max_payload(lo, hi, ok, "rne"), [7.5, 0.01, 0.01, 0.01, 0.0, inf])
    np.testing.assert_array_equal(engine.max_payload(lo, hi, ok, "nov", 0.5), [7.5, 0.5, 0.5, 0.5, 0.0, inf])
    np.testing.assert_array_equal(engine.max_payload(lo, hi, ok, "dyn"), [7.5, 0.0, 0.0, 0.0, 0.0, inf])
    np.testing.assert_array_equal(engine.max_payload(lo, hi, ok, "base"), [inf] * 6)
    # a mass at or below the threshold is not attached: the unloaded verdict
    np.testing.assert_array_equal(engine.payload_passes(lo, hi, ok, 0.01, "rne"), ok.astype(bool))
    np.testing.assert_array_equal(engine.payload_passes(lo, hi, ok, 3.0, "rne"), [1, 0, 1, 0, 1, 1])
    np.testing.assert_array_equal(engine.payload_passes(lo, hi, ok, 0.0, "dyn"), [1, 0, 0, 0, 1, 1])
    np.testing.assert_array_equal(engine.payload_passes(lo, hi, ok, 7.5, "dyn"), [0, 0, 1, 0, 0, 1])
    np.testing.assert_array_equal(engine.payload_passes(lo, hi, ok, 1e9, "base"), [1] * 6)
    per_state = np.array([0.0, 0.02, 3.0, -2.0, 1.0, 50.0])
    np.testing.assert_array_equal(engine.payload_passes(lo, hi, ok, per_state, "nov"), [1, 0, 1, 1, 1, 1])
    # every mass in [0, max_payload) passes
    for mode in ("rne", "nov", "dyn"):
        M = engine.max_payload(lo, hi, ok, mode)
        for f in (0.0, 0.25, 0.5, 0.999):
            m = np.where(np.isfinite(M), M, 1e6) * f
            assert engine.payload_passes(lo, hi, ok, m, mode)[M > 0].all(), (mode, f)


# ---- the C ABI, without a GPU -------------------------------------------------------------------------------------
def test_argument_validation_without_gpu():
    from torque_constrained_motion_planning_b200 import _lib, engine
    lib = _lib.load()
    f, e = lib.tcmp_payload_interval_batch, lib.tcmp_edge_payload_interval
    p = ctypes.c_void_p(0x1000)      # never dereferenced: every call below is rejected or empty
    assert f(None, 4, 8, p, None, None, p, p, p, None) == -1 and b"mode" in lib.tcmp_last_error()
    assert f(None, -1, 8, p, None, None, p, p, p, None) == -1
    assert f(None, 0, -1, p, None, None, p, p, p, None) == -1 and b"negative" in lib.tcmp_last_error()
    assert f(None, 0, 8, None, None, None, p, p, p, None) == -1 and b"q" in lib.tcmp_last_error()
    assert f(None, 0, 8, p, None, None, None, None, None, None) == -1 and b"output" in lib.tcmp_last_error()
    assert f(None, 0, 8, p, p, None, p, None, None, None) == -1 and b"qdd" in lib.tcmp_last_error()
    bad = engine.InertialModel.default()
    bad.mass[2] = -1.0
    assert f(bad.record.ctypes.data, 0, 8, p, None, None, p, None, None, None) == -1
    assert b"mass" in lib.tcmp_last_error()
    for mode in range(4):   # an empty batch is a no-op whatever the buffers
        assert f(None, mode, 0, None, None, None, None, None, None, None) == 0
        assert e(None, mode, 0, 64, None, None, 0, None, None, None, None) == 0
    assert e(None, 4, 8, 64, p, p, 0, p, p, p, None) == -1 and b"mode" in lib.tcmp_last_error()
    assert e(None, 0, -1, 64, p, p, 0, p, p, p, None) == -1
    assert e(None, 0, 8, 0, p, p, 0, p, p, p, None) == -1 and b"n_waypoints" in lib.tcmp_last_error()
    assert e(None, 0, 0, 0, None, None, 0, None, None, None, None) == -1     # n_waypoints is checked first
    assert e(None, 0, 8, 64, None, p, 0, p, p, p, None) == -1 and b"edge" in lib.tcmp_last_error()
    assert e(None, 0, 8, 64, p, p, 0, None, None, None, None) == -1 and b"output" in lib.tcmp_last_error()
    assert e(bad.record.ctypes.data, 0, 8, 64, p, p, 0, p, p, p, None) == -1


def test_velocities_come_in_pairs_without_gpu():
    """qd without qdd (or the reverse) is an error, not a static call: raised before any CUDA call."""
    from torque_constrained_motion_planning_b200 import engine
    q, qd, qdd, _ = sample_states(8, seed=85)
    with pytest.raises(ValueError, match="both"):
        engine.payload_interval_batch(q, qd, None)
    with pytest.raises(ValueError, match="both"):
        engine.payload_interval_batch(q, None, qdd, mode="nov")


def test_library_carries_the_payload_kernels_as_sm_100a_code():
    from torque_constrained_motion_planning_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    usage = subprocess.run([cuobjdump, "-res-usage", _lib.LIB_PATH], capture_output=True, text=True).stdout
    blocks = re.findall(r"Function (\S*(?:payload_interval_kernel|edge_payload_kernel)\S*):\s*\n\s*"
                        r"(REG:\d+ STACK:\d+ SHARED:\d+ LOCAL:\d+)", usage)
    # K11: {int, int64 offsets} x {dyn, static} x {tool, no tool} x {compiled-in, record}; K12: the last three
    assert len(blocks) == 24, usage[:2000]
    for name, res in blocks:
        assert "LOCAL:0" in res, (name, res)       # (STACK holds the libm slow path's frame, as in K1)
    log = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "build", "payload_kernels.cu.ptxas.log")
    if os.path.exists(log):
        props = re.findall(r"Function properties for (\S*(?:payload_interval_kernel|edge_payload_kernel)\S*)\n\s*"
                           r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", open(log).read())
        assert len(props) == 24 and all(st == "0" and ld == "0" for _, _, st, ld in props), props
    elfs = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert {arch for _, arch in re.findall(r"(\w+)\.(sm_\w+)\.cubin", elfs)} == {"sm_100a"}
