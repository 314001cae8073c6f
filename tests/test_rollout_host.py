"""CPU: K14's forward-dynamics rollouts (csrc/rollout_core.cuh -- the same per-rollout source rollout_kernels.cu
instantiates) built for the host by tests/native/rollout_host.cpp.  Checked bit for bit against a NumPy RK4 over K13's
host build, for fourth-order convergence against scipy's DOP853, static equilibrium under the oracle's static torque,
energy drift under free motion, the limit compare at its exact boundary, the non-finite rules, the argument validation
of tcmp_rollout_batch and the sm_100a code of the kernel."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from conftest import Q_HI, Q_LO, ROOT, V_LIM, load_golden, sample_states

NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "csrc")
_dp = ctypes.POINTER(ctypes.c_double)
MODE = {"rne": 0, "dyn": 2}
STOCK_LIMIT = np.array([87.0, 87.0, 87.0, 87.0, 12.0, 12.0, 12.0])
MODELS = {"stock": None, "override": "model_override.npz"}
G = 9.81


def load_rollout_host():
    so = os.path.join(NATIVE, "librollout_host.so")
    src = os.path.join(NATIVE, "rollout_host.cpp")
    deps = [src, os.path.join(NATIVE, "fd_host.cpp"), os.path.join(NATIVE, "dynamics_host.cpp"),
            os.path.join(CSRC, "rollout_core.cuh"), os.path.join(CSRC, "fd_core.cuh"),
            os.path.join(CSRC, "dynamics_core.cuh"), os.path.join(CSRC, "panda_model.cuh"),
            os.path.join(CSRC, "sincos_table.inc"), os.path.join(ROOT, "include", "tcmp.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                               "-Wno-unknown-pragmas", "-o", so, src])
    L = ctypes.CDLL(so)
    L.host_fd_flops.restype = ctypes.c_int64
    L.host_sincos_flops.restype = ctypes.c_int64
    L.host_rollout_combination_flops.restype = ctypes.c_int64
    return L


def _arr(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return None if a is None else a.ctypes.data_as(_dp)


def host_rollout(L, q0, qd0=None, tau=None, dt=1e-3, n_steps=1, mass=0.0, mode="rne", tau_per_step=False,
                 q_lo=None, q_hi=None, qd_max=None, model=None):
    """-> {"q", "qd", "q_traj", "qd_traj", "first_violation"} from the host build (every output requested)."""
    q0, qd0, tau = _arr(q0), _arr(qd0), _arr(tau)
    n = q0.shape[1]
    pm = None if np.ndim(mass) == 0 else _arr(mass)
    lim = [None if a is None else _arr(np.broadcast_to(a, (7,))) for a in (q_lo, q_hi, qd_max)]
    out = {"q": np.empty((7, n)), "qd": np.empty((7, n)), "q_traj": np.empty((n_steps, 7, n)),
           "qd_traj": np.empty((n_steps, 7, n)), "first_violation": np.empty(n, dtype=np.int32)}
    L.host_rollout_batch(_p(_arr(model)), MODE[mode], ctypes.c_int64(n), n_steps, ctypes.c_double(dt), _p(q0),
                         _p(qd0), _p(tau), int(tau_per_step), _p(pm),
                         ctypes.c_double(0.0 if pm is not None else float(mass)), *(_p(a) for a in lim),
                         _p(out["q"]), _p(out["qd"]), _p(out["q_traj"]), _p(out["qd_traj"]),
                         out["first_violation"].ctypes.data_as(ctypes.POINTER(ctypes.c_int32)))
    return out


def fd(L, q, qd, tau, mass, mode, model):
    """K13's host qdd (fd_host.cpp, which rollout_host.cpp includes)."""
    q, qd, tau = _arr(q), _arr(qd), _arr(tau)
    n = q.shape[1]
    pm = None if np.ndim(mass) == 0 else _arr(mass)
    qdd = np.empty((7, n))
    L.host_forward_dynamics_batch(_p(_arr(model)), MODE[mode], ctypes.c_int64(n), _p(q), _p(qd), _p(tau), _p(pm),
                                  ctypes.c_double(0.0 if pm is not None else float(mass)), _p(qdd), None)
    return qdd


def numpy_rk4(f, q, v, tau_at, dt, n_steps):
    """include/tcmp.h's RK4 in its exact order of operations; f(q, v, tau) -> qdd; tau_at(k) -> the step's torque."""
    h2, h6 = 0.5 * dt, dt / 6.0
    qs, vs = [], []
    for k in range(n_steps):
        u = tau_at(k)
        a1 = f(q, v, u)
        q2 = q + h2 * v
        v2 = v + h2 * a1
        a2 = f(q2, v2, u)
        q3 = q + h2 * v2
        v3 = v + h2 * a2
        a3 = f(q3, v3, u)
        q4 = q + dt * v3
        v4 = v + dt * a3
        a4 = f(q4, v4, u)
        q = q + h6 * (((v + 2 * v2) + 2 * v3) + v4)
        v = v + h6 * (((a1 + 2 * a2) + 2 * a3) + a4)
        qs.append(q)
        vs.append(v)
    return np.stack(qs), np.stack(vs)


def first_violation(q_traj, qd_traj, q_lo=None, q_hi=None, qd_max=None):
    """The first stored state failing a requested check (NaN fails), or n_steps."""
    T = q_traj.shape[0]
    bad = np.zeros(q_traj.shape[::2], dtype=bool)          # [T][n]
    if q_lo is not None:
        ok = (q_traj >= np.asarray(q_lo)[None, :, None]) & (q_traj <= np.asarray(q_hi)[None, :, None])
        bad |= ~ok.all(axis=1)
    if qd_max is not None:
        bad |= ~(np.abs(qd_traj) <= np.asarray(qd_max)[None, :, None]).all(axis=1)
    return np.where(bad.any(axis=0), bad.argmax(axis=0), T).astype(np.int32)


def model_record(name):
    return None if MODELS[name] is None else load_golden(MODELS[name])["model"]


def limits(model):
    return STOCK_LIMIT if model is None else oracle.model_fields(np.ascontiguousarray(model))["torque_limit"].copy()


def rollout_inputs(n, seed, model=None, n_steps=1, per_step=False, payload="per_state"):
    q, qd, _, mass = sample_states(n, seed=seed)
    lim = limits(model)[:, None]
    rng = np.random.default_rng(seed + 1)
    tau = rng.uniform(-lim, lim, size=(n_steps, 7, n) if per_step else (7, n))
    return q, qd, tau, (3.0 if payload == "scalar" else mass)


# Limits that some of the sampled states cross within a few steps, others never
TIGHT_LO, TIGHT_HI, TIGHT_V = 0.99 * Q_LO + 0.01 * Q_HI, 0.01 * Q_LO + 0.99 * Q_HI, V_LIM


@pytest.fixture(scope="module")
def L():
    return load_rollout_host()


CASES = [(mode, name, payload, per_step) for mode in ("rne", "dyn") for name in MODELS
         for payload in ("scalar", "per_state") for per_step in (False, True)]


@pytest.mark.parametrize("mode,model_name,payload,per_step", CASES)
def test_rollout_is_the_numpy_rk4_over_k13_bit_for_bit(L, mode, model_name, payload, per_step):
    model = model_record(model_name)
    for T in (1, 2, 7, 32):
        q, qd, tau, mass = rollout_inputs(48, 300 + T, model, T, per_step, payload)
        dt = 1e-3
        out = host_rollout(L, q, qd, tau, dt, T, mass, mode, per_step, TIGHT_LO, TIGHT_HI, TIGHT_V, model)
        ref_q, ref_v = numpy_rk4(lambda a, b, u: fd(L, a, b, u, mass, mode, model), q, qd,
                                 (lambda k: tau[k]) if per_step else (lambda k: tau), dt, T)
        assert np.array_equal(out["q_traj"], ref_q) and np.array_equal(out["qd_traj"], ref_v), (mode, T)
        assert np.array_equal(out["q"], ref_q[-1]) and np.array_equal(out["qd"], ref_v[-1])
        fv = first_violation(ref_q, ref_v, TIGHT_LO, TIGHT_HI, TIGHT_V)
        assert np.array_equal(out["first_violation"], fv)
        if T == 32:
            assert ((fv > 0) & (fv < T)).any(), np.bincount(fv)


def test_fourth_order_against_dop853(L):
    """Median over 64 config-2 states of err(dt) / err(dt/2) lies in [12, 20] (16 for a fourth-order method)."""
    from scipy.integrate import solve_ivp
    n = 64
    q, qd, _, mass = sample_states(n, seed=310)
    qd = 0.3 * qd
    z = np.zeros_like(q)
    grav, _ = oracle.torque_test_batch("rne", q, z, z, mass, payload_threshold=0.0)
    tau = grav + np.random.default_rng(311).uniform(-0.05, 0.05, size=q.shape) * STOCK_LIMIT[:, None]
    horizon, dt = 0.32, 0.02

    def rhs(_, y):
        x = y.reshape(2, 7, n)
        return np.concatenate([x[1], fd(L, x[0], x[1], tau, mass, "rne", None)]).ravel()

    ref = solve_ivp(rhs, (0.0, horizon), np.concatenate([q, qd]).ravel(), method="DOP853", rtol=1e-12,
                    atol=1e-12).y[:, -1].reshape(2, 7, n)
    err = []
    for h in (dt, dt / 2):
        out = host_rollout(L, q, qd, tau, h, int(round(horizon / h)), mass)
        err.append(np.maximum(np.abs(out["q"] - ref[0]).max(axis=0), np.abs(out["qd"] - ref[1]).max(axis=0)))
    ratio = err[0] / err[1]
    print("error at dt: median %.3e; ratio median %.2f, range [%.2f, %.2f]" % (np.median(err[0]), np.median(ratio),
                                                                           ratio.min(), ratio.max()))
    assert np.median(err[1]) > 1e-9          # well above round-off and DOP853's tolerance
    assert 12.0 <= np.median(ratio) <= 20.0


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_static_equilibrium_holds(L, mode):
    """tau = the oracle's static torque at (q, 0, 0) (threshold 0): 1000 steps of 1 ms stay within 1e-10."""
    q, _, _, mass = sample_states(16, seed=320)
    z = np.zeros_like(q)
    tau, _ = oracle.torque_test_batch(mode, q, z, z, mass, payload_threshold=0.0)
    out = host_rollout(L, q, None, tau, 1e-3, 1000, mass, mode)
    dq, dv = np.abs(out["q_traj"] - q).max(), np.abs(out["qd_traj"]).max()
    print("static drift %s: |q - q0| %.3e, |qd| %.3e" % (mode, dq, dv))
    # the residual of the oracle's torque (~1e-13 N.m) accelerates unstable equilibria: qd reaches ~2e-10 in dyn
    assert dq <= 1e-10 and dv <= 1e-9


def dh_link_frames(q):
    """The dense DH chain of test_dynamics_host.dh_frames, returning each link's full 4x4 frame: [8][4][4][n], link
    frames 1..7 (index 0..6) and the flange frame (index 7)."""
    from test_dynamics_host import DH_A, DH_ALPHA, DH_D
    n = q.shape[1]
    T = np.broadcast_to(np.eye(4)[:, :, None], (4, 4, n)).copy()
    frames = []
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
        frames.append(T)
    return np.stack(frames)


def potential(q):
    """V(q) = sum m_i g z_i of the stock record: links 1..7 in their frames, link8 and the hand in the flange frame."""
    f = oracle.model_fields(oracle.default_model())
    F = dh_link_frames(q)
    V = np.zeros(q.shape[1])
    for b in range(9):
        T = F[b] if b < 7 else F[7]
        z = T[2, 0] * f["com"][b][0] + T[2, 1] * f["com"][b][1] + T[2, 2] * f["com"][b][2] + T[2, 3]
        V += f["mass"][b] * G * z
    return V


def host_dynamics(L, q):
    """K10's host M and g (no payload)."""
    q = _arr(q)
    n = q.shape[1]
    M, g = np.empty((7, 7, n)), np.empty((7, n))
    L.host_dynamics_batch(None, ctypes.c_int64(n), _p(q), None, None, ctypes.c_double(0.0), _p(M), None, _p(g), None)
    return M, g


def test_energy_is_conserved_in_free_motion(L):
    q, qd, _, _ = sample_states(32, seed=330)
    qd = 0.3 * qd
    # V first: its central-difference gradient is K10's g
    _, g = host_dynamics(L, q)
    h = 1e-6
    grad = np.stack([(potential(q + h * np.eye(7)[j][:, None]) - potential(q - h * np.eye(7)[j][:, None])) / (2 * h)
                     for j in range(7)])
    assert np.abs(grad - g).max() <= 1e-7, np.abs(grad - g).max()

    def energy(qq, vv):
        M, _ = host_dynamics(L, qq)
        return 0.5 * np.einsum("in,ijn,jn->n", vv, M, vv) + potential(qq)

    E0 = energy(q, qd)
    drift = []
    for dt, T in ((1e-3, 1000), (5e-4, 2000)):
        out = host_rollout(L, q, qd, None, dt, T, 0.0)
        drift.append(max(np.abs(energy(out["q_traj"][k], out["qd_traj"][k]) - E0).max()
                         for k in (T // 4, T // 2, T - 1)))
    print("energy drift over 1 s of free motion: %.3e J at 1 ms, %.3e J at 0.5 ms (|E0| up to %.1f J, |qd| up to "
          "%.0f rad/s)" % (drift[0], drift[1], np.abs(E0).max(), np.abs(out["qd_traj"]).max()))
    # the arm falls freely and joint 7 spins up to ~80 rad/s: the drift is RK4's truncation, and it shrinks as dt^4
    assert drift[0] <= 1e-4
    assert drift[0] / drift[1] >= 8.0


def monotone_case(run, T, seed):
    """Rollouts and joints whose position and |velocity| move strictly monotonically over the T stored states:
    -> q_traj, qd_traj and a list of (rollout, joint, increasing position?)."""
    q, qd, tau, mass = rollout_inputs(256, seed, n_steps=T)
    q_traj, qd_traj = run(q, qd, tau, mass)
    picks = []
    for i in range(q.shape[1]):
        for j in range(7):
            dq = np.diff(q_traj[:, j, i])
            dv = np.diff(np.abs(qd_traj[:, j, i]))
            if (dv > 0).all() and ((dq > 0).all() or (dq < 0).all()):
                picks.append((i, j, bool(dq[0] > 0)))
    assert len(picks) >= 4, len(picks)
    return (q, qd, tau, mass), q_traj, qd_traj, picks


def check_limit_boundaries(run, run_fv, T, seed):
    """CPU test 5 on any rollout implementation: run(q, qd, tau, mass) -> (q_traj, qd_traj); run_fv(inputs, q_lo, q_hi,
    qd_max) -> first_violation.  A limit equal to a stored value passes; one ulp inward fails at exactly that step."""
    inputs, q_traj, qd_traj, picks = monotone_case(run, T, seed)
    inf = np.full(7, np.inf)
    for i, j, up in picks[:4]:
        for k in sorted({0, 1, T - 1}):
            x, v = q_traj[k, j, i], abs(qd_traj[k, j, i])
            lo, hi = -inf.copy(), inf.copy()
            (hi if up else lo)[j] = x
            assert run_fv(inputs, lo, hi, None)[i] > k, (i, j, k, up)
            (hi if up else lo)[j] = np.nextafter(x, -np.inf if up else np.inf)
            assert run_fv(inputs, lo, hi, None)[i] == k, (i, j, k, up)
            vmax = inf.copy()
            vmax[j] = v
            assert run_fv(inputs, None, None, vmax)[i] > k
            vmax[j] = np.nextafter(v, 0.0)
            assert run_fv(inputs, None, None, vmax)[i] == k
    # no check at all: n_steps; checks that cannot fail: n_steps
    assert (run_fv(inputs, None, None, None) == T).all()
    assert (run_fv(inputs, -inf, inf, inf) == T).all()


def test_limit_compare_at_its_exact_boundary(L):
    T = 8
    run = lambda q, qd, tau, m: (lambda o: (o["q_traj"], o["qd_traj"]))(host_rollout(L, q, qd, tau, 1e-3, T, m))
    run_fv = lambda x, lo, hi, vm: host_rollout(L, *x[:3], 1e-3, T, x[3], q_lo=lo, q_hi=hi,
                                                qd_max=vm)["first_violation"]
    check_limit_boundaries(run, run_fv, T, 340)


def test_nan_states_violate_and_the_rollout_continues(L):
    q, qd, tau, mass = rollout_inputs(8, 350, n_steps=6, per_step=True)
    tau[3, 2, 5] = np.nan                       # rollout 5 turns NaN at step 3
    inf = np.full(7, np.inf)
    out = host_rollout(L, q, qd, tau, 1e-3, 6, mass, tau_per_step=True, q_lo=-inf, q_hi=inf)
    assert out["first_violation"][5] == 3 and (np.delete(out["first_violation"], 5) == 6).all()
    assert np.isfinite(out["q_traj"][:3, :, 5]).all() and np.isnan(out["q_traj"][3:, :, 5]).all()
    out = host_rollout(L, q, qd, tau, 1e-3, 6, mass, tau_per_step=True, qd_max=inf)
    assert out["first_violation"][5] == 3
    # a rollout that fails at step 0 still runs all its steps: same trajectory as the unchecked call
    lo = Q_HI.copy()
    checked = host_rollout(L, q, qd, tau, 1e-3, 6, mass, tau_per_step=True, q_lo=lo, q_hi=Q_HI)
    assert (checked["first_violation"] == 0).all()
    assert np.array_equal(checked["q_traj"], out["q_traj"], equal_nan=True)


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_nonfinite_inputs(L, mode):
    T = 5
    q, qd, tau, mass = rollout_inputs(9, 360, n_steps=T, per_step=True)
    base = host_rollout(L, q, qd, tau, 1e-3, T, mass, mode, True)
    assert np.isfinite(base["q_traj"]).all()
    k = 4
    for what in ("q", "qd", "tau", "mass", "tau_step"):
        for j in (0, 3, 6):
            for v in (np.nan, np.inf, -np.inf):
                a = {"q": q.copy(), "qd": qd.copy(), "tau": tau.copy(), "mass": mass.copy()}
                if what == "mass":
                    a["mass"][k] = v
                elif what == "tau":
                    a["tau"][:, j, k] = v
                elif what == "tau_step":
                    a["tau"][2, j, k] = v
                else:
                    a[what][j, k] = v
                out = host_rollout(L, a["q"], a["qd"], a["tau"], 1e-3, T, a["mass"], mode, True)
                others = np.arange(q.shape[1]) != k
                for key in ("q_traj", "qd_traj"):
                    assert np.array_equal(out[key][:, :, others], base[key][:, :, others])
                s0 = 2 if what == "tau_step" else 0
                assert np.array_equal(out["q_traj"][:s0, :, k], base["q_traj"][:s0, :, k])
                assert np.isnan(out["q_traj"][s0:, :, k]).all() and np.isnan(out["qd_traj"][s0:, :, k]).all(), \
                    (what, j, v)


def test_operation_counts(L):
    """What bench_rollout.py reports: 4 x K13's qdd count (sincos of joints 2..7 included) + the RK4 combination."""
    comb = L.host_rollout_combination_flops()
    assert comb == 7 * 26
    assert L.host_fd_flops(0) + L.host_fd_flops(1) > 10 * comb


# ---- the C ABI, without a GPU -------------------------------------------------------------------------------------
def test_argument_validation_without_gpu():
    from torque_constrained_motion_planning_b200 import _lib, engine
    lib = _lib.load()
    f = lib.tcmp_rollout_batch
    p = ctypes.c_void_p(0x1000)      # never dereferenced: every call below is rejected or empty
    lo, hi, vm = (np.ascontiguousarray(a) for a in (Q_LO, Q_HI, V_LIM))
    L7 = lambda a: a.ctypes.data

    def call(mode=0, n=4, T=3, dt=1e-3, q0=p, lo_=None, hi_=None, vm_=None, outs=(p, None, None, None, None),
             model=None):
        return f(model, mode, n, T, dt, q0, None, None, 0, None, 0.0, lo_, hi_, vm_, *outs, None)

    def rejected(why, **kw):
        ns = (kw.pop("n"),) if "n" in kw else (4,) if why in ("q0 is NULL", "output") else (4, 0)
        for n in ns:
            assert call(n=n, **kw) == -1, (why, n)
            assert why.encode() in lib.tcmp_last_error(), (why, lib.tcmp_last_error())

    for mode in (1, 3, 4, -1):
        rejected("mode", mode=mode)
    rejected("negative", n=-1)
    for T in (0, -3):
        rejected("n_steps", T=T)
    for dt in (0.0, -1e-3, np.nan, np.inf, -np.inf):
        rejected("dt", dt=dt)
    bad = engine.InertialModel.default()
    bad.mass[2] = -1.0
    rejected("mass", model=bad.record.ctypes.data)
    rejected("q0 is NULL", q0=None)
    rejected("output", outs=(None,) * 5)
    rejected("both", lo_=L7(lo))
    rejected("both", hi_=L7(hi))
    for arr, key in ((lo, "lo_"), (hi, "hi_")):
        nanl = arr.copy()
        nanl[3] = np.nan
        kw = {"lo_": L7(lo), "hi_": L7(hi)}
        kw[key] = L7(nanl)
        rejected("NaN", **kw)
    for v in (-1e-9, np.nan):
        bad_vm = vm.copy()
        bad_vm[6] = v
        rejected("qd_max", vm_=L7(bad_vm))
    # accepted limits: infinite ones, zero velocity limits; n == 0 is OK whatever the buffers
    zero = np.zeros(7)
    inf = np.full(7, np.inf)
    assert call(n=0, q0=None, lo_=L7(-inf), hi_=L7(inf), vm_=L7(zero), outs=(None,) * 5) == 0
    assert call(n=0, q0=None, outs=(None,) * 5, model=engine.InertialModel.default().record.ctypes.data) == 0
    with pytest.raises(ValueError):
        engine.rollout_batch(np.zeros((7, 1)), q_lo=Q_LO)


def test_library_carries_the_rollout_kernel_as_sm_100a_code():
    from torque_constrained_motion_planning_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    usage = subprocess.run([cuobjdump, "-res-usage", _lib.LIB_PATH], capture_output=True, text=True).stdout
    blocks = re.findall(r"Function (\S*rollout_kernel\S*):\s*\n\s*(REG:\d+ STACK:\d+ SHARED:\d+ LOCAL:\d+)", usage)
    assert len(blocks) == 8, usage[:2000]      # {int, int64 offsets} x {rne, dyn} x {compiled-in, record}
    for name, res in blocks:
        assert "LOCAL:0" in res, (name, res)
    log = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "build", "rollout_kernels.cu.ptxas.log")
    if os.path.exists(log):
        props = re.findall(r"Function properties for (\S*rollout_kernel\S*)\n\s*(\d+) bytes stack frame, "
                           r"(\d+) bytes spill stores, (\d+) bytes spill loads", open(log).read())
        assert len(props) == 8 and all(st == "0" and ld == "0" for _, _, st, ld in props), props
