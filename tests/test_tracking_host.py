"""CPU: K15's closed-loop tracking rollouts (csrc/track_core.cuh -- the same per-rollout source track_kernels.cu
instantiates) built for the host by tests/native/track_host.cpp.  Checked bit for bit against a NumPy composition of
the pinned reference, the exported controller torque, a NumPy clamp and K14's host build one step at a time; the
controller torque against K1's host build and the oracle; the closed loop against DOP853 for fourth order; the
physics of the error (zero-order hold, PD decay, payload mismatch); saturation against the torque test's designed edge
cases; the saturation compare at its exact boundary; the non-finite rules; the argument validation of
tcmp_track_batch and the sm_100a code of the kernel."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import minjerk_reference as mj
import oracle
from conftest import Q_HI, Q_LO, ROOT, V_LIM, sample_edges, sample_states
from test_rollout_host import MODE, MODELS, _arr, _p, fd, first_violation, host_rollout, limits, model_record

NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "csrc")
_i32p = ctypes.POINTER(ctypes.c_int32)
KP, KD = np.full(7, 100.0), np.full(7, 20.0)           # critically damped: kd = 2 sqrt(kp)


def load_track_host():
    so = os.path.join(NATIVE, "libtrack_host.so")
    src = os.path.join(NATIVE, "track_host.cpp")
    deps = [src] + [os.path.join(NATIVE, f) for f in ("rollout_host.cpp", "fd_host.cpp", "dynamics_host.cpp")] + \
        [os.path.join(CSRC, f) for f in ("track_core.cuh", "rollout_core.cuh", "fd_core.cuh", "dynamics_core.cuh",
                                         "panda_model.cuh", "sincos_table.inc")] + [os.path.join(ROOT, "include", "tcmp.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                               "-Wno-unknown-pragmas", "-o", so, src])
    L = ctypes.CDLL(so)
    for f in ("host_fd_flops", "host_sincos_flops", "host_rollout_combination_flops", "host_track_flops"):
        getattr(L, f).restype = ctypes.c_int64
    return L


@pytest.fixture(scope="module")
def L():
    return load_track_host()


def host_track(L, coeffs, dt, n_steps, kp=KP, kd=KD, q0=None, qd0=None, mass=0.0, ctrl_mass=None, mode="rne",
               q_lo=None, q_hi=None, qd_max=None, model=None, n=None):
    """-> every output of the host build; coeffs [n_seg][7][6] (shared) or [n_seg][7][6][n]."""
    coeffs = _arr(coeffs)
    q0, qd0 = _arr(q0), _arr(qd0)
    n = coeffs.shape[3] if coeffs.ndim == 4 else n if n is not None else (q0 if q0 is not None else qd0).shape[1]
    ctrl_mass = mass if ctrl_mass is None else ctrl_mass
    pm, cm = (None if np.ndim(m) == 0 else _arr(m) for m in (mass, ctrl_mass))
    lim = [None if a is None else _arr(np.broadcast_to(a, (7,))) for a in (q_lo, q_hi, qd_max)]
    T = n_steps
    out = {"q": np.empty((7, n)), "qd": np.empty((7, n)), "q_traj": np.empty((T, 7, n)),
           "qd_traj": np.empty((T, 7, n)), "tau_traj": np.empty((T, 7, n)),
           "first_violation": np.empty(n, np.int32), "first_saturation": np.empty(n, np.int32),
           "max_err": np.empty(n)}
    L.host_track_batch(_p(_arr(model)), MODE[mode], ctypes.c_int64(n), T, ctypes.c_double(dt), coeffs.shape[0],
                       _p(coeffs), int(coeffs.ndim == 3), _p(q0), _p(qd0), _p(_arr(np.broadcast_to(kp, (7,)))),
                       _p(_arr(np.broadcast_to(kd, (7,)))), _p(pm), ctypes.c_double(0.0 if pm is not None else mass),
                       _p(cm), ctypes.c_double(0.0 if cm is not None else ctrl_mass), *(_p(a) for a in lim),
                       *(_p(out[k]) for k in ("q", "qd", "q_traj", "qd_traj", "tau_traj")),
                       *(out[k].ctypes.data_as(_i32p) for k in ("first_violation", "first_saturation")),
                       _p(out["max_err"]))
    return out


def control(L, q, qd, acmd, ctrl_mass, mode="rne", model=None):
    """The exported controller torque (unsaturated)."""
    q, qd, acmd = _arr(q), _arr(qd), _arr(acmd)
    n = q.shape[1]
    cm = None if np.ndim(ctrl_mass) == 0 else _arr(ctrl_mass)
    tau = np.empty((7, n))
    L.host_track_control(_p(_arr(model)), MODE[mode], ctypes.c_int64(n), _p(q), _p(qd), _p(acmd), _p(cm),
                         ctypes.c_double(0.0 if cm is not None else float(ctrl_mass)), _p(tau))
    return tau


def reference(coeffs, t, n, want_va=True):
    """include/tcmp.h's reference at time t for n rollouts -> x, v, a [7][n] (v = a = 0 in the hold)."""
    c = np.asarray(coeffs)
    n_seg = c.shape[0]
    hold = not (t < float(n_seg))
    s = n_seg - 1 if hold else int(t)
    u = 1.0 if hold else t - float(s)
    cs = c[s] if c.ndim == 4 else np.broadcast_to(c[s][:, :, None], (7, 6, n))
    c0, c1, c2, c3, c4, c5 = (cs[:, k] for k in range(6))
    x = c0 + u * (c1 + u * (c2 + u * (c3 + u * (c4 + u * c5))))
    if hold:
        return x, np.zeros_like(x), np.zeros_like(x)
    v = c1 + u * (2.0 * c2 + u * (3.0 * c3 + u * (4.0 * c4 + u * (5.0 * c5))))
    a = 2.0 * c2 + u * (6.0 * c3 + u * (12.0 * c4 + u * (20.0 * c5)))
    return x, v, a


def saturate(tau, lim):
    L7 = np.asarray(lim)[:, None]
    over = np.abs(tau) > L7
    return np.where(over, np.copysign(np.broadcast_to(L7, tau.shape), tau), tau), over.any(axis=0)


def composed(L, coeffs, dt, T, kp, kd, q0, qd0, mass, ctrl_mass, mode, model, n):
    """Step by step: the NumPy reference, the exported controller torque, a NumPy clamp, host_rollout_batch(1)."""
    lim = limits(model)
    x0, v0, _ = reference(coeffs, 0.0, n)
    q = x0.copy() if q0 is None else np.array(q0)
    qd = v0.copy() if qd0 is None else np.array(qd0)
    qs, vs, taus = [], [], []
    first_sat = np.full(n, T, np.int32)
    err = np.zeros(n)
    for k in range(T):
        x, v, a = reference(coeffs, k * dt, n)
        acmd = (a + kp[:, None] * (x - q)) + kd[:, None] * (v - qd)
        tau, sat = saturate(control(L, q, qd, acmd, ctrl_mass, mode, model), lim)
        first_sat = np.where(sat & (first_sat == T), k, first_sat).astype(np.int32)
        o = host_rollout(L, q, qd, tau, dt, 1, mass, mode, model=model)
        q, qd = o["q"], o["qd"]
        err = np.maximum(err, np.abs(q - reference(coeffs, (k + 1) * dt, n)[0]).max(axis=0))
        qs.append(q)
        vs.append(qd)
        taus.append(tau)
    return np.stack(qs), np.stack(vs), np.stack(taus), first_sat, err


def edge_chain(n, seed, n_seg=2):
    """Per-rollout references [n_seg][7][6][n]: min-jerk edges chained through random waypoints."""
    pts = [sample_edges(n, seed)[0]]
    for s in range(n_seg):
        pts.append(sample_edges(n, seed + 1 + s)[1] * 0.3 + pts[-1] * 0.7)
    # C order: np.concatenate keeps the transposed views' layout, and the raw C ABI reads the buffer as it lies
    return np.ascontiguousarray(np.concatenate([mj.edge_coeffs(pts[s], pts[s + 1]).transpose(1, 2, 0)[None]
                                                for s in range(n_seg)]))


CASES = [(mode, name, payload, ctrl, bcast, start)
         for mode in ("rne", "dyn") for name in MODELS
         for payload, ctrl in (("scalar", "same"), ("per_rollout", "same"), ("scalar", "other"),
                               ("per_rollout", "other"))
         for bcast, start in ((True, "given"), (False, "null"), (True, "null"), (False, "given"))]


@pytest.mark.parametrize("mode,model_name,payload,ctrl,broadcast,start", CASES)
def test_track_is_the_numpy_composition_bit_for_bit(L, mode, model_name, payload, ctrl, broadcast, start):
    model = model_record(model_name)
    n, dt = 24, 0.07                      # 32 steps reach t = 2.24: both segment boundaries and the hold
    coeffs = edge_chain(n, 500)
    if broadcast:
        coeffs = np.ascontiguousarray(coeffs[..., 3])
    q, qd, _, mass = sample_states(n, seed=501)
    x0, v0, _ = reference(coeffs, 0.0, n)
    q0, qd0 = (x0 + 0.05 * np.tanh(q), v0 + 0.1 * np.tanh(qd)) if start == "given" else (None, None)
    m_p = 3.0 if payload == "scalar" else mass
    m_c = m_p if ctrl == "same" else (1.5 if payload == "scalar" else mass[::-1].copy())
    saw_sat = False
    for T in (1, 2, 7, 32):
        out = host_track(L, coeffs, dt, T, KP, KD, q0, qd0, m_p, m_c, mode, Q_LO, Q_HI, V_LIM, model, n=n)
        rq, rv, rt, fs, err = composed(L, coeffs, dt, T, KP, KD, q0, qd0, m_p, m_c, mode, model, n)
        same = lambda a, b: np.array_equal(a, b, equal_nan=True)
        assert same(out["q_traj"], rq) and same(out["qd_traj"], rv), (mode, T)
        assert same(out["tau_traj"], rt), T
        assert same(out["q"], rq[-1]) and same(out["qd"], rv[-1])
        assert np.array_equal(out["first_saturation"], fs) and same(out["max_err"], err)
        assert np.array_equal(out["first_violation"], first_violation(rq, rv, Q_LO, Q_HI, V_LIM))
        saw_sat = saw_sat or bool((fs < T).any())
    assert saw_sat or broadcast           # the edges saturate somewhere; one shared edge need not


def test_controller_torque_is_k1s_and_the_oracles(L):
    so = os.path.join(NATIVE, "librne_host.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                           "-o", so, os.path.join(NATIVE, "rne_host.cpp")])
    R = ctypes.CDLL(so)
    q, qd, qdd, mass = sample_states(5000, seed=510)
    tau = control(L, q, qd, qdd, mass)
    ref, ok = np.empty((7, q.shape[1])), np.empty(q.shape[1], np.uint8)
    R.host_rne_batch_table(ctypes.c_int64(q.shape[1]), *(_p(_arr(a)) for a in (q, qd, qdd, mass)), ctypes.c_double(0.0),
                           _p(ref), ok.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
    assert np.array_equal(tau, ref)
    worst = 0.0
    for mode in ("rne", "dyn"):
        for name in MODELS:
            model = model_record(name)
            t = control(L, q, qd, qdd, mass, mode, model)
            t_o, _ = oracle.torque_test_batch(mode, q, qd, qdd, mass, payload_threshold=0.0, model=model)
            worst = max(worst, float(np.abs(t - t_o).max()))
    print("controller torque vs oracle: max |diff| %.3e N.m" % worst)
    assert worst <= 1e-9


def test_closed_loop_is_fourth_order_against_dop853(L):
    """The plant between control instants by DOP853 (rtol 1e-12) under the torque that the oracle's inverse dynamics
    and the same clamp give at each step's start; err(dt) / err(dt/2), each against its own reference, is ~16."""
    from scipy.integrate import solve_ivp
    n = 16
    coeffs = edge_chain(n, 520, n_seg=1)
    x0, v0, _ = reference(coeffs, 0.0, n)
    q0 = x0 + 0.02
    mass, lim = 2.0, limits(None)
    horizon = 0.32

    def dop853(dt):
        q, v = q0.copy(), v0.copy()
        for k in range(int(round(horizon / dt))):
            x, vr, a = reference(coeffs, k * dt, n)
            acmd = (a + KP[:, None] * (x - q)) + KD[:, None] * (vr - v)
            tau, _ = oracle.torque_test_batch("rne", q, v, acmd, mass, payload_threshold=0.0)
            tau, _ = saturate(tau, lim)

            def rhs(_, y, tau=tau):
                s = y.reshape(2, 7, n)
                return np.concatenate([s[1], fd(L, s[0], s[1], tau, mass, "rne", None)]).ravel()
            y = solve_ivp(rhs, (0.0, dt), np.concatenate([q, v]).ravel(), method="DOP853", rtol=1e-12,
                          atol=1e-12).y[:, -1].reshape(2, 7, n)
            q, v = y[0], y[1]
        return q, v

    err = []
    for dt in (0.04, 0.02):
        rq, rv = dop853(dt)
        out = host_track(L, coeffs, dt, int(round(horizon / dt)), q0=q0, mass=mass)
        err.append(np.maximum(np.abs(out["q"] - rq).max(axis=0), np.abs(out["qd"] - rv).max(axis=0)))
    ratio = err[0] / err[1]
    print("closed loop vs DOP853: err at dt median %.3e; ratio median %.2f, range [%.2f, %.2f]"
          % (np.median(err[0]), np.median(ratio), ratio.min(), ratio.max()))
    assert np.median(err[1]) > 1e-10
    assert 12.0 <= np.median(ratio) <= 20.0


def test_zero_order_hold_error_is_first_order_in_dt(L):
    """Exact model, kp = kd = 0, a start on the reference, no saturation: max_err is the hold's error, ~ dt."""
    n = 32
    coeffs = edge_chain(n, 530, n_seg=1) * np.array([1, 1, 1, 0.3, 0.3, 0.3])[None, None, :, None]
    coeffs[0, :, 0] = edge_chain(n, 530, n_seg=1)[0, :, 0]
    errs = []
    for dt in (4e-3, 2e-3, 1e-3):
        out = host_track(L, coeffs, dt, int(round(1.0 / dt)), kp=0.0, kd=0.0, mass=1.0)
        assert (out["first_saturation"] == int(round(1.0 / dt))).all()
        errs.append(out["max_err"])
    r1, r2 = errs[0] / errs[1], errs[1] / errs[2]
    print("hold error at 1 ms: median %.3e rad; ratios per halving: median %.3f, %.3f"
          % (np.median(errs[2]), np.median(r1), np.median(r2)))
    assert 1.8 <= np.median(r1) <= 2.2 and 1.8 <= np.median(r2) <= 2.2


def test_pd_offset_decays_as_the_linear_closed_loop(L):
    """Critically damped PD (kp = w^2, kd = 2 w), exact model, an offset e0 at rest on a held reference: the error is
    e(t) = e0 (1 + w t) exp(-w t) up to the hold's O(dt) effect, down to the round-off floor."""
    n, w, dt = 16, 10.0, 1e-3
    q, _, _, _ = sample_states(n, seed=540)
    c = np.zeros((1, 7, 6, n))
    c[0, :, 0] = q
    e0 = 0.01
    T = 1500
    out = host_track(L, c, dt, T, kp=w * w, kd=2 * w, q0=q + e0, qd0=np.zeros_like(q), mass=1.0)
    t = (np.arange(T) + 1) * dt
    pred = e0 * (1 + w * t) * np.exp(-w * t)
    got = np.abs(out["q_traj"] - q[None]).max(axis=1)                      # [T][n]
    dev = np.abs(got - pred[:, None]).max()
    print("PD decay: |e(t) - e0 (1 + wt) exp(-wt)| <= %.3e rad (e0 = %.0e), final %.3e" % (dev, e0, got[-1].max()))
    assert dev <= 2e-2 * e0
    assert got[-1].max() <= 1e-6


def test_error_grows_with_payload_mismatch(L):
    n = 8
    coeffs = edge_chain(n, 550, n_seg=1)
    x0, v0, _ = reference(coeffs, 0.0, n)
    err = []
    masses = (0.0, 0.5, 1.0, 2.0, 3.0)
    for mp in masses:
        err.append(host_track(L, coeffs, 1e-3, 1200, mass=mp, ctrl_mass=0.0)["max_err"])
    err = np.array(err)
    matched = host_track(L, coeffs, 1e-3, 1200, mass=2.0, ctrl_mass=2.0)["max_err"]
    print("max_err by plant mass %s (controller 0 kg), median over rollouts: %s; matched at 2 kg: %.3e"
          % (masses, np.median(err, axis=1), np.median(matched)))
    assert (np.diff(err, axis=0) > 0).all()
    assert np.abs(matched - err[0]).max() <= 0.5 * err[1].min()


def unlimited_record():
    """The stock robot's record with torque limits no torque reaches: its tau_traj is the commanded torque."""
    rec = oracle.default_model()
    oracle.model_fields(rec)["torque_limit"][:] = 1e9
    return rec


def check_edge_saturation(run, mode):
    """CPU check 5 on any implementation: run(coeffs [1][7][6][1], dt, n_steps, mass, model) -> (tau_traj [T][7],
    first_saturation).  Each designed edge as a one-segment reference, dt = 1/W, W + 1 steps (step k samples waypoint
    k - 1), plant mass = controller mass = the case's, kp = kd = 0: a case feasible by delta never saturates joints
    0..5; one failing at `first` saturates first at step first + 1.  Asserted where the commanded torque (a run without
    reachable limits, identical up to the first saturation) stays within delta of the oracle torque on the reference
    up to the deciding step, step 0 (t = 0, not a waypoint) does not saturate, and joint 7 stays delta inside its
    limit (first_saturation counts joint 7, the torque test does not).  -> (checked, excluded)."""
    lim = limits(None)
    used = excluded = 0
    for case in mj.edge_family(mode):
        W = case.W
        c = np.ascontiguousarray(mj.edge_coeffs(case.qa[:, None], case.qb[:, None]).transpose(1, 2, 0)[None])
        tau, fs = run(c, 1.0 / W, W + 1, case.mass, None)
        cmd, _ = run(c, 1.0 / W, W + 1, case.mass, unlimited_record())
        (x, v, a), _ = mj.edge_samples(case.qa[:, None], case.qb[:, None], W)
        tau_o = mj.torques(mode, x.reshape(-1, 7), v.reshape(-1, 7), a.reshape(-1, 7), case.mass)   # [W][7]
        upto = W if case.first == W else case.first + 1
        ok = (np.abs(cmd[1:upto + 1] - tau_o[:upto]).max() < case.delta and (np.abs(cmd[0]) <= lim).all()
              and (np.abs(tau_o[:upto, 6]) <= lim[6] - case.delta).all())
        if not ok:
            excluded += 1
            continue
        used += 1
        assert fs == (W + 1 if case.first == W else case.first + 1), (W, case.first, case.delta)
    return used, excluded


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_saturation_against_the_torque_tests_edge_cases(L, mode):
    def run(c, dt, T, mass, model):
        o = host_track(L, c, dt, T, kp=0.0, kd=0.0, mass=mass, mode=mode, model=model)
        return o["tau_traj"][:, :, 0], int(o["first_saturation"][0])
    used, excluded = check_edge_saturation(run, mode)
    print("%s: %d designed edge cases checked, %d excluded by the preconditions" % (mode, used, excluded))
    assert used >= 10


def test_saturation_compare_at_its_exact_boundary(L):
    """A record whose limit equals |tau_cmd_j| exactly: no saturation, tau unchanged; one ulp below: tau = +-L."""
    n = 6
    coeffs = edge_chain(n, 560, n_seg=1)
    x0, v0, a0 = reference(coeffs, 0.0, n)
    q0 = x0 + 0.1                         # a_cmd = -1 rad/s^2 on every joint: no torque is exactly 0
    acmd = (a0 + 10.0 * (x0 - q0)) + 0.0 * (v0 - v0)
    tau = control(L, q0, v0, acmd, 1.0, model=oracle.default_model())     # the record's torques (limits unused)
    assert (tau != 0).all()
    for j in (0, 4, 6):
        for i in range(n):
            rec = oracle.default_model()
            f = oracle.model_fields(rec)
            f["torque_limit"][:] = 1e6
            run = lambda: host_track(L, coeffs[..., i:i + 1], 1e-3, 1, kp=10.0, kd=0.0, q0=q0[:, i:i + 1], mass=1.0,
                                     model=rec)
            f["torque_limit"][j] = abs(tau[j, i])
            out = run()
            assert out["first_saturation"][0] == 1 and out["tau_traj"][0, j, 0] == tau[j, i]
            f["torque_limit"][j] = np.nextafter(abs(tau[j, i]), 0.0)
            out = run()
            assert out["first_saturation"][0] == 0
            assert out["tau_traj"][0, j, 0] == np.copysign(f["torque_limit"][j], tau[j, i])


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_nonfinite_inputs(L, mode):
    n, T = 9, 68
    coeffs = edge_chain(n, 570)
    x0, v0, _ = reference(coeffs, 0.0, n)
    q0, qd0 = x0 + 0.01, v0.copy()
    mass, cmass = np.full(n, 2.0), np.full(n, 1.0)
    dt, kp, kd = 1.0 / 64, KP, KD         # steps 0..63 in segment 0, 64.. in segment 1
    base = host_track(L, coeffs, dt, T, kp, kd, q0=q0, qd0=qd0, mass=mass, ctrl_mass=cmass, mode=mode)
    assert np.isfinite(base["q_traj"]).all() and np.isfinite(base["max_err"]).all()
    k = 4
    for what in ("q0", "qd0", "mass", "cmass", "coeff0", "coeff1"):
        for v in (np.nan, np.inf, -np.inf):
            a = {"q0": q0.copy(), "qd0": qd0.copy(), "mass": mass.copy(), "cmass": cmass.copy(), "c": coeffs.copy()}
            if what in ("q0", "qd0"):
                a[what][3, k] = v
            elif what in ("mass", "cmass"):
                a[what][k] = v
            else:
                a["c"][int(what[-1]), 2, 5, k] = v
            out = host_track(L, a["c"], dt, T, kp, kd, q0=a["q0"], qd0=a["qd0"], mass=a["mass"],
                             ctrl_mass=a["cmass"], mode=mode)
            others = np.arange(n) != k
            for key in ("q_traj", "qd_traj", "tau_traj", "max_err", "first_saturation"):
                assert np.array_equal(out[key][..., others], base[key][..., others]), (what, key)
            s0 = 64 if what == "coeff1" else 0    # segment 1 is first read at step 64 (t = 1)
            t0 = s0 + (what == "mass")            # the plant's mass reaches the torque through the state
            assert np.array_equal(out["tau_traj"][:t0, :, k], base["tau_traj"][:t0, :, k]), what
            assert np.isnan(out["tau_traj"][t0:, :, k]).all(), (what, v)
            assert np.isnan(out["q_traj"][s0:, :, k]).all() and np.isnan(out["max_err"][k]), (what, v)


def test_operation_counts(L):
    """What bench_tracking.py adds to K14's count: the controller's rne_body, the reference and a_cmd, the error."""
    assert L.host_track_flops(1) == 7 * 38 and L.host_track_flops(2) == 7 * 11
    assert L.host_track_flops(0) > L.host_track_flops(1) + L.host_track_flops(2)


# ---- the C ABI, without a GPU -------------------------------------------------------------------------------------
def test_argument_validation_without_gpu():
    from torque_constrained_motion_planning_b200 import _lib, engine
    lib = _lib.load()
    f = lib.tcmp_track_batch
    p = ctypes.c_void_p(0x1000)      # never dereferenced: every call below is rejected or empty
    kp, kd = np.ascontiguousarray(KP), np.ascontiguousarray(KD)
    lo, hi, vm = (np.ascontiguousarray(a) for a in (Q_LO, Q_HI, V_LIM))
    A = lambda a: a.ctypes.data

    def call(mode=0, n=4, T=3, dt=1e-3, n_seg=1, coeffs=p, kp_=A(kp), kd_=A(kd), lo_=None, hi_=None, vm_=None,
             outs=(p,) + (None,) * 7, model=None):
        return f(model, mode, n, T, dt, n_seg, coeffs, 1, None, None, kp_, kd_, None, 0.0, None, 0.0, lo_, hi_, vm_,
                 *outs, None)

    def rejected(why, ns=(4, 0), **kw):
        for n in ns:
            assert call(n=n, **kw) == -1, (why, n)
            assert why.encode() in lib.tcmp_last_error(), (why, lib.tcmp_last_error())

    for mode in (1, 3, 4, -1):
        rejected("mode", mode=mode)
    rejected("negative", ns=(-1,))
    for T in (0, -3):
        rejected("n_steps", T=T)
    for dt in (0.0, -1e-3, np.nan, np.inf):
        rejected("dt", dt=dt)
    bad = engine.InertialModel.default()
    bad.mass[2] = -1.0
    rejected("mass", model=bad.record.ctypes.data)
    rejected("both", lo_=A(lo))
    nanl = lo.copy()
    nanl[3] = np.nan
    rejected("NaN", lo_=A(nanl), hi_=A(hi))
    bad_vm = vm.copy()
    bad_vm[6] = -1.0
    rejected("qd_max", vm_=A(bad_vm))
    for ns in (0, -2):
        rejected("n_seg", n_seg=ns)
    rejected("kp and kd", kp_=None)
    rejected("kp and kd", kd_=None)
    for v in (-1.0, np.nan, np.inf):
        for which in ("kp_", "kd_"):
            g = kp.copy()
            g[5] = v
            rejected("gains", **{which: A(g)})
    rejected("coeffs is NULL", ns=(4,), coeffs=None)
    rejected("output", ns=(4,), outs=(None,) * 8)
    # n == 0 is OK whatever the buffers; q0 may be NULL
    assert call(n=0, coeffs=None, outs=(None,) * 8) == 0
    assert call(n=0, coeffs=None, lo_=A(lo), hi_=A(hi), vm_=A(np.zeros(7)), outs=(None,) * 8) == 0
    with pytest.raises(ValueError):
        engine.track_batch(np.zeros((1, 7, 6)), 1e-3, 1, 1.0, 1.0)            # shared coefficients, no n
    with pytest.raises(ValueError):
        engine.track_batch(np.zeros((1, 7, 5)), 1e-3, 1, 1.0, 1.0, n=1)
    with pytest.raises(ValueError):
        engine.track_batch(np.zeros((1, 7, 6)), 1e-3, 1, 1.0, 1.0, n=1, q_lo=Q_LO)


def test_edge_coefficients_are_the_edge_kernels_min_jerk():
    from torque_constrained_motion_planning_b200 import engine
    qa, qb = sample_edges(5, 580)
    c = engine.edge_coefficients(qa, qb)
    assert c.shape == (1, 7, 6, 5)
    assert np.array_equal(c[0].transpose(2, 0, 1), mj.edge_coeffs(qa, qb))


def test_library_carries_the_track_kernel_as_sm_100a_code():
    from torque_constrained_motion_planning_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    usage = subprocess.run([cuobjdump, "-res-usage", _lib.LIB_PATH], capture_output=True, text=True).stdout
    blocks = re.findall(r"Function (\S*track_kernel\S*):\s*\n\s*(REG:\d+ STACK:\d+ SHARED:\d+ LOCAL:\d+)", usage)
    assert len(blocks) == 8, usage[:2000]      # {int, int64 offsets} x {rne, dyn} x {compiled-in, record}
    for name, res in blocks:
        assert "LOCAL:0" in res, (name, res)
    log = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "build", "track_kernels.cu.ptxas.log")
    if os.path.exists(log):
        props = re.findall(r"Function properties for (\S*track_kernel\S*)\n\s*(\d+) bytes stack frame, "
                           r"(\d+) bytes spill stores, (\d+) bytes spill loads", open(log).read())
        assert len(props) == 8 and all(st == "0" and ld == "0" for _, _, st, ld in props), props
