"""CPU: the long-double min-jerk reference (tests/minjerk_reference.py) against the C oracle and the golden vectors, its
boundary-case generators against the oracle's edge and trajectory checks, and a non-finite joint-1 angle through the
host build of csrc/panda_model.cuh (the recursion every torque kernel runs)."""
import ctypes

import numpy as np
import pytest

import minjerk_reference as R
import oracle
from conftest import load_golden, sample_states
from test_rne_core_host import host_rne  # noqa: F401  (fixture: the host build of panda_model.cuh)

MODES = ("rne", "nov", "dyn")


def test_oracle_linspace_sample_is_numpy_linspace():
    f = oracle.lib().oracle_linspace_sample
    f.restype = ctypes.c_double
    f.argtypes = [ctypes.c_int, ctypes.c_int]
    for S in range(1, 4097):
        want = R.linspace_times(S)
        got = np.array([f(S, i) for i in range(S)])
        assert np.array_equal(got, want), S


def _within(got, want, bound):
    err = np.abs(np.asarray(got, np.float64).astype(R.LD) - want).astype(np.float64)
    return bool((err <= bound).all())


def test_long_double_sampling_agrees_with_oracle_and_golden():
    g = load_golden("minjerk.npz")
    for p in ("p2", "p5", "p20", "p3_1"):
        c, S = g[p + "_coeffs"], int(g[p + "_n"])
        assert np.abs(oracle.minjerk_coefficients(g[p + "_points"]) - c).max() == 0
        ref, bounds = R.traj_samples(c, S)
        ox, ov, oa = oracle.minjerk_trajectory(c, S)
        for got_g, got_o, want, b in zip((g[p + "_x"], g[p + "_v"], g[p + "_a"]), (ox, ov, oa), ref, bounds):
            assert _within(got_g, want, b) and _within(got_o, want, b), p
    t = load_golden("traj.npz")
    c = oracle.minjerk_coefficients(t["points"])
    ref, bounds = R.traj_samples(c, int(t["n_int"]))
    for got, want, b in zip((t["x"], t["v"], t["a"]), ref, bounds):
        assert _within(got, want, b)
    # the two-point edge form and the general quintic on the edge's coefficients describe the same samples
    qa, qb = R.sample_edges(64, 3)
    for W in (1, 7, 64, 1000):
        (ex, ev, ea), eb = R.edge_samples(qa, qb, W)
        (tx, tv, ta), _ = R.traj_samples(R.edge_coeffs(qa, qb), W)
        ox, ov, oa = oracle.minjerk_trajectory(R.edge_coeffs(qa, qb)[:1], W)
        for e_, t_, b in zip((ex, ev, ea), (tx, tv, ta), eb):
            assert (np.abs(e_.reshape(-1, 7) - t_).astype(np.float64) <= b.reshape(-1, 7)).all()
        for o_, e_, b in zip((ox, ov, oa), (ex, ev, ea), eb):
            assert _within(o_, e_[0], b[0])


@pytest.mark.parametrize("model_name", [None, "override"])
@pytest.mark.parametrize("mode", MODES)
def test_edge_cases_give_the_designed_first_failure(mode, model_name):
    model = None if model_name is None else R.override_model()
    cases = R.edge_family(mode, model_name)
    R.check_edge_cases(cases, lambda qa, qb, W, m: oracle.edge_feasibility(mode, qa, qb, W, m, model=model))
    assert all(c.clearance >= 0.5 * c.delta for c in cases)
    # the shapes of failure the kernels' warp reduction must get right are all present
    assert any(c.first == 31 and c.lanes_in_first_round == 1 for c in cases)
    assert any(len(c.fail_rounds) >= 2 for c in cases)
    assert any(c.lanes_in_first_round >= 3 for c in cases)
    assert any(c.delta == 1.0 and c.first < c.W for c in cases) and any(c.delta == 1.0 and c.first == c.W for c in cases)


@pytest.mark.parametrize("mode", ["rne", "dyn"])
def test_threshold_edges_flip_at_the_payload_threshold(mode):
    found = R.threshold_edge(mode)
    assert found is not None
    qa, qb, (m_lo, f_lo), (m_hi, f_hi) = found
    assert f_lo != f_hi
    for m, f in ((m_lo, f_lo), (m_hi, f_hi)):
        assert oracle.edge_feasibility(mode, qa[:, None], qb[:, None], 64, m, 0.01)[0] == f


@pytest.mark.parametrize("mode", MODES)
def test_trajectory_cases_give_the_designed_first_failure(mode):
    by_key = {(c.W, c.first, c.delta): c for c in R.edge_family(mode)}
    S = 64
    for first_local, n_seg, at_seg in ((0, 20, 0), (S - 1, 20, 0), (0, 20, 1), (30, 20, 19), (S - 1, 20, 19),
                                      (S, 20, 5)):
        case = by_key[(S, first_local, R.DELTAS[0])]
        ref = R.traj_reference(mode, R.traj_with_failure(case, S, n_seg, at_seg), S, case.mass)
        want = n_seg * S if first_local == S else at_seg * S + first_local
        assert ref["first_fail"] == want and not ref["in_band"].any()
        if first_local < S and at_seg < n_seg - 1:
            assert (~ref["feasible"]).sum() > 1


@pytest.mark.parametrize("model_name", [None, "override"])
@pytest.mark.parametrize("mode", MODES)
def test_nonfinite_joint1_gives_nan_torques_like_the_oracle(host_rne, mode, model_name):  # noqa: F811
    """rne.py rotates by joint 1's angle although gravity lies along its axis: q[0] = NaN or +-inf makes every torque
    NaN there, and NaN never compares >= a limit, so the state is feasible.  The recursion must do the same."""
    model = None if model_name is None else R.override_model()
    q, qd, qdd, mass = sample_states(2000, seed=50)
    for v in (np.nan, np.inf, -np.inf):
        q[0] = v
        tau_o, ok_o = oracle.torque_test_batch(mode, q, qd, qdd, mass, model=model)
        tau, ok = host_rne(mode, q, qd, qdd, mass, model=model)
        assert np.isnan(tau_o).all() and ok_o.all()
        assert np.isnan(tau).all() and np.array_equal(ok, ok_o), (mode, v)
