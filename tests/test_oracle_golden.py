"""CPU: the C oracle (oracle/rne_oracle.c) against golden vectors produced by the UNMODIFIED
reference (oracle/make_golden.py) and against SURVEY.md Appendix B known answers."""
import math

import numpy as np
import pytest

import oracle
from conftest import load_golden

Q_HOME = [0, -math.pi / 4, 0.0, -3 * math.pi / 4, 0, math.pi / 2, math.pi / 4]

# SURVEY.md Appendix B, captured from the reference during the survey
KAT = [
    (Q_HOME, [0] * 7, [0] * 7, 0.0,
     [4.116468857429579e-18, -3.8185811407630106, -0.6440003196651124, 21.722207990949524, 0.6338461854898331,
      2.2807151301040953, 8.482515890803612e-18], True),
    (Q_HOME, [0] * 7, [0] * 7, 1.0,
     [6.875373572988104e-17, -6.829177599039773, -0.644000319665112, 26.352527990949525, 0.6338461854898331,
      3.1439951301040954, 8.482515890803612e-18], True),
    (Q_HOME, [0] * 7, [0] * 7, 5.0,
     [3.62777831858652e-17, -18.871563432146786, -0.6440003196651103, 44.87380799094953, 0.633846185489833,
      6.597115130104095, 8.482515890803612e-18], True),
    (Q_HOME, [0.1] * 7, [0.2] * 7, 1.0,
     [0.28705338153374077, -6.717120688516587, -0.251006678143913, 26.46715515507654, 0.694375126666447,
      3.19981432844381, -0.017970786750102868], True),
    ([0.5, 0.9, -0.3, -1.2, 0.7, 2.5, -1.0], [1, -0.5, 0.8, -1.2, 0.3, 0.9, -2], [3, -4, 2, 5, -1, 2.5, -6], 5.0,
     [32.97269121922599, -135.2546094950906, 1.256744471212042, 75.8608410279572, -0.7007246594455788,
      12.381408550524942, -1.3170570244757673], False),
    ([0] * 7, [0] * 7, [0] * 7, 0.0,
     [8.510968221163834e-32, -4.021462307689471, 7.654655230781446e-32, -3.22053441196239, -1.5106557604274467e-32,
      2.28124719855189, 9.293245291771726e-18], True),
]


@pytest.mark.parametrize("case", range(len(KAT)))
def test_appendix_b_kats(case):
    q, qd, qdd, m, tau_ref, ok_ref = KAT[case]
    col = lambda v: np.asarray(v, dtype=np.float64).reshape(7, 1)
    tau, ok = oracle.torque_test_batch("rne", col(q), col(qd), col(qdd), m)
    assert np.abs(tau[:, 0] - np.array(tau_ref)).max() < 1e-12
    assert bool(ok[0]) == ok_ref


def test_kat_file_and_payload_rule():
    g = load_golden("kat_rne.npz")
    tau, ok = oracle.torque_test_batch("rne", g["q"], g["qd"], g["qdd"], g["mass"])
    assert np.abs(tau - g["tau"]).max() < 1e-12
    assert (ok == g["feasible"]).all()
    # raw rne.add_payload rule (m > 0) differs from the torque-test rule (m > 0.01) for 0 < m <= 0.01
    tau_raw, _ = oracle.torque_test_batch("rne", g["q"], g["qd"], g["qdd"], g["mass"], payload_threshold=0.0)
    assert np.abs(tau_raw - g["tau_raw"]).max() < 1e-12
    assert np.abs(g["tau"][:, 6] - g["tau_raw"][:, 6]).max() > 1e-6  # the 0.005 kg case really differs


@pytest.mark.parametrize("mode", ["rne", "nov"])
def test_states_cfg2(mode):
    g = load_golden("states_cfg2.npz")
    tau, ok = oracle.torque_test_batch(mode, g["q"], g["qd"], g["qdd"], g["mass"])
    assert np.abs(tau - g["tau_" + mode]).max() < 1e-12
    assert (ok == g["feasible_" + mode]).all()
    assert 0.05 < 1.0 - ok.mean() < 0.5 or mode == "nov"  # the set exercises both outcomes


def test_model_override_vs_reference():
    """The model-parametrised oracle against rne.py run with its module-level inertial lists overwritten
    (oracle/make_golden.py gen_model): every link perturbed, link8 massive with an off-axis COM, another payload
    lever, tighter limits."""
    g = load_golden("model_override.npz")
    tau, ok = oracle.torque_test_batch("rne", g["q"], g["qd"], g["qdd"], g["mass"], model=g["model"])
    assert np.abs(tau - g["tau_rne"]).max() < 1e-12 and (ok == g["feasible_rne"]).all()
    tau, ok = oracle.torque_test_batch("nov", g["q"], None, None, g["mass"], model=g["model"])
    assert np.abs(tau - g["tau_nov"]).max() < 1e-12 and (ok == g["feasible_nov"]).all()
    # and it is a different robot: the stock tables give other torques on the same states
    tau0, _ = oracle.torque_test_batch("rne", g["q"], g["qd"], g["qdd"], g["mass"])
    assert np.abs(tau0 - g["tau_rne"]).max() > 1.0
    assert np.array_equal(oracle.torque_test_batch("rne", g["q"], g["qd"], g["qdd"], g["mass"],
                                                   model=oracle.default_model())[0], tau0)


def test_base_mode_is_constant_true():
    g = load_golden("states_cfg2.npz")
    tau, ok = oracle.torque_test_batch("base", g["q"], g["qd"], g["qdd"], g["mass"])
    assert ok.all()


def test_minjerk():
    m = load_golden("minjerk.npz")
    for name in ["p2", "p5", "p20", "p3_1"]:
        c = oracle.minjerk_coefficients(m[name + "_points"])
        x, v, a = oracle.minjerk_trajectory(c, int(m[name + "_n"]))
        assert np.abs(c - m[name + "_coeffs"]).max() < 1e-12
        assert np.abs(x - m[name + "_x"]).max() < 1e-12
        assert np.abs(v - m[name + "_v"]).max() < 1e-12
        assert np.abs(a - m[name + "_a"]).max() < 1e-11


def test_edges_cfg4():
    e = load_golden("edges_cfg4.npz")
    ff = oracle.edge_feasibility("rne", e["qa"], e["qb"], int(e["W"]), float(e["mass"]))
    assert (ff == e["first_fail"]).all()
    assert (ff == int(e["W"])).any() and (ff < int(e["W"])).any()


def test_traj():
    t = load_golden("traj.npz")
    tau, mask, ff = oracle.traj_feasibility("rne", t["points"], int(t["n_int"]), float(t["mass"]))
    assert np.abs(tau - t["tau"]).max() < 1e-12
    assert (mask == t["feasible"]).all()
    bad = np.nonzero(t["feasible"] == 0)[0]
    assert ff == (bad[0] if len(bad) else len(mask))
    # Conf logging pass (utils.py:3376-3378): rne without payload on the same samples
    tau0, _, _ = oracle.traj_feasibility("rne", t["points"], int(t["n_int"]), 0.0)
    assert np.abs(tau0 - t["tau_nopayload"]).max() < 1e-12


def test_dyn_defined_oracle_consistency():
    """`dyn` is a DEFINED oracle (parity unpinned): check its two defining identities.
    (1) zero payload -> equals rne without payload; (2) the tool-force term is linear in the mass and
    equals a finite-difference of the potential energy of a point mass at the grasp target."""
    g = load_golden("states_cfg2.npz")
    q, qd, qdd = g["q"][:, :200], g["qd"][:, :200], g["qdd"][:, :200]
    t0, _ = oracle.torque_test_batch("dyn", q, qd, qdd, 0.0)
    tr, _ = oracle.torque_test_batch("rne", q, qd, qdd, 0.0)
    assert np.abs(t0 - tr).max() < 1e-12
    t2, _ = oracle.torque_test_batch("dyn", q, qd, qdd, 2.0)
    t4, _ = oracle.torque_test_batch("dyn", q, qd, qdd, 4.0)
    assert np.abs((t4 - t0) - 2 * (t2 - t0)).max() < 1e-10
    # d(height of tool)/dq_i * m g == J^T F; tool = link8 origin + 0.105 along its z axis (FK of ComputeFk's
    # convention, checked against the reference's golden poses in test_ik_core_host)
    import ik_reference

    def tool_z(qq):
        tr_, rot = ik_reference.fk_batch(qq)
        return tr_[2] + 0.105 * rot[8]
    h = 1e-6
    for i in range(7):
        dq = np.zeros((7, 1)); dq[i] = h
        num = (tool_z(q + dq) - tool_z(q - dq)) / (2 * h) * 2.0 * 9.81
        assert np.abs(num - (t2 - t0)[i]).max() < 1e-6


def test_ref_ikfast_kats():
    """SURVEY.md Appendix B FK/IK known answers through the compiled, unmodified reference."""
    if not oracle.have_ref():
        pytest.skip("oracle/_ref not built")
    q = np.array(Q_HOME).reshape(7, 1)
    trans, rot = oracle.ref_fk_batch(q)
    assert np.abs(trans[:, 0] - [0.3068905665929411, 0.0, 0.5902820523028393]).max() < 1e-15
    sols, counts = oracle.ref_ik_batch(rot, trans, np.array([math.pi / 4]))
    assert counts[0] == 8
    assert np.abs(sols[0] - np.array(Q_HOME)).max(axis=1).min() < 1e-12
    g = load_golden("ik_cfg3.npz")
    sols, counts = oracle.ref_ik_batch(g["rot"], g["trans"], g["free"])
    assert (counts == g["counts"]).all()
    assert np.abs(sols - g["sols"]).max() < 1e-12


def test_numpy_port_at_reference_granularity():
    """oracle/rne_numpy_port.py (the per-call cost model bench.py times) reproduces the unmodified rne.py."""
    from oracle import rne_numpy_port as P
    g = load_golden("states_cfg2.npz")
    for i in range(60):
        ok, tau = P.torque_test(g["q"][:, i], g["qd"][:, i], g["qdd"][:, i], g["mass"][i])
        assert np.abs(tau - g["tau_rne"][:, i]).max() < 1e-12
        assert ok == bool(g["feasible_rne"][i])
    k = load_golden("kat_rne.npz")
    for i in range(k["q"].shape[1]):
        tau = P.rne(k["q"][:, i], k["qd"][:, i], k["qdd"][:, i], float(k["mass"][i]))
        assert np.abs(tau - k["tau_raw"][:, i]).max() < 1e-12
