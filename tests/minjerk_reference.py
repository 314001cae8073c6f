"""Long-double reference of the min-jerk sampling of K4 (edge_kernel: tcmp_edge_feasibility[_model|_host|_scatter];
traj_kernel: tcmp_traj_feasibility[_model]) and the boundary-case generators shared by
tests/test_minjerk_reference_cpu.py (the generators against the C oracle) and tests/test_gpu_minjerk.py (the kernels).
Test-side only: nothing in the package imports it.

Sampling.  Sample i of S sits at np.linspace(1/S, 1, S)[i]; NumPy's own result is the reference for the times.
An edge qa -> qb is the two-point min-jerk of min_jerk_v2.py:121-130 (x = qa, v = a = 0, t = 1): with A = qb - qa
(a double, as every implementation forms it) the waypoint is x = qa + A (10 t^3 - 15 t^4 + 6 t^5), v = A x'(t),
a = A x''(t).  A trajectory segment is the quintic sum c_i t^i on the caller's double coefficients
(min_jerk_v2.py:216-220).  Both are evaluated in np.longdouble (64-bit mantissa) from the double inputs.  A double
implementation that evaluates the same polynomial with a few roundings per term stays within
SAMPLE_ULPS * 2^-53 * sum |c_i| t^i (and of the derivative sums): the bounds edge_samples and traj_samples return.

Torques.  The pinned C oracle (oracle.torque_test_batch, within 1.4e-13 N.m of rne.py) evaluated on the reference
samples rounded to double.  No verdict is asserted where a torque lies within BAND = 1e-9 N.m of its limit (the
torque contract of include/tcmp.h); every check reports how many samples fell there.

Boundary cases.  The payload mass is the only run-time knob of the compiled-in kernels, and each waypoint's torque
is affine in it (above the payload threshold in rne / nov, for every mass in dyn).  From two oracle evaluations the
generator solves for the mass that puts joint j at waypoint k exactly delta above its limit with every earlier
waypoint at least delta inside (first failure k), or every waypoint at least delta inside with one at exactly -delta
(first failure W), then re-verifies the margins with the oracle at that mass.
"""
import numpy as np

import oracle
from conftest import sample_edges

LD = np.longdouble
BAND = 1e-9
DELTAS = (1e-8, 1e-5, 1.0)
SAMPLE_ULPS = 16
_EPS = 2.0 ** -53
MASS_RANGE = (0.05, 40.0)          # solved masses stay well above the 0.01 kg payload threshold


def linspace_times(S):
    return np.linspace(1.0 / S, 1.0, S)


def limits(model=None):
    if model is None:
        return np.array([87.0, 87.0, 87.0, 87.0, 12.0, 12.0])
    return np.array(oracle.model_fields(np.asarray(model))["torque_limit"][:6])


# ---- sampling -------------------------------------------------------------------------------------------------------
def edge_samples(qa, qb, W):
    """qa, qb [7][n] double -> (x, v, a) [n][W][7] longdouble and the matching rounding bounds (double)."""
    t = linspace_times(W).astype(LD)[None, :, None]
    q0 = np.asarray(qa, np.float64).T.astype(LD)[:, None, :]
    A = (np.asarray(qb, np.float64) - np.asarray(qa, np.float64)).T.astype(LD)[:, None, :]
    px = t ** 3 * (10 + t * (-15 + 6 * t))
    pv = t ** 2 * (30 + t * (-60 + 30 * t))
    pa = t * (60 + t * (-180 + 120 * t))
    x, v, a = q0 + A * px, A * pv, A * pa
    absA = np.abs(A)
    bx = np.abs(q0) + absA * (10 * t ** 3 + 15 * t ** 4 + 6 * t ** 5)
    bv = absA * (30 * t ** 2 + 60 * t ** 3 + 30 * t ** 4)
    ba = absA * (60 * t + 180 * t ** 2 + 120 * t ** 3)
    return (x, v, a), tuple((SAMPLE_ULPS * _EPS * b).astype(np.float64) for b in (bx, bv, ba))


def traj_samples(coeffs, S):
    """coeffs [n_seg][7][6] double -> (x, v, a) [n_seg * S][7] longdouble and the rounding bounds (double)."""
    c = np.asarray(coeffs, np.float64).astype(LD)
    t = linspace_times(S).astype(LD)[None, :, None]
    cs = [c[:, None, :, i] for i in range(6)]
    x = sum(cs[i] * t ** i for i in range(6))
    v = sum(i * cs[i] * t ** (i - 1) for i in range(1, 6))
    a = sum(i * (i - 1) * cs[i] * t ** (i - 2) for i in range(2, 6))
    bx = sum(np.abs(cs[i]) * t ** i for i in range(6))
    bv = sum(i * np.abs(cs[i]) * t ** (i - 1) for i in range(1, 6))
    ba = sum(i * (i - 1) * np.abs(cs[i]) * t ** (i - 2) for i in range(2, 6))
    n = c.shape[0] * S
    out = tuple(y.reshape(n, 7) for y in (x, v, a))
    return out, tuple((SAMPLE_ULPS * _EPS * b).reshape(n, 7).astype(np.float64) for b in (bx, bv, ba))


def edge_coeffs(qa, qb):
    """The single-segment coefficients [n][7][6] of edges qa -> qb, as oracle.minjerk_coefficients forms them."""
    A = np.asarray(qb, np.float64) - np.asarray(qa, np.float64)
    c = np.zeros((A.shape[1], 7, 6))
    c[:, :, 0] = np.asarray(qa).T
    c[:, :, 3], c[:, :, 4], c[:, :, 5] = 10 * A.T, -15 * A.T, 6 * A.T
    return c


# ---- torques ----------------------------------------------------------------------------------------------------------
def torques(mode, x, v, a, mass, threshold=0.01, model=None):
    """Oracle torques of [m][7] samples (rounded to double) -> tau [m][7]."""
    X, V, A = (np.ascontiguousarray(np.asarray(y, np.float64).T) for y in (x, v, a))
    tau, _ = oracle.torque_test_batch(mode, X, V, A, mass, threshold, model=model)
    return tau.T


def margins(tau, model=None):
    """|tau_j| - limit_j for the six tested joints -> [..., 6] (NaN torques give NaN, i.e. within limits)."""
    return np.abs(tau[..., :6]) - limits(model)


def first_fail_from_margins(mg):
    """mg [..., W, 6] -> first waypoint with a margin >= 0 (W if none), and whether any margin lies in the band."""
    fails = (mg >= 0).any(-1)
    W = fails.shape[-1]
    ff = np.where(fails.any(-1), fails.argmax(-1), W)
    return ff, (np.abs(mg) < BAND).any(-1)


def edge_reference(mode, qa, qb, W, mass, threshold=0.01, model=None):
    """Oracle margins [n][W][6] on the long-double waypoints of edges qa -> qb ('nov' for static_only)."""
    (x, v, a), _ = edge_samples(qa, qb, W)
    n = x.shape[0]
    tau = torques(mode, x.reshape(-1, 7), v.reshape(-1, 7), a.reshape(-1, 7), mass, threshold, model)
    return margins(tau.reshape(n, W, 7), model), tau.reshape(n, W, 7)


def traj_reference(mode, coeffs, S, mass, threshold=0.01, model=None):
    """-> dict(x, v, a longdouble [n][7], bounds, tau [n][7], margin [n][6], feasible [n], first_fail, in_band [n])."""
    (x, v, a), bounds = traj_samples(coeffs, S)
    tau = torques(mode, x, v, a, mass, threshold, model)
    mg = margins(tau, model)
    fails = (mg >= 0).any(-1)
    return {"x": x, "v": v, "a": a, "bounds": bounds, "tau": tau, "margin": mg, "feasible": ~fails,
            "first_fail": int(fails.argmax()) if fails.any() else len(fails),
            "in_band": (np.abs(mg) < BAND).any(-1)}


# ---- boundary cases: edges ---------------------------------------------------------------------------------------------
class EdgeCase:
    """One edge (qa, qb [7] each) at one payload mass with a designed first failure `first` (W = feasible) whose
    deciding margins are at least `delta` N.m away from the limits, as verified with the oracle."""

    def __init__(self, qa, qb, W, mass, first, delta, mg):
        self.qa, self.qb, self.W, self.mass, self.first, self.delta = qa, qb, W, mass, first, delta
        fails = (mg >= 0).any(-1)
        self.fail_rounds = sorted({int(w) // 32 for w in np.nonzero(fails)[0]})
        self.lanes_in_first_round = int(fails[(first // 32) * 32:(first // 32) * 32 + 32].sum()) if first < W else 0
        # distance of the verdict from the boundary: the failing margin at `first`, the safe margins before it
        parts = ([float(mg[first].max())] if first < W else []) + ([float(-mg[:first].max())] if first else [])
        self.clearance = min(parts)


def _affine(mode, qa, qb, W, model, m1=2.0, m2=6.0):
    """Torque of every waypoint of every edge as a + b m (joints 0..5) -> a, b [n][W][6]."""
    t1 = edge_reference(mode, qa, qb, W, m1, model=model)[1][..., :6]
    t2 = edge_reference(mode, qa, qb, W, m2, model=model)[1][..., :6]
    b = (t2 - t1) / (m2 - m1)
    return t1 - b * m1, b


def _solve(a, b, level):
    """Masses with |a + b m| = level (both signs) inside MASS_RANGE -> list."""
    out = []
    if b == 0:
        return out
    for s in (1.0, -1.0):
        m = (s * level - a) / b
        if MASS_RANGE[0] <= m <= MASS_RANGE[1]:
            out.append(m)
    return out


def find_edge_cases(mode, W, targets, deltas=DELTAS, model=None, n_edges=256, seed=0, feasible=True):
    """For each first-failure target k in `targets` and each delta, an EdgeCase found among `n_edges` random edges
    (conftest.sample_edges(n_edges, seed)); with `feasible` also one case per delta whose first failure is W (every
    margin <= -delta, one at exactly -delta).  -> dict (k or W, delta) -> EdgeCase; missing targets are absent."""
    qa, qb = sample_edges(n_edges, seed)
    a, b = _affine(mode, qa, qb, W, model)
    lim = limits(model)
    found = {}
    want = [(k, d) for k in targets for d in deltas] + ([(W, d) for d in deltas] if feasible else [])
    grid = np.linspace(*MASS_RANGE, 256)
    for e in range(n_edges):
        if len(found) == len(want):
            break
        for key in [kd for kd in want if kd not in found]:
            k, d = key
            hit = None
            if k < W:
                for j in range(6):
                    for m in _solve(a[e, k, j], b[e, k, j], lim[j] + d):
                        pre = np.abs(a[e, :k] + b[e, :k] * m) - lim
                        if pre.size == 0 or pre.max() <= -d:
                            hit = m
                            break
                    if hit is not None:
                        break
            else:
                # G(m) = max over waypoints and joints of |a + b m| - limit is convex: bisect G = -d from its minimum
                G = lambda m: (np.abs(a[e] + b[e] * m) - lim).max()
                gs = (np.abs(a[e][None] + b[e][None] * grid[:, None, None]) - lim).max(axis=(1, 2))
                lo = grid[int(gs.argmin())]
                if G(lo) < -d and G(MASS_RANGE[1]) > -d:
                    hi = MASS_RANGE[1]
                    for _ in range(80):
                        mid = 0.5 * (lo + hi)
                        lo, hi = (mid, hi) if G(mid) < -d else (lo, mid)
                    hit = lo
            if hit is None:
                continue
            case = _verify(mode, qa[:, e], qb[:, e], W, hit, k, d, model)
            if case is not None:
                found[key] = case
    return found


EDGE_WS = (1, 2, 31, 32, 33, 63, 64, 65, 96, 97, 100, 1000)
EDGE_KS = (0, 1, 30, 31, 32, 33, 63, 64, 95, 96)


def edge_targets(W):
    return sorted({k for k in EDGE_KS + (W - 1,) if k < W})


_FAMILIES = {}


def edge_family(mode, model_name=None):
    """Every boundary case of one torque mode ('nov' also serves rne with static_only) for every W in EDGE_WS, against
    the compiled-in Panda (model_name None) or the robot of tests/golden/model_override.npz ('override').  Cached.
    Every target k is found at delta = 1e-8 and every W has its feasible-by-delta cases (asserted); the larger deltas
    are kept where adjacent waypoints leave room for them."""
    key = (mode, model_name)
    if key not in _FAMILIES:
        model = None if model_name is None else override_model()
        cases = []
        for W in EDGE_WS:
            found = find_edge_cases(mode, W, edge_targets(W), model=model)
            for k in edge_targets(W) + [W]:
                assert (k, DELTAS[0]) in found, (mode, model_name, W, k)
            cases += [found[kd] for kd in sorted(found)]
        _FAMILIES[key] = cases
    return _FAMILIES[key]


def override_model():
    from conftest import load_golden
    return np.ascontiguousarray(load_golden("model_override.npz")["model"], dtype=np.float64)


def _verify(mode, qa, qb, W, mass, k, d, model):
    """Re-evaluate the candidate with the oracle at `mass`; keep it if the first failure is k (or W) with every
    deciding margin outside max(BAND, d / 2)."""
    mg = edge_reference(mode, qa[:, None], qb[:, None], W, mass, model=model)[0][0]
    ff, _ = first_fail_from_margins(mg[None])
    if int(ff[0]) != k:
        return None
    tol = max(BAND, 0.5 * d)
    if k < W:
        if mg[:k].size and mg[:k].max() > -tol or mg[k].max() < tol:
            return None
    elif mg.max() > -tol:
        return None
    return EdgeCase(qa.copy(), qb.copy(), W, float(mass), k, d, mg)


def threshold_edge(mode, W=64, model=None, n_edges=4000, seed=7):
    """An edge whose verdict at payload mass nextafter(0.01, 1) (payload attached, rne/nov) differs from its verdict
    at exactly 0.01 (no payload), or in dyn, at 0.01 from that at 0 (the tool force is applied unconditionally), with
    every deciding margin outside BAND at both masses.  -> (qa [7], qb [7], (m_lo, ff_lo), (m_hi, ff_hi))."""
    # The payload of 0.01 kg moves a torque by a few 1e-2 N.m.  So the edge qa -> qa + s (qb - qa), 0 <= s <= 8, is
    # scaled until its largest margin without the payload is -GAP (bisection on s), and kept if the payload then
    # makes it fail.  Only the dynamic modes get there: the arm's static torques stay far inside the limits.
    GAP = 2e-3
    qa, qb = sample_edges(n_edges, seed)
    m_lo, m_hi = (0.0, 0.01) if mode == "dyn" else (0.01, float(np.nextafter(0.01, 1.0)))
    worst = lambda a, b: edge_reference(mode, a[:, None], b[:, None], W, m_lo, model=model)[0][0].max()
    for e in range(min(n_edges, 64)):
        a, d = qa[:, e], qb[:, e] - qa[:, e]
        if not (worst(a, a) < -GAP < worst(a, a + 8 * d)):
            continue
        lo, hi = 0.0, 8.0
        for _ in range(60):
            mid = 0.5 * (lo + hi)
            lo, hi = (mid, hi) if worst(a, a + mid * d) < -GAP else (lo, mid)
        b = a + lo * d
        out = []
        for m in (m_lo, m_hi):
            mg = edge_reference(mode, a[:, None], b[:, None], W, m, model=model)[0][0]
            ff = int(first_fail_from_margins(mg[None])[0][0])
            out.append((m, ff, not (np.abs(mg[: min(ff, W - 1) + 1]) < BAND).any()))
        if out[0][1] != out[1][1] and out[0][2] and out[1][2]:
            return a.copy(), b, out[0][:2], out[1][:2]
    return None


# ---- boundary cases: trajectories ----------------------------------------------------------------------------------------
# arm up with the flange pointing down its axis: at 40 kg every torque is still > 11 N.m inside its limit (checked)
SAFE_Q = np.array([0.0, 0.0, 0.0, -0.07, 0.0, 2.49, 0.0])


def safe_segment():
    c = np.zeros((7, 6))
    c[:, 0] = SAFE_Q
    return c


def traj_with_failure(case, S, n_seg, at_seg, repeat_after=3):
    """Coefficients [n_seg][7][6]: safe segments, the case's edge (sampled with S = case.W) as segment `at_seg`, and
    `repeat_after` more copies of it after that, so later samples fail too.  Expected first failure:
    at_seg * S + case.first (n_seg * S when the case is feasible)."""
    assert case.W == S
    c = np.broadcast_to(safe_segment(), (n_seg, 7, 6)).copy()
    seg = edge_coeffs(case.qa[:, None], case.qb[:, None])[0]
    for s in range(at_seg, min(n_seg, at_seg + 1 + repeat_after * 7), 7):
        c[s] = seg
    return c


# ---- checks shared by the CPU and GPU tests ---------------------------------------------------------------------------------
def check_edge_cases(cases, run, static_only=False):
    """run(qa [7][n], qb [7][n], W, mass) -> first failures [n]; every case's designed first failure, the case run
    alone and tiled with itself so that its lanes share a warp with other copies."""
    for case in cases:
        qa, qb = case.qa[:, None], case.qb[:, None]
        ff = np.asarray(run(np.repeat(qa, 3, 1), np.repeat(qb, 3, 1), case.W, case.mass))
        assert (ff == case.first).all(), (case.W, case.first, case.delta, case.mass, ff)


def check_times(S, q, dtype=np.float64):
    """q [7][n] of the c = (0, 1, 0, 0, 0, 0) trajectory: every sample equals linspace(1/S, 1, S) bit for bit."""
    want = linspace_times(S).astype(dtype)
    q = np.asarray(q)
    assert q.dtype == dtype
    for j in range(7):
        assert np.array_equal(q[j].reshape(-1, S), np.broadcast_to(want, (q.shape[1] // S, S))), (S, j)


def check_samples(ref, q, qd, qdd):
    """Kernel samples [7][n] against the long-double reference within its rounding bound."""
    for got, want, bound in zip((q, qd, qdd), (ref["x"], ref["v"], ref["a"]), ref["bounds"]):
        err = np.abs(np.asarray(got, np.float64).T.astype(LD) - want).astype(np.float64)
        assert (err <= bound).all(), float((err - bound).max())


def check_traj(ref, feasible, first_fail):
    """Kernel feasibility [n] and first failure against the reference outside the band."""
    feasible = np.asarray(feasible).astype(bool)
    out = ~ref["in_band"]
    assert np.array_equal(feasible[out], ref["feasible"][out])
    assert not ref["in_band"][: ref["first_fail"] + 1].any()
    assert first_fail == ref["first_fail"]
