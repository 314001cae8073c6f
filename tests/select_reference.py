"""Reference and case generators for goal-IK selection (K7, tcmp_ik_select[_model], engine.ik_select).

The reference composes the semantics of include/tcmp.h at tcmp_ik_select from pieces pinned elsewhere:
* candidates: the solutions and counts of a given IK output, min(count, 8) per solve (the host build of
  csrc/ik_core.cuh on the CPU, the kernel's own tcmp_ik_batch on the GPU);
* the limit filter lo <= q <= hi, exactly (a NaN limit bounds nothing);
* the static torque test of the pinned oracle (qd = qdd = 0), on the stock robot or a tcmp_model record;
* the cost: the max norm in float64 is exact (one rounded subtraction per joint and a max; NaN propagates), the L2
  norm is not (nvcc contracts the sum of squares into FMAs), so an L2 selection is decidable only where the
  runner-up is more than 1e-12 (relative) behind the winner, and its cost is compared to 4 ulps;
* the arg-min over (cost, key = 8 f + s): a NaN cost ranks after every number, equal costs by the smaller key.

Joint 7 of every solution is the free value bit for bit, which the generators use to build exact cases without
relying on the last bits of joints 1-6: joint-7 limit cases, exact max-norm ties, sweep-round placements.  Torque
cases place the payload mass so that the nearest candidate fails or passes by delta N m on its binding joint (static
torques are affine in the mass) and re-verify every case with the oracle at that mass.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np

import oracle
from conftest import Q_HI, Q_LO, ROOT, load_golden
from ik_reference import fk_batch, host_ik

NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "torque_constrained_motion_planning_b200", "csrc")
MODE = {"rne": 0, "nov": 1, "dyn": 2, "base": 3}
BAND = 1e-9            # no torque verdict is asserted within this distance of a limit (N m)
L2_GAP = 1e-12         # relative lead an L2 winner needs over the runner-up to be decidable
J7_MARGIN = 1e-6       # joint 7 exceeds every other joint's distance by this much in the tie cases (rad)
THRESHOLD = 0.01
DELTAS = (1e-8, 1e-5, 1e-2)
INF7 = np.full(7, np.inf)
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int32)

# ---- host build of K7 (tests/native/select_host.cpp) -------------------------------------------------------------
_lib = None


def _host():
    global _lib
    if _lib is None:
        so = os.path.join(NATIVE, "libselect_host.so")
        src = os.path.join(NATIVE, "select_host.cpp")
        deps = [src] + [os.path.join(CSRC, h) for h in ("select_core.cuh", "ik_core.cuh", "panda_model.cuh",
                                                        "sincos_table.inc")] + [os.path.join(ROOT, "include", "tcmp.h")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
            subprocess.check_call([shutil.which("g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-fopenmp",
                                   "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", so, src])
        _lib = ctypes.CDLL(so)
    return _lib


def host_select(rot, trans, free, q_ref, lo=Q_LO, hi=Q_HI, mode="base", mass=0.0, threshold=THRESHOLD, norm="inf",
                model=None):
    """The host build of K7 -> (best_q [7][n], best_cost [n], n_valid int32 [n], n_redo int32 [n])."""
    f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    rot, trans, free, q_ref, lo, hi = (f64(a) for a in (rot, trans, free, q_ref, lo, hi))
    model = None if model is None else f64(model)
    n = rot.shape[1]
    best, cost = np.empty((7, n)), np.empty(n)
    nv, redo = np.empty(n, np.int32), np.empty(n, np.int32)
    _host().host_select(None if model is None else model.ctypes.data_as(_dp), ctypes.c_int64(n),
                        rot.ctypes.data_as(_dp), trans.ctypes.data_as(_dp), free.ctypes.data_as(_dp),
                        ctypes.c_int(free.shape[0]), ctypes.c_int(int(free.ndim == 1)), q_ref.ctypes.data_as(_dp),
                        ctypes.c_int(int(q_ref.ndim == 1)), lo.ctypes.data_as(_dp), hi.ctypes.data_as(_dp),
                        ctypes.c_int(MODE[mode]), ctypes.c_double(mass), ctypes.c_double(threshold),
                        ctypes.c_int(int(norm == "inf")), best.ctypes.data_as(_dp), cost.ctypes.data_as(_dp),
                        nv.ctypes.data_as(_ip), redo.ctypes.data_as(_ip))
    return best, cost, nv, redo


# ---- the reference ------------------------------------------------------------------------------------------------
def torque_limits(model):
    return np.array([87.0, 87.0, 87.0, 87.0, 12.0, 12.0]) if model is None else \
        np.array(oracle.model_fields(model)["torque_limit"][:6])


def candidates(sols, counts, n, n_free):
    """Every emitted solution -> (q [m][7], pose [m], key [m]) in (pose, free value, solver order)."""
    c = np.minimum(np.asarray(counts).reshape(n, n_free), 8)
    live = np.arange(8)[None, None, :] < c[:, :, None]
    p, f, s = np.nonzero(live)
    q = np.asarray(sols).reshape(n, n_free, 8, 7)[p, f, s]
    return q, p, f * 8 + s


def reference_select(sols, counts, n_free, q_ref, lo=Q_LO, hi=Q_HI, mode="base", mass=0.0, threshold=THRESHOLD,
                     norm="inf", model=None):
    """The composed reference on the IK output (sols [n*n_free][8][7], counts [n*n_free]) -> dict of
    best [7][n], cost [n], nv [n], key [n] (-1 = none), band [n] (a verdict within BAND of a limit: only the limit
    filter's survivors count) and decidable [n] (the winner is decided whatever the rounding of an L2 cost)."""
    n = np.asarray(counts).size // n_free
    q, pose, key = candidates(sols, counts, n, n_free)
    lo, hi = np.asarray(lo, np.float64), np.asarray(hi, np.float64)
    inl = (~(q < lo) & ~(q > hi)).all(1)
    ok = inl.copy()
    band = np.zeros(n, bool)
    if mode != "base" and inl.any():
        tau, passed = oracle.torque_test_batch(mode, np.ascontiguousarray(q[inl].T), None, None, mass, threshold,
                                               model=model)
        ok[inl] = passed.astype(bool)
        near = (np.abs(np.abs(tau[:6]) - torque_limits(model)[:, None]) < BAND).any(0)
        band[pose[inl][near]] = True
    ref = np.asarray(q_ref, np.float64)
    ref = np.broadcast_to(ref[:, None], (7, n)) if ref.ndim == 1 else ref
    d = np.abs(q - ref.T[pose])
    cost = np.max(d, axis=1) if norm == "inf" else np.sqrt((d * d).sum(1))
    q, pose, key, cost = q[ok], pose[ok], key[ok], cost[ok]
    nv = np.bincount(pose, minlength=n).astype(np.int32)
    nan = np.isnan(cost)
    order = np.lexsort((key, np.where(nan, 0.0, cost), nan, pose))
    first = np.ones(order.size, bool)
    first[1:] = pose[order][1:] != pose[order][:-1]
    win = order[first]
    out = {"best": np.zeros((7, n)), "cost": np.full(n, np.inf), "nv": nv, "key": np.full(n, -1), "band": band,
           "decidable": np.ones(n, bool)}
    out["best"][:, pose[win]] = q[win].T
    out["cost"][pose[win]] = cost[win]
    out["key"][pose[win]] = key[win]
    if norm != "inf":   # the runner-up of each pose directly follows its winner in `order`
        st = np.flatnonzero(first)
        st = st[st + 1 < order.size]
        st = st[~first[st + 1]]
        w, r = cost[order[st]], cost[order[st + 1]]
        close = np.isfinite(w) & ~(r > w * (1 + L2_GAP))
        out["decidable"][pose[order[st[close]]]] = False
    return out


def check_select(got, want, norm, exact_q=True):
    """Assert a selection (best [7][n], cost [n], nv [n]) equals the reference outside its band -> poses skipped."""
    best, cost, nv = (np.asarray(a) for a in got)
    keep = ~want["band"]
    assert np.array_equal(nv[keep], want["nv"][keep]), np.flatnonzero(nv[keep] != want["nv"][keep])[:10]
    dec = keep & want["decidable"]
    if exact_q:
        assert np.array_equal(best[:, dec], want["best"][:, dec], equal_nan=True), \
            np.flatnonzero((best[:, dec] != want["best"][:, dec]).any(0))[:10]
    else:
        assert np.abs(best[:, dec] - want["best"][:, dec]).max(initial=0) < 1e-9
    c, w = cost[dec], want["cost"][dec]
    if norm == "inf" and exact_q:
        assert np.array_equal(c, w, equal_nan=True)
    else:
        assert np.array_equal(np.isnan(c), np.isnan(w)) and np.array_equal(np.isinf(c), np.isinf(w))
        fin = np.isfinite(w)
        tol = 4 * np.spacing(w[fin]) if exact_q else 1e-9
        assert (np.abs(c[fin] - w[fin]) <= tol).all(), np.abs(c[fin] - w[fin]).max()
    return int((~keep).sum())


# ---- case generators -----------------------------------------------------------------------------------------------
# A case is a dict: rot [9][n], trans [3][n], free [n_free][n], q_ref [7][n], lo, hi [7], mode, mass, threshold, norm,
# model (record or None) and what the generator designed (want_key [n] where it fixes the winner).
def _poses(rng, n):
    q = rng.uniform(Q_LO[:, None] + 0.05, Q_HI[:, None] - 0.05, size=(7, n))
    trans, rot = fk_batch(q)
    return q, rot, trans


def _case(rot, trans, free, q_ref, **kw):
    c = {"rot": rot, "trans": trans, "free": np.ascontiguousarray(free), "q_ref": np.ascontiguousarray(q_ref),
         "lo": Q_LO, "hi": Q_HI, "mode": "base", "mass": 0.0, "threshold": THRESHOLD, "norm": "inf", "model": None}
    c.update(kw)
    return c


def ik_of(case):
    sols, counts, status = host_ik(case["rot"], case["trans"], case["free"])
    return sols, counts, status


def reference_of(case, sols=None, counts=None):
    if sols is None:
        sols, counts, _ = ik_of(case)
    return reference_select(sols, counts, case["free"].shape[0], case["q_ref"], case["lo"], case["hi"], case["mode"],
                            case["mass"], case["threshold"], case["norm"], case["model"])


def host_of(case):
    return host_select(case["rot"], case["trans"], case["free"], case["q_ref"], case["lo"], case["hi"], case["mode"],
                       case["mass"], case["threshold"], case["norm"], case["model"])


def joint7_limit_cases(seed=1, n=64):
    """Free values at Q_LO[6] and Q_HI[6], one ulp outside and one ulp inside; q_ref = a solution at the limit itself,
    so the limit candidate wins at cost 0 iff the filter keeps it."""
    rng = np.random.default_rng(seed)
    out = []
    for side in (0, 1):
        lim = Q_HI[6] if side else Q_LO[6]
        outward = np.inf if side else -np.inf
        vals = np.array([np.nextafter(lim, -outward), lim, np.nextafter(lim, outward)])
        q, rot, trans = _poses(rng, 4 * n)
        q[6] = lim
        trans, rot = fk_batch(q)
        for k, v in enumerate(vals):
            # the limit value first, then two in-range values 0.2-0.6 rad inside it
            inner = lim - np.sign(outward) * rng.uniform(0.2, 0.6, size=(2, q.shape[1]))
            free = np.vstack([np.full((1, q.shape[1]), v), inner])
            s, c, _ = host_ik(rot, trans, free)
            sols = s.reshape(-1, 3, 8, 7)
            cnt = c.reshape(-1, 3)
            in6 = ((sols[:, 0, :, :6] >= Q_LO[:6]) & (sols[:, 0, :, :6] <= Q_HI[:6])).all(2) & \
                (np.arange(8)[None] < cnt[:, :1])
            good = np.flatnonzero(in6.any(1))[:n]
            if good.size == 0:
                continue
            first = in6[good].argmax(1)
            q_ref = sols[good, 0, first].T.copy()
            case = _case(rot[:, good], trans[:, good], free[:, good], q_ref, family="j7_limit",
                         label="%s%+d" % ("hi" if side else "lo", k - 1), limit_value=v,
                         want_key=np.where(k < 2, first, -2))
            out.append(case)
    return out


def _tie_pose(rng, idx, n_free):
    """One pose and its free sweep with an exact max-norm tie between the first solutions of the free values at sweep
    indices idx = (i1, i2): f1, r7 = f1 + h, f2 = f1 + 2 h, all multiples of 2^-20, so |f1 - r7| == |f2 - r7| exactly
    -> (rot, trans, free [n_free], q_ref [7]) or None."""
    q, rot, trans = _poses(rng, 1)
    f1 = np.round(q[6, 0] * 2**20) / 2**20
    h = rng.integers(2**16, 2**17) / 2**20             # 0.06 .. 0.12 rad, exact multiples of 2^-20
    f2 = f1 + 2 * h
    r7 = f1 + h
    if not (Q_LO[6] < min(f1, f2) and max(f1, f2, r7) < Q_HI[6]):
        return None
    pair = np.array([f1, f2])
    s, c, _ = host_ik(rot, trans, pair)
    if c[0] < 1 or c[1] < 1:
        return None
    c1, c2 = s[0, 0], s[1, 0]
    ref = np.empty(7)
    ref[:6] = (c1[:6] + c2[:6]) / 2
    ref[6] = r7
    # filler free values: further from r7 than the tie by > 1 mrad, so their candidates lose whatever joints 1-6 do
    fill = r7 + np.where(rng.random(n_free) < 0.5, -1, 1) * rng.uniform(h + 1e-3, h + 0.5, n_free)
    fill = np.clip(fill, Q_LO[6], Q_HI[6])
    bad = np.abs(fill - r7) <= h + 1e-3
    if bad.any():
        return None
    free = fill
    free[idx[0]], free[idx[1]] = f1, f2
    return rot, trans, free, ref


def _tie_ok(rot, trans, free, ref):
    """The designed tie is the winner and exact: every candidate within 1e-6 of the best cost has its max attained
    by joint 7 with a J7_MARGIN lead."""
    s, c, _ = host_ik(rot, trans, free)
    q, _, key = candidates(s, c, 1, free.size)
    d = np.abs(q - ref)
    cost = d.max(1)
    best = cost.min()
    near = cost < best + 1e-6
    j7 = d[:, 6] >= d[:, :6].max(1) + J7_MARGIN
    return bool((j7[near]).all()), key[np.argmin(np.where(cost == best, key, 1 << 30))], q, cost


def tie_cases(seed=2, pairs=((0, 1), (1, 0), (0, 31), (31, 32), (3, 35), (40, 8)), n_frees=(33, 64, 65), per=4):
    """Cross-free exact ties at sweep indices (i1, i2): the smaller index wins; r7 one ulp towards the other value
    makes that one strictly nearer."""
    rng = np.random.default_rng(seed)
    out = []
    for nf in n_frees:
        for i1, i2 in pairs:
            if max(i1, i2) >= nf:
                continue
            got = 0
            for _ in range(400):
                if got >= per:
                    break
                t = _tie_pose(rng, (i1, i2), nf)
                if t is None:
                    continue
                rot, trans, free, ref = t
                ok, wkey, q, cost = _tie_ok(rot, trans, free, ref)
                f1, f2 = free[i1], free[i2]
                if not ok or abs(f1 - ref[6]) != abs(f2 - ref[6]) or wkey // 8 != min(i1, i2):
                    continue
                # one ulp of r7 towards the later index's value
                late = max(i1, i2)
                flip = ref.copy()
                flip[6] = np.nextafter(ref[6], free[late])
                ok2, wkey2, _, _ = _tie_ok(rot, trans, free, flip)
                if not ok2 or wkey2 // 8 != late:
                    continue
                for r, lab, wk in ((ref, "tie", wkey), (flip, "flip", wkey2)):
                    out.append(_case(rot, trans, free[:, None], r[:, None], lo=-INF7, hi=INF7, family="tie",
                                     label="nf%d_%d_%d_%s" % (nf, i1, i2, lab), want_key=np.array([wk])))
                got += 1
    return out


def solver_tie_cases(seed=3, n=2000):
    """Two solutions of one free value at an exact tie: with limits +-inf and q_ref = a solution's joints 1-6 shifted
    to the midpoint of two solutions of the same free value, whose joint-7 distances are equal by construction (one
    free value): the smaller solver index wins whenever joint 7 dominates."""
    rng = np.random.default_rng(seed)
    q, rot, trans = _poses(rng, n)
    free = q[6:7]
    s, c, _ = host_ik(rot, trans, free)
    out_idx, refs, keys = [], [], []
    for p in range(n):
        if c[p] < 2:
            continue
        a, b = s[p, 0], s[p, 1]
        ref = np.empty(7)
        ref[:6] = (a[:6] + b[:6]) / 2
        span = np.abs(a[:6] - b[:6]).max() / 2
        ref[6] = free[0, p] + span + 0.01          # joint 7 dominates both by >= 0.01 - rounding
        ref[6] = free[0, p] - span - 0.01 if ref[6] > Q_HI[6] else ref[6]
        qs, _, key = candidates(s[p:p + 1], c[p:p + 1], 1, 1)
        d = np.abs(qs - ref)
        cost = d.max(1)
        if not (d[:2, 6] >= d[:2, :6].max(1) + J7_MARGIN).all() or cost[0] != cost[1]:
            continue
        if (cost[2:] < cost[0] + 1e-6).any():
            continue
        out_idx.append(p)
        refs.append(ref)
        keys.append(0)
        if len(out_idx) >= 32:
            break
    idx = np.array(out_idx)
    return [_case(rot[:, idx], trans[:, idx], free[:, idx], np.array(refs).T, lo=-INF7, hi=INF7, family="solver_tie",
                  label="s0_s1", want_key=np.array(keys))]


def full_list_case(seed=4, tries=4000):
    """32 copies of one free value on a pose with 8 solutions: the 256-row candidate list fills exactly; q_ref =
    solution 5's configuration, so solver index 5 of the first copy wins at cost 0."""
    rng = np.random.default_rng(seed)
    q, rot, trans = _poses(rng, tries)
    s, c, _ = host_ik(rot, trans, q[6:7])
    p = np.flatnonzero(c >= 8)
    assert p.size, "no pose with 8 solutions"
    p = p[:8]
    free = np.repeat(q[6:7, p], 32, axis=0)
    ref = s[p, 5].T.copy()
    return [_case(rot[:, p], trans[:, p], free, ref, lo=-INF7, hi=INF7, family="full_list", label="32x8",
                  want_key=np.full(p.size, 5))]


def sweep_round_cases(seed=5, n_frees=(1, 2, 31, 32, 33, 63, 64, 65, 100), n=16):
    """The winner (the pose's own j7, q_ref = the pose's configuration) at index 0, 31, 32, 33 or n_free - 1, with
    worse candidates before it: filler free values 0.1-0.5 rad away from the pose's j7."""
    rng = np.random.default_rng(seed)
    out = []
    for nf in n_frees:
        for w in sorted({i for i in (0, 31, 32, 33, nf - 1) if i < nf}):
            q, rot, trans = _poses(rng, n)
            q[5] = np.minimum(q[5], 3.1)
            trans, rot = fk_batch(q)
            off = rng.uniform(0.1, 0.5, size=(nf, n)) * np.where(q[6] > 0, -1, 1)
            free = q[6] + off
            free[w] = q[6]
            out.append(_case(rot, trans, free, q, lo=-INF7, hi=INF7, family="sweep_round",
                             label="nf%d_w%d" % (nf, w), winner_index=w))
    return out


def affine_terms(mode, q, model):
    """Static torques tau(m) = a + m b [7][m] (m > 0 attached in rne / nov, every m in dyn), from the oracle at 2 and
    6 kg with threshold 0."""
    t1, _ = oracle.torque_test_batch(mode, q, None, None, 2.0, 0.0, model=model)
    t2, _ = oracle.torque_test_batch(mode, q, None, None, 6.0, 0.0, model=model)
    b = (t2 - t1) / 4.0
    return t1 - 2.0 * b, b


def torque_cases(mode, model=None, norm="inf", seed=6, n=64, n_free=4):
    """Masses at which the nearest in-limit candidate of each pose passes, or fails, by delta on its binding joint ->
    one case per (delta, side): all poses of a case share the mass, so each case holds one pose."""
    rng = np.random.default_rng(seed)
    q, rot, trans = _poses(rng, n)
    free = np.vstack([q[6:7], np.clip(q[6:7] + rng.uniform(-0.4, 0.4, size=(n_free - 1, n)), Q_LO[6], Q_HI[6])])
    q_ref = np.clip(q + rng.normal(0, 0.3, size=q.shape), Q_LO[:, None], Q_HI[:, None])
    s, c, _ = host_ik(rot, trans, free)
    base = reference_select(s, c, n_free, q_ref, norm=norm)
    lim = torque_limits(model)
    out = []
    for p in np.flatnonzero(base["key"] >= 0):
        cq = base["best"][:, p:p + 1]
        a, b = affine_terms(mode, cq, model)
        a, b = a[:6, 0], b[:6, 0]
        # masses where |a_j + m b_j| == lim_j, m > THRESHOLD: the first one above the threshold binds
        roots = []
        for j in range(6):
            if b[j] == 0:
                continue
            for sgn in (1, -1):
                m = (sgn * lim[j] - a[j]) / b[j]
                if m > 0.05:
                    roots.append((m, j))
        if not roots:
            continue
        m0, j = min(roots)
        for delta in DELTAS:
            for side in (-1, 1):    # -1: passes by delta, +1: fails by delta
                m = m0 + side * delta / abs(b[j])
                if m <= 0.05:
                    continue
                tau, _ = oracle.torque_test_batch(mode, cq, None, None, m, THRESHOLD, model=model)
                margin = abs(tau[j, 0]) - lim[j]
                if abs(margin - side * delta) > 1e-3 * delta + 1e-11:
                    continue
                case = _case(rot[:, p:p + 1], trans[:, p:p + 1], free[:, p:p + 1], q_ref[:, p:p + 1], mode=mode,
                             mass=float(m), norm=norm, model=model, family="torque_%s" % mode,
                             label="p%d_d%g_%s" % (p, delta, "fail" if side > 0 else "pass"), margin=margin)
                out.append(case)
    return out


def threshold_model(seed=7, n=32):
    """A tcmp_model record whose joint-j limit sits halfway between |tau_j| at 0.01 kg (payload not attached) and at
    nextafter(0.01, 1) (attached), for the nearest candidate of pose 0, plus the cases at the two masses and at
    threshold 0 with mass 0 and 5e-324, in rne and nov."""
    rng = np.random.default_rng(seed)
    q, rot, trans = _poses(rng, n)
    free = q[6:7]
    s, c, _ = host_ik(rot, trans, free)
    base = reference_select(s, c, 1, q, norm="inf")
    p = int(np.flatnonzero(base["key"] >= 0)[0])
    cq = base["best"][:, p:p + 1]
    model = oracle.default_model()
    up = float(np.nextafter(0.01, 1.0))
    t0, _ = oracle.torque_test_batch("rne", cq, None, None, 0.01, 0.01, model=model)
    t1, _ = oracle.torque_test_batch("rne", cq, None, None, up, 0.01, model=model)
    j = int(np.argmax(np.abs(np.abs(t1[:6, 0]) - np.abs(t0[:6, 0]))))
    oracle.model_fields(model)["torque_limit"][j] = (abs(t0[j, 0]) + abs(t1[j, 0])) / 2
    out = []
    for mode in ("rne", "nov"):
        for mass, thr, lab in ((0.01, 0.01, "at"), (up, 0.01, "above"), (0.0, 0.0, "zero"), (5e-324, 0.0, "denorm")):
            out.append(_case(rot[:, p:p + 1], trans[:, p:p + 1], free[:, p:p + 1], q[:, p:p + 1], mode=mode,
                             mass=mass, threshold=thr, model=model.copy(), family="threshold",
                             label="%s_%s" % (mode, lab), limit_gap=abs(abs(t1[j, 0]) - abs(t0[j, 0])) / 2))
    return out


def nonfinite_ref_cases(seed=8, n=64, n_free=4):
    """NaN, +inf or -inf in one joint of q_ref (joint 0, 3 or 6), each norm; q_ref otherwise the pose's own
    configuration, stock limits, base mode."""
    rng = np.random.default_rng(seed)
    q, rot, trans = _poses(rng, n)
    free = np.vstack([q[6:7], np.clip(q[6:7] + rng.uniform(-0.4, 0.4, size=(n_free - 1, n)), Q_LO[6], Q_HI[6])])
    out = []
    for bad, lab in ((np.nan, "nan"), (np.inf, "pinf"), (-np.inf, "minf")):
        for j in (0, 3, 6):
            for norm in ("inf", "l2"):
                ref = q.copy()
                ref[j] = bad
                out.append(_case(rot, trans, free, ref, norm=norm, family="nonfinite_ref",
                                 label="%s_j%d_%s" % (lab, j, norm)))
    return out


def nan_limit_cases(seed=9, n=64, n_free=4):
    """A NaN caller limit (lo or hi of one joint) bounds nothing: equal to the same limits with that bound at +-inf."""
    rng = np.random.default_rng(seed)
    q, rot, trans = _poses(rng, n)
    free = np.vstack([q[6:7], rng.uniform(Q_LO[6], Q_HI[6], size=(n_free - 1, n))])
    out = []
    for j in (1, 3, 6):
        for which in ("lo", "hi"):
            lo, hi = Q_LO.copy(), Q_HI.copy()
            lo[j] = (lo[j] + hi[j]) / 2 if which == "hi" else lo[j]      # make the finite side bind
            hi[j] = (Q_LO[j] + hi[j]) / 2 if which == "lo" else hi[j]
            (lo if which == "lo" else hi)[j] = np.nan
            out.append(_case(rot, trans, free, q, lo=lo, hi=hi, family="nan_limit", label="%s%d" % (which, j)))
    return out


def all_cases():
    """Every family of designed cases (no torque families: torque_families())."""
    fams = {}
    for c in (joint7_limit_cases() + tie_cases() + solver_tie_cases() + full_list_case() + sweep_round_cases() +
              threshold_model() + nonfinite_ref_cases() + nan_limit_cases()):
        fams.setdefault(c["family"], []).append(c)
    return fams


MODELS = {"stock": None, "override": "model_override.npz"}


def model_record(name):
    return None if MODELS[name] is None else np.ascontiguousarray(load_golden(MODELS[name])["model"], np.float64)


def torque_families():
    """(mode, model name, norm) -> torque boundary cases."""
    out = {}
    for mode in ("rne", "nov", "dyn"):
        for mname in MODELS:
            for norm in ("inf", "l2"):
                out[(mode, mname, norm)] = torque_cases(mode, model_record(mname), norm)
    return out
