"""Long-double reference of the synthetic-scene collision predicate (collision.get_collision_fn, K8, K9) and the case
generators shared by tests/test_collision_core_host.py (host build of csrc/collision_core.cuh) and
tests/test_gpu_collision.py (the kernels).  Test-side only: nothing in the package imports it.

The reference restates the link-sphere model from the robot description, not from collision.py or the kernel: the
modified-DH chain of the Panda with the twists alpha in {0, +-pi/2} taken exactly, spheres strung along the segments
between the origins of DH frames 2..7, the flange and the grasp target (frame 7 + (0.107 + 0.105) along z7), and the
payload sphere at the grasp target.  Everything is evaluated in np.longdouble (64-bit mantissa) from the double inputs.

Verdict: a configuration collides iff a joint is outside its limits or some sphere's signed clearance to some
obstacle is < 0.  The double-precision forward kinematics of the implementations round at about 1e-15 m, so a
configuration whose smallest clearance lies within EPS = 1e-12 m of zero is in the band where no verdict is
asserted; every check reports how many fell there.  The boundary cases put an obstacle at |delta| >= 1e-9 m, 1000x
EPS, from the sphere they test.
"""
import numpy as np

from conftest import Q_HI, Q_LO

LD = np.longdouble
EPS = LD("1e-12")
DELTAS = (-1e-6, -1e-9, 1e-9, 1e-6)

# Panda modified-DH rows 1..7 (a, d, twist code: alpha = code * pi/2) and the flange row (d = 0.107)
_DH_A = [LD(s) for s in ("0", "0", "0", "0.0825", "-0.0825", "0", "0.088")]
_DH_D = [LD(s) for s in ("0.333", "0", "0.316", "0", "0.384", "0", "0")]
_DH_TWIST = [0, -1, 1, 1, -1, 1, 1]
_FLANGE_D = LD("0.107")
_TOOL_D = LD("0.105")
# (origin_from, origin_to, samples, radius) of the link-sphere model, indices into frame_origins()
SEGMENTS = [(1, 2, 3, "0.07"), (2, 3, 2, "0.07"), (3, 4, 4, "0.065"), (4, 5, 2, "0.06"), (5, 6, 2, "0.055"),
            (6, 7, 2, "0.05"), (7, 8, 3, "0.05")]
N_LINK_SPHERES = sum(m for _, _, m, _ in SEGMENTS)          # 18; index 18 is the payload sphere
LINK_RADII = np.array([LD(r) for _, _, m, r in SEGMENTS for _ in range(m)])
# Spheres that no boundary case can pin: each sits at the same centre as a larger one (origins 4 and 5 coincide, and
# consecutive segments share their end points), so the larger one is always nearer to any obstacle.
DOMINATED = {5, 9, 10, 11, 13}


def frame_origins(qs):
    """qs [n][7] (double) -> origins [n][9][3] (longdouble): index k < 7 is the origin after DH row k (frame k + 1),
    7 the flange, 8 the grasp target (collision.link_frames)."""
    qs = np.asarray(qs, dtype=np.float64).astype(LD)
    n = qs.shape[0]
    R = np.broadcast_to(np.eye(3, dtype=LD), (n, 3, 3)).copy()
    p = np.zeros((n, 3), dtype=LD)
    out = np.empty((n, 9, 3), dtype=LD)
    for k in range(7):
        tw = _DH_TWIST[k]
        # translation (a, -sin(alpha) d, cos(alpha) d) in frame k-1, then R <- R Rx(alpha) Rz(q_k)
        t = np.array([_DH_A[k], -tw * _DH_D[k], _DH_D[k] if tw == 0 else LD(0)], dtype=LD)
        p = p + np.einsum("nij,j->ni", R, t)
        rx = np.array([[1, 0, 0], [0, 0, -tw], [0, tw, 0]] if tw else np.eye(3), dtype=LD)
        c, s = np.cos(qs[:, k]), np.sin(qs[:, k])
        rz = np.zeros((n, 3, 3), dtype=LD)
        rz[:, 0, 0], rz[:, 0, 1], rz[:, 1, 0], rz[:, 1, 1], rz[:, 2, 2] = c, -s, s, c, 1
        R = np.einsum("nij,njk->nik", np.einsum("nij,jk->nik", R, rx), rz)
        out[:, k] = p
    z = R[:, :, 2]
    out[:, 7] = p + _FLANGE_D * z
    out[:, 8] = p + (_FLANGE_D + _TOOL_D) * z
    return out


def sphere_centres(qs):
    """-> centres [n][19][3] longdouble: the 18 link spheres in collision.py's order, then the grasp target."""
    o = frame_origins(qs)
    cs = []
    for a, b, m, _ in SEGMENTS:
        for i in range(m):
            t = LD(i) / LD(m - 1)
            cs.append((1 - t) * o[:, a] + t * o[:, b])
    cs.append(o[:, 8])
    return np.stack(cs, axis=1)


def clearance(centres, radii, ob):
    """Signed clearance [n][S] of spheres (centres [n][S][3], radii [S]) to one obstacle, longdouble; NaN stays NaN."""
    d = centres - np.asarray(ob.center, dtype=np.float64).astype(LD)
    if hasattr(ob, "radius"):
        return np.sqrt((d * d).sum(axis=-1)) - (radii + LD(float(ob.radius)))
    e = np.abs(d) - np.asarray(ob.half, dtype=np.float64).astype(LD)
    e = np.where(e < 0, LD(0), e)                                   # NaN kept, as np.maximum(delta, 0) does
    return np.sqrt((e * e).sum(axis=-1)) - radii


def min_clearance(qs, obstacles, payload_radius=0.0):
    """Smallest signed clearance of each configuration over every sphere and obstacle (+inf with no obstacle or
    where every clearance is NaN)."""
    qs = np.atleast_2d(np.asarray(qs, dtype=np.float64))
    out = np.full(qs.shape[0], np.inf, dtype=LD)
    if not obstacles:
        return out
    C = sphere_centres(qs)
    radii = LINK_RADII
    if payload_radius > 0:
        radii = np.concatenate([radii, [LD(float(payload_radius))]])
    else:
        C = C[:, :N_LINK_SPHERES]
    for ob in obstacles:
        c = clearance(C, radii, ob)
        c = np.where(np.isnan(c), LD(np.inf), c)
        out = np.minimum(out, c.min(axis=1))
    return out


def verdict(qs, obstacles, q_lo=Q_LO, q_hi=Q_HI, payload_radius=0.0):
    """-> (hit bool[n], in_band bool[n]): the true verdict and whether it is too close to call (never for a
    configuration outside its limits: that comparison is exact)."""
    qs = np.atleast_2d(np.asarray(qs, dtype=np.float64))
    limits = np.any(qs < q_lo, axis=1) | np.any(qs > q_hi, axis=1)
    mc = min_clearance(qs, obstacles, payload_radius)
    hit = limits | (mc < 0)
    band = ~limits & (np.abs(mc) < EPS)
    return hit, band


def assert_verdicts(got, qs, obstacles, q_lo=Q_LO, q_hi=Q_HI, payload_radius=0.0, what=""):
    """got bool[n] must equal the reference outside the band; returns the number of configurations in the band."""
    hit, band = verdict(qs, obstacles, q_lo, q_hi, payload_radius)
    got = np.asarray(got, dtype=bool)
    bad = np.flatnonzero((got != hit) & ~band)
    assert bad.size == 0, (what, bad[:10], got[bad[:10]], hit[bad[:10]])
    return int(band.sum())


# ---- case generators and checks shared by the host-build and the kernel tests ----------------------------------------
# collide(qs [n][7], obstacles, q_lo, q_hi, payload_radius) -> bool [n]
# extend(q1 [n][7], q2 [n][7], resolutions [7], obstacles, q_lo, q_hi, payload_radius) -> (n_steps [n], prefix [n])
WIDE_LO, WIDE_HI = np.full(7, -np.inf), np.full(7, np.inf)
PAYLOAD_R = 0.06            # > 0.05, so the payload sphere is never hidden behind the last link sphere
CONTACT_KINDS = ("sphere", "face", "edge", "corner", "point_sphere", "point_box")


def _unit(rng, n_axes):
    """A unit vector with exactly n_axes nonzero components (each >= 0.25 in magnitude before normalising)."""
    u = np.zeros(3)
    axes = rng.choice(3, size=n_axes, replace=False)
    u[axes] = rng.uniform(0.25, 1.0, size=n_axes) * rng.choice([-1.0, 1.0], size=n_axes)
    return u.astype(LD) / np.sqrt((u.astype(LD) ** 2).sum())


def contact_cases(n_configs, seed):
    """One obstacle at clearance delta (DELTAS) from one sphere (link spheres 0..17 with no payload, the payload
    sphere 18 with payload radius PAYLOAD_R) of a seeded configuration.  Sphere obstacles are reached along a random
    direction; boxes through a face (1 axis), an edge (2 axes) or a corner (3 axes), the three Voronoi regions of the
    box distance; point_sphere / point_box are a zero-radius sphere and a zero-size box.  The obstacle is built in
    long double and rounded to double; the reference recomputes the clearance from the rounded values.
    -> list of (q [7], obstacle, payload_radius, sphere, kind, delta)."""
    from torque_constrained_motion_planning_b200.collision import Box, Sphere
    rng = np.random.default_rng(seed)
    qs = rng.uniform(Q_LO, Q_HI, size=(n_configs, 7))
    C = sphere_centres(qs)
    cases = []
    for i in range(n_configs):
        for s in range(N_LINK_SPHERES + 1):
            r = LINK_RADII[s] if s < N_LINK_SPHERES else LD(PAYLOAD_R)
            pr = 0.0 if s < N_LINK_SPHERES else PAYLOAD_R
            c = C[i, s]
            for kind in CONTACT_KINDS:
                n_axes = {"face": 1, "edge": 2, "corner": 3}.get(kind, int(rng.integers(1, 4)))
                u = _unit(rng, n_axes)
                rad = LD(rng.uniform(0.01, 0.05))
                h = rng.uniform(0.01, 0.05, size=3).astype(LD)
                lateral = rng.uniform(-0.5, 0.5, size=3).astype(LD) * h       # inside the face for unused axes
                for delta in DELTAS:
                    near = c + u * (r + LD(delta))                             # nearest point of the obstacle
                    if kind == "sphere":
                        ob = Sphere((c + u * (r + LD(delta) + rad)).astype(np.float64), float(rad))
                    elif kind == "point_sphere":
                        ob = Sphere(near.astype(np.float64), 0.0)
                    elif kind == "point_box":
                        ob = Box(near.astype(np.float64), np.zeros(3))
                    else:
                        centre = np.where(u != 0, near + np.sign(u) * h, c + lateral)
                        ob = Box(centre.astype(np.float64), h.astype(np.float64))
                    cases.append((qs[i], ob, pr, s, kind, delta))
    return cases


def check_contacts(collide, n_configs=8, seed=11):
    """Every contact case against the reference; returns (band count, {sphere: pinned count}).  A case group
    (configuration, sphere, kind) pins the sphere when the reference flips from hit at delta < 0 to free at delta > 0,
    so an implementation that passes is within 1e-9 m of the reference's clearance for it."""
    cases = contact_cases(n_configs, seed)
    band = 0
    truth = {}
    for q, ob, pr, s, kind, delta in cases:
        got = collide(q[None], [ob], Q_LO, Q_HI, pr)
        band += assert_verdicts(got, q[None], [ob], payload_radius=pr, what=(s, kind, delta))
        truth.setdefault((tuple(q), s, kind), []).append(bool(verdict(q[None], [ob], payload_radius=pr)[0][0]))
    pinned = {}
    for (_, s, _), v in truth.items():
        pinned[s] = pinned.get(s, 0) + (v == [True, True, False, False])
    for s in range(N_LINK_SPHERES + 1):
        if s not in DOMINATED:
            assert pinned.get(s, 0) > 0, ("sphere never decides its own contact", s, pinned)
    return band, pinned


def check_obstacle_table(collide, seed=12):
    """Slot 31 and slot 0 of a full table, mixed kinds, an infinite floor slab, and an empty scene with a payload
    radius.  Returns the band count."""
    from torque_constrained_motion_planning_b200 import collision
    from torque_constrained_motion_planning_b200.collision import Box, Sphere
    rng = np.random.default_rng(seed)
    band = 0
    # one hitting obstacle in slot 31 or slot 0 of 32; the other 31 are far away
    far = [Sphere([5.0 + i, 0.0, 0.0], 0.1) if i % 2 else Box([0.0, 5.0 + i, 0.0], [0.1, 0.1, 0.1]) for i in range(31)]
    qs = rng.uniform(Q_LO, Q_HI, size=(64, 7))
    C, O = sphere_centres(qs[:1]), frame_origins(qs[:1])
    for s, (a, b) in ((1, (1, 2)), (16, (7, 8))):                 # mid-segment spheres, reached at right angles
        u = np.cross((O[0, b] - O[0, a]).astype(np.float64), rng.normal(size=3)).astype(LD)
        u /= np.sqrt((u * u).sum())
        for delta in (-1e-6, 1e-6):
            near = Sphere((C[0, s] + u * (LINK_RADII[s] + LD(0.02) + LD(delta))).astype(np.float64), 0.02)
            for table in (far + [near], [near] + far):
                assert len(table) == 32
                got = collide(qs, table, Q_LO, Q_HI, 0.0)
                band += assert_verdicts(got, qs, table, what=("slot", s, delta))
                assert bool(got[0]) == (delta < 0)
    # mixed kinds: the demo scenes, and 32 random boxes and spheres in the workspace, over random configurations
    qs = rng.uniform(Q_LO - 0.05, Q_HI + 0.05, size=(3000, 7))
    mixed = []
    for i in range(32):
        c = rng.uniform([-0.8, -0.8, -0.2], [0.8, 0.8, 1.2])
        mixed.append(Sphere(c, rng.uniform(0.01, 0.1)) if i % 3 else Box(c, rng.uniform(0.005, 0.1, size=3)))
    for scene, pr in ((collision.hiro_scene(), 0.0), (collision.cluttered_scene(), 0.04), (mixed, 0.0),
                      (mixed[:7], PAYLOAD_R)):
        got = collide(qs, scene, Q_LO, Q_HI, pr)
        band += assert_verdicts(got, qs, scene, payload_radius=pr, what="mixed")
        hit = verdict(qs, scene, payload_radius=pr)[0]
        assert 0.02 < hit.mean() < 0.98
    # an infinite floor slab whose top is delta below the lowest sphere
    qs = rng.uniform(Q_LO, Q_HI, size=(40, 7))
    C = sphere_centres(qs)[:, :N_LINK_SPHERES]
    bottom = (C[:, :, 2] - LINK_RADII).min(axis=1)
    for i in range(len(qs)):
        for delta in DELTAS:
            top = bottom[i] - LD(delta)
            slab = Box([0.0, 0.0, float(top - 1)], [np.inf, np.inf, 1.0])
            got = collide(qs[i:i + 1], [slab], Q_LO, Q_HI, 0.0)
            band += assert_verdicts(got, qs[i:i + 1], [slab], what=("slab", i, delta))
            assert bool(got[0]) == (delta < 0)
    # empty scene: only the joint limits count, the payload radius is ignored
    qs = rng.uniform(Q_LO - 0.05, Q_HI + 0.05, size=(2000, 7))
    got = collide(qs, [], Q_LO, Q_HI, PAYLOAD_R)
    assert np.array_equal(got, np.any(qs < Q_LO, axis=1) | np.any(qs > Q_HI, axis=1))
    return band


def check_joint_limits(collide, seed=13):
    """Limits are inclusive, the first double outside is a hit, caller limits replace the defaults, +-inf joints hit,
    and NaN joints follow the NumPy stand-in."""
    from torque_constrained_motion_planning_b200 import collision
    from torque_constrained_motion_planning_b200.collision import Sphere
    rng = np.random.default_rng(seed)
    far = [Sphere([9.0, 9.0, 9.0], 0.1)]                     # a scene the arm never reaches: the FK path still runs
    tight_lo, tight_hi = Q_LO + rng.uniform(0.1, 0.5, 7), Q_HI - rng.uniform(0.1, 0.5, 7)
    for lo, hi in ((Q_LO, Q_HI), (tight_lo, tight_hi)):
        mid = 0.5 * (lo + hi)
        qs, want = [], []
        for j in range(7):
            for v, hit in ((lo[j], False), (hi[j], False), (np.nextafter(lo[j], -np.inf), True),
                           (np.nextafter(hi[j], np.inf), True), (-np.inf, True), (np.inf, True)):
                q = mid.copy()
                q[j] = v
                qs.append(q)
                want.append(hit)
        qs, want = np.array(qs), np.array(want)
        for scene in ([], far):
            assert np.array_equal(collide(qs, scene, lo, hi, 0.0), want)
    # NaN joints: the stand-in's verdict, in scenes where the finite spheres before the NaN joint do and do not hit
    base = [0.5 * (Q_LO + Q_HI), rng.uniform(Q_LO, Q_HI), rng.uniform(Q_LO, Q_HI)]
    qs = []
    for q in base:
        for j in range(7):
            qn = q.copy()
            qn[j] = np.nan
            qs.append(qn)
    qs = np.array(qs)
    shoulder = [Sphere([0.0, 0.0, 0.333], 0.01)]             # at origin 1, the centre of the first link sphere
    for scene, pr in ((collision.hiro_scene(), 0.0), (collision.cluttered_scene(), PAYLOAD_R), (shoulder, 0.0),
                      (shoulder + collision.hiro_scene(), 0.0)):
        want = collision.get_collision_fn(obstacles=scene, payload_radius=pr).batch(qs)
        assert np.array_equal(collide(qs, scene, Q_LO, Q_HI, pr), want), scene
    # NaN in joint 0 or 1 leaves no sphere finite: the first sphere is 1 * origin 1 + 0 * origin 2, and 0 * NaN = NaN
    first_two = np.tile(np.arange(7) < 2, len(base))
    assert np.array_equal(collision.get_collision_fn(obstacles=shoulder).batch(qs), ~first_two)
    assert not collision.get_collision_fn(obstacles=collision.hiro_scene()).batch(qs).any()


def monotone_edges(seed, n=2, res=0.01):
    """Edges that move every joint monotonically by 0.3..0.6 rad, so > 96 configurations at resolution 0.01."""
    rng = np.random.default_rng(seed)
    q1 = rng.uniform(-1.0, 1.0, size=(n, 7))
    q2 = q1 + rng.uniform(0.3, 0.6, size=(n, 7)) * rng.choice([-1.0, 1.0], size=(n, 7))
    return q1, q2, np.full(7, res)


def extend_sequence(q1, q2, res):
    from torque_constrained_motion_planning_b200 import utils
    return np.array(list(utils.get_extend_fn(None, list(range(7)), resolutions=res)(tuple(q1), tuple(q2))))


def check_extend_steps(extend, seed=14):
    """Pins configuration k of the implementation's extend sequence to the host's ExtendSequence bit for bit: with
    the limit of joint j set to x_k[j] the safe prefix is k + 1, with the limit one ulp inside it is k.  Returns the
    number of calls made."""
    q1s, q2s, res = monotone_edges(seed)
    calls = 0
    for q1, q2 in zip(q1s, q2s):
        X = extend_sequence(q1, q2, res)
        N = len(X)
        assert N > 96
        for j in range(7):
            up = q2[j] > q1[j]
            steps = np.diff(X[:, j])
            assert (steps > 0).all() if up else (steps < 0).all()
            for k in sorted({0, 31, 32, 33, 63, 64, N - 1}):
                x = X[k, j]
                for limit, want in ((x, k + 1), (np.nextafter(x, -np.inf if up else np.inf), k)):
                    lo, hi = WIDE_LO.copy(), WIDE_HI.copy()
                    (hi if up else lo)[j] = limit
                    ns, pre = extend(q1[None], q2[None], res, [], lo, hi, 0.0)
                    calls += 1
                    assert int(ns[0]) == N and int(pre[0]) == want, (j, k, N, int(ns[0]), int(pre[0]), want)
    return calls


def sequential_num_configs(q1, q2, res):
    """int(sqrt(sum of squares)) + 1 with the sum rounded in joint order (Python floats are IEEE doubles)."""
    s = 0.0
    for j in range(7):
        d = (float(q2[j]) - float(q1[j])) / float(res[j])
        s = s + d * d
    n = float(np.sqrt(s))
    return int(n) + 1 if n == n and n < 1.0e6 else 0


def step_count_edges(seed=15):
    """Axis-aligned moves by multiples of the resolution 0.1 along Pythagorean triples and quadruples, whose exact
    norm is an integer, so rounding decides which side of it the computed norm lands on; random edges; and
    zero-length edges."""
    from torque_constrained_motion_planning_b200 import utils  # noqa: F401  (ExtendSequence is what is compared)
    rng = np.random.default_rng(seed)
    combos = [(3, 4), (6, 8), (5, 12), (1, 2, 2), (2, 3, 6), (1, 4, 8), (2, 6, 9), (4, 4, 7), (2, 10, 11), (1, 1, 1, 1),
              (2, 4, 5, 6)]
    q1, q2 = [], []
    for _ in range(300):
        for cmb in combos:
            a = rng.uniform(-2.0, 2.0, size=7)
            b = a.copy()
            axes = rng.choice(7, size=len(cmb), replace=False)
            b[axes] = a[axes] + 0.1 * np.array(cmb) * rng.choice([-1.0, 1.0], size=len(cmb))
            q1.append(a)
            q2.append(b)
    a = rng.uniform(-2.0, 2.0, size=(500, 7))
    q1 += list(a)
    q2 += list(a + rng.normal(0, 0.6, size=a.shape))
    q1 += list(a[:50])
    q2 += list(a[:50])                                            # zero length: 1 configuration
    return np.array(q1), np.array(q2), np.full(7, 0.1)


def check_step_count(extend):
    """n_steps equals the sequentially rounded count everywhere, and ExtendSequence.num_configs() except where
    np.linalg.norm's own summation order lands on the other side of an integer.  Non-finite end points and norms
    >= 1e6 give 0 configurations and a prefix of 0.  Returns the number of edges where the two counts differ."""
    from torque_constrained_motion_planning_b200 import utils
    q1, q2, res = step_count_edges()
    ns, pre = extend(q1, q2, res, [], WIDE_LO, WIDE_HI, 0.0)
    want = np.array([sequential_num_configs(a, b, res) for a, b in zip(q1, q2)])
    assert np.array_equal(ns, want) and np.array_equal(pre, ns)
    assert (ns[-50:] == 1).all()
    ext = utils.get_extend_fn(None, list(range(7)), resolutions=res)
    host = np.array([ext(tuple(a), tuple(b)).num_configs() for a, b in zip(q1, q2)])
    differ = np.flatnonzero(host != ns)
    for e in differ:
        nrm = np.linalg.norm((q2[e] - q1[e]) / res)
        assert abs(host[e] - ns[e]) == 1 and abs(nrm - round(nrm)) < 1e-12, (e, host[e], ns[e], nrm)
    # no step count: NaN / inf end points, and norms >= 1e6
    a = np.zeros((6, 7))
    b = np.zeros((6, 7))
    b[0, 2], a[1, 5], b[2, 0], a[3, 6] = np.nan, np.nan, np.inf, -np.inf
    b[4, 0] = 2.0e5                         # norm 2e6 at resolution 0.1
    b[5, 3] = 3.0e7
    ns, pre = extend(a, b, res, [], WIDE_LO, WIDE_HI, 0.0)
    assert (ns == 0).all() and (pre == 0).all(), (ns, pre)
    return int(differ.size)
