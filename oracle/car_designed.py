"""Designed car states and float64 references for the car step-kernel parity tests -- TEST INFRASTRUCTURE ONLY.

Rows are in get_state()'s (24,) layout per car: hull x, y, angle, vx, vy, w; per wheel k joint angle, omega, gas,
#tiles; reward; tiles visited.  set_state (crl_car_set_state, car_oracle_set_state) uses x .. w, the joint angles, omega,
rear gas and the reward.  Each generator has an explicit list of corner rows, cycled by `app` (the how-many-th
application this is) so that small batches still reach every corner, and fills the other rows from a seeded numpy
Generator.

References (float64, restated from the reference's Python and Box2D's published algorithm):
  * tile_polygons: the 5 listed vertices of every tile (_create_track :399-445), then their convex hull;
  * sat_margin: the largest face separation of a wheel box and a tile polygon minus 2 * b2_polygonRadius
    (touching <=> margin < 0, the sensor test of b2ContactManager::Collide without the broadphase);
  * wheel_omega_step1: omega of every wheel after the first sub-step that follows set_state.  set_state clears the
    wheels' tile sets on both sides, so this sub-step always uses the grass friction limit (0.6 x).
"""
import numpy as np

SIZE = 0.02
TRACK_WIDTH = 40 / 6.0
PLAYFIELD = 2000 / 6.0
FPS = 50
ENGINE_POWER = 100000000 * SIZE * SIZE
WHEEL_MOI = 4000 * SIZE * SIZE
FRICTION_LIMIT = 1000000 * SIZE * SIZE
WHEEL_R, WHEEL_W = 27, 14
POLY_SKIN = 2 * float(np.float32(0.01))           # 2 * b2_polygonRadius (float32 0.01)
WHEELPOS = np.array([[-55, 80], [55, 80], [-55, -82], [55, -82]], np.float64)
MAX_TRANSLATION, MAX_ROTATION = 2.0, 0.5 * np.pi
f32 = np.float32


# ---------------------------------------------------------------------------------------------------------------- tracks
def _pts3(track):
    t = np.asarray(track, np.float64)
    return t[:, 1:4] if t.shape[1] == 4 else t


def tile_raw(track, i):
    """The 5 vertices build_tile / build_tiles list for tile i (fp64): l1, bump, r1 of point i, r2, l2 of point i - 1."""
    p = _pts3(track)
    n = len(p)
    b1, x1, y1 = p[i]
    b2, x2, y2 = p[(i - 1) % n]
    W = TRACK_WIDTH
    return np.array([[x1 - W * np.cos(b1), y1 - W * np.sin(b1)],
                     [x1 - W / 2 * np.cos(b1 - np.pi / 2), y1 - W / 2 * np.sin(b1 - np.pi / 2)],
                     [x1 + W * np.cos(b1), y1 + W * np.sin(b1)],
                     [x2 + W * np.cos(b2), y2 + W * np.sin(b2)],
                     [x2 - W * np.cos(b2), y2 - W * np.sin(b2)]])


def convex_hull(pts):
    """CCW convex hull (monotone chain), points closer than 0.5 * b2_linearSlop welded as b2PolygonShape::Set does."""
    q = []
    for v in pts:
        if all(np.hypot(*(v - u)) >= 0.0025 for u in q):
            q.append(np.asarray(v, np.float64))
    q = sorted(q, key=lambda v: (v[0], v[1]))
    cross = lambda o, a, b: (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])   # noqa: E731
    lo, hi = [], []
    for v in q:
        while len(lo) >= 2 and cross(lo[-2], lo[-1], v) <= 0:
            lo.pop()
        lo.append(v)
    for v in reversed(q):
        while len(hi) >= 2 and cross(hi[-2], hi[-1], v) <= 0:
            hi.pop()
        hi.append(v)
    return np.array(lo[:-1] + hi[:-1])


def tile_polygons(track):
    return [convex_hull(tile_raw(track, i)) for i in range(len(track))]


def tile_reach(track):
    """(n,) largest distance from each tile's track point to one of its listed vertices."""
    p = _pts3(track)
    return np.array([np.hypot(*(tile_raw(track, i) - p[i, 1:3]).T).max() for i in range(len(p))])


def seam_gap(track):
    """length of the seam (point n - 1 to point 0) along the direction of point 0, and across it"""
    p = _pts3(track)
    d = p[0, 1:3] - p[-1, 1:3]
    fwd = np.array([-np.sin(p[0, 0]), np.cos(p[0, 0])])
    return float(d @ fwd), float(abs(d @ np.array([np.cos(p[0, 0]), np.sin(p[0, 0])])))


def long_seam_tracks(count, seed=1, min_gap=11.0):
    """The first `count` tracks of RandomState(seed) (car_oracle.make_track) whose seam is longer than min_gap along the
    track: there the middle of the seam tile lies more than 9 units from every track point."""
    import car_oracle as C
    rng = np.random.RandomState(seed)
    out = []
    while len(out) < count:
        tr, bd, d = C.make_track(rng)
        if seam_gap(tr)[0] > min_gap:
            out.append((tr, bd, d))
    return out


# ---------------------------------------------------------------------------------------------------------------- wheels
def _rot(a):
    return np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])


def wheel_poses(row):
    """(4, 3) wheel centre x, y and angle right after set_state(row), from the float32-rounded inputs (fp64 arithmetic)."""
    org = np.array([f32(row[0]), f32(row[1])], np.float64)
    a = float(f32(row[2]))
    out = np.zeros((4, 3))
    for k in range(4):
        out[k, :2] = org + _rot(a) @ np.array([float(f32(WHEELPOS[k, 0] * SIZE)), float(f32(WHEELPOS[k, 1] * SIZE))])
        out[k, 2] = a + float(f32(row[6 + 4 * k]))
    return out


def wheel_box(pose):
    hw, hr = WHEEL_W * SIZE, WHEEL_R * SIZE
    loc = np.array([[-hw, -hr], [hw, -hr], [hw, hr], [-hw, hr]])
    return loc @ _rot(pose[2]).T + pose[:2]


def _max_sep(A, B):
    best = -np.inf
    for i in range(len(A)):
        e = A[(i + 1) % len(A)] - A[i]
        ln = np.hypot(*e)
        if ln < 1e-12:
            continue
        nrm = np.array([e[1], -e[0]]) / ln
        best = max(best, ((B - A[i]) @ nrm).min())
    return best


def sat_margin(A, B):
    """largest separation over the faces of both convex CCW polygons, minus the two skins: < 0 = the sensors touch"""
    return max(_max_sep(A, B), _max_sep(B, A)) - POLY_SKIN


def wheel_tile_margins(polys, row):
    """(4, n) margins of every wheel of the car in `row` against every tile (tiles farther than 20 units: +inf)."""
    wp = wheel_poses(row)
    out = np.full((4, len(polys)), np.inf)
    for k in range(4):
        box = wheel_box(wp[k])
        for t, P in enumerate(polys):
            if np.hypot(*(P.mean(0) - wp[k, :2])) < 20.0:
                out[k, t] = sat_margin(box, P)
    return out


def sensor_reference(polys, row, eps=1e-4):
    """(counts (4,), touched tile set, near-zero flag): what the four wheels of a car set to `row` overlap."""
    m = wheel_tile_margins(polys, row)
    touch = m < 0
    return touch.sum(1), set(np.nonzero(touch.any(0))[0].tolist()), bool((np.abs(m) <= eps).any())


# ---------------------------------------------------------------------------------------------------------- wheel model
def _hull_local_centre():
    """centroid of the hull's four polygons (density 1), body frame"""
    polys = [[(-60, 130), (60, 130), (60, 110), (-60, 110)], [(-15, 120), (15, 120), (20, 20), (-20, 20)],
             [(25, 20), (50, -10), (50, -40), (20, -90), (-20, -90), (-50, -40), (-50, -10), (-25, 20)],
             [(-50, -120), (50, -120), (50, -90), (-50, -90)]]
    area, c = 0.0, np.zeros(2)
    for P in polys:
        P = np.array(P, np.float64) * SIZE
        if sum(P[i - 1, 0] * P[i, 1] - P[i, 0] * P[i - 1, 1] for i in range(len(P))) < 0:
            P = P[::-1]                                  # the listed polygons wind both ways
        for i in range(len(P)):
            a, b = P[i], P[(i + 1) % len(P)]
            cr = a[0] * b[1] - a[1] * b[0]
            area += cr / 2
            c += cr * (a + b) / 6
    return c / area


HULL_LC = _hull_local_centre()


def process_action(a0, a1):
    """process_action (:527-540) -> (steer, gas, brake)"""
    a0 = max(min(float(a0), 1.0), -1.0)
    a1 = max(min(float(a1), 1.0), -1.0)
    if a1 > 0:
        a2 = 0.0
    else:
        a2, a1 = a1, 0.0
    return -a0, abs(a1), abs(a2)


def wheel_omega_step1(row, action):
    """(4,) omega after the first sub-step after set_state(row) with `action` (float32 as the env receives it): Car.gas /
    brake, then Car.step's wheel model with the grass friction limit.  Wheel velocity, forward and side axes in float32
    from the float32-rounded state as set_state and Box2D compute them; the model itself in float64."""
    a = f32(row[2])
    q = _rot(float(a))
    org = np.array([f32(row[0]), f32(row[1])], np.float64)
    com = org + q @ HULL_LC
    v0 = np.array([f32(row[3]), f32(row[4])], np.float64)
    w0 = float(f32(row[5]))
    _, g, brake = process_action(f32(action[0]), f32(action[1]))
    wp = wheel_poses(row)
    out = np.zeros(4)
    for k in range(4):
        d = wp[k, :2] - com
        vw = v0 + w0 * np.array([-d[1], d[0]])
        wa = float(f32(wp[k, 2]))
        forw = np.array([-np.sin(wa), np.cos(wa)], np.float32).astype(np.float64)
        side = np.array([np.cos(wa), np.sin(wa)], np.float32).astype(np.float64)
        vf, vs = float(forw @ vw), float(side @ vw)
        om = float(row[7 + 4 * k])
        gas = 0.0
        if k >= 2:
            gk = float(row[8 + 4 * k])
            gas = gk + min(g - gk, 0.1)
        om += (1.0 / FPS) * ENGINE_POWER * gas / WHEEL_MOI / (abs(om) + 5.0)
        if brake >= 0.9:
            om = 0.0
        elif brake > 0:
            bval = min(15 * brake, abs(om))
            om += -np.sign(om) * bval
        ff = (-vf + om * WHEEL_R * SIZE) * 205000 * SIZE * SIZE
        pf = -vs * 205000 * SIZE * SIZE
        frc = np.hypot(ff, pf)
        lim = FRICTION_LIMIT * 0.6
        if frc > lim:
            ff = ff / frc * lim
        om -= (1.0 / FPS) * ff * (WHEEL_R * SIZE) / WHEEL_MOI
        out[k] = om
    return out


# -------------------------------------------------------------------------------------------------------- designed rows
def placed_row(target, wheel, hull_angle, joint=0.0):
    """A row whose wheel `wheel` has its centre at `target` (x, y) with the hull at `hull_angle` (front joints `joint`)."""
    r = np.zeros(24)
    r[2] = hull_angle
    r[0:2] = np.asarray(target, np.float64) - _rot(hull_angle) @ (WHEELPOS[wheel] * SIZE)
    r[6] = r[10] = joint
    return r


def _edge_normal(P, i):
    e = P[(i + 1) % len(P)] - P[i]
    return np.array([e[1], -e[0]]) / np.hypot(*e)


SENSOR_KINDS = ("edge", "corner", "bump", "seam", "inner", "off_road", "random")


def sensor_rows(rng, track, n, app=0, polys=None):
    """n rows of one car placed around the tiles of `track` (n, 4): each corner puts one wheel (cycled 0..3) straddling a
    tile edge, on a hull corner, on the bump vertex (W/2 ahead of the track point), on the seam tile at fractions of the
    seam gap, on the inner side of the sharpest turn, or parallel to a road edge at +-0.005 / 0.05 / 0.5 off the touching
    distance; the remaining rows are random poses near the road.  Front joint angles in [-0.5, 0.5]."""
    p = _pts3(track)
    nt = len(p)
    polys = tile_polygons(track) if polys is None else polys
    db = np.abs((p[:, 0] - np.roll(p[:, 0], 1) + np.pi) % (2 * np.pi) - np.pi)
    db[0] = 0.0
    sharp = int(np.argmax(db))
    corners = []
    for f in (0.05, 0.15, 0.25, 0.35, 0.5, 0.65, 0.8, 0.95):
        for lat in (-0.8, -0.3, 0.0, 0.4, 0.85):
            corners.append(("seam", f, lat))
    for d in (0.005, -0.005, 0.05, -0.05, 0.5, -0.5):
        corners.append(("off_road", d, None))
    corners += [("edge", None, None), ("corner", None, None), ("bump", None, None), ("inner", None, None)]
    rows = np.zeros((n, 24))
    for i in range(n):
        wheel = (i + app) % 4
        ang = rng.uniform(-np.pi, np.pi)
        joint = rng.uniform(-0.5, 0.5)
        kind, a1, a2 = corners[(i + app * n) % len(corners)] if i < max(len(corners), n // 2) else ("random", None, None)
        t = int(rng.integers(0, nt))
        if kind == "seam":
            c = p[-1, 1:3] + a1 * (p[0, 1:3] - p[-1, 1:3])
            lat = np.array([np.cos(p[0, 0]), np.sin(p[0, 0])])
            rows[i] = placed_row(c + a2 * TRACK_WIDTH * lat, wheel, ang, joint)
        elif kind == "off_road":
            P = polys[t]
            outer = tile_raw(track, t)[[2, 3]] if rng.random() < 0.5 else tile_raw(track, t)[[4, 0]]
            e = outer[1] - outer[0]
            nrm = np.array([e[1], -e[0]]) / np.hypot(*e)
            if (P.mean(0) - outer[0]) @ nrm > 0:
                nrm = -nrm
            mid = 0.5 * (outer[0] + outer[1])
            wa = np.arctan2(-e[0], e[1])               # wheel's long axis along the edge
            hw = WHEEL_W * SIZE
            r = placed_row(mid + (hw + POLY_SKIN + a1) * nrm, wheel, ang, 0.0)
            r[2] = wa - (joint if wheel < 2 else 0.0)
            r[0:2] = mid + (hw + POLY_SKIN + a1) * nrm - _rot(r[2]) @ (WHEELPOS[wheel] * SIZE)
            r[6] = r[10] = joint
            rows[i] = r
        elif kind in ("edge", "corner"):
            P = polys[t]
            j = int(rng.integers(0, len(P)))
            c = P[j] if kind == "corner" else 0.5 * (P[j] + P[(j + 1) % len(P)])
            rows[i] = placed_row(c, wheel, ang, joint)
        elif kind == "bump":
            rows[i] = placed_row(tile_raw(track, t)[1], wheel, ang, joint)
        elif kind == "inner":
            v = tile_raw(track, sharp)
            rows[i] = placed_row(v[0] if rng.random() < 0.5 else v[2], wheel, ang, joint)
        else:
            c = p[t, 1:3] + rng.uniform(-9, 9, 2)
            rows[i] = placed_row(c, wheel, ang, joint)
        if rng.random() < 0.5:                          # the other front wheel at its own angle
            rows[i, 10] = rng.uniform(-0.5, 0.5)
    return rows


def at_rest(rows):
    """The same placements with the car at rest and both front wheels at the angle the steering holds (|joint| < 0.4):
    through further sub-steps of the same action (action_repeat > 1) the wheels stay where they were put.  Returns the
    rows and the (n, 2) actions that hold them."""
    r = np.array(rows, np.float64).copy()
    r[:, 3:6] = 0.0
    j = np.clip(r[:, 6], -0.39, 0.39)
    r[:, 6] = r[:, 10] = j
    for k in range(4):
        r[:, 7 + 4 * k] = 0.0
        r[:, 8 + 4 * k] = 0.0
    return r, np.stack([-j, np.zeros_like(j)], axis=1)


WHEEL_CORNERS = [  # (speed, heading of the velocity relative to the hull, w, omega, gas)
    (0.0, 0.0, 0.0, 0.0, 0.0), (0.0, 0.0, 0.0, -300.0, 1.0), (0.0, 0.0, 0.0, 400.0, 0.0), (5.0, 0.0, 0.0, 0.0, 0.5),
    (30.0, 0.0, 0.0, 60.0, 1.0), (30.0, np.pi / 2, 0.0, 0.0, 0.0), (99.0, 0.0, 0.0, 150.0, 0.9),
    (101.0, 0.3, 0.0, -50.0, 0.2), (150.0, -1.0, 0.0, 400.0, 1.0), (20.0, 0.0, 78.0, 0.0, 0.0),
    (0.0, 0.0, -80.0, 10.0, 0.0), (40.0, 2.5, 120.0, -300.0, 0.7), (1e-3, 0.0, 1e-3, 1e-3, 0.0),
]


def wheel_rows(rng, track, n, app=0):
    """Cars on the road (hull origin on a random track point, heading along it) with the wheel-model corners: omega in
    [-300, 400], gas 0..1, speeds from 0 to above b2_maxTranslation * FPS (100), |w| above b2_maxRotation * FPS (78.5)."""
    p = _pts3(track)
    rows = np.zeros((n, 24))
    for i in range(n):
        t = int(rng.integers(0, len(p)))
        r = rows[i]
        r[0:2] = p[t, 1:3] + rng.uniform(-2, 2, 2)
        r[2] = p[t, 0] + rng.uniform(-0.3, 0.3)
        j = i + app * n
        if i < len(WHEEL_CORNERS):
            sp, hd, w, om, g = WHEEL_CORNERS[j % len(WHEEL_CORNERS)]
            oms = np.full(4, om)
            gs = np.full(4, g)
        else:
            sp, hd, w = rng.uniform(0, 160), rng.uniform(-np.pi, np.pi), rng.choice([0.0, rng.uniform(-100, 100)])
            oms, gs = rng.uniform(-300, 400, 4), rng.uniform(0, 1, 4)
        fwd = r[2] + hd
        r[3:5] = sp * np.array([-np.sin(fwd), np.cos(fwd)])
        r[5] = w
        for k in range(4):
            r[6 + 4 * k] = rng.uniform(-0.5, 0.5) if k < 2 else 0.0
            r[7 + 4 * k] = oms[k]
            r[8 + 4 * k] = gs[k] if k >= 2 else 0.0
        r[22] = rng.uniform(-50, 500)
    return rows


WHEEL_ACTIONS = np.array([[0.0, 0.0], [-0.0, -0.0], [0.0, 1.0], [0.3, 0.5], [-0.3, -0.3], [0.6, -0.89], [-0.6, -0.9],
                          [1.0, -1.0], [-1.0, 0.2], [1.7, 2.5], [-3.0, -1.2], [0.0, -0.3], [0.0, -0.89], [0.0, -0.9]],
                         np.float32)


def playfield_rows(rng, n, deltas=(-1.0, -0.01, 0.01, 1.0)):
    """The hull at +-(2000/6 + delta) in x or y (delta < 0: still inside), at rest, heading random."""
    rows = np.zeros((n, 24))
    for i in range(n):
        d = deltas[i % len(deltas)]
        axis, sgn = (i // len(deltas)) % 2, (-1.0, 1.0)[(i // (2 * len(deltas))) % 2]
        rows[i, axis] = sgn * (PLAYFIELD + d)
        rows[i, 1 - axis] = rng.uniform(-200, 200)
        rows[i, 2] = rng.uniform(-np.pi, np.pi)
    return rows


def road_row(track, t, lateral=0.0):
    """the car at rest with its hull origin on the middle of tile t (between points t - 1 and t), facing along the track"""
    p = _pts3(track)
    c = 0.5 * (p[t, 1:3] + p[t - 1, 1:3]) + lateral * np.array([np.cos(p[t, 0]), np.sin(p[t, 0])])
    r = np.zeros(24)
    r[0:2] = c
    r[2] = p[t, 0]
    return r
