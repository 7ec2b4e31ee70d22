"""The game step's numeric decisions at their boundaries, one teacher-forced step against the oracle.

Each GPU case builds crafted states, puts them on one handle (sf_set_state), takes ONE sf_step with key mask 0 and
compares with the oracle's SSF_Env.step from the same states. Ships and projectiles stand still unless a case needs
motion, so the points that are tested are the points that were chosen. The cases:

* aiming: the autoturn heading ceil(angleTo) and the fortress sector ceil(angle / 10) * 10 (sf_ceil_angle<1> / <10>), on
  every integer position of the big hexagon's bounding box, the same moved by one ulp, exact octants, random doubles and
  the doubles nearest the rays at every integer degree. Outside a band of 1e-12 degrees around the multiples of the step
  the device equals the oracle. Inside it the reference's own rounding decides, so the device is held to the exact
  ceiling (the direction computed to 60 digits) down to ANGLE_SIGN_BAND, and to one of the two neighbouring multiples
  below that: the sign test compares against a host-libm cos / sin table whose argument a * pi / 180 is itself rounded,
  an angle error of up to ~1e-13 degrees at 359 degrees;
* collisions at the radii 13 (shell / ship), 23 (missile / fortress) and 21 (shells hidden near the fortress, frames):
  squared distances at the host-built threshold T(r) (SfHot::touch2) and a few ulps either side;
* the ship on the edges of both hexagons (inclusive) and one ulp off them;
* the shell the fortress fires (device fp64 atan2 / cos / sin): bit-exact angles at octants, 1e-12 elsewhere;
* feature rows (sf_features_f64 / sf_features) where aim and ndist sit on their monitor thresholds.

The tests without the gpu marker show, from the oracle and host arithmetic alone, that these sets can catch a wrong
kernel."""
import ctypes as C
import decimal
import math

import numpy as np
import pytest

from gpu_helpers import KINDS, oracle_features, torch_cuda, vp
from oracle.oracle import MAX_MISSILES, MAX_SHELLS, Record, draw_native, record_dtype, step_records, OracleEnv

DT = record_dtype()
FX, FY = 355.0, 315.0
STEP_BAND = 1e-12        # degrees: outside it the device decides like the reference
ANGLE_SIGN_BAND = 2e-13  # degrees: beyond it (inside STEP_BAND) the device gives the exact ceiling
SHELL_TOL = 1e-12        # |d shell_angle| (degrees) and |d shell_v| of a fresh shell (CUDA: <= 2 ulp atan2 / cos / sin)
EV_FORTRESS_FIRED, EV_HIT_FORTRESS, EV_SHELL_HIT_SHIP = 1 << 1, 1 << 2, 1 << 9
EV_BIGHEX, EV_SMALLHEX, EV_COL_MISSILE = 1 << 7, 1 << 8, 1 << 14
INF = float("inf")
AIM_FIELDS = ("ship_angle", "fortress_angle", "fortress_last_angle", "fortress_timer")   # what the aiming decides

# ---------------------------------------------------------------------------------------------------------------------
# exact arithmetic: directions to 60 digits (stdlib decimal, exact Decimal(float) inputs)
# ---------------------------------------------------------------------------------------------------------------------
_CTX = decimal.Context(prec=60)
_D = decimal.Decimal
PI = _D("3.14159265358979323846264338327950288419716939937510582097494459230781640628620899863")


def _series(x):
    """(cos x, sin x) by their Taylor series, |x| <= 2 pi, to the context's 60 digits"""
    with decimal.localcontext(_CTX):
        c, s, t, k = _D(0), _D(0), _D(1), 0
        while abs(t) > _D("1e-75"):
            c += t; k += 2; t = -t * x * x / (k * (k - 1))
        t, k = x, 1
        while abs(t) > _D("1e-75"):
            s += t; k += 2; t = -t * x * x / (k * (k - 1))
        return c, s


_CS = None


def cs_deg(k):
    """exact (cos, sin) of k degrees, k integer"""
    global _CS
    if _CS is None:
        with decimal.localcontext(_CTX):
            _CS = [_series(_D(a) * PI / 180) for a in range(360)]
    return _CS[int(k) % 360]


def ceil_exact(dx, dy, step):
    """For directions (dx, dy) (float arrays, computed exactly from the chosen points): the exact ceil of the direction
    theta in [0, 360) to a multiple of `step`, mod 360, and the distance (degrees) from theta to the nearest multiple
    (inf when it is more than 1e-9, where float64 decides). (0, 0) counts as direction 0, like atan2."""
    dx, dy = np.asarray(dx, np.float64), np.asarray(dy, np.float64)
    th = np.degrees(np.arctan2(dy, dx)) % 360.0
    out = (step * np.ceil(th / step)).astype(np.int64) % 360
    dist = np.full(len(dx), INF)
    m = step * np.round(th / step)
    near = np.abs(th - m) < 1e-9
    with decimal.localcontext(_CTX):
        for i in np.nonzero(near)[0]:
            if dx[i] == 0 and dy[i] == 0:
                out[i], dist[i] = 0, 0.0
                continue
            c, s = cs_deg(m[i])
            f = c * _D(float(dy[i])) - s * _D(float(dx[i]))   # sin(theta - m) * r
            r = (_D(float(dx[i])) ** 2 + _D(float(dy[i])) ** 2).sqrt()
            dist[i] = float(abs(f) / r * 180 / PI)
            out[i] = (int(m[i]) + (0 if f <= 0 else step)) % 360
    return out, dist


def heading_dir(x, y):   # angleTo(ship -> fortress) (vector.cpp:48-52)
    return FX - x, FY - y


def sector_dir(x, y):    # the fortress's angle to the ship (game.cpp:197)
    return x - FX, y - FY


def octant(dx, dy):
    """the directions sf_ceil_angle hands to the reference's own libm values (sf_atan2)"""
    return (dx == 0) | (dy == 0) | (np.abs(dx) == np.abs(dy))


# ---------------------------------------------------------------------------------------------------------------------
# records
# ---------------------------------------------------------------------------------------------------------------------
def records(x, y):
    """live ship at (x, y), at rest, heading 90; live fortress, not about to fire; tick 1000"""
    r = np.zeros(len(x), DT)
    r["ship_x"], r["ship_y"] = x, y
    r["ship_angle"] = 90.0
    r["ship_alive"] = 1; r["fortress_alive"] = 1
    r["ship_death_timer"] = 5000; r["fortress_death_timer"] = 5000; r["fortress_vuln_timer"] = 250
    r["tick"] = 1000; r["time"] = 34000
    r["rng_seed"] = 1
    return r


def to_record(row):
    return Record.from_buffer_copy(row.tobytes())


def _live(mask, n):
    return ((mask[:, None].astype(np.int64) >> np.arange(n)) & 1).astype(bool)


def mismatch(exp, got, skip=(), shell_tol=0.0):
    """per record: True where a field of the states differs (projectile arrays: live slots only; shells within
    shell_tol, everything else exact)"""
    bad = np.zeros(len(exp), bool)
    lm, ls = _live(exp["missile_mask"], MAX_MISSILES), _live(exp["shell_mask"], MAX_SHELLS)
    for name in DT.names:
        if name in skip or name == "_pad":   # _pad is the device's ep_return
            continue
        a, b = exp[name], got[name]
        if name.startswith("missile_") and name != "missile_mask":
            bad |= ((a != b) & lm).any(1)
        elif name.startswith("shell_") and name != "shell_mask":
            bad |= ((np.abs(a - b) > shell_tol) & ls).any(1)
        else:
            d = a != b
            bad |= d.reshape(len(a), -1).any(1)
    return bad


def first(idx, k=5):
    return [int(i) for i in np.nonzero(idx)[0][:k]]


class Device:
    """one handle of n envs for the crafted states of a case"""

    def __init__(self, gametype, n):
        torch = torch_cuda()
        from spacefortress_b200 import SFVecEnv, _lib
        self.torch, self._lib = torch, _lib
        self.env = SFVecEnv(gametype, num_envs=n, device=0, render=False)
        self.n = n

    def set(self, recs):
        assert len(recs) == self.n and recs.dtype == DT
        recs = np.ascontiguousarray(recs)
        self._lib.check(self.env.L.sf_set_state(self.env.h, 0, self.n, C.c_void_p(recs.ctypes.data)))

    def get(self):
        out = np.zeros(self.n, DT)
        self._lib.check(self.env.L.sf_get_state(self.env.h, 0, self.n, C.c_void_p(out.ctypes.data)))
        return out

    def step(self, recs, native=False):
        """sf_step with key mask 0 from `recs`: (states after, int [n, 4] reward / done / kill / events, frames or None)"""
        torch, L = self.torch, self._lib
        self.set(recs)
        back = self.get()
        assert not mismatch(recs, back).any(), "sf_set_state / sf_get_state round trip"
        n = self.n
        act = torch.zeros(n, dtype=torch.int32, device="cuda")
        rew, ev = torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda")
        done, kill = torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
        obs = torch.empty((n, 92, 90), dtype=torch.uint8, device="cuda") if native else None
        flags = L.FLAG_ACTIONS_ARE_KEYMASKS | L.FLAG_NO_AUTORESET | ((L.FLAG_RENDER | L.FLAG_NATIVE_OBS) if native else 0)
        L.check(self.env.L.sf_step(self.env.h, vp(act), vp(obs), vp(rew), vp(done), vp(kill), vp(ev), flags, None))
        torch.cuda.synchronize()
        outs = np.stack([t.cpu().numpy().astype(np.int64) for t in (rew, done, kill, ev)], 1)
        return self.get(), outs, (obs.cpu().numpy() if native else None)

    def render_native(self):
        return self.env.render_frames(native=True)

    def close(self):
        self.env.close()


def oracle_step(gametype, recs):
    after, out = step_records(gametype, recs)
    out = out.astype(np.int64)
    out[:, 3] &= 0xFFFFFFFF   # the event bits as unsigned
    return after, out


def compare(gametype, recs, dev, ctx, skip=(), shell_tol=0.0, native=False):
    """one step (youturn game types) on the device and in the oracle; asserts everything but `skip` equal, and the
    fortress's aim too unless its direction to the ship is in the aiming band (test_aiming_decisions_against_the_oracle);
    returns both"""
    assert "autoturn" not in gametype
    exp, eout = oracle_step(gametype, recs)
    got, gout, frames = dev.step(recs, native=native)
    gout[:, 3] &= 0xFFFFFFFF
    dx, dy = sector_dir(recs["ship_x"], recs["ship_y"])
    band = ~octant(dx, dy) & (ceil_exact(dx, dy, 10)[1] <= STEP_BAND)
    bad = mismatch(exp, got, skip + AIM_FIELDS, shell_tol) | (eout != gout).any(1)
    bad |= ~band & mismatch(exp, got, skip, shell_tol)
    assert not bad.any(), (ctx, int(bad.sum()), [(i, recs[i]["ship_x"], recs[i]["ship_y"], eout[i].tolist(), gout[i].tolist()) for i in first(bad)])
    return exp, eout, got, gout, frames


# ---------------------------------------------------------------------------------------------------------------------
# aiming sets
# ---------------------------------------------------------------------------------------------------------------------
def _nextafter(v, k):
    """v moved by k ulps (a float for a float, an array for an array)"""
    if np.ndim(v) == 0:
        v = float(v)
        for _ in range(abs(k)):
            v = math.nextafter(v, INF if k > 0 else -INF)
        return v
    v = np.asarray(v, np.float64).copy()
    for _ in range(abs(k)):
        v = np.nextafter(v, INF if k > 0 else -INF)
    return v


def aiming_sets():
    xs, ys = np.arange(155.0, 556.0), np.arange(141.0, 489.0)   # the big hexagon's bounding box (vertices floored)
    X, Y = np.meshgrid(xs, ys)
    gx, gy = X.ravel(), Y.ravel()
    sets = {"integer": (gx, gy)}
    sets["integer_ulp"] = (np.concatenate([_nextafter(gx, 1), _nextafter(gx, -1), gx, gx]),
                           np.concatenate([gy, gy, _nextafter(gy, 1), _nextafter(gy, -1)]))
    ox, oy = [FX], [FY]   # the fortress centre itself: atan2(0, 0)
    for d in (1.0, 2.0, 3.0, 7.0, 0.5, 0.25, 40.0, 41.0, 100.0, 199.0, 200.0, 201.5):
        for cx, cy in ((1, 0), (1, 1), (0, 1), (-1, 1), (-1, 0), (-1, -1), (0, -1), (1, -1)):
            ox.append(FX + cx * d); oy.append(FY + cy * d)
    sets["octants"] = (np.array(ox), np.array(oy))
    rng = np.random.RandomState(20)
    sets["random"] = (rng.uniform(150, 560, 100000), rng.uniform(110, 520, 100000))
    sets["near_ray"] = near_ray_set()
    return sets


def near_ray_set():
    """for every integer degree k and several radii: the doubles nearest the ray from the fortress at k and at
    k +- {1e-13, 1e-11, 1e-9} degrees; and the ship at x = 100 / 600 with y = 315 +- 1..4 ulp"""
    px, py = [], []
    with decimal.localcontext(_CTX):
        for k in range(360):
            c, s = cs_deg(k)
            for dd in ("0", "1e-13", "-1e-13", "1e-11", "-1e-11", "1e-9", "-1e-9"):
                e = _D(dd) * PI / 180
                ce, se = 1 - e * e / 2 + e ** 4 / 24, e - e ** 3 / 6 + e ** 5 / 120   # |e| < 2e-11: exact to 60 digits
                cc, ss = c * ce - s * se, s * ce + c * se
                for rad in (45, 100, 170, 230):
                    px.append(float(_D(FX) + rad * cc)); py.append(float(_D(FY) + rad * ss))
    for x in (100.0, 600.0):
        for k in (-4, -3, -2, -1, 1, 2, 3, 4):
            px.append(x); py.append(float(_nextafter(FY, k)))
    return np.array(px), np.array(py)


def aiming_expectations(x, y):
    """per record and per decision (heading step 1, sector step 10): exact ceiling, distance to the nearest multiple,
    octant flag"""
    out = {}
    for key, step, (dx, dy) in (("heading", 1, heading_dir(x, y)), ("sector", 10, sector_dir(x, y))):
        ex, dist = ceil_exact(dx, dy, step)
        out[key] = (ex, dist, octant(dx, dy), step)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# collision sets
# ---------------------------------------------------------------------------------------------------------------------
def touch_threshold(r):
    """SfHot::touch2 (sf_tables.cpp): the largest double x with sqrt(x) <= r (math.sqrt is correctly rounded)"""
    x = float(r * r)
    while math.sqrt(x) > r:
        x = math.nextafter(x, 0.0)
    while math.sqrt(math.nextafter(x, INF)) <= r:
        x = math.nextafter(x, INF)
    return x


def d2(ax, ay, bx, by):
    dx, dy = ax - bx, ay - by
    return dx * dx + dy * dy   # float64, two roundings and one, no contraction: what the kernel and the oracle compute


def points_on_cut(cx, cy, r, rng, n_dirs=4000, ulps=3):
    """points p near the circle of radius r around (cx, cy) with d2(p, c) equal to T(r) moved by -ulps..ulps ulps:
    random directions (p rounded to doubles, then y walked over its neighbouring doubles), (5, 12)-type exact points
    and the axes. Returns x, y, k (the ulp offset of d2 from T(r), or None for the axis / exact points)."""
    T = touch_threshold(r)
    targets = {float(_nextafter(T, k)): k for k in range(-ulps, ulps + 1)}
    xs, ys, ks = [], [], []
    phi = rng.uniform(0, 2 * np.pi, n_dirs)
    bx = cx + r * np.cos(phi)
    for x0, p in zip(bx, phi):
        dx = x0 - cx
        rest = T - dx * dx
        if rest <= 0:
            continue
        x0 = float(x0)
        y = _nextafter(cy + math.copysign(math.sqrt(rest), math.sin(p)), -40)
        for j in range(81):
            k = targets.get(d2(x0, y, cx, cy))
            if k is not None:
                xs.append(x0); ys.append(y); ks.append(k)
            y = math.nextafter(y, INF)
    for ex, ey in ((5.0, 12.0), (12.0, 5.0), (-5.0, 12.0), (5.0, -12.0)) if r == 13 else ():
        for j in range(-2, 3):
            xs.append(cx + ex); ys.append(float(_nextafter(cy + ey, j))); ks.append(None)
    for ax, ay in ((1, 0), (0, 1), (-1, 0), (0, -1)):
        for j in range(-3, 4):
            xs.append(float(_nextafter(cx + ax * r, j)) if ax else cx)
            ys.append(float(_nextafter(cy + ay * r, j)) if ay else cy)
            ks.append(None)
    return np.array(xs), np.array(ys), ks


def shell_ship_set(rng):
    """a live ship at integer points of the hexagon ring and a zero-velocity shell in slot 0 at distance ~13"""
    ships = [(455.0, 315.0), (300.0, 200.0), (410.0, 430.0), (250.0, 330.0)]
    parts = []
    for sx, sy in ships:
        x, y, _ = points_on_cut(sx, sy, 13, rng, n_dirs=1500)
        r = records(np.full(len(x), sx), np.full(len(x), sy))
        r["shell_mask"] = 1; r["shell_x"][:, 0] = x; r["shell_y"][:, 0] = y; r["shell_angle"][:, 0] = 30.0
        parts.append(r)
    return np.concatenate(parts)


def missile_fortress_set(rng):
    """a missile at heading 0 or 90 placed 20 back, so that after its move it stands at distance ~23 from the fortress;
    the fortress in the states that make a hit count (vulnerability up, reset, destruction) and dead"""
    x, y, _ = points_on_cut(FX, FY, 23, rng, n_dirs=6000)
    n = len(x)
    parts = []
    for ang in (0, 90):
        r = records(np.full(n, 455.0), np.full(n, 315.0))
        c, s = math.cos(ang * math.pi / 180), math.sin(ang * math.pi / 180)   # deg2rad (vector.cpp:34-36), libm
        r["missile_mask"] = 1
        r["missile_x"][:, 0] = x - (20.0 if ang == 0 else 0.0); r["missile_y"][:, 0] = y - (20.0 if ang == 90 else 0.0)
        r["missile_vx"][:, 0] = 20 * c; r["missile_vy"][:, 0] = 20 * s; r["missile_angle"][:, 0] = float(ang)
        case = np.arange(n) % 4
        r["fortress_vuln_timer"] = np.where(case == 0, 250, 100)
        r["vulnerability"] = np.where(case == 1, 11, np.where(case == 2, 4, 7))
        r["fortress_alive"] = (case != 3).astype(np.int32)
        r["stats"][:, 12] = 11
        parts.append(r)
    recs = np.concatenate(parts)
    # the move is exact: missile + 20 * (cos, sin) lands on the chosen point (the 1e-15 of 20 * cos 90 vanishes)
    mx = recs["missile_x"][:, 0] + recs["missile_vx"][:, 0]
    my = recs["missile_y"][:, 0] + recs["missile_vy"][:, 0]
    assert np.array_equal(mx, np.concatenate([x, x])) and np.array_equal(my, np.concatenate([y, y]))
    return recs


def hide_set(rng):
    """a zero-velocity shell at distance ~21 from the fortress (drawn only when further than 21); the ship far away"""
    x, y, _ = points_on_cut(FX, FY, 21, rng, n_dirs=3000)
    r = records(np.full(len(x), 255.0), np.full(len(x), 250.0))
    r["shell_mask"] = 1; r["shell_x"][:, 0] = x; r["shell_y"][:, 0] = y
    r["shell_angle"][:, 0] = rng.randint(0, 360, len(x)).astype(np.float64)
    return r


# ---------------------------------------------------------------------------------------------------------------------
# hexagon, shell launch and feature sets
# ---------------------------------------------------------------------------------------------------------------------
def hex_vertices(radius):   # hexagon.cpp:13-35, vertices floored
    x1, x2 = math.floor(355 - radius), math.floor(355 - radius * 0.5)
    x3, x4 = math.floor(355 + radius * 0.5), math.floor(355 + radius)
    y2, y3 = math.floor(315 - radius * math.sin(math.pi * 2 / 3)), math.floor(315 + radius * math.sin(math.pi * 2 / 3))
    return [(x1, 315), (x2, y2), (x3, y2), (x4, 315), (x3, y3), (x2, y3)]


def hex_edge_set():
    """points exactly on each edge of both hexagons (dyadic fractions of the integer edges: exact), and one ulp off in
    x and in y"""
    xs, ys = [], []
    for radius in (200, 40):
        v = hex_vertices(radius)
        for i in range(6):
            (ax, ay), (bx, by) = v[i], v[(i + 1) % 6]
            for t in np.arange(17) / 16.0:
                px, py = ax + t * (bx - ax), ay + t * (by - ay)
                for ox, oy in ((0, 0), (1, 0), (-1, 0), (0, 1), (0, -1)):
                    xs.append(float(_nextafter(px, ox))); ys.append(float(_nextafter(py, oy)))
    return np.array(xs), np.array(ys)


def shell_launch_set(rng):
    """ship positions from which the fortress fires this tick: octant directions, near-octant ones and random doubles
    of the hexagon ring. fortress_last_angle is the sector the oracle computes, so the lock timer (1000) fires."""
    xs, ys, octs = [], [], []
    for d in (45.0, 60.0, 80.0, 100.0, 120.0, 150.0):
        for cx, cy in ((1, 0), (1, 1), (0, 1), (-1, 1), (-1, 0), (-1, -1), (0, -1), (1, -1)):
            xs.append(FX + cx * d); ys.append(FY + cy * d); octs.append(True)
            for ex, ey in ((1, 0), (0, 1), (-1, 0), (0, -1)):
                xs.append(FX + cx * d + ex); ys.append(FY + cy * d + ey); octs.append(False)
                xs.append(float(_nextafter(FX + cx * d, ex))); ys.append(float(_nextafter(FY + cy * d, ey))); octs.append(False)
    phi, rad = rng.uniform(0, 2 * np.pi, 4000), rng.uniform(42, 170, 4000)
    xs += list(FX + rad * np.cos(phi)); ys += list(FY + rad * np.sin(phi)); octs += [False] * 4000
    r = records(np.array(xs), np.array(ys))
    r["fortress_timer"] = 1000
    pre, _ = oracle_step("youturn", r)
    r["fortress_last_angle"] = pre["fortress_angle"]
    after, out = oracle_step("youturn", r)
    # a sector decided inside the aiming band may differ from the reference's (test_aiming_decisions_against_the_oracle),
    # and then the lock timer restarts instead of firing: those positions are left to that test
    _, dist = ceil_exact(*sector_dir(r["ship_x"], r["ship_y"]), 10)
    octs = np.array(octs)
    keep = ((out[:, 3] & EV_FORTRESS_FIRED) != 0) & (octs | (dist > STEP_BAND))
    return r[keep], octs[keep]


def feature_set(rng):
    """crafted states at the feature thresholds; `integer` marks states with integer dx and dy"""
    rows = []   # (x, y, vx, vy, angle, vulnerability, vuln_timer, tick)
    for d in (60.0, 100.0, 140.0, 180.0):
        for cx, cy in ((1, 0), (1, 1), (0, 1), (-1, 1), (-1, 0), (-1, -1), (0, -1), (1, -1)):
            x, y = FX + cx * d, FY + cy * d
            o = math.degrees(math.atan2(cy, cx)) % 360
            for da in (-1, 0, 1):   # aim = o - angle + 180 == 3 + da
                rows.append((x, y, 1.0, 0.0, float(round(o + 180 - 3 - da) % 360), 5, 300, 100))
            for ey in (-1, 1):      # aim 3 +- ulp-scale
                rows.append((x, _nextafter(y, ey), 0.0, 1.0, float(round(o + 180 - 3) % 360), 5, 300, 100))
    for dx in (60.0, 100.0, 140.0, 180.0):   # ndist exactly -0.75 / -0.25 / 0.25 / 0.75 (Q11: dx only)
        for sx in (1, -1):
            for dy in (0.0, 7.0, -30.0, 55.0):
                rows.append((FX + sx * dx, FY + dy, 0.5, -0.5, 90.0, 3, 300, 100))
            for e in (-1, 1):
                rows.append((float(_nextafter(FX + sx * dx, e)), FY + 20.0, 0.5, -0.5, 90.0, 3, 300, 100))
    for (x, y) in ((455.0, 315.0), (255.0, 315.0), (355.0, 415.0), (355.0, 215.0), (425.0, 385.0), (285.0, 245.0)):
        for vx, vy in ((1.0, 0.0), (-1.0, 0.0), (0.0, 1.0), (0.0, -1.0), (1.0, 1.0), (-1.0, -1.0), (2.0, -0.0), (-2.0, -0.0)):
            rows.append((x, y, vx, vy, 0.0, 2, 300, 100))   # v - o at 0 / +-pi
    for v in (9, 10, 11, 12):
        for t in (249, 250):
            rows.append((400.0, 260.0, 0.3, 0.2, 45.0, v, t, 100))
    for _ in range(40):
        rows.append((float(rng.randint(160, 550)), float(rng.randint(150, 480)), float(rng.uniform(-3, 3)), float(rng.uniform(-3, 3)),
                     float(rng.randint(360)), int(rng.randint(13)), int(rng.choice([249, 250, 400])), 100))
    for (x, y) in ((455.0, 315.0), (400.0, 260.0)):
        rows.append((x, y, 0.7, 0.1, 30.0, 11, 100, 0))   # tick 0: vdir = aim = ndist = 0
    a = np.array(rows, dtype=object)
    r = records(a[:, 0].astype(np.float64), a[:, 1].astype(np.float64))
    r["ship_vx"], r["ship_vy"], r["ship_angle"] = a[:, 2].astype(np.float64), a[:, 3].astype(np.float64), a[:, 4].astype(np.float64)
    r["vulnerability"], r["fortress_vuln_timer"], r["tick"] = a[:, 5].astype(np.int32), a[:, 6].astype(np.int32), a[:, 7].astype(np.int32)
    r["time"] = r["tick"] * 34
    r["missile_mask"] = np.arange(len(r)) % 3 == 0
    r["fire_timer"], r["thrust_timer"], r["left_timer"], r["right_timer"] = 3, -40, 17, -5
    integer = (np.floor(r["ship_x"]) == r["ship_x"]) & (np.floor(r["ship_y"]) == r["ship_y"])
    return r, integer


# =====================================================================================================================
# CPU self-checks: the sets reach the decisions they are meant to test
# =====================================================================================================================
def test_threshold_restatement():
    """T(r) as sf_tables.cpp builds it: a cut of sqrt(x) <= r; T(21) is not 441"""
    for r in (13, 23, 21):
        T = touch_threshold(r)
        assert math.sqrt(T) <= r < math.sqrt(math.nextafter(T, INF))
    assert touch_threshold(13) == 169.0 and touch_threshold(23) == 529.0
    assert touch_threshold(21) == 441.00000000000006


@pytest.mark.parametrize("which", ["shell_ship", "missile_fortress", "hide"])
def test_collision_sets_straddle_the_cut(which):
    """Each set holds squared distances on both sides of T(r) that the oracle decides differently, and exactly T(r),
    which the oracle counts as touching (so `<` instead of `<=` changes a decision)."""
    rng = np.random.RandomState(7)
    recs = {"shell_ship": shell_ship_set, "missile_fortress": missile_fortress_set, "hide": hide_set}[which](rng)
    after, out = oracle_step("youturn", recs)
    if which == "shell_ship":
        r, cx, cy = 13, recs["ship_x"], recs["ship_y"]
        px, py = recs["shell_x"][:, 0], recs["shell_y"][:, 0]
        hit = (out[:, 3] & EV_SHELL_HIT_SHIP) != 0
    elif which == "missile_fortress":
        r, cx, cy = 23, FX, FY
        px = recs["missile_x"][:, 0] + recs["missile_vx"][:, 0]; py = recs["missile_y"][:, 0] + recs["missile_vy"][:, 0]
        hit = (out[:, 3] & EV_COL_MISSILE) != 0
    else:
        r, cx, cy = 21, FX, FY
        px, py = recs["shell_x"][:, 0], recs["shell_y"][:, 0]
        assert (after["shell_mask"] == 1).all()
        blank = after.copy(); blank["shell_mask"] = 0   # hidden: the frame is that of the state without the shell
        hit = np.array([np.array_equal(draw_native(to_record(after[i])), draw_native(to_record(blank[i]))) for i in range(len(recs))])
    T = touch_threshold(r)
    dd = d2(px, py, cx, cy)
    assert np.array_equal(hit, dd <= T), which    # the oracle's decision is the cut at T(r), both sides present
    assert (dd == T).any() and (dd == math.nextafter(T, INF)).any() and (dd == math.nextafter(T, 0)).any()
    assert hit[dd == T].all() and not hit[dd == math.nextafter(T, INF)].any()
    # at least 20 points on each of T - 1 ulp, T, T + 1 ulp
    for v in (math.nextafter(T, 0), T, math.nextafter(T, INF)):
        assert (dd == v).sum() >= 20, (which, v, int((dd == v).sum()))


def test_float32_cos_breaks_the_shell_bar():
    """A shell velocity from a float32 cos / sin, or a float32 deg2rad, misses SHELL_TOL at most angles."""
    rng = np.random.RandomState(3)
    a = rng.uniform(0, 360, 20000)
    rad = a * np.pi / 180
    v64 = 6 * np.cos(rad)
    v32 = 6 * np.cos(rad.astype(np.float32)).astype(np.float64)
    v32b = 6 * np.cos(rad.astype(np.float32).astype(np.float64))
    assert (np.abs(v32 - v64) > SHELL_TOL).mean() > 0.9
    assert (np.abs(v32b - v64) > SHELL_TOL).mean() > 0.9


def test_aiming_sets_straddle_every_multiple():
    """The aiming set has directions just below and just above every multiple of 1 degree (heading) and of 10 degrees
    (sector), and directions inside the 1e-12 band where the reference's rounded formula and the exact ceiling differ,
    among them y = 315 - 1 ulp at x = 100 (sector: reference 180, exact 190)."""
    x, y = near_ray_set()
    exp = aiming_expectations(x, y)
    after, _ = oracle_step("autoturn", records(x, y))
    for key, got in (("heading", after["ship_angle"]), ("sector", after["fortress_angle"])):
        ex, dist, octs, step = exp[key]
        dx, dy = heading_dir(x, y) if key == "heading" else sector_dir(x, y)
        th = np.degrees(np.arctan2(dy, dx)) % 360
        near = dist < 1e-8
        m = (step * np.round(th / step)).astype(np.int64) % 360
        below = near & (ex == m) & (dist > 0)
        above = near & (ex == (m + step) % 360)
        for k in range(0, 360, step):
            assert below[m == k].any() and above[m == k].any(), (key, k)
        alive = after["ship_alive"] == 1 if key == "sector" else np.ones(len(x), bool)
        differ = alive & (dist <= STEP_BAND) & ~octs & (got.astype(np.int64) != ex)
        assert differ.sum() > 0, key
    # The ship at x = 100 has left the big hexagon, so the step does not turn the fortress to it; the reference's
    # formula for the sector (game.cpp:197,206), evaluated here with the same libm, rounds the direction to 180.
    i = np.nonzero((x == 100.0) & (y == _nextafter(FY, -1)))[0][0]
    ang = math.atan2(y[i] - FY, x[i] - FX) / math.pi * 180 + 360
    assert exp["sector"][0][i] == 190 and math.ceil(ang / 10) * 10 == 180


# =====================================================================================================================
# GPU
# =====================================================================================================================
@pytest.mark.gpu
def test_aiming_decisions_against_the_oracle():
    sets = aiming_sets()
    report = {}
    for name, (x, y) in sets.items():
        recs = records(x, y)
        n = len(recs)
        dev = Device("autoturn", n)
        exp, eout = oracle_step("autoturn", recs)
        got, gout, _ = dev.step(recs)
        dev.close()
        gout[:, 3] &= 0xFFFFFFFF
        bad = mismatch(exp, got, skip=AIM_FIELDS) | (eout != gout).any(1)
        assert not bad.any(), (name, int(bad.sum()), first(bad))
        e = aiming_expectations(x, y)
        alive = exp["ship_alive"] == 1   # the fortress only turns to a live ship
        band_count, band_max = 0, 0.0
        for key, field, decided in (("heading", "ship_angle", np.ones(n, bool)), ("sector", "fortress_angle", alive)):
            ex, dist, octs, step = e[key]
            g, o = got[field].astype(np.int64), exp[field].astype(np.int64)
            outside = decided & (octs | (dist > STEP_BAND))
            wrong = outside & (g != o)
            assert not wrong.any(), (name, key, int(wrong.sum()), [(float(x[i]), float(y[i]), int(g[i]), int(o[i]), float(dist[i])) for i in first(wrong)])
            band = decided & ~octs & (dist <= STEP_BAND)
            wrong = band & (dist > ANGLE_SIGN_BAND) & (g != ex)
            assert not wrong.any(), (name, key, [(float(x[i]), float(y[i]), int(g[i]), int(ex[i]), float(dist[i])) for i in first(wrong)])
            # closer than ANGLE_SIGN_BAND: one of the two multiples next to the direction
            dx, dy = heading_dir(x, y) if key == "heading" else sector_dir(x, y)
            th = np.degrees(np.arctan2(dy, dx)) % 360
            m = (step * np.round(th / step)).astype(np.int64)
            wrong = band & (g != m % 360) & (g != (m + step) % 360)
            assert not wrong.any(), (name, key, first(wrong))
            if key == "sector":   # the rest of the fortress's state follows its angle
                same = decided & (g == o)
                assert np.array_equal(got["fortress_last_angle"][same], exp["fortress_last_angle"][same])
                assert np.array_equal(got["fortress_timer"][same], exp["fortress_timer"][same])
            dis = band & (g != o)
            band_count += int(dis.sum())
            if dis.any():
                band_max = max(band_max, float(dist[dis].max()))
            report[(name, key)] = (n, int(decided.sum()), int(band.sum()), int(dis.sum()), int((band & (g != ex)).sum()))
        report[name] = (n, band_count, band_max)
    print("\naiming: (set, decision) -> records, decided, in band, band disagreements with the oracle, with the exact ceiling")
    for k, v in report.items():
        print("  ", k, v)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["shell_ship", "missile_fortress"])
def test_collision_cuts(which):
    rng = np.random.RandomState(7)
    recs = {"shell_ship": shell_ship_set, "missile_fortress": missile_fortress_set}[which](rng)
    dev = Device("youturn", len(recs))
    exp, eout, got, gout, _ = compare("youturn", recs, dev, which)
    dev.close()
    bit = EV_SHELL_HIT_SHIP if which == "shell_ship" else EV_COL_MISSILE
    hits = int(((gout[:, 3] & bit) != 0).sum())
    assert 0 < hits < len(recs)
    print("\n%s: %d records, %d hits" % (which, len(recs), hits))


@pytest.mark.gpu
def test_hide_radius_in_frames():
    """A shell at distance ~21 from the fortress: the frame of the step and sf_render's frame of the same state equal the
    oracle's, bit for bit (the step decides visibility in the step kernel, the draw mode in sf_load_group)."""
    rng = np.random.RandomState(7)
    recs = hide_set(rng)
    dev = Device("youturn", len(recs))
    exp, eout, got, gout, frames = compare("youturn", recs, dev, "hide", native=True)
    rendered = dev.render_native()
    dev.close()
    shown = 0
    for i in range(len(recs)):
        want = draw_native(to_record(exp[i]))
        assert np.array_equal(frames[i], want), ("step frame", i, float(d2(recs[i]["shell_x"][0], recs[i]["shell_y"][0], FX, FY)))
        assert np.array_equal(rendered[i], want), ("sf_render frame", i, float(d2(recs[i]["shell_x"][0], recs[i]["shell_y"][0], FX, FY)))
        shown += int(d2(recs[i]["shell_x"][0], recs[i]["shell_y"][0], FX, FY) > touch_threshold(21))
    assert 0 < shown < len(recs)
    print("\nhide radius: %d records, %d shells drawn" % (len(recs), shown))


@pytest.mark.gpu
def test_hexagon_edges():
    x, y = hex_edge_set()
    recs = records(x, y)
    dev = Device("youturn", len(recs))
    exp, eout, got, gout, _ = compare("youturn", recs, dev, "hexagon edges")
    dev.close()
    big, small = (gout[:, 3] & EV_BIGHEX) != 0, (gout[:, 3] & EV_SMALLHEX) != 0
    assert big.any() and small.any() and (~big & ~small).any()
    on_edge, half = np.arange(len(recs)) % 5 == 0, len(recs) // 2   # the big hexagon's points first, then the small one's
    assert not big[:half][on_edge[:half]].any() and not small[:half].any()   # inclusive: on the edge is inside
    assert small[half:][on_edge[half:]].all() and not big[half:].any()
    print("\nhexagon edges: %d records, %d big-hexagon deaths, %d small-hexagon deaths" % (len(recs), int(big.sum()), int(small.sum())))


@pytest.mark.gpu
def test_shell_launch():
    rng = np.random.RandomState(9)
    recs, octs = shell_launch_set(rng)
    assert octs.sum() >= 40 and (~octs).sum() >= 1000
    dev = Device("youturn", len(recs))
    exp, eout, got, gout, _ = compare("youturn", recs, dev, "shell launch", shell_tol=1e-9)
    dev.close()
    assert ((gout[:, 3] & EV_FORTRESS_FIRED) != 0).all()
    da = np.abs(got["shell_angle"][:, 0] - exp["shell_angle"][:, 0])
    dv = np.maximum(np.abs(got["shell_vx"][:, 0] - exp["shell_vx"][:, 0]), np.abs(got["shell_vy"][:, 0] - exp["shell_vy"][:, 0]))
    print("\nshell launch: %d records (%d octants); max |d angle| %.3g deg, max |d v| %.3g" % (len(recs), int(octs.sum()), da.max(), dv.max()))
    assert (da[octs] == 0).all(), first(octs & (da != 0))
    assert da.max() <= SHELL_TOL and dv.max() <= SHELL_TOL, (da.max(), dv.max())


@pytest.mark.gpu
@pytest.mark.parametrize("gametype", ["youturn", "autoturn"])
def test_feature_rows_at_thresholds(gametype):
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    youturn = gametype == "youturn"
    recs, integer = feature_set(np.random.RandomState(4))
    n = len(recs)
    dev = Device(gametype, n)
    dev.set(recs)
    o = OracleEnv(gametype, 1)
    for kind in KINDS:
        nf = dev.env.L.sf_num_features(dev.env.h, _lib.OBS_TYPES[kind])
        f64 = torch.full((n, nf), float("nan"), dtype=torch.float64, device="cuda")
        f32 = torch.full((n, nf), float("nan"), dtype=torch.float32, device="cuda")
        _lib.check(dev.env.L.sf_features_f64(dev.env.h, _lib.OBS_TYPES[kind], vp(f64), None))
        _lib.check(dev.env.L.sf_features(dev.env.h, _lib.OBS_TYPES[kind], vp(f32), None))
        torch.cuda.synchronize()
        f64, f32 = f64.cpu().numpy(), f32.cpu().numpy()
        assert np.array_equal(f32.view(np.uint32), f64.astype(np.float32).view(np.uint32)), kind
        for i in range(n):
            o.set_state(to_record(recs[i]))
            exp = oracle_features(o, kind, youturn)
            if kind == "monitors":
                _, _, ndist, aim = o.extra()
                near = min(abs(aim - 3), abs(abs(ndist) - .75), abs(abs(ndist) - .25)) < 1e-9
                assert (near and not integer[i]) or np.array_equal(f64[i], exp), (kind, i, recs[i]["ship_x"], recs[i]["ship_y"], f64[i], exp)
            else:
                assert np.allclose(f64[i], exp, rtol=0, atol=1e-9), (kind, i, f64[i] - exp)
    dev.close()
