"""The renderer's geometry at its edges, bit for bit against the restatement (oracle/sf_draw_oracle.c).

Every GPU case is a set of crafted records: sf_set_state, then sf_render into 84x84 observations and into 92x90 native
frames, each compared with draw_obs / draw_native of the same record. Frames must be equal; a failure names the case,
the env, the number of differing pixels, the first differing pixel and the largest delta. The sets:

1. every integer angle of the ship, a missile and a shell (the shell also at 360.0, at the doubles next to every
   integer and just below 360), each centre at 24.8 phases 0, 1, 127, 128, 129, 255 in x and y;
2. rounding ties: centres at which the fp64 CTM puts a corner of the model exactly on a half unit of 24.8
   (nearbyint: half to even), and the doubles either side;
3. the view's borders: each kind at 8 angles swept across the 4 edges and the 4 corners of the 90x92 view in steps of
   1/32 px, from fully outside to fully inside, plus the centres at which a corner of a stroked quad lies on the edge;
4. the dead ship's 28x28 explosion box clipped by each edge and corner at y phases spread over 0..255, rendered twice
   (the second render takes the sprite path);
5. a missile and a shell crossing the ship, each other, the fortress (36 sectors and its explosion), the hexagons,
   the vulnerability bar and the score strip, windows overlapping partially;
6. the score's (int) truncation and its clamps to [0, 9999999], the bar at every vulnerability with the kill window
   on and off;
7. one crowded state and one dead-ship state copied into every env of a 4737-env handle.

Coordinates: native x = (x - 130) * 90/450, native y = (y - 80) * 92/460 (both scales are the double 0.2); the view is
x in [130, 580], y in [80, 540] and the world [0, 710] x [0, 626], so objects beyond the view are reachable states.

The tests without the gpu marker show from the oracle alone that the sets can catch a wrong kernel, and check the
bounds that the kernel's shortcuts rely on (sf_render.cuh) over every integer angle and every 24.8 phase."""
import ctypes as C
import functools
import math
import time

import numpy as np
import pytest

from gpu_helpers import frame_diff, torch_cuda
from oracle.oracle import Record, oracle_lib, record_dtype

DT = record_dtype()
SCALE = 90 / 450                    # == 92 / 460, the base CTM (sf_draw_oracle.c:92-98)
X0, Y0 = -130 * SCALE, -80 * SCALE  # -26.0, -16.0
HW = (3 * 0.5) * SCALE              # half the line width in device px (sf_draw_oracle.c:205)
NAT_W, NAT_H = 90, 92
OFF_VIEW = (680.0, 600.0)           # a live ship here is culled: native (110, 104)
FX, FY = 355.0, 315.0
BATCH = 4096
MODELS = {   # wireframe.cpp:8-70 as sf_draw_oracle.c:252-254: lines from.x, from.y, to.x, to.y
    "ship": ((-18, 0, 18, 0), (-18, 18, 0, 0), (0, 0, -18, -18)),
    "missile": ((0, 0, -25, 0), (0, 0, -5, 5), (0, 0, -5, -5)),
    "shell": ((-8, 0, 0, -6), (0, -6, 16, 0), (16, 0, 0, 6), (0, 6, -8, 0)),
}
KINDS = tuple(MODELS)
PHASES = (0, 1, 127, 128, 129, 255)
PHASE_PAIRS = [(PHASES[i], PHASES[(i + 2) % 6]) for i in range(6)] + [(0, 0), (128, 128), (255, 255), (127, 129)]
BORDER_ANGLES = (0, 37, 90, 128, 180, 219, 270, 301)
BORDERS = ("left", "right", "top", "bottom", "top-left", "top-right", "bottom-left", "bottom-right")
INF = float("inf")


# ---------------------------------------------------------------------------------------------------------------------
# M1 restated in numpy: the same double operations in the same order as base_ctm / mat_mul / xform
# (sf_draw_oracle.c:69-98) and sf_wire_xf / sf_xform_wire (csrc/sf_geom.h:63-79). numpy does not contract a * b + c.
# ---------------------------------------------------------------------------------------------------------------------
def ctm(angle):
    """xx, yx, xy, yy of translate(pos) then rotate(deg2rad((int)angle)) after the base CTM; angle an int"""
    rad = angle * math.pi / 180   # (double)angle * M_PI / 180, host libm like the oracle and the device table
    c, s = math.cos(rad), math.sin(rad)
    return c * SCALE, s * SCALE, -s * SCALE, c * SCALE


def origin(px, py):
    """x0, y0 of the CTM after cairo_translate(px, py): px * 0.2 + py * 0 + (-26) == fl(fl(px * 0.2) - 26)"""
    return np.asarray(px, np.float64) * SCALE + X0, np.asarray(py, np.float64) * SCALE + Y0


def to_fixed(v):
    return np.rint(np.asarray(v, np.float64) * 256.0).astype(np.int64)   # nearbyint: half to even


def xform(m, x0, y0, mx, my):
    xx, yx, xy, yy = m
    return to_fixed((xx * mx + xy * my) + x0), to_fixed((yx * mx + yy * my) + y0)


def stroke_quads(kind, angle, px, py):
    """[(4 corners x, 4 corners y)] per line of the model: the stroked segments (slope_of / stroke_segment,
    sf_draw_oracle.c:193-213), int64 arrays of 24.8 device coordinates, each [4, n]"""
    m = ctm(int(angle))
    x0, y0 = origin(px, py)
    out = []
    for (ax, ay, bx, by) in MODELS[kind]:
        pax, pay = xform(m, x0, y0, ax, ay)
        pbx, pby = xform(m, x0, y0, bx, by)
        dx, dy = (pbx - pax) / 256.0, (pby - pay) / 256.0
        with np.errstate(invalid="ignore", divide="ignore"):
            mag = np.sqrt(dx * dx + dy * dy)
            ux = np.where(dy == 0, np.sign(dx), np.where(dx == 0, 0.0, dx / mag))
            uy = np.where(dx == 0, np.sign(dy), np.where(dy == 0, 0.0, dy / mag))
        assert not ((dx == 0) & (dy == 0)).any()   # no model line is shorter than one pixel
        ox, oy = to_fixed(-uy * HW), to_fixed(ux * HW)
        out.append((np.stack([pax + ox, pbx + ox, pbx - ox, pax - ox]), np.stack([pay + oy, pby + oy, pby - oy, pay - oy])))
    return out


def grid_y(y):
    return (y * 15 + 128) >> 8   # sf_geom.h:109, round half up to 1/15 px


def world(c, axis):
    """the user coordinate whose centre lands on 24.8 device coordinate c (the inverse of the base CTM; exact doubles)"""
    return 5.0 * (np.asarray(c, np.float64) / 256.0 + (26.0 if axis == "x" else 16.0))


def _next(v, k):
    """doubles moved by k ulps"""
    v = np.asarray(v, np.float64).copy()
    for _ in range(abs(k)):
        v = np.nextafter(v, INF if k > 0 else -INF)
    return v


# ---------------------------------------------------------------------------------------------------------------------
# records
# ---------------------------------------------------------------------------------------------------------------------
def blank(n):
    """live fortress at angle 0, live ship off the view, nothing else; tick 1000"""
    r = np.zeros(n, DT)
    r["ship_x"], r["ship_y"] = OFF_VIEW
    r["ship_alive"] = 1; r["fortress_alive"] = 1
    r["ship_death_timer"] = 5000; r["fortress_death_timer"] = 5000; r["fortress_vuln_timer"] = 250
    r["tick"] = 1000; r["time"] = 34000; r["rng_seed"] = 1
    return r


def with_stroke(kind, angle, px, py):
    """one stroke of `kind` at (px, py), angle (per record or one for all); everything else as blank()"""
    px, py = np.asarray(px, np.float64), np.asarray(py, np.float64)
    r = blank(len(px))
    if kind == "ship":
        r["ship_x"], r["ship_y"], r["ship_angle"] = px, py, angle
    elif kind == "missile":
        r["missile_mask"] = 1
        r["missile_x"][:, 0], r["missile_y"][:, 0], r["missile_angle"][:, 0] = px, py, angle
    else:
        r["shell_mask"] = 1
        r["shell_x"][:, 0], r["shell_y"][:, 0], r["shell_angle"][:, 0] = px, py, angle
    return r


def interior(rng, n, margin=12, away_from_fortress=False):
    """native pixel positions (cx, cy) whose strokes lie inside the view; optionally further than 40 units (8 px) from
    the fortress, so that a shell is drawn"""
    cx, cy = rng.randint(margin, NAT_W - margin, n), rng.randint(margin, NAT_H - margin, n)
    if away_from_fortress:
        near = np.hypot(cx - 45, cy - 47) < 9
        while near.any():
            cx[near], cy[near] = rng.randint(margin, NAT_W - margin, near.sum()), rng.randint(margin, NAT_H - margin, near.sum())
            near = np.hypot(cx - 45, cy - 47) < 9
    return cx, cy


def shell_angles():
    """every integer 0..360 and the doubles either side of each (among them the double just below 360)"""
    k = np.arange(361, dtype=np.float64)
    return np.unique(np.concatenate([k, _next(k, 1), _next(k, -1)]))


# ---- set 1: every angle x sub-pixel phase ---------------------------------------------------------------------------
def angle_set():
    """{kind: records}: every angle at every phase pair of PHASE_PAIRS, one stroke per frame"""
    rng = np.random.RandomState(1)
    out = {}
    for kind in KINDS:
        angles = shell_angles() if kind == "shell" else np.arange(360, dtype=np.float64)
        parts = []
        for phx, phy in PHASE_PAIRS:
            cx, cy = interior(rng, len(angles), away_from_fortress=kind == "shell")
            parts.append(with_stroke(kind, angles, world(cx * 256 + phx, "x"), world(cy * 256 + phy, "y")))
        out[kind] = np.concatenate(parts)
    return out


# ---- set 2: rounding ties ------------------------------------------------------------------------------------------
def model_points(kind):
    return sorted({(l[0], l[1]) for l in MODELS[kind]} | {(l[2], l[3]) for l in MODELS[kind]})


def find_ties(angles, mx, my, axis, base):
    """For each angle: a world coordinate (along `axis`, others from `base`) at which the model point (mx, my) lands
    exactly on a half unit of 24.8, or NaN where none was found next to the base."""
    base = np.asarray(base, np.float64)
    sh = X0 if axis == "x" else Y0
    A = np.array([(ctm(a)[0] * mx + ctm(a)[2] * my) if axis == "x" else (ctm(a)[1] * mx + ctm(a)[3] * my) for a in angles])
    found = np.full(len(angles), np.nan)
    o0 = base * SCALE + sh
    for k in range(12):   # half units above the base's, until one is reachable by the doubles of px
        T = (np.floor((A + o0) * 256.0) + k + 0.5) / 256.0
        p0 = (T - A - sh) / SCALE
        for j in range(-6, 7):
            p = _next(p0, j)
            hit = np.isnan(found) & (((p * SCALE + sh) + A) == T) & np.isfinite(p)
            found[hit] = p[hit]
    return found


def tie_set():
    """{kind: (records, role)}: role 0 at a tie, -1 / +1 the double below / above it; ties of every model point along
    x and along y, every integer angle (the shell also at 360)"""
    rng = np.random.RandomState(2)
    out = {}
    for kind in KINDS:
        angles = np.arange(361 if kind == "shell" else 360)
        recs, roles = [], []
        for (mx, my) in model_points(kind):
            for axis in ("x", "y"):
                cx, cy = interior(rng, len(angles), away_from_fortress=kind == "shell")
                bx, by = world(cx * 256 + rng.randint(256, size=len(angles)), "x"), world(cy * 256 + rng.randint(256, size=len(angles)), "y")
                t = find_ties(angles, mx, my, axis, bx if axis == "x" else by)
                ok = ~np.isnan(t)
                for role in (-1, 0, 1):
                    p = _next(t[ok], role)
                    recs.append(with_stroke(kind, angles[ok].astype(np.float64), p if axis == "x" else bx[ok], by[ok] if axis == "x" else p))
                    roles.append(np.full(ok.sum(), role))
        out[kind] = (np.concatenate(recs), np.concatenate(roles))
    return out


# ---- set 3: the view's borders -------------------------------------------------------------------------------------
EDGE = {"left": (0, None), "right": (NAT_W * 256, None), "top": (None, 0), "bottom": (None, NAT_H * 256)}
SWEEP = np.arange(-7 * 32, 7 * 32 + 1) * 8   # -7 px .. +7 px in 1/32 px (24.8 units), outside to inside


def border_centres(border, along):
    """24.8 centres (cx, cy) of the sweep across `border` (inward is +); `along`: the other coordinate of an edge"""
    parts = border.split("-")
    cx = np.full(len(SWEEP), along[0]); cy = np.full(len(SWEEP), along[1])
    for p in parts:
        if p == "left": cx = SWEEP.copy()
        if p == "right": cx = NAT_W * 256 - SWEEP
        if p == "top": cy = SWEEP.copy()
        if p == "bottom": cy = NAT_H * 256 - SWEEP
    return cx, cy


def corner_on_edge(kind, angle, border, along):
    """24.8 centres at which a corner of a stroked quad lies exactly on the edge(s) of `border`"""
    cxs, cys = [], []
    for p in border.split("-"):
        ex, ey = EDGE[p]
        axis = "x" if ex is not None else "y"
        e = ex if ex is not None else ey
        cx0, cy0 = (np.array([e]), np.array([along[1]])) if axis == "x" else (np.array([along[0]]), np.array([e]))
        quads = stroke_quads(kind, angle, world(cx0, "x"), world(cy0, "y"))
        for qx, qy in quads:
            for k in range(4):
                d = int((qx if axis == "x" else qy)[k, 0]) - e   # the corner relative to the centre on the edge
                for shift in (-2, -1, 0, 1, 2):                  # the corner moves with the centre up to rounding
                    cx, cy = (cx0 - d + shift, cy0) if axis == "x" else (cx0, cy0 - d + shift)
                    qq = stroke_quads(kind, angle, world(cx, "x"), world(cy, "y"))
                    c = [int((q[0] if axis == "x" else q[1])[k, 0]) for q in qq]
                    if e in c:
                        cxs.append(int(cx[0])); cys.append(int(cy[0]))
    return np.array(cxs, np.int64), np.array(cys, np.int64)


def border_set():
    """{kind: (records, sweep id, step)}: step -1 marks the corner-on-edge centres"""
    out = {}
    for kind in KINDS:
        recs, sid, steps = [], [], []
        for b, border in enumerate(BORDERS):
            along = (45 * 256 + 77, 30 * 256 + 201) if kind == "shell" else (45 * 256 + 77, 46 * 256 + 201)
            for a, angle in enumerate(BORDER_ANGLES):
                cx, cy = border_centres(border, along)
                ex, ey = corner_on_edge(kind, angle, border, along)
                recs.append(with_stroke(kind, float(angle), world(np.concatenate([cx, ex]), "x"), world(np.concatenate([cy, ey]), "y")))
                sid.append(np.full(len(cx) + len(ex), b * 8 + a))
                steps.append(np.concatenate([np.arange(len(cx)), np.full(len(ex), -1)]))
        out[kind] = (np.concatenate(recs), np.concatenate(sid), np.concatenate(steps))
    return out


# ---- set 4: the explosion at the borders ---------------------------------------------------------------------------
def explosion_border_set():
    """a dead ship whose 28x28 box (centre pixel - 13 .. + 14) is clipped by each edge and corner, at 8 y phases"""
    rows = []
    for border in BORDERS:
        for off in range(-14, 15):   # centre pixel from 14 px outside to 14 px inside
            for k, phy in enumerate((0, 37, 73, 110, 146, 183, 219, 255)):
                phx = (off * 37 + k * 91) % 256
                cx, cy = 45 * 256 + phx, 46 * 256 + phy
                for p in border.split("-"):
                    if p == "left": cx = off * 256 + phx
                    if p == "right": cx = (NAT_W - 1 - off) * 256 + phx
                    if p == "top": cy = off * 256 + phy
                    if p == "bottom": cy = (NAT_H - 1 - off) * 256 + phy
                rows.append((cx, cy))
    c = np.array(rows)
    r = blank(len(c))
    r["ship_x"], r["ship_y"] = world(c[:, 0], "x"), world(c[:, 1], "y")
    r["ship_alive"] = 0; r["ship_death_timer"] = 10
    r["ship_angle"] = np.arange(len(c)) % 360
    r["points"] = np.where(np.arange(len(c)) % 3 == 0, 4321.0, 0.0)
    r["vulnerability"] = np.arange(len(c)) % 13
    return r


# ---- set 5: overlaps -----------------------------------------------------------------------------------------------
def hexagon_points(radius):   # hexagon.cpp:13-35, vertices floored (sf_draw_oracle.c:271-273)
    x1, x2, x3, x4 = math.floor(355 - radius), math.floor(355 - radius * 0.5), math.floor(355 + radius * 0.5), math.floor(355 + radius)
    y2, y3 = math.floor(315 - radius * math.sin(math.pi * 2 / 3)), math.floor(315 + radius * math.sin(math.pi * 2 / 3))
    return [(x1, 315), (x2, y2), (x3, y2), (x4, 315), (x3, y3), (x2, y3)]


def overlap_set():
    """{zone: records}: a missile (slot 3) and a shell (slot 1) near each other and near the zone's object"""
    rng = np.random.RandomState(5)
    zones = {}

    def place(n, cx, cy, spread, ship=True):
        r = blank(n)
        if ship:
            r["ship_x"], r["ship_y"] = cx + rng.uniform(-spread, spread, n), cy + rng.uniform(-spread, spread, n)
            r["ship_angle"] = rng.randint(360, size=n)
        r["missile_mask"] = 1 << 3; r["shell_mask"] = 1 << 1
        r["missile_x"][:, 3], r["missile_y"][:, 3] = cx + rng.uniform(-spread, spread, n), cy + rng.uniform(-spread, spread, n)
        r["missile_angle"][:, 3] = rng.randint(360, size=n)
        r["shell_x"][:, 1], r["shell_y"][:, 1] = r["missile_x"][:, 3] + rng.uniform(-25, 25, n), r["missile_y"][:, 3] + rng.uniform(-25, 25, n)
        r["shell_angle"][:, 1] = rng.uniform(0, 360, n)
        r["points"] = rng.choice([0.0, 7.0, 123456.0], n)
        r["vulnerability"] = rng.randint(15, size=n); r["fortress_vuln_timer"] = rng.choice([100, 249, 250], n)
        return r

    zones["ship"] = place(600, rng.uniform(200, 510, 600), rng.uniform(150, 470, 600), 20)
    # the fortress: every sector and its explosion; shells inside the hide radius are not drawn
    r = place(37 * 24, FX, FY, 45)
    r["fortress_angle"] = 10.0 * (np.arange(len(r)) % 37 % 36); r["fortress_last_angle"] = r["fortress_angle"]
    r["fortress_alive"] = (np.arange(len(r)) % 37 != 36).astype(np.int32)
    zones["fortress"] = r
    pts = np.array([p for rad in (200, 40) for p in hexagon_points(rad)], np.float64)
    nxt = np.roll(pts.reshape(2, 6, 2), -1, axis=1).reshape(12, 2)
    t = rng.uniform(0, 1, 720)
    k = rng.randint(12, size=720)
    e = pts[k] + t[:, None] * (nxt[k] - pts[k])
    zones["hexagons"] = place(720, e[:, 0], e[:, 1], 12)
    zones["bar"] = place(400, rng.uniform(245, 465, 400), rng.uniform(515, 540, 400), 12)
    r = place(400, rng.uniform(270, 440, 400), rng.uniform(80, 112, 400), 12)
    r["points"] = rng.choice([1.0, 4444444.0, 9999999.0, 88.5], 400)
    zones["score"] = r
    return zones


# ---- set 6: score and bar ------------------------------------------------------------------------------------------
def score_values():
    """float32 points: 0, d * 10^k, the clamp at 9999999 and above it up to the largest float below 2^31, negative and
    fractional values. (int) of a float outside the int range is undefined in C (and the reference's score is a float
    that never gets there), so that range is not part of the set."""
    v = [0.0] + [d * 10.0 ** k for k in range(7) for d in range(1, 10)]
    v += [9999999.0, 9999999.99, 1e7, 1e7 + 1, 12345678.0, 99999999.0, 1e9, 2147483520.0]   # float32(2^31 - 65) = 2147483520
    v += [-0.5, -0.99, -1.0, -7.0, -123456.0, -2147483648.0, 0.5, 0.99, 1.5, 9.99, 99.5, 1234567.5, -0.0]
    return np.array(v, np.float32)


def score_bar_set():
    """every score value with every bar state (vulnerability 0..14, fortress vulnerability timer 249 / 250)"""
    pts = score_values()
    bars = [(v, t) for v in range(15) for t in (249, 250)]
    r = blank(len(pts) * len(bars))
    r["points"] = np.repeat(pts, len(bars))
    r["vulnerability"] = np.tile([b[0] for b in bars], len(pts))
    r["fortress_vuln_timer"] = np.tile([b[1] for b in bars], len(pts))
    return r


# ---- set 7: position independence ----------------------------------------------------------------------------------
def crowded_states():
    """(crowded: live ship, 20 missiles, 3 shells, a score, a full bar in the kill window; dead ship)"""
    rng = np.random.RandomState(7)
    a = blank(1)
    a["ship_x"], a["ship_y"], a["ship_angle"] = 300.0, 250.0, 33.0
    a["missile_mask"] = (1 << 20) - 1
    a["missile_x"][0], a["missile_y"][0] = rng.uniform(200, 520, 20), rng.uniform(150, 480, 20)
    a["missile_angle"][0] = rng.randint(360, size=20)
    a["shell_mask"] = 0b111
    a["shell_x"][0, :3], a["shell_y"][0, :3] = [250.0, 420.0, 300.5], [400.0, 200.25, 260.0]
    a["shell_angle"][0, :3] = [12.5, 360.0, 199.99]
    a["points"], a["vulnerability"], a["fortress_vuln_timer"] = 1234.5, 12, 100
    a["fortress_angle"] = 70.0
    b = blank(1)
    b["ship_x"], b["ship_y"], b["ship_alive"], b["ship_death_timer"] = 402.3, 205.7, 0, 12
    b["missile_mask"] = 0b101
    b["missile_x"][0, [0, 2]], b["missile_y"][0, [0, 2]] = [395.0, 410.0], [200.0, 215.0]
    b["missile_angle"][0, [0, 2]] = [45.0, 300.0]
    b["points"], b["vulnerability"] = 98765.0, 7
    b["fortress_alive"] = 0
    return a, b


# ---------------------------------------------------------------------------------------------------------------------
# the oracle's frames
# ---------------------------------------------------------------------------------------------------------------------
def oracle_frames(recs, native):
    """draw_native (92x90) or draw_obs (84x84) of every record"""
    L = oracle_lib()
    recs = np.ascontiguousarray(recs, DT)
    f = L.sfo_draw_native if native else L.sfo_draw_obs
    out = np.zeros((len(recs),) + ((NAT_H, NAT_W) if native else (84, 84)), np.uint8)
    base, step, ob, ostep = recs.ctypes.data, DT.itemsize, out.ctypes.data, out[0].nbytes if len(out) else 0
    P = C.POINTER(Record)
    for i in range(len(recs)):
        f(C.cast(base + i * step, P), C.c_void_p(ob + i * ostep))
    return out


def differ(a, b):
    """per frame: True where the two stacks of frames differ"""
    return (a != b).reshape(len(a), -1).any(1)


# =====================================================================================================================
# CPU: the sets reach what they are meant to test
# =====================================================================================================================
def test_placements_land_where_intended():
    """the centres of the phase, border and explosion sets are the intended 24.8 device points"""
    for kind, r in angle_set().items():
        x, y = (r["ship_x"], r["ship_y"]) if kind == "ship" else ((r["missile_x"][:, 0], r["missile_y"][:, 0]) if kind == "missile" else (r["shell_x"][:, 0], r["shell_y"][:, 0]))
        fx, fy = to_fixed(origin(x, y)[0]), to_fixed(origin(x, y)[1])
        n = len(r) // len(PHASE_PAIRS)
        for k, (phx, phy) in enumerate(PHASE_PAIRS):
            assert ((fx[k * n:(k + 1) * n] & 255) == phx).all() and ((fy[k * n:(k + 1) * n] & 255) == phy).all(), (kind, phx, phy)
    for cx in (SWEEP, NAT_W * 256 - SWEEP):
        assert np.array_equal(to_fixed(origin(world(cx, "x"), 0.0)[0]), cx)
    r = explosion_border_set()
    phy = to_fixed(origin(r["ship_x"], r["ship_y"])[1]) & 255
    assert set(phy.tolist()) == {0, 37, 73, 110, 146, 183, 219, 255}


def test_every_angle_changes_the_frame():
    """Neighbouring integer angles give different frames (so an angle off by one, or a wrong cos / sin entry, shows),
    and the shell at 360 (and at the doubles just above it) gives the frame of 0, as (int) and a rotation by 360 degrees
    do in the restatement: the device aliases 360 to 0 (sf_render.cuh, sf_gather_strokes)."""
    for kind in KINDS:
        for phx, phy in PHASE_PAIRS:
            px, py = world(np.full(360, 40 * 256 + phx), "x"), world(np.full(360, 30 * 256 + phy), "y")
            f = oracle_frames(with_stroke(kind, np.arange(360, dtype=np.float64), px, py), native=True)
            assert differ(f, np.roll(f, -1, axis=0)).all(), (kind, phx, phy)
    r = angle_set()["shell"]
    at360 = r["shell_angle"][:, 0] >= 360
    assert at360.sum() == 2 * len(PHASE_PAIRS)   # 360.0 and the double above it, at every phase pair
    same = r[at360].copy()
    same["shell_angle"][:, 0] = 0.0
    assert np.array_equal(oracle_frames(r[at360], native=True), oracle_frames(same, native=True))
    # and on the tie set, where a rotation by 360 degrees (sin = -2.4e-16) could move a point off its tie
    r, role = tie_set()["shell"]
    at360 = r["shell_angle"][:, 0] == 360
    same = r[at360].copy()
    same["shell_angle"][:, 0] = 0.0
    assert at360.sum() > 0 and np.array_equal(oracle_frames(r[at360], native=True), oracle_frames(same, native=True))


def test_ties_are_ties_and_decide_frames():
    """Each tie record puts its model point exactly on a half unit; its neighbours one ulp away do not. For a useful
    share of the ties that nearbyint rounds down (to even), the frame differs from the frame one ulp above: a kernel
    that rounded half up would draw the latter."""
    for kind, (r, role) in tie_set().items():
        assert (role == 0).sum() >= 360 * len(model_points(kind)), (kind, int((role == 0).sum()))   # about one per point and axis
        nat = oracle_frames(r, native=True)
        n = (role == 0).sum()
        lo, tie, hi = r[role == -1], r[role == 0], r[role == 1]
        assert len(lo) == len(tie) == len(hi)
        f_lo, f_tie, f_hi = nat[role == -1], nat[role == 0], nat[role == 1]
        ch_hi = differ(f_tie, f_hi)
        ch_lo = differ(f_tie, f_lo)
        print("\n%s: %d ties; frame at the tie != one ulp above: %d, != one ulp below: %d" % (kind, n, ch_hi.sum(), ch_lo.sum()))
        assert ch_hi.sum() >= 0.1 * n and ch_lo.sum() >= 0.1 * n, kind


@pytest.mark.parametrize("kind", KINDS)
def test_border_steps_change_the_frame(kind):
    """7 px outside the view a stroke is not drawn; from the first step that draws it, most 1/32 px steps change the
    frame (at least half of every sweep, 95 % over all sweeps: a step that moves no edge over a 1/256 px boundary that
    matters can leave every pixel as it was)."""
    r, sid, step = border_set()[kind]
    nat = oracle_frames(r, native=True)
    empty = oracle_frames(blank(1), native=True)[0]
    frac = []
    for s in np.unique(sid):
        m = (sid == s) & (step >= 0)
        f = nat[m]
        assert np.array_equal(f[0], empty), (kind, s)                   # 7 px outside: nothing
        drawn = differ(f, np.broadcast_to(empty, f.shape))
        first = np.nonzero(drawn)[0][0]
        ch = differ(f[first:-1], f[first + 1:])
        frac.append(ch.mean())
        assert ch.mean() >= 0.5, (kind, s, float(ch.mean()))
    assert np.mean(frac) >= 0.95, (kind, float(np.mean(frac)))
    print("\n%s: border sweeps, share of steps that change the frame: min %.3f, mean %.3f" % (kind, min(frac), np.mean(frac)))


# ---- the bounds the kernel's shortcuts rely on ----------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def stroke_extents(kind):
    """over every integer angle and every pair of 24.8 phases (x, y) of the centre: the largest extent in grid rows
    and in 24.8 x of a stroke, and the largest region in pixels (w, h) that sf_open_regions opens for it"""
    ph = np.arange(256)
    PX, PY = np.meshgrid(ph, ph, indexing="ij")
    cx, cy = world((40 * 256 + PX).ravel(), "x"), world((40 * 256 + PY).ravel(), "y")
    worst = dict(rows=0, x=0, w=0, h=0, cells=0)
    for angle in range(360):
        q = stroke_quads(kind, angle, cx, cy)
        xs = np.concatenate([a for a, _ in q]); ys = np.concatenate([b for _, b in q])
        xmin, xmax = xs.min(0), xs.max(0)
        gmin, gmax = grid_y(ys).min(0), grid_y(ys).max(0)
        w = ((xmax - 1) >> 8) - (xmin >> 8) + 1
        h = np.floor_divide(gmax - 1, 15) - np.floor_divide(gmin, 15) + 1   # sf_row_of
        worst["rows"] = max(worst["rows"], int((gmax - gmin).max())); worst["x"] = max(worst["x"], int((xmax - xmin).max()))
        worst["w"] = max(worst["w"], int(w.max())); worst["h"] = max(worst["h"], int(h.max())); worst["cells"] = max(worst["cells"], int((w * h).max()))
    return worst


def area_tab(ssize, dsize):
    """(dst, src) pairs of cv2 INTER_AREA (sf_draw_oracle.c:446-462, weights left out)"""
    scale = ssize / dsize
    tab = []
    for dx in range(dsize):
        f1 = dx * scale; f2 = f1 + scale
        cell = min(scale, ssize - f1)
        s1, s2 = math.ceil(f1), math.floor(f2)
        s2 = min(s2, ssize - 1); s1 = min(s1, s2)
        if s1 - f1 > 1e-3: tab.append((dx, s1 - 1))
        tab += [(dx, s) for s in range(s1, s2)]
        if f2 - s2 > 1e-3: tab.append((dx, s2))
    return tab


def window_size(x0, x1, ssize):
    """the native footprint closure of native columns x0..x1 (sf_phase_window: col_out0 / col_out1, then the taps of
    the first and last output column)"""
    tab = area_tab(ssize, 84)
    j0 = min(d for d, s in tab if s == x0); j1 = max(d for d, s in tab if s == x1)
    return max(s for d, s in tab if d == j1) - min(s for d, s in tab if d == j0) + 1


def test_stroke_bounds_fit_the_pools_and_windows():
    """SF_CELLS_SHIP / _MISSILE / _SHELL (sf_render.cuh:59-63, the round scan admits envs by this worst-case need),
    windows of at most 30 x 32 native pixels (sf_render.cuh:39-45; the explosion box is 28 x 28 and the score strip
    27 x 5), over every angle and phase"""
    cells = {"ship": 144, "missile": 49, "shell": 49}
    worst = {}
    for kind in KINDS:
        e = stroke_extents(kind)
        worst[kind] = e
        assert e["cells"] <= cells[kind], (kind, e)
        # the window of a region of the largest size, at every position of the view
        ww = max(window_size(x, min(x + e["w"] - 1, NAT_W - 1), NAT_W) for x in range(NAT_W))
        wh = max(window_size(y, min(y + e["h"] - 1, NAT_H - 1), NAT_H) for y in range(NAT_H))
        assert ww <= 30 and wh <= 32, (kind, ww, wh)
    ww = max(window_size(x, min(x + 27, NAT_W - 1), NAT_W) for x in range(NAT_W))
    wh = max(window_size(y, min(y + 27, NAT_H - 1), NAT_H) for y in range(NAT_H))
    assert ww <= 30 and wh <= 32, ("explosion box", ww, wh)
    assert window_size(32, 58, NAT_W) <= 30 and window_size(1, 5, NAT_H) <= 32
    # "at most 44 user units (8.8 px) + the line width in any direction" (sf_render.cuh:59-60)
    assert worst["ship"]["x"] <= (8.8 + 2 * HW) * 256 + 2 and worst["ship"]["rows"] <= (8.8 + 2 * HW) * 15 + 2
    print("\nstroke extents over every angle and phase:", worst)


def test_scan_converter_arithmetic_is_exact_where_reached():
    """Exhaustively over the reachable range: the magic reciprocal of sf_make_edge / sf_edge_x (sf_render.cuh:330-345,
    M = floor((2^32 - 1) / dy) + 1 as sf_tables.cpp builds it: umulhi(n, M) == n // dy for every edge height dy and
    every n = rows * |dx| of a stroke edge), sf_div15 (sf_render.cuh:240: the sub-row of a region over 15) and the
    k / 7 of the cached sprite rows (sf_render.cuh:613). sf_div_small (sf_render.cuh:237) has no caller, so it has no
    reachable range to check."""
    rows = max(stroke_extents(k)["rows"] for k in KINDS)
    xext = max(stroke_extents(k)["x"] for k in KINDS)
    assert rows < 512   # SF_MAGIC_N: every edge has its own reciprocal
    for dy in range(2, rows + 1):
        M = np.uint64(0xFFFFFFFF // dy + 1)
        n = np.arange(dy * xext + 1, dtype=np.uint64)
        assert int(dy * xext) * int(M) < 2 ** 64
        assert np.array_equal((n * M) >> np.uint64(32), n // np.uint64(dy)), dy
    # sf_div15(d) = (d * 2185) >> 15 for d = sub-row - region top, d < 15 * (the tallest region)
    h = max(stroke_extents(k)["h"] for k in KINDS)
    d = np.arange(15 * h)
    assert np.array_equal((d * 2185) >> 15, d // 15)
    d = np.arange(4694)
    assert np.array_equal((d * 2185) >> 15, d // 15) and (4694 * 2185) >> 15 != 4694 // 15
    k = np.arange(196)   # 32-bit words of the 28 rows of a sprite: 7 per row
    assert np.array_equal((k * 9363) >> 16, k // 7)


# =====================================================================================================================
# GPU
# =====================================================================================================================
class Renderer:
    """one handle for the crafted states of a case; sf_render of up to `n` records at a time"""

    def __init__(self, gametype, n=BATCH):
        torch_cuda()
        from spacefortress_b200 import SFVecEnv, _lib
        self._lib = _lib
        self.env = SFVecEnv(gametype, num_envs=n, device=0, render=False)
        self.n = n

    def frames(self, recs, twice=False):
        """(obs, native) of `recs`; twice: render the observations again and require the same frames (the second
        render of a dead ship takes the sprite and resampled-box caches)"""
        obs, nat = [], []
        for b in range(0, len(recs), self.n):
            part = np.ascontiguousarray(recs[b:b + self.n])
            self._lib.check(self.env.L.sf_set_state(self.env.h, 0, len(part), C.c_void_p(part.ctypes.data)))
            o = self.env.render_frames(native=False)[:len(part)]
            nat.append(self.env.render_frames(native=True)[:len(part)])
            if twice:
                again = self.env.render_frames(native=False)[:len(part)]
                bad = differ(o, again)
                assert not bad.any(), ("second render", b + int(np.nonzero(bad)[0][0]))
            obs.append(o)
        return np.concatenate(obs), np.concatenate(nat)

    def close(self):
        self.env.close()


def assert_frames_equal(label, recs, got_obs, got_nat):
    """every frame equal to the oracle's; on a failure: label, env, differing pixels, first pixel, largest delta"""
    for native, got in ((False, got_obs), (True, got_nat)):
        exp = oracle_frames(recs, native)
        bad = np.nonzero(differ(exp, got))[0]
        assert len(bad) == 0, (label, "native" if native else "obs", "%d of %d frames differ" % (len(bad), len(recs)),
                               [(int(i),) + frame_diff(exp[i], got[i]) for i in bad[:5]])
    return 2 * len(recs)


REPORT = {}


def _run(label, gametype, recs, twice=False):
    t = time.time()
    dev = Renderer(gametype)
    obs, nat = dev.frames(recs, twice)
    dev.close()
    REPORT[label] = (assert_frames_equal(label, recs, obs, nat), time.time() - t)
    print("\n%s: %d frames equal (%.1f s)" % (label, *REPORT[label]))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_every_angle_at_every_phase(kind):
    _run("angles x phases, " + kind, "youturn", angle_set()[kind])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_rounding_ties(kind):
    r, _ = tie_set()[kind]
    _run("ties, " + kind, "youturn", r)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_border_sweeps(kind):
    r, _, _ = border_set()[kind]
    _run("borders, " + kind, "youturn", r)


@pytest.mark.gpu
def test_explosion_at_the_borders():
    _run("explosion at the borders", "youturn", explosion_border_set(), twice=True)


@pytest.mark.gpu
@pytest.mark.parametrize("zone", ["ship", "fortress", "hexagons", "bar", "score"])
def test_overlaps(zone):
    _run("overlaps, " + zone, "youturn", overlap_set()[zone], twice=True)


@pytest.mark.gpu
def test_score_and_bar():
    _run("score and bar", "youturn", score_bar_set())


@pytest.mark.gpu
@pytest.mark.parametrize("gametype", ["youturn", "autoturn"])
def test_position_independence(gametype):
    """the same state in every env of 4737 (148 groups of 32 and a partial one) gives the oracle's one frame"""
    n = 4737
    for which, state in zip(("crowded", "dead ship"), crowded_states()):
        t = time.time()
        dev = Renderer(gametype, n)
        obs, nat = dev.frames(np.repeat(state, n), twice=True)
        dev.close()
        for native, got in ((False, obs), (True, nat)):
            exp = oracle_frames(state, native)[0]
            bad = np.nonzero(differ(np.broadcast_to(exp, got.shape), got))[0]
            assert len(bad) == 0, (gametype, which, "native" if native else "obs", len(bad), [(int(i),) + frame_diff(exp, got[i]) for i in bad[:5]])
        print("\nposition independence, %s, %s: %d frames equal (%.1f s)" % (gametype, which, 2 * n, time.time() - t))
