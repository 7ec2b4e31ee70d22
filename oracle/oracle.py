"""TEST INFRASTRUCTURE ONLY (oracle/): ctypes bindings for

* ``libsforacle.so`` — the plain-C restatement (sf_oracle.c, sf_draw_oracle.c), class ``OracleEnv``;
* ``_ref/libsfref.so`` — the UNMODIFIED reference game core compiled in place from
  /root/reference (ref_harness.cpp), class ``RefEnv`` (state/step only; the cairo
  renderer cannot be built offline).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference arm may import this.
The product package (spacefortress_b200/) never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
MAX_MISSILES = 20
MAX_SHELLS = 20
NUM_STATS = 13

STAT_NAMES = ["bigHexDeaths", "smallHexDeaths", "shellDeaths", "shipDeaths", "resets", "destroyedFortresses",
              "missedShots", "totalShots", "totalThrusts", "totalLefts", "totalRights", "vlnerIncs", "maxVlner"]


class Record(C.Structure):
    """Mirror of sfr_record (oracle/sf_record.h) == sf_state_record (include/sf_b200.h)."""
    _fields_ = [
        ("ship_x", C.c_double), ("ship_y", C.c_double), ("ship_vx", C.c_double), ("ship_vy", C.c_double),
        ("ship_angle", C.c_double), ("fortress_angle", C.c_double), ("fortress_last_angle", C.c_double),
        ("missile_x", C.c_double * MAX_MISSILES), ("missile_y", C.c_double * MAX_MISSILES),
        ("missile_vx", C.c_double * MAX_MISSILES), ("missile_vy", C.c_double * MAX_MISSILES),
        ("missile_angle", C.c_double * MAX_MISSILES),
        ("shell_x", C.c_double * MAX_SHELLS), ("shell_y", C.c_double * MAX_SHELLS),
        ("shell_vx", C.c_double * MAX_SHELLS), ("shell_vy", C.c_double * MAX_SHELLS),
        ("shell_angle", C.c_double * MAX_SHELLS),
        ("points", C.c_float), ("raw_points", C.c_float),
        ("missile_mask", C.c_uint32), ("shell_mask", C.c_uint32),
        ("ship_alive", C.c_int32), ("fortress_alive", C.c_int32),
        ("ship_death_timer", C.c_int32), ("fire_timer", C.c_int32), ("thrust_timer", C.c_int32),
        ("left_timer", C.c_int32), ("right_timer", C.c_int32),
        ("thrust_flag", C.c_int32), ("fire_flag", C.c_int32), ("left_flag", C.c_int32), ("right_flag", C.c_int32),
        ("turn_flag", C.c_int32),
        ("fortress_timer", C.c_int32), ("fortress_death_timer", C.c_int32), ("fortress_vuln_timer", C.c_int32),
        ("vulnerability", C.c_int32), ("tick", C.c_int32), ("time", C.c_int32),
        ("stats", C.c_int32 * NUM_STATS),
        ("prev_vlner", C.c_int32), ("rng_seed", C.c_uint32), ("rng_count", C.c_uint32), ("_pad", C.c_int32),
    ]

    INT_FIELDS = ["missile_mask", "shell_mask", "ship_alive", "fortress_alive", "ship_death_timer", "fire_timer",
                  "thrust_timer", "left_timer", "right_timer", "thrust_flag", "fire_flag", "left_flag", "right_flag",
                  "turn_flag", "fortress_timer", "fortress_death_timer", "fortress_vuln_timer", "vulnerability",
                  "tick", "time", "prev_vlner", "rng_seed", "rng_count"]
    SCALAR_FLOAT_FIELDS = ["ship_x", "ship_y", "ship_vx", "ship_vy", "ship_angle", "fortress_angle",
                           "fortress_last_angle", "points", "raw_points"]

    def copy(self):
        r = Record()
        C.memmove(C.byref(r), C.byref(self), C.sizeof(Record))
        return r

    def int_state(self):
        """Integer / event-driven state as a plain dict (bit-exact comparison)."""
        d = {k: int(getattr(self, k)) for k in self.INT_FIELDS}
        d["stats"] = [int(v) for v in self.stats]
        return d

    def float_state(self):
        """Continuous state; projectile arrays only for live slots."""
        d = {k: float(getattr(self, k)) for k in self.SCALAR_FLOAT_FIELDS}
        for name, mask, n in (("missile", self.missile_mask, MAX_MISSILES), ("shell", self.shell_mask, MAX_SHELLS)):
            for f in ("x", "y", "vx", "vy", "angle"):
                arr = getattr(self, "%s_%s" % (name, f))
                d["%s_%s" % (name, f)] = [float(arr[i]) if (mask >> i) & 1 else 0.0 for i in range(n)]
        return d


def record_dtype():
    """numpy structured dtype with the same layout as Record (for batched get/set state)."""
    fields = []
    for name, ct in Record._fields_:
        if hasattr(ct, "_length_"):
            fields.append((name, np.dtype(ct._type_), (ct._length_,)))
        else:
            fields.append((name, np.dtype(ct)))
    dt = np.dtype(fields, align=True)
    assert dt.itemsize == C.sizeof(Record), (dt.itemsize, C.sizeof(Record))
    return dt


def step_records(gametype, recs, keymask=0):
    """One teacher-forced SSF_Env.step(keymask) from each state of `recs` (a record_dtype() array). Returns (the states
    after the step, int32 [n, 4] of reward, done, fort_kill, events)."""
    L = oracle_lib()
    gt = L.sfo_gametype_from_name(gametype.encode())
    if gt < 0:
        raise RuntimeError("Unknown config value: `%s'" % gametype)
    after = np.ascontiguousarray(recs, dtype=record_dtype()).copy()
    out = np.zeros((len(after), 4), np.int32)
    L.sfo_step_records(gt, after.ctypes.data, len(after), int(keymask), out.ctypes.data)
    return after, out


def build(force=False):
    """Compile libsforacle.so (always possible: gcc only) and _ref/libsfref.so (only where
    /root/reference exists; the prebuilt .so travels to the GPU box)."""
    if force:
        subprocess.run(["make", "-C", HERE, "clean"], check=True, capture_output=True)
    subprocess.run(["make", "-C", HERE, "all"], check=True, capture_output=True)


_ORACLE = None
_REF = None


def oracle_lib():
    global _ORACLE
    if _ORACLE is None:
        path = os.path.join(HERE, "libsforacle.so")
        if not os.path.exists(path):
            build()
        L = C.CDLL(path)
        L.sfo_gametype_from_name.argtypes = [C.c_char_p]
        L.sfo_create.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
        L.sfo_reset.argtypes = [C.c_void_p]
        L.sfo_core_step.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_uint32)]
        L.sfo_env_step.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.sfo_set_state.argtypes = [C.c_void_p, C.POINTER(Record)]
        L.sfo_step_records.argtypes = [C.c_int, C.c_void_p, C.c_long, C.c_int, C.c_void_p]
        L.sfo_get_extra.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.sfo_dump.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_char_p, C.c_int]
        L.sfo_run.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_void_p]
        L.sfo_run.restype = C.c_long
        L.sfo_rand.argtypes = [C.c_void_p]
        L.sfo_srand.argtypes = [C.c_void_p, C.c_uint32]
        L.sfo_action_to_keymask.argtypes = [C.c_int, C.c_int, C.c_int]
        L.sfo_num_actions.argtypes = [C.c_int, C.c_int]
        L.sfo_draw_native.argtypes = [C.POINTER(Record), C.c_void_p]
        L.sfo_draw_obs.argtypes = [C.POINTER(Record), C.c_void_p]
        L.sfo_resize_area.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]
        L.sfo_set_glyph_masks.argtypes = [C.c_void_p, C.c_void_p]
        _ORACLE = L
    return _ORACLE


def ref_available():
    return os.path.exists(os.path.join(HERE, "_ref", "libsfref.so"))


def ref_lib():
    global _REF
    if _REF is None:
        path = os.path.join(HERE, "_ref", "libsfref.so")
        if not os.path.exists(path):
            raise RuntimeError("oracle/_ref/libsfref.so missing: run `make -C oracle ref` where /root/reference exists")
        L = C.CDLL(path)
        L.sfref_create.restype = C.c_void_p
        L.sfref_create.argtypes = [C.c_char_p, C.c_uint32]
        for name in ("sfref_destroy", "sfref_reset"):
            getattr(L, name).argtypes = [C.c_void_p]
        L.sfref_core_step.argtypes = [C.c_void_p, C.c_int]
        L.sfref_env_step.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.sfref_get_state.argtypes = [C.c_void_p, C.POINTER(Record)]
        L.sfref_set_state.argtypes = [C.c_void_p, C.POINTER(Record)]
        L.sfref_dump.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.sfref_get_extra.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.sfref_hexagons.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.sfref_wireframe.argtypes = [C.c_int, C.POINTER(C.c_double), C.c_int]
        L.sfref_events.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.sfref_collisions.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.sfref_run.argtypes = [C.c_void_p, C.c_void_p, C.c_long]
        L.sfref_run.restype = C.c_long
        L.sfref_run_render.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p]
        L.sfref_run_render.restype = C.c_long
        _REF = L
    return _REF


class _OEnvStruct(C.Structure):
    _fields_ = [("s", Record), ("gametype", C.c_int), ("r", C.c_int32 * 34), ("rng_i", C.c_int)]


class OracleEnv:
    """C restatement behind an SSF_Env-like interface (key masks instead of action ids)."""

    def __init__(self, gametype="youturn", seed=1):
        self.L = oracle_lib()
        self.gametype = gametype
        self.gt = self.L.sfo_gametype_from_name(gametype.encode())
        if self.gt < 0:
            raise RuntimeError("Unknown config value: `%s'" % gametype)
        self.e = _OEnvStruct()
        self.L.sfo_create(C.byref(self.e), self.gt, seed)

    @property
    def state(self):
        return self.e.s

    def reset(self):
        self.L.sfo_reset(C.byref(self.e))

    def step(self, keymask):
        out = (C.c_int * 4)()
        self.L.sfo_env_step(C.byref(self.e), int(keymask), out)
        return out[0], bool(out[1]), bool(out[2]), out[3] & 0xFFFFFFFF

    def core_step(self, keymask):
        ev = C.c_uint32(0)
        r = self.L.sfo_core_step(C.byref(self.e), int(keymask), C.byref(ev))
        return r, ev.value

    def get_state(self):
        return self.e.s.copy()

    def set_state(self, rec):
        self.L.sfo_set_state(C.byref(self.e), C.byref(rec))

    def extra(self):
        out = (C.c_double * 4)()
        self.L.sfo_get_extra(C.byref(self.e), out)
        return list(out)

    def dump(self):
        b = C.create_string_buffer(8192)
        self.L.sfo_dump(C.byref(self.e), 0, 0, b, 8192)
        return b.value.decode()

    def rand(self):
        return self.L.sfo_rand(C.byref(self.e))

    def keymask(self, action, action_set=1):
        return self.L.sfo_action_to_keymask(self.gt, action_set, int(action))

    def num_actions(self, action_set=1):
        return self.L.sfo_num_actions(self.gt, action_set)

    def native_frame(self, rec=None):
        img = np.zeros((92, 90), np.uint8)
        self.L.sfo_draw_native(C.byref(rec if rec is not None else self.e.s), img.ctypes.data)
        return img

    def obs(self, rec=None):
        img = np.zeros((84, 84), np.uint8)
        self.L.sfo_draw_obs(C.byref(rec if rec is not None else self.e.s), img.ctypes.data)
        return img

    def run(self, keymasks, render=False):
        km = np.ascontiguousarray(keymasks, dtype=np.uint8)
        obs = np.zeros((84, 84), np.uint8)
        return self.L.sfo_run(C.byref(self.e), km.ctypes.data, km.size, obs.ctypes.data if render else None)


def set_glyph_masks(alpha=None, slot=None):
    """Digits from a real cairo + font (same format as the product's sf_set_glyph_masks); None restores the 7-segment face."""
    L = oracle_lib()
    if alpha is None:
        L.sfo_set_glyph_masks(None, None)
        return
    a = np.ascontiguousarray(alpha, dtype=np.uint8).reshape(10, 5 * 27)
    s = np.ascontiguousarray(slot, dtype=np.uint8).reshape(27)
    L.sfo_set_glyph_masks(a.ctypes.data, s.ctypes.data)


def resize_area(img, dh=84, dw=84):
    L = oracle_lib()
    src = np.ascontiguousarray(img, dtype=np.uint8)
    dst = np.zeros((dh, dw), np.uint8)
    L.sfo_resize_area(src.ctypes.data, src.shape[0], src.shape[1], dst.ctypes.data, dh, dw)
    return dst


def draw_native(rec):
    img = np.zeros((92, 90), np.uint8)
    oracle_lib().sfo_draw_native(C.byref(rec), img.ctypes.data)
    return img


def draw_obs(rec):
    img = np.zeros((84, 84), np.uint8)
    oracle_lib().sfo_draw_obs(C.byref(rec), img.ctypes.data)
    return img


class RefEnv:
    """The compiled reference core (unmodified), same interface as OracleEnv."""

    def __init__(self, gametype="youturn", seed=1):
        self.L = ref_lib()
        self.gametype = gametype
        self.h = self.L.sfref_create(gametype.encode(), seed)
        if not self.h:
            raise RuntimeError("Unknown config value: `%s'" % gametype)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.L.sfref_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def reset(self):
        self.L.sfref_reset(self.h)

    def step(self, keymask):
        out = (C.c_int * 4)()
        self.L.sfref_env_step(self.h, int(keymask), out)
        return out[0], bool(out[1]), bool(out[2]), out[3] & 0xFFFFFFFF

    def core_step(self, keymask):
        return self.L.sfref_core_step(self.h, int(keymask))

    def get_state(self):
        r = Record()
        self.L.sfref_get_state(self.h, C.byref(r))
        return r

    def set_state(self, rec):
        self.L.sfref_set_state(self.h, C.byref(rec))

    def extra(self):
        out = (C.c_double * 4)()
        self.L.sfref_get_extra(self.h, out)
        return list(out)

    def dump(self):
        b = C.create_string_buffer(8192)
        self.L.sfref_dump(self.h, b, 8192)
        return b.value.decode()

    def events(self):
        """Game.events of the last tick (pymodule.cpp:136-143)."""
        b = C.create_string_buffer(4096)
        self.L.sfref_events(self.h, b, 4096)
        return tuple(x for x in b.value.decode().split(",") if x)

    def collisions(self):
        """Game.collisions of the last tick, in pymodule.cpp:182-197's order."""
        b = C.create_string_buffer(256)
        self.L.sfref_collisions(self.h, b, 256)
        return tuple(x for x in b.value.decode().split(",") if x)

    def hexagons(self):
        big = (C.c_double * 12)()
        small = (C.c_double * 12)()
        self.L.sfref_hexagons(self.h, big, small)
        return np.array(big).reshape(6, 2), np.array(small).reshape(6, 2)

    def run(self, keymasks, render=False):
        """Bulk loop in C: reference tick + shaping + auto-reset (+ restated frame when render=True)."""
        km = np.ascontiguousarray(keymasks, dtype=np.uint8)
        if not render:
            return self.L.sfref_run(self.h, km.ctypes.data, km.size)
        obs = np.zeros((84, 84), np.uint8)
        draw = C.cast(oracle_lib().sfo_draw_obs, C.c_void_p)
        return self.L.sfref_run_render(self.h, km.ctypes.data, km.size, draw, obs.ctypes.data)


def wireframe(which):
    out = (C.c_double * 64)()
    n = ref_lib().sfref_wireframe(which, out, 64)
    return np.array(out[:4 * n]).reshape(n, 4)
