"""`Game` — same constructor, methods and read-only properties as the reference's CPython type
`spacefortress.core.Game` (python/spacefortress/src/pymodule.cpp:319-411), backed by a one-env slab of the
batched CUDA simulator. It exists so single-env callers (evaluation, trace tools, the SSF_Env facade) keep
working; throughput comes from SFVecEnv.

Supported render configuration = the one the gym env uses (ssf_env.py:50,164): width 90, height 92,
viewport (130,80,450,460), lw 3, grayscale. Anything else raises (the kernels are specialised for it).
Known binding defects of the reference are NOT replicated (SURVEY.md §8(b)): `shells` returns shells,
`vulnerability_timer`/`vulnerability_time` return real numbers.
"""
import ctypes as C

import numpy as np

from . import _lib

NO_KEY, FIRE_KEY, THRUST_KEY, LEFT_KEY, RIGHT_KEY = 0, 1, 2, 3, 4  # game.hh:15-17, pymodule.cpp:467-471
MAX_MISSILES = 20
MAX_SHELLS = 20
_KEY_BIT = {FIRE_KEY: _lib.KEY_FIRE, THRUST_KEY: _lib.KEY_THRUST, LEFT_KEY: _lib.KEY_LEFT, RIGHT_KEY: _lib.KEY_RIGHT}

_CONFIG = {  # configs.cpp:3-49 (baseConfig) and the per-preset overrides :51-89
    "width": 710, "height": 626, "gameTime": 180000, "destroyFortress": 100, "shipDeathPenalty": 100,
    "missilePenalty": 2.0, "missPenalty": 0, "incRewardInvulnerable": 0, "incRewardVulnerable": 0, "maxPoints": 3748,
    "maxBonus": 90, "shellSpeed": 6, "shellCollisionRadius": 3, "missileSpeed": 20, "missileCollisionRadius": 5,
    "autoTurn": 0, "staircase": 0, "fortressPointsPerContraction": 10, "fortressSectorSize": 10,
    "fortressLockTime": 1000, "fortressVulnerabilityTime": 250, "fortressVulnerabilityThreshold": 10,
    "fortressCollisionRadius": 18, "bigHex": 200, "smallHex": 40, "hexContraction": 5, "hexExpansion": 15,
    "minHexDistance": 20, "shipExplodeDuration": 1000, "shipStartX": 235.0, "shipStartY": 315.0,
    "shipStartVelX": float(np.cos(-60 * np.pi / 180)), "shipStartVelY": float(np.sin(-60 * np.pi / 180)),
    "shipStartAngle": 0.0, "shipCollisionRadius": 10, "shipAcceleration": 0.3, "shipTurnSpeed": 6,
}
_TRAIN = {"destroyFortress": 1, "shipDeathPenalty": 1, "missilePenalty": 0.05}


def config_of(gametype):
    c = dict(_CONFIG)
    if gametype in ("autoturn", "test-autoturn"):
        c["autoTurn"] = 1
    if gametype in ("autoturn", "youturn"):
        c.update(_TRAIN)
    return c


class Game(object):
    def __init__(self, config, lw=2.0, grayscale=0, width=-1, height=-1, viewport=(0, 0, -1, -1), device=0, _shaped=False):
        if config not in ("autoturn", "youturn", "test-youturn", "test-autoturn"):
            raise RuntimeError("cannot initialize Game. Unknown config value: `%s'" % config)  # pymodule.cpp:341
        if (width, height, tuple(viewport), float(lw), bool(grayscale)) != (90, 92, (130, 80, 450, 460), 3.0, True):
            raise NotImplementedError("only the gym env's render setup is supported: width=90, height=92, "
                                      "viewport=(130,80,450,460), lw=3, grayscale=True (ssf_env.py:50,164)")
        self.L = _lib.lib()
        self.gametype = config
        self.device = int(device)
        self._config = config_of(config)
        h = C.c_void_p()
        _lib.check(self.L.sf_create(config.encode(), -1, 1, int(device), C.byref(h)))
        self.h = h
        self._shaped = _shaped
        self._flags = _lib.FLAG_NO_AUTORESET | _lib.FLAG_ACTIONS_ARE_KEYMASKS | (0 if _shaped else _lib.FLAG_RAW_REWARD)
        _lib.check(self.L.sf_reset(self.h, None, 1, None, 0, None))
        self._pixels = np.zeros((92, 90, 4), np.uint8)  # BGRX like the cairo RGB24 surface (draw.cpp:62-66)
        self._keys = None  # pending key state for the next tick
        self._touched = []   # (sym, state) of the press_key / release_key calls since the last tick, in call order
        self._logged = ()
        self._rec = None
        self._events = 0
        self._last = (0, False, False)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.L.sf_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ---- state access -------------------------------------------------------------------------
    @property
    def record(self):
        if self._rec is None:
            arr = (_lib.StateRecord * 1)()
            _lib.check(self.L.sf_get_state(self.h, 0, 1, arr))
            self._rec = arr[0]
        return self._rec

    def set_record(self, rec):
        arr = (_lib.StateRecord * 1)(rec)
        _lib.check(self.L.sf_set_state(self.h, 0, 1, arr))
        self._rec = None

    def clone_state(self):
        """The complete game state as a host uint8 array [ENV_BLOB_BYTES] (one sf_save_envs row; it pickles). Unlike
        the record it holds the rand() stream itself, so restore_state does not replay it."""
        import torch
        dev = torch.device("cuda", self.device)
        with torch.cuda.device(dev):
            o = torch.empty((1, _lib.ENV_BLOB_BYTES), dtype=torch.uint8, device=dev)
            _lib.check(self.L.sf_save_envs(self.h, None, 1, C.c_void_p(o.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
            return o[0].cpu().numpy()

    def restore_state(self, blob):
        """Continue from a state clone_state returned (of a Game of the same config). Key presses since the last tick
        are dropped."""
        import torch
        b = np.asarray(blob)
        if b.dtype != np.uint8 or b.shape != (_lib.ENV_BLOB_BYTES,):
            raise ValueError("blob must be a uint8 array of shape (%d,)" % _lib.ENV_BLOB_BYTES)
        dev = torch.device("cuda", self.device)
        with torch.cuda.device(dev):
            t = torch.from_numpy(np.ascontiguousarray(b).reshape(1, -1)).to(dev)
            rejected = torch.zeros(1, dtype=torch.int32, device=dev)
            _lib.check(self.L.sf_load_envs(self.h, C.c_void_p(t.data_ptr()), None, 1, C.c_void_p(rejected.data_ptr()),
                                           C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
            if int(rejected.item()):
                raise _lib.SFError("restore_state: not a state of a %r game (bad magic, version or game type)" % self.gametype)
        self._rec = None
        self._keys = None
        self._touched = []

    def _current_keymask(self):
        r = self.record
        return (_lib.KEY_FIRE if r.fire_flag else 0) | (_lib.KEY_THRUST if r.thrust_flag else 0) | \
               (_lib.KEY_LEFT if r.left_flag else 0) | (_lib.KEY_RIGHT if r.right_flag else 0)

    # ---- methods (pymodule.cpp:361-370) ---------------------------------------------------------
    def _key(self, sym, state):
        if sym not in _KEY_BIT:
            return
        if self._keys is None:
            self._keys = self._current_keymask()
            self._touched = []
        if any(k == sym for k, _ in self._touched):
            raise NotImplementedError("more than one event for the same key inside one tick")
        self._touched.append((sym, bool(state)))
        self._keys = (self._keys | _KEY_BIT[sym]) if state else (self._keys & ~_KEY_BIT[sym])

    def press_key(self, sym):
        self._key(int(sym), True)

    def release_key(self, sym):
        self._key(int(sym), False)

    def step_one_tick(self, ms):
        if int(ms) != 34:
            raise NotImplementedError("the tick is fixed at 34 ms (ssf_env.py:61)")
        km = self._keys if self._keys is not None else self._current_keymask()
        self._keys = None
        self._logged, self._touched = tuple(self._touched), []
        a = np.array([km], np.int32)
        rew = np.zeros(1, np.int32)
        done = np.zeros(1, np.uint8)
        kill = np.zeros(1, np.uint8)
        ev = np.zeros(1, np.uint32)
        _lib.check(self.L.sf_step_host(self.h, a.ctypes.data_as(C.c_void_p), None, rew.ctypes.data_as(C.c_void_p),
                                       done.ctypes.data_as(C.c_void_p), kill.ctypes.data_as(C.c_void_p),
                                       ev.ctypes.data_as(C.c_void_p), self._flags))
        self._rec = None
        self._events = int(ev[0])
        self._last = (int(rew[0]), bool(done[0]), bool(kill[0]))
        return int(rew[0])

    def is_game_over(self):
        return self.record.time >= self._config["gameTime"]

    def _render(self, native):
        import torch
        shape = (1, 92, 90) if native else (1, 84, 84)
        dev = torch.device("cuda", self.device)  # the device the slab lives on (sf_create), not the current one
        with torch.cuda.device(dev):
            o = torch.empty(shape, dtype=torch.uint8, device=dev)
            _lib.check(self.L.sf_render(self.h, C.c_void_p(o.data_ptr()), _lib.FLAG_NATIVE_OBS if native else 0,
                                        C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
            return o[0].cpu().numpy()

    def features(self, obs_type="features"):
        """SSF_Env._get_features (ssf_env.py:95-157) as float64, computed on the device (sf_features_f64)."""
        import torch
        kind = _lib.OBS_TYPES[obs_type]
        dev = torch.device("cuda", self.device)
        with torch.cuda.device(dev):
            o = torch.empty((1, self.L.sf_num_features(self.h, kind)), dtype=torch.float64, device=dev)
            _lib.check(self.L.sf_features_f64(self.h, kind, C.c_void_p(o.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
            return o[0].cpu().numpy()

    def draw(self):
        g = self._render(True)
        self._pixels[..., 0] = g
        self._pixels[..., 1] = g
        self._pixels[..., 2] = g

    def gray_frame(self):
        """(92,90) u8: what cv2.cvtColor(pb_pixels, RGBA2GRAY) gives in ssf_env.py:205."""
        return self._render(True)

    def obs84(self):
        """(84,84) u8: gray_frame() after cv2.resize(..., INTER_AREA) (rl/envs.py:29), computed on the GPU."""
        return self._render(False)

    def config(self, key):
        if key not in self._config:
            raise ValueError("No config value for `%s'" % key)  # pymodule.cpp:273
        return self._config[key]

    def dump(self):
        """Game::dumpState (game.cpp:519-576)."""
        r = self.record
        ms = ",".join("%.3f,%.3f,%.1f" % (r.missile_x[i], r.missile_y[i], r.missile_angle[i]) for i in range(MAX_MISSILES) if (r.missile_mask >> i) & 1)
        ss = ",".join("%.3f,%.3f,%.1f" % (r.shell_x[i], r.shell_y[i], r.shell_angle[i]) for i in range(MAX_SHELLS) if (r.shell_mask >> i) & 1)
        ev = ",".join('"%s"' % e for e in self.events)
        return "[%d,%d,%.3f,%.3f,%.3f,%.3f,%.1f,%d,%.1f,[%s],[%s],%.1f,%d,%d,%d,[%s]]" % (
            r.time, r.ship_alive, r.ship_x, r.ship_y, r.ship_vx, r.ship_vy, r.ship_angle, r.fortress_alive, r.fortress_angle,
            ms, ss, r.points, r.vulnerability, r.thrust_flag, r.turn_flag, ev)

    # ---- read-only properties (pymodule.cpp:372-411) -----------------------------------------------
    tick = property(lambda s: s.record.tick)
    time = property(lambda s: s.record.time)
    max_time = property(lambda s: s._config["gameTime"])
    ship_alive = property(lambda s: bool(s.record.ship_alive))
    ship_x = property(lambda s: s.record.ship_x)
    ship_y = property(lambda s: s.record.ship_y)
    ship_vx = property(lambda s: s.record.ship_vx)
    ship_vy = property(lambda s: s.record.ship_vy)
    ship_angle = property(lambda s: s.record.ship_angle)
    fortress_alive = property(lambda s: bool(s.record.fortress_alive))
    fortress_angle = property(lambda s: s.record.fortress_angle)
    bighex = property(lambda s: s._config["bigHex"])
    smallhex = property(lambda s: s._config["smallHex"])
    points = property(lambda s: float(s.record.points))
    max_points = property(lambda s: float(s._config["maxPoints"]))
    raw_points = property(lambda s: float(s.record.raw_points))
    vulnerability = property(lambda s: s.record.vulnerability)
    vulnerability_time = property(lambda s: float(s._config["fortressVulnerabilityTime"]))
    vulnerability_timer = property(lambda s: float(s.record.fortress_vuln_timer))
    thrust_flag = property(lambda s: bool(s.record.thrust_flag))
    turn_flag = property(lambda s: s.record.turn_flag)
    pb_pixels = property(lambda s: memoryview(s._pixels.reshape(-1)))
    pb_width = property(lambda s: 90)
    pb_height = property(lambda s: 92)
    thrust_durations = property(lambda s: ())   # S20: unbounded per-episode logs are not kept on the device
    shot_durations = property(lambda s: ())
    shot_intervals_invul = property(lambda s: ())
    shot_intervals_vul = property(lambda s: ())

    @property
    def missiles(self):
        r = self.record
        return tuple((r.missile_x[i], r.missile_y[i], r.missile_angle[i]) for i in range(MAX_MISSILES) if (r.missile_mask >> i) & 1)

    @property
    def shells(self):
        r = self.record
        return tuple((r.shell_x[i], r.shell_y[i], r.shell_angle[i]) for i in range(MAX_SHELLS) if (r.shell_mask >> i) & 1)

    @property
    def events(self):
        """The tick's event strings in the order Game::stepOneTick logs them (game.cpp:124-127 call sites): one
        press-/release- entry per press_key / release_key call in call order (game.cpp:223) with missile-fired right
        after the press-fire that caused it (:186), then ship-respawn (:155), explode-* (:342,348), fortress-respawn
        (:202), fortress-fired (:169), shell-hit-ship (:417) and the missile loop's hit events (:363-393). The device
        keeps one bit per event kind, so a kind that occurs twice in a tick (two missiles hitting) is listed once."""
        ev, out = self._events, []
        names = {FIRE_KEY: "fire", THRUST_KEY: "thrust", LEFT_KEY: "left", RIGHT_KEY: "right"}
        for sym, state in self._logged:
            out.append(("press-" if state else "release-") + names[sym])
            if sym == FIRE_KEY and state and ev & _lib.EVENT_BITS["missile-fired"]:
                out.append("missile-fired")
        for name in ("ship-respawn", "explode-bighex", "explode-smallhex", "fortress-respawn", "fortress-fired", "shell-hit-ship",
                     "hit-fortress", "vlner-increased", "fortress-destroyed", "vlner-reset", "hit-dead-fortress"):
            if ev & _lib.EVENT_BITS[name]:
                out.append(name)
        return tuple(out)

    @property
    def collisions(self):
        """pymodule.cpp:182-197 fills its tuple from the back: the order is shell, missile, smallhex, bighex."""
        return tuple(name for name in ("shell", "missile", "smallhex", "bighex") if self._events & _lib.COLLISION_BITS[name])

    @property
    def stats(self):
        r = self.record
        return tuple(int(v) for v in r.stats) + (float(r.points), float(r.raw_points))

    @property
    def timers(self):
        r = self.record
        return (r.fire_timer, r.thrust_timer, r.left_timer, r.right_timer)

    # computeExtra (game.cpp:282-312): evaluated on the device (sf_features_f64, columns 6..8 of 'features')
    def _extra(self):
        f = self.features("features")
        return float(f[7]), float(f[6]), float(f[8])

    vdir = property(lambda s: s._extra()[0])
    aim = property(lambda s: s._extra()[1])
    ndist = property(lambda s: s._extra()[2])
