"""SFVecEnv — batched drop-in for the reference's vectorised env usage.

The reference trains through ``gym_vecenv.SubprocVecEnv([make_env(...)] * N)`` (rl/train.py:30-34): one OS
process per env, one pipe round-trip per env per step, numpy in/out. SFVecEnv keeps that interface
(``reset() -> [N,1,84,84] u8``, ``step(actions) -> (obs, rew, done, infos)``, ``close()``,
``observation_space``/``action_space``, ``num_envs``, ``step_async/step_wait``; rl/train.py:35-41,60,80-85,179)
but all N envs live in one SoA slab on one GPU and one kernel launch advances them.

* ``step(np.ndarray)``  -> numpy results through the C-ABI host path (sf_step_host): literal drop-in.
* ``step(torch.Tensor on cuda)`` -> torch CUDA tensors, no host round trip (sf_step).
* ``rollout(T, actions=None)`` -> T steps in one launch (sf_rollout), time-major outputs.

With ``obs_type`` 'features' / 'normalized-features' / 'monitors' the observation of every step is a feature row written
by the same state-only kernel that steps the envs (sf_step_host_features, sf_rollout_features).

Auto-reset follows gym_vecenv's worker loop: when an env is done its returned observation is the first
frame of the next episode; reward/done/info belong to the terminal step.
"""
import ctypes as C

import sys

import numpy as np

from . import _lib
from .spaces import Box, Discrete

GAMETYPE_OF_ENV_ID = {
    "SpaceFortress-youturn-image-v0": "youturn",
    "SpaceFortress-autoturn-image-v0": "autoturn",
    "SpaceFortress-testyouturn-image-v0": "test-youturn",
    "SpaceFortress-testautoturn-image-v0": "test-autoturn",
}
GAMETYPES = ("youturn", "autoturn", "test-youturn", "test-autoturn")


def _gametype(name):
    if name in GAMETYPE_OF_ENV_ID:
        return GAMETYPE_OF_ENV_ID[name]
    return name  # unknown names are rejected by sf_create like pymodule.cpp:341


def _torch():
    import torch
    return torch


class SFVecEnv(object):
    def __init__(self, env_id="SpaceFortress-youturn-image-v0", num_envs=16, device=0, action_set=1, seeds=None,
                 render=True, native_obs=False, autoreset=True, first_global_env=0, copy_outputs=False, obs_type="image",
                 host_delta=True, action_repeat=1, repeat_action_probability=0.0, sticky_seed=0):
        """copy_outputs (numpy path): False = step() returns views of the env's page-locked output buffers, which the
        next step() overwrites, and `infos` as a bool ndarray (the fast path); True = fresh arrays every step and
        `infos` as a tuple of N bools, exactly what gym_vecenv's np.stack returns; "ring" (SubprocVecEnv / DummyVecEnv
        default) = the same contract without the host-side copy: the observations come from a rotation of page-locked
        buffers, each updated in place by the GPU (host_delta), and a buffer is reused only when nobody holds a
        reference to the array that was handed out (or to a view / torch.from_numpy tensor of it), so an observation
        a caller keeps is never overwritten; those arrays are read-only (in-place edits would corrupt the next update). obs_type: 'image' (default), or 'features' / 'normalized-features' / 'monitors' (ssf_env.py:95-157):
        step() / reset() then return the [N, F] float32 feature matrix computed on the device: reset() reads the new
        state (sf_features), step() and rollout() get the rows from the kernel that steps the envs (sf_step_host_features,
        sf_rollout_features), one launch per step or rollout.
        host_delta (numpy path): the frames reach the page-locked observation buffer as SF_FLAG_HOST_DELTA updates (only
        the bytes that changed since the previous step cross PCIe; the buffer's contents are those of a full copy). The
        views step() returns are then read-only, because the next update builds on them. False: whole frames every step.
        action_repeat: game ticks per agent step (gym's `frameskip`, sf_set_action_repeat): every step() and each of the T
        steps of rollout(T) repeats its action for up to action_repeat ticks, stopping at the tick an episode ends; the
        reward is the sum over those ticks, done / infos / events are set by any of them, and the observation is that of
        the state after the last one. 1 (default) is the plain one-tick step.
        repeat_action_probability, sticky_seed: sticky actions (ALE's repeat_action_probability, sf_set_sticky_actions):
        every game tick keeps the keys the env already holds with probability p instead of taking the action's, drawn on
        the device from (sticky_seed, the env's global index, its rand() count and tick). 0.0 (default) never sticks."""
        self.L = _lib.lib()
        self.gametype = _gametype(env_id)
        self.num_envs = int(num_envs)
        self.device_index = int(device) if not isinstance(device, str) else int(device.split(":")[1]) if ":" in device else 0
        self.render_on = bool(render)
        self.native_obs = bool(native_obs)
        self.autoreset = bool(autoreset)
        self.copy_outputs = copy_outputs if copy_outputs == "ring" else bool(copy_outputs)
        self.host_delta = bool(host_delta)
        self._ring = []
        if obs_type not in _lib.OBS_TYPES:
            raise ValueError("obs_type must be one of %r" % (tuple(_lib.OBS_TYPES),))  # ssf_env.py:51
        self.obs_type = obs_type
        if obs_type != "image":
            render = False
            self.render_on = False
        h = C.c_void_p()
        _lib.check(self.L.sf_create(self.gametype.encode(), int(action_set), self.num_envs, self.device_index, C.byref(h)))
        self.h = h
        self.action_repeat = int(action_repeat)
        rc = self.L.sf_set_action_repeat(self.h, self.action_repeat)
        if rc != _lib.SF_OK:
            msg = self.L.sf_last_error()
            self.L.sf_destroy(self.h)
            self.h = None
            raise ValueError("action_repeat must be in [1, %d]: %s" % (_lib.MAX_ACTION_REPEAT, msg.decode() if msg else "?"))
        self.repeat_action_probability = float(repeat_action_probability)
        self.sticky_seed = int(sticky_seed)
        if not 0 <= self.sticky_seed < 1 << 32:  # the draw takes a uint32 seed: anything else would alias another seed
            self.L.sf_destroy(self.h)
            self.h = None
            raise ValueError("sticky_seed must be in [0, 2**32)")
        rc = self.L.sf_set_sticky_actions(self.h, self.repeat_action_probability, self.sticky_seed)
        if rc != _lib.SF_OK:
            msg = self.L.sf_last_error()
            self.L.sf_destroy(self.h)
            self.h = None
            raise ValueError("repeat_action_probability must be in [0, 1]: %s" % (msg.decode() if msg else "?"))
        self.num_actions = self.L.sf_num_actions(self.h)
        self.action_space = Discrete(self.num_actions)
        self.obs_shape = (1, _lib.NATIVE_H, _lib.NATIVE_W) if native_obs else (1, _lib.OBS_H, _lib.OBS_W)
        self.observation_space = Box(0, 255, self.obs_shape, dtype=np.uint8)  # rl/envs.py:21-25
        if obs_type != "image":
            self.num_features = self.L.sf_num_features(self.h, _lib.OBS_TYPES[obs_type])
            self.obs_shape = (self.num_features,)
            self.observation_space = Box(-np.inf, np.inf, self.obs_shape, dtype=np.float32)  # ssf_env.py:176
        self.first_global_env = int(first_global_env)
        if seeds is not None or first_global_env:
            self.seed_streams(seeds, first_global_env)
        self._flags = (_lib.FLAG_RENDER if render else 0) | (_lib.FLAG_NATIVE_OBS if native_obs else 0) | \
                      (0 if autoreset else _lib.FLAG_NO_AUTORESET)
        self._t = 0
        self._pending = None
        self._bufs = None
        self._np = None
        self._constructed = False
        self._device_work = False
        self.closed = False

    # ------------------------------------------------------------------ helpers
    def _device(self):
        return _torch().device("cuda", self.device_index)

    def _torch_bufs(self):
        if self._bufs is None:
            torch = _torch()
            dev = self._device()
            n = self.num_envs
            self._bufs = dict(
                obs=torch.empty((n,) + self.obs_shape, dtype=torch.uint8, device=dev),
                reward=torch.empty(n, dtype=torch.int32, device=dev),
                done=torch.empty(n, dtype=torch.uint8, device=dev),
                kill=torch.empty(n, dtype=torch.uint8, device=dev),
                events=torch.empty(n, dtype=torch.int32, device=dev),
            )
        return self._bufs

    def _np_bufs(self):
        if self._np is None:
            n = self.num_envs
            self._np = {}
            obs_dt = np.uint8 if self.obs_type == "image" else np.float32  # features: the kernel writes the rows in place
            for k, shape, dt in (("obs", (n,) + self.obs_shape, obs_dt), ("reward", (n,), np.int32), ("done", (n,), np.uint8),
                                 ("kill", (n,), np.uint8), ("events", (n,), np.uint32), ("actions", (n,), np.int32)):
                self._np[k] = _lib.pinned_array(shape, dt)  # page-locked: D2H lands directly in what step() returns
            self._np_ptr = {k: C.c_void_p(v.ctypes.data) for k, v in self._np.items()}  # (building these per step costs ~10 us)
            self._obs_ro = self._np["obs"].view()  # what step() hands out under host_delta: the next update builds on its contents
            self._obs_ro.flags.writeable = False
        return self._np

    def _feature_flags(self):
        """the step flags for the feature steps, which draw no frames"""
        return self._flags & ~(_lib.FLAG_RENDER | _lib.FLAG_NATIVE_OBS)

    def _stream_ptr(self):
        torch = _torch()
        self._device_work = True  # something of this env may now be in flight on torch's stream (see _step_numpy)
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    # ------------------------------------------------------------------ API
    def set_ticks(self, ticks):
        """Extension (BASELINE.json configs[4]): env i continues its episode from tick ticks[i], so that the envs of
        the batch reach the fixed episode end (5295 ticks, game.cpp:487-489) at different steps."""
        arr = np.ascontiguousarray(ticks, dtype=np.int32)
        assert arr.shape == (self.num_envs,)
        _lib.check(self.L.sf_set_ticks(self.h, arr.ctypes.data_as(C.c_void_p)))

    def seed_streams(self, seeds=None, first_global_env=0):
        """Per-env libc-rand() stream seeds (default: 1 for every env, the reference's behaviour since it
        never calls srand — game.cpp:137-148). An int s gives seeds s+i (rl/envs.py:13 `seed + rank`)."""
        if seeds is None:
            ptr = None
        else:
            if np.isscalar(seeds):
                seeds = int(seeds) + self.first_global_env + np.arange(self.num_envs)
            arr = np.ascontiguousarray(seeds, dtype=np.uint32)
            assert arr.shape == (self.num_envs,)
            ptr = arr.ctypes.data_as(C.c_void_p)
        _lib.check(self.L.sf_seed(self.h, ptr, int(first_global_env), None))
        self.first_global_env = int(first_global_env)
        return [seeds]

    def reset(self, to_numpy=True, clear_prev_vlner=None):
        """SSF_Env.reset for every env. The first call also plays the role of SSF_Env.__init__ (prev_vlner=0);
        later calls keep prev_vlner (quirk Q7, ssf_env.py:92)."""
        if clear_prev_vlner is None:
            clear_prev_vlner = not self._constructed
        self._constructed = True
        torch = _torch()
        b = self._torch_bufs()
        obs_ptr = C.c_void_p(b["obs"].data_ptr()) if self.render_on else None
        _lib.check(self.L.sf_reset(self.h, None, int(bool(clear_prev_vlner)), obs_ptr, self._flags, self._stream_ptr()))
        self._t = 0
        if self.obs_type != "image":
            return self.features(to_numpy=to_numpy)
        if not self.render_on:
            return None
        if to_numpy:
            return b["obs"].cpu().numpy()
        return b["obs"]

    def step_async(self, actions):
        self._pending = actions

    def step_wait(self):
        a, self._pending = self._pending, None
        return self.step(a)

    def step(self, actions, out_obs=None):
        if isinstance(actions, np.ndarray) or isinstance(actions, (list, tuple)):
            return self._step_numpy(np.asarray(actions))
        return self._step_torch(actions, out_obs)

    def _step_numpy(self, actions):
        n = self.num_envs
        b = self._np_bufs()
        a = b["actions"]
        a[:] = actions.reshape(n)
        if self._device_work:  # device-path work may be in flight on torch's stream: sf_step_host runs on its own streams
            _torch().cuda.synchronize(self._device())
            self._device_work = False
        p = self._np_ptr
        ring = self._ring_buffer() if (self.copy_outputs == "ring" and self.render_on and self.host_delta) else None
        if self.obs_type != "image":  # the step kernel writes the feature rows into the page-locked buffer
            _lib.check(self.L.sf_step_host_features(self.h, _lib.OBS_TYPES[self.obs_type], p["actions"], p["obs"], p["reward"], p["done"],
                                                    p["kill"], p["events"], self._feature_flags()))
        else:
            _lib.check(self.L.sf_step_host(self.h, p["actions"], (ring[3] if ring else p["obs"]) if self.render_on else None, p["reward"], p["done"], p["kill"], p["events"],
                                           self._flags | (_lib.FLAG_HOST_DELTA if self.host_delta and self.render_on else 0)))
        self._t += 1
        if self.obs_type != "image":
            obs = b["obs"].copy()  # a new array every step, as gym_vecenv gives
        elif not self.render_on:
            obs = None
        elif ring:
            obs = ring[0].view()
            obs.flags.writeable = False
        else:
            obs = b["obs"].copy() if self.copy_outputs else (self._obs_ro if self.host_delta else b["obs"])
        if self.copy_outputs:  # literal gym_vecenv: fresh arrays, info = tuple of N bools (ssf_env.py:233,250)
            self.last_events = b["events"].copy()
            return obs, b["reward"].astype(np.int64), b["done"].astype(bool), tuple(b["kill"].astype(bool).tolist())
        # fast path: views of the page-locked buffers (valid until the next step()); sum(infos) works like rl/train.py:81
        self.last_events = b["events"]
        return obs, b["reward"], b["done"].view(np.bool_), b["kill"].view(np.bool_)

    def _ring_buffer(self):
        """copy_outputs="ring": a page-locked observation buffer that nobody outside holds a view of — the most recently
        written one first (the smallest update). In a loop like rl/train.py:79-90, where the previous observation is
        dropped when the next one is bound, two buffers alternate and each update spans two steps."""
        ring = self._ring
        for k, e in enumerate(ring):
            if sys.getrefcount(e[1]) == e[2]:
                ring.insert(0, ring.pop(k))
                return e
        if len(ring) >= _lib.MAX_HOST_MIRRORS:  # every buffer is still held by the caller: let the oldest go (the caller's views keep it alive)
            old = ring.pop()
            _lib.check(self.L.sf_host_forget(self.h, old[3]))
        arr = _lib.pinned_array((self.num_envs,) + self.obs_shape, np.uint8)
        e = [arr, arr.base if isinstance(arr.base, np.ndarray) else arr, 0, C.c_void_p(arr.ctypes.data)]
        del arr
        e[2] = sys.getrefcount(e[1])  # the references this entry itself accounts for
        ring.insert(0, e)
        return e

    def _step_torch(self, actions, out_obs=None):
        """Device path. out_obs: optional contiguous uint8 CUDA tensor [N,1,84,84] to receive the frames (e.g.
        a slice of a time-major rollout buffer) instead of the env's own buffer."""
        torch = _torch()
        b = self._torch_bufs()
        a = actions.to(device=self._device(), dtype=torch.int32).reshape(self.num_envs).contiguous()
        if self.obs_type != "image":  # one launch: the step kernel writes the feature rows (a new tensor every step)
            obs = torch.empty((self.num_envs,) + self.obs_shape, dtype=torch.float32, device=self._device())
            _lib.check(self.L.sf_rollout_features(
                self.h, _lib.OBS_TYPES[self.obs_type], 1, C.c_void_p(a.data_ptr()), 0, int(self._t), C.c_void_p(obs.data_ptr()),
                C.c_void_p(b["reward"].data_ptr()), C.c_void_p(b["done"].data_ptr()), C.c_void_p(b["kill"].data_ptr()),
                C.c_void_p(b["events"].data_ptr()), self._feature_flags(), self._stream_ptr()))
            self._t += 1
            return obs, b["reward"], b["done"].bool(), b["kill"].bool()
        if out_obs is not None:
            assert out_obs.is_contiguous() and out_obs.dtype == torch.uint8 and out_obs.numel() == b["obs"].numel()
            b = dict(b, obs=out_obs)
        _lib.check(self.L.sf_step(
            self.h, C.c_void_p(a.data_ptr()), C.c_void_p(b["obs"].data_ptr()) if self.render_on else None,
            C.c_void_p(b["reward"].data_ptr()), C.c_void_p(b["done"].data_ptr()), C.c_void_p(b["kill"].data_ptr()),
            C.c_void_p(b["events"].data_ptr()), self._flags, self._stream_ptr()))
        self._t += 1
        obs = b["obs"] if self.render_on else None
        return obs, b["reward"], b["done"].bool(), b["kill"].bool()

    def host_delta_stats(self):
        """(observation bytes written to host buffers by delta updates, number of delta updates, number of whole-frame steps)."""
        out = (C.c_ulonglong * 3)()
        _lib.check(self.L.sf_host_delta_stats(self.h, out))
        return int(out[0]), int(out[1]), int(out[2])

    def features(self, obs_type=None, to_numpy=False, out=None):
        """[N, F] float32 feature observations of the current state (ssf_env.py:95-157: 'features' and
        'normalized-features' have 17 columns for autoturn, 19 for youturn; 'monitors' 10), one thread per env."""
        torch = _torch()
        kind = _lib.OBS_TYPES[obs_type or (self.obs_type if self.obs_type != "image" else "features")]
        nf = self.L.sf_num_features(self.h, kind)
        if out is None:
            out = torch.empty((self.num_envs, nf), dtype=torch.float32, device=self._device())
        _lib.check(self.L.sf_features(self.h, kind, C.c_void_p(out.data_ptr()), self._stream_ptr()))
        return out.cpu().numpy() if to_numpy else out

    def rollout(self, T, actions=None, action_seed=0, out=None, want=("obs", "reward", "done", "kill")):
        """T steps in one launch. actions: int32 CUDA tensor [T,N] or None for the synthetic counter-hash
        policy. Returns a dict of time-major CUDA tensors. With obs_type != 'image', "obs" is float32 [T, N, F]: row t
        holds the features after step t (auto-reset included), written by the kernel that steps the envs."""
        torch = _torch()
        dev = self._device()
        n = self.num_envs
        features = self.obs_type != "image"
        if out is None:
            out = {}
            if "obs" in want and (self.render_on or features):
                out["obs"] = torch.empty((T, n) + self.obs_shape, dtype=torch.float32 if features else torch.uint8, device=dev)
            if "reward" in want:
                out["reward"] = torch.empty((T, n), dtype=torch.int32, device=dev)
            if "done" in want:
                out["done"] = torch.empty((T, n), dtype=torch.uint8, device=dev)
            if "kill" in want:
                out["kill"] = torch.empty((T, n), dtype=torch.uint8, device=dev)
        aptr = None
        if actions is not None:
            actions = actions.to(device=dev, dtype=torch.int32).reshape(T, n).contiguous()
            aptr = C.c_void_p(actions.data_ptr())

        def p(k):
            return C.c_void_p(out[k].data_ptr()) if k in out else None
        if features and "obs" in out:
            o = out["obs"]
            if o.dtype != torch.float32 or not o.is_contiguous() or o.numel() != T * n * self.num_features:
                raise ValueError("out['obs'] must be a contiguous float32 tensor of shape %r" % ((T, n) + self.obs_shape,))
            _lib.check(self.L.sf_rollout_features(self.h, _lib.OBS_TYPES[self.obs_type], int(T), aptr, int(action_seed), int(self._t),
                                                  p("obs"), p("reward"), p("done"), p("kill"), None, self._feature_flags(), self._stream_ptr()))
        else:
            flags = self._flags if "obs" in out else (self._flags & ~_lib.FLAG_RENDER)
            _lib.check(self.L.sf_rollout(self.h, int(T), aptr, int(action_seed), int(self._t), p("obs"), p("reward"), p("done"),
                                         p("kill"), flags, self._stream_ptr()))
        self._t += T
        return out

    def synthetic_actions(self, T, action_seed=0, t0=None):
        """Host materialisation of the stream sf_rollout(actions=None) uses (parity runs)."""
        t0 = self._t if t0 is None else t0
        a = np.empty((T, self.num_envs), np.int32)
        for t in range(T):
            for i in range(self.num_envs):
                a[t, i] = self.L.sf_synthetic_action(int(action_seed), self.first_global_env + i, t0 + t, self.num_actions)
        return a

    def render_frames(self, native=False, to_numpy=True):
        """Game.draw() of the current state without stepping."""
        torch = _torch()
        shape = (self.num_envs, _lib.NATIVE_H, _lib.NATIVE_W) if native else (self.num_envs, _lib.OBS_H, _lib.OBS_W)
        o = torch.empty(shape, dtype=torch.uint8, device=self._device())
        _lib.check(self.L.sf_render(self.h, C.c_void_p(o.data_ptr()), _lib.FLAG_NATIVE_OBS if native else 0, self._stream_ptr()))
        return o.cpu().numpy() if to_numpy else o

    def get_state(self, first=0, count=None):
        count = self.num_envs - first if count is None else count
        arr = (_lib.StateRecord * count)()
        _lib.check(self.L.sf_get_state(self.h, first, count, arr))
        return arr

    def set_state(self, records, first=0):
        count = len(records)
        arr = records if isinstance(records, C.Array) else (_lib.StateRecord * count)(*records)
        _lib.check(self.L.sf_set_state(self.h, first, count, arr))

    def _env_index(self, idx):
        """idx (None, a sequence, a numpy array or a tensor of env indices) -> None or an int32 CUDA tensor on the env's
        device. Host indices are range-checked here (SFError), device indices by the kernels: save_envs writes an all-zero
        row for an index outside [0, num_envs), load_envs rejects the row."""
        torch = _torch()
        if idx is None:
            return None
        if isinstance(idx, torch.Tensor):
            if idx.dtype.is_floating_point or idx.dtype == torch.bool:
                raise TypeError("env indices must be integers")
            return idx.to(device=self._device(), dtype=torch.int32).reshape(-1).contiguous()
        arr = np.asarray(idx).reshape(-1)
        if arr.size and not np.issubdtype(arr.dtype, np.integer):
            raise TypeError("env indices must be integers")
        if arr.size and (arr.min() < 0 or arr.max() >= self.num_envs):
            raise _lib.SFError("env index out of range [0, %d)" % self.num_envs)
        return torch.from_numpy(arr.astype(np.int32)).to(self._device())

    def save_envs(self, idx=None, out=None):
        """Complete game state of envs idx (None: all) as a uint8 CUDA tensor [k, ENV_BLOB_BYTES] on the env's device,
        one canonical row per env (layout: SF_ENV_BLOB_BYTES in include/sf_b200.h). The result is an ordinary tensor:
        index it, torch.save it, move it to another GPU. out: a contiguous uint8 tensor of that shape to write into."""
        torch = _torch()
        ix = self._env_index(idx)
        k = self.num_envs if ix is None else ix.numel()
        shape = (k, _lib.ENV_BLOB_BYTES)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=self._device())
        elif out.dtype != torch.uint8 or tuple(out.shape) != shape or out.device != self._device() or not out.is_contiguous():
            raise ValueError("out must be a contiguous uint8 tensor of shape %r on %s" % (shape, self._device()))
        _lib.check(self.L.sf_save_envs(self.h, C.c_void_p(ix.data_ptr()) if ix is not None else None, k,
                                       C.c_void_p(out.data_ptr()), self._stream_ptr()))
        return out

    def load_envs(self, blob, idx=None, check=True):
        """Env idx[k] <- row k of blob (rows from save_envs of a handle of the same game type, on any device; idx=None:
        row i -> env i, which needs one row per env). Target indices must not repeat. The loaded envs continue exactly
        where the saved ones were; the render caches are rebuilt on the next frame. check=True waits for the load and
        raises SFError if any row had a bad header or target index (those rows are skipped either way)."""
        torch = _torch()
        dev = self._device()
        if isinstance(blob, np.ndarray):
            blob = torch.from_numpy(blob)
        if blob.dtype != torch.uint8 or blob.dim() != 2 or blob.shape[1] != _lib.ENV_BLOB_BYTES:
            raise ValueError("blob must be a uint8 tensor of shape [k, %d]" % _lib.ENV_BLOB_BYTES)
        blob = blob.to(dev).contiguous()
        k = blob.shape[0]
        ix = self._env_index(idx)
        if ix is None:
            if k != self.num_envs:
                raise ValueError("%d rows for %d envs: pass idx to load a subset" % (k, self.num_envs))
        else:
            if ix.numel() != k:
                raise ValueError("%d rows for %d target indices" % (k, ix.numel()))
            if torch.unique(ix).numel() != k:
                raise ValueError("repeated target index")
        rejected = torch.zeros(1, dtype=torch.int32, device=dev) if check else None
        _lib.check(self.L.sf_load_envs(self.h, C.c_void_p(blob.data_ptr()), C.c_void_p(ix.data_ptr()) if ix is not None else None, k,
                                       C.c_void_p(rejected.data_ptr()) if check else None, self._stream_ptr()))
        if check:
            bad = int(rejected.item())
            if bad:
                raise _lib.SFError("load_envs: %d of %d rows rejected (bad magic, version or game type, or target index out of "
                                   "range); the other rows were loaded" % (bad, k))

    def episode_stats(self, reset=True, all_reduce=True):
        """Finished-episode statistics since the last reset of the accumulators, summed over all ranks when
        torch.distributed is initialised (one small all-reduce per rollout; replaces rl/train.py:81-88)."""
        torch = _torch()
        out = torch.zeros(_lib.NUM_EPISODE_STATS, dtype=torch.int64, device=self._device())
        _lib.check(self.L.sf_episode_stats(self.h, C.c_void_p(out.data_ptr()), int(bool(reset)), self._stream_ptr()))
        from .dist import all_reduce_episode_stats
        if all_reduce:
            out = all_reduce_episode_stats(out)
        vals = out.cpu().tolist()
        return dict(zip(_lib.EPISODE_STAT_NAMES, vals))

    def set_glyph_masks(self, alpha=None, slot=None):
        """Install score-digit masks rendered by a real cairo + font (tools/dump_cairo_glyphs.py): alpha uint8 [10, 5, 27]
        (digit d in all 7 slots over native rows 1..5 x columns 32..58), slot uint8 [27]. None: the built-in 7-segment face."""
        if alpha is None:
            _lib.check(self.L.sf_set_glyph_masks(self.h, None, None))
            return
        a = np.ascontiguousarray(alpha, dtype=np.uint8).reshape(10, 5 * 27)
        s = np.ascontiguousarray(slot, dtype=np.uint8).reshape(27)
        _lib.check(self.L.sf_set_glyph_masks(self.h, a.ctypes.data_as(C.c_void_p), s.ctypes.data_as(C.c_void_p)))

    def state_bytes(self):
        return self.L.sf_state_bytes(self.h)

    def close(self):
        if not self.closed and getattr(self, "h", None):
            self._np = None  # the page-locked buffers free themselves when the last array handed out dies
            self._np_ptr = None
            self.L.sf_destroy(self.h)
            self.h = None
            self.closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EnvThunk(object):
    """What make_env() returns: rl/envs.py:10-16 builds a closure; here it only carries the parameters."""

    def __init__(self, env_id, seed, rank):
        self.env_id, self.seed, self.rank = env_id, seed, rank

    def __call__(self):
        from .gym.envs import SSF_Env
        from .rl_envs import WrapPyTorch
        env = SSF_Env(gametype=_gametype(self.env_id))
        env.seed(self.seed + self.rank)
        return WrapPyTorch(env)


class SubprocVecEnv(SFVecEnv):
    """gym_vecenv.SubprocVecEnv(list_of_thunks) look-alike (rl/train.py:32): the thunks are not called,
    one batched GPU env replaces the N worker processes."""

    def __init__(self, env_fns, device=0, **kw):
        kw.setdefault("copy_outputs", "ring")  # literal drop-in: fresh (read-only) arrays and a tuple of bools every step
        env_fns = list(env_fns)
        ids = set(getattr(f, "env_id", None) for f in env_fns)
        if len(ids) != 1 or None in ids:
            raise ValueError("SubprocVecEnv expects thunks from spacefortress_b200.make_env for ONE env id")
        SFVecEnv.__init__(self, env_id=ids.pop(), num_envs=len(env_fns), device=device, **kw)


class DummyVecEnv(SubprocVecEnv):
    """gym_vecenv.DummyVecEnv look-alike (rl/train.py:34, rl/evaluate.py:40-47)."""
    pass
