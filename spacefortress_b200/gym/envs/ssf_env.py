"""SSF_Env — the reference's gym environment (python/spacefortress.gym/spacefortress/gym/envs/ssf_env.py:43-269)
as a facade over a one-env slab of the batched CUDA simulator: same constructor arguments, action tables,
reset/step return values, reward shaping (done on the device, sf_step.cuh) and quirks:
  * step returns (obs (92,90) u8, reward:int, done:bool, fort_kill:bool) — info is a bool (ssf_env.py:250);
  * reset() does not clear prev_vlner (ssf_env.py:92,163-178);
  * seed() only creates np_random, which nothing reads (ssf_env.py:159-161);
  * no auto-reset: stepping past `done` keeps ticking the same game.
The pyglet viewer (ssf_env.py:18-41) is out of scope; render('rgb_array') returns the grey frame as RGB.
"""
import ctypes as C

import numpy as np

from ... import _lib
from ...core import Game
from ...spaces import Box, Discrete


class SSF_Env(object):
    metadata = {"render.modes": ["human", "rgb_array"], "video.frames_per_second": 30}

    def __init__(self, gametype="youturn", scale=.2, viewport=(130, 80, 450, 460), ls=3, action_set=1, obs_type="image", device=0):
        assert obs_type in ("image", "features", "normalized-features", "monitors")
        self.obs_type = obs_type
        self.seed()
        self.viewer = None
        self.last_action = None
        self.gametype = gametype
        self.w = int(viewport[2] * scale)
        self.h = int(viewport[3] * scale)
        self.viewport = viewport
        self.ls = ls
        self.tickdur = int(np.ceil(1. / self.metadata["video.frames_per_second"] * 1000))
        self.action_set = action_set
        self.youturn = gametype in ("youturn", "test-youturn")
        self.device = device
        # action tables (ssf_env.py:65-90); columns FIRE, THRUST[, LEFT, RIGHT]
        if self.youturn:
            if action_set in (-1, 0):
                self.action_combinations = np.array(np.meshgrid([0, 1], [0, 1], [0, 1], [0, 1])).T.reshape(-1, 4)
            elif action_set == 1:
                self.action_combinations = np.array([[0, 0, 0, 0], [1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1]])
        elif gametype in ("autoturn", "test-autoturn"):
            if action_set == -1:
                self.action_combinations = np.array(np.meshgrid([0, 1], [0, 1], [0, 1], [0, 1])).T.reshape(-1, 4)
            elif action_set == 0:
                self.action_combinations = np.array(np.meshgrid([0, 1], [0, 1])).T.reshape(-1, 2)
            elif action_set == 1:
                self.action_combinations = np.array([[0, 0], [1, 0], [0, 1]])
        else:
            raise RuntimeError("cannot initialize Game. Unknown config value: `%s'" % gametype)
        self.action_space = Discrete(len(self.action_combinations))
        self.actions_taken = {i: 0 for i in range(len(self.action_combinations))}
        self.g = None
        self.reset()

    # ssf_env.py:159-161 — has no effect on the game (the C++ core uses libc rand(), never seeded)
    def seed(self, seed=None):
        self.np_random = np.random.RandomState(seed)
        return [seed]

    def reset(self):
        if self.g is None:
            # one slab for the life of the env; the kernel's new-game path replaces `sf.Game(...)` per episode
            self.g = Game(self.gametype, width=self.w, height=self.h, viewport=tuple(self.viewport), lw=self.ls, grayscale=True,
                          device=self.device, _shaped=True)
        else:
            _lib.check(self.g.L.sf_reset(self.g.h, None, 0, None, 0, None))
            self.g._rec = None
        self.max_ticks = np.floor(self.g.max_time / self.tickdur)
        if self.obs_type == "image":
            self.observation_space = Box(low=0, high=255, shape=(self.g.pb_height, self.g.pb_width, 3), dtype=np.uint8)
            self.game_state = self.g.gray_frame()
            self.game_gray_rgb = np.repeat(self.game_state[..., None], 3, axis=2)
            return self.game_state
        self.observation_space = Box(low=-np.inf, high=np.inf, shape=self._get_features().shape, dtype=np.float32)
        self.game_state = np.array([])
        return self._get_features()

    def step(self, action):
        self.actions_taken[action] += 1
        keystate = self.action_combinations[action]
        g = self.g
        (g.press_key if keystate[0] else g.release_key)(1)
        (g.press_key if keystate[1] else g.release_key)(2)
        if self.youturn:
            (g.press_key if keystate[2] else g.release_key)(3)
            (g.press_key if keystate[3] else g.release_key)(4)
        reward = g.step_one_tick(self.tickdur)  # shaped on the device for the train presets (ssf_env.py:233-244)
        _, done, fort_kill = g._last
        self.last_action = action
        if self.obs_type == "image":
            self.game_state = g.gray_frame()
            self.game_gray_rgb = np.repeat(self.game_state[..., None], 3, axis=2)
            return self.game_state, reward, done, fort_kill
        self.game_state = np.array([])
        return self._get_features(), reward, done, fort_kill

    def clone_state(self):
        """ALE-style snapshot of the game (Game.clone_state): a host uint8 array that restore_state takes back."""
        return self.g.clone_state()

    def restore_state(self, blob):
        self.g.restore_state(blob)
        if self.obs_type == "image":
            self.game_state = self.g.gray_frame()
            self.game_gray_rgb = np.repeat(self.game_state[..., None], 3, axis=2)
        else:
            self.game_state = np.array([])  # render() draws the restored frame

    def obs84(self):
        return self.g.obs84()

    def render(self, mode="human", close=False):
        if close:
            return None
        if self.obs_type != "image" and self.game_state.shape == (0,):
            self.game_state = self.g.gray_frame()
            self.game_gray_rgb = np.repeat(self.game_state[..., None], 3, axis=2)
        if mode == "rgb_array":
            return self.game_gray_rgb
        return None  # the pyglet window of the reference is not provided

    def close(self):
        self.g = None

    # ssf_env.py:95-157: computed on the device (sf_features_f64), float64 like np.array(f) in the reference
    def _get_features(self):
        return self.g.features(self.obs_type)
