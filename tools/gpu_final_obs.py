"""Final observations at auto-reset (sf_set_final_obs): what keeping them costs, at action repeat k = 1 and 4.
usage: python tools/gpu_final_obs.py OUT_DIR   -> OUT_DIR/r08_final_obs_n1.json

Every variant is a setting (final observations off / on, k) with k in {1, 4}. Off at k = 1 is the plain step (the fused
rollout kernel with frames); on takes the route of k > 1. With frames each agent step is then four launches: the repeat
kernel with a deferred reset, a masked draw of the finished states, sf_final_reset_kernel and the draw of the step.
Without frames the repeat kernel stores final_step and the final rows just before the new game.
  rollout16   autoturn, 4096 and 65 536 envs, sf_rollout T = 16 with 84x84 frames, synthetic actions
  host_step   autoturn, 4096 envs, SFVecEnv.step(np.ndarray) with delta updates (sf_step_host, SF_FLAG_HOST_DELTA), wall time
  features    youturn, 131 072 envs, sf_rollout_features 'features' (19 columns), T = 64
The envs first run 400 state-only ticks, then their clocks are staggered over a whole episode, so that about n / 5295
envs end per tick. Device variants are timed with CUDA events, five windows per variant, the variants alternating window
by window; the host step with a host clock around windows that end in a device synchronise. Medians."""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ctypes as C  # noqa: E402

from spacefortress_b200 import _lib  # noqa: E402
# the timing harness of the action-repeat measurement: nvidia-smi query, CUDA-event and host-clock windows, alternation
# of variants window by window, the mid-episode env mix
from gpu_action_repeat import WINDOWS, alternate, event_ms, mixed_env, smi, vp, wall_ms  # noqa: E402

SETTINGS = [(on, k) for k in (1, 4) for on in (False, True)]


def name(on, k):
    return "%s_k%d" % ("on" if on else "off", k)


class Finals(object):
    """device final buffers for n envs (frames big enough for either layout, rows of the widest kind, final_step)"""

    def __init__(self, n):
        self.frames = torch.zeros((n, 92 * 90), dtype=torch.uint8, device="cuda")
        self.rows = torch.zeros((n, 19), dtype=torch.float32, device="cuda")
        self.step = torch.full((n,), -1, dtype=torch.int32, device="cuda")

    def set(self, env, on):
        _lib.check(env.L.sf_set_final_obs(env.h, *((vp(self.frames), vp(self.rows), vp(self.step)) if on else (None, None, None))))


def with_setting(env, fin, on, k, fn):
    def run():
        fin.set(env, on)
        _lib.check(env.L.sf_set_action_repeat(env.h, k))
        env.action_repeat = k
        fn()
    return run


def summarise(ms, n, steps_per_call, res):
    """per variant: us per agent step (median and windows), agent steps/s, ticks/s"""
    for v, w in ms.items():
        k = int(v.split("_k")[1])
        med = float(np.median(w))
        res[v] = dict(k=k, final_obs=v.startswith("on"), us_per_agent_step_median=round(med * 1e3 / steps_per_call, 2),
                      us_per_agent_step_windows=[round(x * 1e3 / steps_per_call, 2) for x in w],
                      agent_steps_per_s=int(round(n * steps_per_call / (med * 1e-3))),
                      ticks_per_s=int(round(n * steps_per_call * k / (med * 1e-3))))
    for k in (1, 4):
        res["on_over_off_time_k%d" % k] = round(res[name(True, k)]["us_per_agent_step_median"] / res[name(False, k)]["us_per_agent_step_median"], 3)
    return res


def frames(n):
    env = mixed_env("autoturn", n)
    fin = Finals(n)
    L, h = env.L, env.h
    T = 16
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    obs = torch.empty((T, n, 84, 84), dtype=torch.uint8, device="cuda")
    rew = torch.empty((T, n), dtype=torch.int32, device="cuda")
    done = torch.empty((T, n), dtype=torch.uint8, device="cuda")
    clock = [0]

    def rollout16():
        _lib.check(L.sf_rollout(h, T, None, 0, clock[0], vp(obs), vp(rew), vp(done), None, _lib.FLAG_RENDER, st))
        clock[0] += T
    reps = 2 if n >= 65536 else 10
    ms = alternate({name(on, k): (with_setting(env, fin, on, k, rollout16), reps, 2) for on, k in SETTINGS}, event_ms)
    res = summarise(ms, n, T, dict(n=n, gametype="autoturn", entry="sf_rollout, 84x84 frames", T=T, windows=WINDOWS))
    res["episode_ends_per_agent_step_last_call"] = round(float(done.sum()) / T, 1)
    env.close()
    del obs, rew, done, fin
    torch.cuda.empty_cache()
    return res


def host_step(n=4096):
    env = mixed_env("autoturn", n)
    fin = Finals(n)
    acts = np.random.RandomState(2).randint(env.num_actions, size=(64, n)).astype(np.int32)
    pos = [0]

    def step():
        env.step(acts[pos[0] % 64])
        pos[0] += 1
    ms = alternate({name(on, k): (with_setting(env, fin, on, k, step), 100, 10) for on, k in SETTINGS}, wall_ms)
    res = summarise(ms, n, 1, dict(n=n, gametype="autoturn", entry="SFVecEnv.step(np.ndarray), delta updates", windows=WINDOWS,
                                   steps_per_window=100))
    env.close()
    return res


def features(n=131072, T=64, kind="features"):
    env = mixed_env("youturn", n, render=False)
    fin = Finals(n)
    L, h, kid = env.L, env.h, _lib.OBS_TYPES[kind]
    nf = L.sf_num_features(h, kid)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    feat = torch.empty((T, n, nf), dtype=torch.float32, device="cuda")
    rew = torch.empty((T, n), dtype=torch.int32, device="cuda")
    done = torch.empty((T, n), dtype=torch.uint8, device="cuda")
    kill = torch.empty((T, n), dtype=torch.uint8, device="cuda")

    def rows():
        _lib.check(L.sf_rollout_features(h, kid, T, None, 0, 0, vp(feat), vp(rew), vp(done), vp(kill), None, 0, st))
    ms = alternate({name(on, k): (with_setting(env, fin, on, k, rows), 10, 2) for on, k in SETTINGS}, event_ms)
    res = summarise(ms, n, T, dict(n=n, gametype="youturn", entry="sf_rollout_features", kind=kind, columns=nf, T=T, windows=WINDOWS))
    env.close()
    del feat, rew, done, kill, fin
    torch.cuda.empty_cache()
    return res


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    res = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit_max_sm_clock=smi("name,power.limit,clocks.max.sm"))
    res["sm_clock_before"] = smi("clocks.sm")
    for n in (4096, 65536):
        res["rollout16_%d" % n] = frames(n)
        res["sm_clock_after_rollout16_%d" % n] = smi("clocks.sm")
        print(json.dumps(res["rollout16_%d" % n]), flush=True)
    res["host_step_4096"] = host_step()
    res["sm_clock_after_host_step_4096"] = smi("clocks.sm")
    print(json.dumps(res["host_step_4096"]), flush=True)
    res["features_131072"] = features()
    res["sm_clock_after_features"] = smi("clocks.sm")
    print(json.dumps(res["features_131072"]), flush=True)
    with open(os.path.join(out_dir, "r08_final_obs_n1.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1])
