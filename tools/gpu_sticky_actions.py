"""Sticky actions (sf_set_sticky_actions): what p > 0 costs, at action repeat k = 1 and 4.
usage: python tools/gpu_sticky_actions.py OUT_DIR   -> OUT_DIR/r07_sticky_actions_n1.json

Every variant is a setting (p, k) with p in {0, 0.25} and k in {1, 4}. p = 0 at k = 1 is the plain step (the fused
rollout kernel with frames); p > 0 takes the route of k > 1: the repeat kernel with its per-tick draws, and with frames
one draw launch per agent step.
  rollout16   autoturn, 4096 and 65 536 envs, sf_rollout T = 16 with 84x84 frames, synthetic actions
  host_step   autoturn, 4096 envs, SFVecEnv.step(np.ndarray) with delta updates (sf_step_host, SF_FLAG_HOST_DELTA), wall time
  features    youturn, 131 072 envs, sf_rollout_features 'features' (19 columns), T = 64
The envs first run 400 state-only ticks, then their clocks are staggered over a whole episode (a mid-episode mix with
auto-resets inside the runs). Device variants are timed with CUDA events, five windows per variant, the variants
alternating window by window; the host step with a host clock around windows that end in a device synchronise. Medians.
ticks/s = agent steps/s x k (an episode end cuts its agent step short: < 0.1 % at one end per 5295 ticks per env)."""
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

SETTINGS = [(p, k) for k in (1, 4) for p in (0.0, 0.25)]
STICKY_SEED = 1


def name(p, k):
    return "p%g_k%d" % (p, k)


def with_setting(env, p, k, fn):
    def run():
        _lib.check(env.L.sf_set_sticky_actions(env.h, p, STICKY_SEED))
        _lib.check(env.L.sf_set_action_repeat(env.h, k))
        env.action_repeat = k
        fn()
    return run


def summarise(ms, n, steps_per_call, res):
    """per variant: us per agent step (median and windows), agent steps/s, ticks/s"""
    for v, w in ms.items():
        k = int(v.split("_k")[1])
        med = float(np.median(w))
        res[v] = dict(k=k, p=float(v.split("_")[0][1:]), us_per_agent_step_median=round(med * 1e3 / steps_per_call, 2),
                      us_per_agent_step_windows=[round(x * 1e3 / steps_per_call, 2) for x in w],
                      agent_steps_per_s=int(round(n * steps_per_call / (med * 1e-3))),
                      ticks_per_s=int(round(n * steps_per_call * k / (med * 1e-3))))
    for k in (1, 4):
        res["p0.25_over_p0_time_k%d" % k] = round(res[name(0.25, k)]["us_per_agent_step_median"] / res[name(0.0, k)]["us_per_agent_step_median"], 3)
    return res


def frames(n):
    env = mixed_env("autoturn", n)
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
    ms = alternate({name(p, k): (with_setting(env, p, k, rollout16), reps, 2) for p, k in SETTINGS}, event_ms)
    res = summarise(ms, n, T, dict(n=n, gametype="autoturn", entry="sf_rollout, 84x84 frames", T=T, windows=WINDOWS))
    env.close()
    del obs, rew, done
    torch.cuda.empty_cache()
    return res


def host_step(n=4096):
    env = mixed_env("autoturn", n)
    acts = np.random.RandomState(2).randint(env.num_actions, size=(64, n)).astype(np.int32)
    pos = [0]

    def step():
        env.step(acts[pos[0] % 64])
        pos[0] += 1
    ms = alternate({name(p, k): (with_setting(env, p, k, step), 100, 10) for p, k in SETTINGS}, wall_ms)
    res = summarise(ms, n, 1, dict(n=n, gametype="autoturn", entry="SFVecEnv.step(np.ndarray), delta updates", windows=WINDOWS,
                                   steps_per_window=100))
    env.close()
    return res


def features(n=131072, T=64, kind="features"):
    env = mixed_env("youturn", n, render=False)
    L, h, kid = env.L, env.h, _lib.OBS_TYPES[kind]
    nf = L.sf_num_features(h, kid)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    feat = torch.empty((T, n, nf), dtype=torch.float32, device="cuda")
    rew = torch.empty((T, n), dtype=torch.int32, device="cuda")
    done = torch.empty((T, n), dtype=torch.uint8, device="cuda")
    kill = torch.empty((T, n), dtype=torch.uint8, device="cuda")

    def rows():
        _lib.check(L.sf_rollout_features(h, kid, T, None, 0, 0, vp(feat), vp(rew), vp(done), vp(kill), None, 0, st))
    ms = alternate({name(p, k): (with_setting(env, p, k, rows), 10, 2) for p, k in SETTINGS}, event_ms)
    res = summarise(ms, n, T, dict(n=n, gametype="youturn", entry="sf_rollout_features", kind=kind, columns=nf, T=T, windows=WINDOWS))
    env.close()
    del feat, rew, done, kill
    torch.cuda.empty_cache()
    return res


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    res = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit_max_sm_clock=smi("name,power.limit,clocks.max.sm"),
               sticky_seed=STICKY_SEED)
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
    with open(os.path.join(out_dir, "r07_sticky_actions_n1.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1])
