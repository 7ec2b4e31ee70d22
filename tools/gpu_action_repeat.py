"""Action repeat (sf_set_action_repeat): what an agent step and a game tick cost at k = 1, 2, 4.
usage: python tools/gpu_action_repeat.py OUT_DIR   -> OUT_DIR/action_repeat.json

Autoturn envs at 4096 and 65 536, 400 state-only ticks first and clocks staggered over a whole episode (a mid-episode mix
with auto-resets inside the runs), synthetic actions:
  rollout16   sf_rollout T = 16 with 84x84 frames (k = 1: the fused kernel; k > 1: per agent step the repeat kernel and a
              draw launch)
  step        a loop of sf_step with frames, 16 calls per repetition
  host_step   SFVecEnv.step(np.ndarray) with delta updates (sf_step_host, SF_FLAG_HOST_DELTA), wall time
  split_k1    k = 1 only: sf_step without frames (the state-only kernel, T = 1) + sf_render, against `step` at k = 1: would the
              two-launch shape also suit the plain one-tick step?
Youturn envs at 131 072, 'features' (19 columns), T = 64: sf_rollout_features, and sf_rollout without frames for reference.
Device variants are timed with CUDA events, five windows per variant, the variants alternating window by window; the
host step with a host clock around windows that end in a device synchronise. Medians. ticks/s = agent steps/s x k: an
episode end cuts its agent step short, which at one end per 5295 ticks per env changes the count by < 0.1 %."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C  # noqa: E402

from spacefortress_b200 import SFVecEnv, _lib  # noqa: E402

END_TICK = 5295
WINDOWS = 5
KS = (1, 2, 4)


def smi(fields):
    return subprocess.run(["nvidia-smi", "--query-gpu=" + fields, "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().split("\n")[0]


def vp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def event_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def wall_ms(fn, reps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / reps


def alternate(variants, timer):
    """variants: name -> (fn, reps, warm-up calls); returns name -> [ms per call of every window]"""
    for fn, reps, warm in variants.values():
        for _ in range(warm):
            fn()
    torch.cuda.synchronize()
    ms = {v: [] for v in variants}
    for _ in range(WINDOWS):
        for v, (fn, reps, _) in variants.items():
            ms[v].append(timer(fn, reps))
    return ms


def mixed_env(gametype, n, **kw):
    env = SFVecEnv(gametype, num_envs=n, device=0, seeds=1, **kw)
    env.reset(to_numpy=False)
    env.rollout(400, action_seed=1, want=("done",))
    env.set_ticks((END_TICK - np.random.RandomState(0).randint(1, END_TICK, size=n)).astype(np.int32))
    return env


def with_repeat(env, k, fn):
    def run():
        _lib.check(env.L.sf_set_action_repeat(env.h, k))
        env.action_repeat = k
        fn()
    return run


def frames(n):
    env = mixed_env("autoturn", n)
    L, h = env.L, env.h
    T = 16
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    obs = torch.empty((T, n, 84, 84), dtype=torch.uint8, device="cuda")
    rew = torch.empty((T, n), dtype=torch.int32, device="cuda")
    done = torch.empty((T, n), dtype=torch.uint8, device="cuda")
    acts = torch.from_numpy(np.random.RandomState(1).randint(env.num_actions, size=(T, n)).astype(np.int32)).cuda()
    frame = torch.empty((n, 84, 84), dtype=torch.uint8, device="cuda")
    clock = [0]

    def rollout16():
        _lib.check(L.sf_rollout(h, T, None, 0, clock[0], vp(obs), vp(rew), vp(done), None, _lib.FLAG_RENDER, st))
        clock[0] += T

    def step16():
        for t in range(T):
            _lib.check(L.sf_step(h, vp(acts[t]), vp(obs[t]), vp(rew[t]), vp(done[t]), None, None, _lib.FLAG_RENDER, st))

    def split16():
        for t in range(T):
            _lib.check(L.sf_step(h, vp(acts[t]), None, vp(rew[t]), vp(done[t]), None, None, 0, st))
            _lib.check(L.sf_render(h, vp(frame), 0, st))

    big = n >= 65536
    variants = {}
    for k in KS:
        variants["rollout16_k%d" % k] = (with_repeat(env, k, rollout16), 2 if big else 10, 2)
        variants["step_k%d" % k] = (with_repeat(env, k, step16), 2 if big else 10, 2)
    variants["split_k1"] = (with_repeat(env, 1, split16), 2 if big else 10, 2)
    ms = alternate(variants, event_ms)
    res = dict(n=n, gametype="autoturn", T_per_call=T, windows=WINDOWS)
    for v, w in ms.items():
        k = 1 if v == "split_k1" else int(v.split("_k")[1])
        med = float(np.median(w))
        res[v] = dict(k=k, us_per_agent_step_median=round(med * 1e3 / T, 2), us_per_agent_step_windows=[round(x * 1e3 / T, 2) for x in w],
                      agent_steps_per_s=int(round(n * T / (med * 1e-3))), ticks_per_s=int(round(n * T * k / (med * 1e-3))))
    res["split_k1_over_step_k1_time"] = round(res["split_k1"]["us_per_agent_step_median"] / res["step_k1"]["us_per_agent_step_median"], 3)
    env.close()
    del obs, rew, done, acts, frame
    torch.cuda.empty_cache()
    return res


def host_step(n):
    env = mixed_env("autoturn", n)
    acts = np.random.RandomState(2).randint(env.num_actions, size=(64, n)).astype(np.int32)
    reps = 20 if n >= 65536 else 100
    pos = [0]

    def step():
        env.step(acts[pos[0] % 64])
        pos[0] += 1
    variants = {"host_step_k%d" % k: (with_repeat(env, k, step), reps, 10) for k in KS}
    ms = alternate(variants, wall_ms)
    res = dict(n=n, gametype="autoturn", delta_updates=True, windows=WINDOWS, steps_per_window=reps)
    for v, w in ms.items():
        k = int(v.split("_k")[1])
        med = float(np.median(w))
        res[v] = dict(k=k, us_per_agent_step_median=round(med * 1e3, 2), us_per_agent_step_windows=[round(x * 1e3, 2) for x in w],
                      agent_steps_per_s=int(round(n / (med * 1e-3))), ticks_per_s=int(round(n * k / (med * 1e-3))))
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

    def state_only():
        _lib.check(L.sf_rollout(h, T, None, 0, 0, None, vp(rew), vp(done), vp(kill), 0, st))
    variants = {}
    for k in KS:
        variants["features_k%d" % k] = (with_repeat(env, k, rows), 10, 2)
        variants["state_only_k%d" % k] = (with_repeat(env, k, state_only), 10, 2)
    ms = alternate(variants, event_ms)
    res = dict(n=n, gametype="youturn", kind=kind, columns=nf, T=T, windows=WINDOWS)
    for v, w in ms.items():
        k = int(v.split("_k")[1])
        med = float(np.median(w))
        res[v] = dict(k=k, ms_per_launch_median=round(med, 4), ms_per_launch_windows=[round(x, 4) for x in w],
                      agent_steps_per_s=int(round(n * T / (med * 1e-3))), ticks_per_s=int(round(n * T * k / (med * 1e-3))))
    env.close()
    del feat, rew, done, kill
    torch.cuda.empty_cache()
    return res


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    res = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit_max_sm_clock=smi("name,power.limit,clocks.max.sm"))
    for n in (4096, 65536):
        res["frames_%d" % n] = frames(n)
        res["sm_clock_after_frames_%d" % n] = smi("clocks.sm")
        print(json.dumps(res["frames_%d" % n]), flush=True)
        res["host_step_%d" % n] = host_step(n)
        res["sm_clock_after_host_step_%d" % n] = smi("clocks.sm")
        print(json.dumps(res["host_step_%d" % n]), flush=True)
    res["features_131072"] = features()
    res["sm_clock_after_features"] = smi("clocks.sm")
    print(json.dumps(res["features_131072"]), flush=True)
    with open(os.path.join(out_dir, "action_repeat.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1])
