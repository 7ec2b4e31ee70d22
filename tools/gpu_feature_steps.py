"""Feature observations from the step kernel: what the rows cost, and what one launch saves over two.
usage: python tools/gpu_feature_steps.py OUT_DIR   -> OUT_DIR/feature_steps.json

1. Device rollout, 131 072 youturn envs ('features', 19 columns), T = 64, given actions, 400 state-only ticks first and
   clocks staggered over a whole episode (a mid-episode mix with auto-resets inside the launches):
     fused      sf_rollout_features: one launch, rows + reward / done / kill
     two_launch 64 x (sf_step without frames + sf_features): the path feature agents had before
     state_only sf_rollout without frames: the same step, no rows (the price of the rows is fused - state_only)
   Timed with CUDA events, five windows of back-to-back calls per variant, the variants alternating; medians.
   Bytes written per env-step are the outputs' bytes from their shapes (the env state is read and written by every
   launch in every variant and is not counted).
2. Host step, 4096 envs: SFVecEnv(obs_type="features").step(np.ndarray) (sf_step_host_features into a page-locked
   buffer + one host copy) against the sequence step() ran before (sf_step_host, sf_features on torch's stream,
   .cpu().numpy(), and the device synchronise the next step started with), rebuilt here from the same C-ABI. Wall time
   per step, five alternating windows of 500 steps; medians."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from spacefortress_b200 import SFVecEnv, _lib  # noqa: E402

END_TICK = 5295
WINDOWS = 5


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


def device_rollout(n=131072, T=64, kind="features"):
    env = SFVecEnv("youturn", num_envs=n, device=0, render=False, seeds=1)
    env.reset()
    env.rollout(400, action_seed=1, want=("done",))
    env.set_ticks((END_TICK - np.random.RandomState(0).randint(1, END_TICK, size=n)).astype(np.int32))
    L, h, k = env.L, env.h, _lib.OBS_TYPES[kind]
    nf = L.sf_num_features(h, k)
    acts = torch.from_numpy(np.random.RandomState(1).randint(env.num_actions, size=(T, n)).astype(np.int32)).cuda()
    feat = torch.empty((T, n, nf), dtype=torch.float32, device="cuda")
    rew = torch.empty((T, n), dtype=torch.int32, device="cuda")
    done = torch.empty((T, n), dtype=torch.uint8, device="cuda")
    kill = torch.empty((T, n), dtype=torch.uint8, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    fp, ap, rp, dp, kp = (C.c_void_p(x.data_ptr()) for x in (feat, acts, rew, done, kill))

    def fused():
        _lib.check(L.sf_rollout_features(h, k, T, ap, 0, 0, fp, rp, dp, kp, None, 0, st))

    def two_launch():
        for t in range(T):
            _lib.check(L.sf_step(h, vp(acts[t]), None, vp(rew[t]), vp(done[t]), vp(kill[t]), None, 0, st))
            _lib.check(L.sf_features(h, k, vp(feat[t]), st))

    def state_only():
        _lib.check(L.sf_rollout(h, T, ap, 0, 0, None, rp, dp, kp, 0, st))

    variants = dict(fused=fused, two_launch=two_launch, state_only=state_only)
    for fn in variants.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    reps = dict(fused=20, two_launch=10, state_only=20)
    ms = {v: [] for v in variants}
    for _ in range(WINDOWS):
        for v, fn in variants.items():
            ms[v].append(event_ms(fn, reps[v]))
    out_bytes = dict(fused=nf * 4 + 4 + 1 + 1, two_launch=nf * 4 + 4 + 1 + 1, state_only=4 + 1 + 1)
    res = dict(n=n, T=T, kind=kind, columns=nf, gametype="youturn", actions="given [T][n]", windows=WINDOWS, reps_per_window=reps)
    for v in variants:
        med = float(np.median(ms[v]))
        res[v] = dict(ms_per_launch_median=round(med, 4), ms_per_launch_windows=[round(x, 4) for x in ms[v]],
                      env_steps_per_s=int(round(n * T / (med * 1e-3))), output_bytes_per_env_step=out_bytes[v],
                      output_gb_per_s=round(n * T * out_bytes[v] / (med * 1e-3) / 1e9, 1))
    res["fused_over_two_launch_speedup"] = round(res["two_launch"]["ms_per_launch_median"] / res["fused"]["ms_per_launch_median"], 3)
    res["fused_over_state_only_time"] = round(res["fused"]["ms_per_launch_median"] / res["state_only"]["ms_per_launch_median"], 3)
    env.close()
    del feat, acts, rew, done, kill
    torch.cuda.empty_cache()
    return res


def host_step(n=4096, kind="features", steps=500):
    env = SFVecEnv("youturn", num_envs=n, device=0, obs_type=kind, seeds=1)
    env.reset()
    env.set_ticks((END_TICK - np.random.RandomState(0).randint(1, END_TICK, size=n)).astype(np.int32))
    rng = np.random.RandomState(2)
    acts = rng.randint(env.num_actions, size=(steps, n)).astype(np.int32)
    L, h, k = env.L, env.h, _lib.OBS_TYPES[kind]
    nf = env.num_features
    b = env._np_bufs()
    p = env._np_ptr
    flags = env._feature_flags()

    def new(a):
        return env.step(a)[0]

    def old(a):  # step() before sf_step_host_features
        torch.cuda.synchronize()  # the device work of the previous step's sf_features (_device_work)
        b["actions"][:] = a
        _lib.check(L.sf_step_host(h, p["actions"], None, p["reward"], p["done"], p["kill"], p["events"], flags))
        out = torch.empty((n, nf), dtype=torch.float32, device="cuda")
        _lib.check(L.sf_features(h, k, C.c_void_p(out.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return out.cpu().numpy()

    variants = dict(new=new, old=old)
    for fn in variants.values():
        for t in range(20):
            fn(acts[t])
    us = {v: [] for v in variants}
    for _ in range(WINDOWS):
        for v, fn in variants.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for t in range(steps):
                fn(acts[t])
            torch.cuda.synchronize()
            us[v].append((time.perf_counter() - t0) * 1e6 / steps)
    res = dict(n=n, kind=kind, columns=nf, steps_per_window=steps, windows=WINDOWS)
    for v in variants:
        res[v] = dict(us_per_step_median=round(float(np.median(us[v])), 2), us_per_step_windows=[round(x, 2) for x in us[v]])
    res["old_over_new"] = round(res["old"]["us_per_step_median"] / res["new"]["us_per_step_median"], 3)
    env.close()
    return res


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    res = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit_max_sm_clock=smi("name,power.limit,clocks.max.sm"))
    res["device_rollout"] = device_rollout()
    res["sm_clock_after_device_rollout"] = smi("clocks.sm")
    print(json.dumps(res["device_rollout"]))
    res["host_step"] = host_step()
    res["sm_clock_after_host_step"] = smi("clocks.sm")
    print(json.dumps(res["host_step"]))
    with open(os.path.join(out_dir, "feature_steps.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1])
