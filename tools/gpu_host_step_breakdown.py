"""Where the time of one host-buffer step (SFVecEnv.step(np.ndarray) -> sf_step_host) goes: the Python wrapper, the C call,
a state-only C call and the device path's kernel. `native`: 92x90 frames, whose delta updates take the separate kernel.
usage: python tools/gpu_host_step_breakdown.py [n] [steps] [native]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from spacefortress_b200 import SFVecEnv, _lib

n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 300
native = sys.argv[3:4] == ["native"]
for gt in ("autoturn", "youturn"):
    env = SFVecEnv(gt, num_envs=n, device=0, native_obs=native)
    env.reset()
    env.rollout(400, want=("reward",), action_seed=7)
    torch.cuda.synchronize()
    acts = np.random.RandomState(0).randint(0, env.num_actions, size=(steps + 5, n)).astype(np.int32)
    for t in range(5):
        env.step(acts[t])
    s0 = env.host_delta_stats()
    t0 = time.perf_counter()
    for t in range(steps):
        env.step(acts[5 + t])
    t_wrap = (time.perf_counter() - t0) / steps
    s1 = env.host_delta_stats()
    p = env._np_ptr
    fl = env._flags | _lib.FLAG_HOST_DELTA
    t0 = time.perf_counter()
    for t in range(steps):
        env._np["actions"][:] = acts[5 + t]
        env.L.sf_step_host(env.h, p["actions"], p["obs"], p["reward"], p["done"], p["kill"], p["events"], fl)
    t_call = (time.perf_counter() - t0) / steps
    t0 = time.perf_counter()
    for t in range(steps):
        env.L.sf_step_host(env.h, p["actions"], None, p["reward"], p["done"], p["kill"], p["events"], fl & ~1)
    t_state = (time.perf_counter() - t0) / steps
    a_dev = torch.from_numpy(acts).cuda()
    env.step(a_dev[0]); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(steps):
        env.step(a_dev[5 + t])
    e1.record(); torch.cuda.synchronize()
    print("%s%s n=%d: wrapper %.1f us/step (%.1f M env-steps/s), C call %.1f us, state-only C call %.1f us, device-path kernel %.1f us, obs bytes/env-step %.0f"
          % (gt, " native" if native else "", n, 1e6 * t_wrap, n / t_wrap / 1e6, 1e6 * t_call, 1e6 * t_state, 1e3 * e0.elapsed_time(e1) / steps, (s1[0] - s0[0]) / steps / n), flush=True)
    env.close()
    for mode, what in (("ring", "SubprocVecEnv look-alike's default: fresh read-only arrays from a rotation of page-locked buffers"),
                       (True, "private writable copies every step")):
        lit = SFVecEnv(gt, num_envs=n, device=0, native_obs=native, copy_outputs=mode)
        lit.reset()
        for t in range(5):
            o, r, d, i = lit.step(acts[t])   # (bound like in the loop below: the ring's second buffer is allocated here)
        s0 = lit.host_delta_stats()
        t0 = time.perf_counter()
        for t in range(100):
            o, r, d, i = lit.step(acts[5 + t])
        dt = time.perf_counter() - t0
        s1 = lit.host_delta_stats()
        print("   copy_outputs=%r (%s): %.1f us/step (%.2f M env-steps/s), obs bytes/env-step %.0f"
              % (mode, what, 1e6 * dt / 100, n * 100 / dt / 1e6, (s1[0] - s0[0]) / 100 / n), flush=True)
        lit.close()
