"""A/B timing of library variants in one GPU session (interleaved runs): usage python tools/gpu_ab.py libA.so libB.so ...
Each run: frames of autoturn 4096 envs (T=20 x 9 launches, T=1 x 60 launches, T=64 x 3), youturn 65536 envs (T=16 x 3) and
youturn 16384 envs at action repeat 4 (T=16 x 5: state kernel + draw per agent step); state only (SF_AB_STATE=1, the
default): youturn and autoturn 65536 envs at T=1 and T=64, and 'features' rows of 131072 youturn envs at T=64."""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
code = r'''
import os, sys
sys.path.insert(0, os.getcwd())
import numpy as np, torch
from spacefortress_b200 import SFVecEnv
def run(gt, n, T, reps, warm=400, k=1):
    env = SFVecEnv(gt, num_envs=n, device=0, action_repeat=k); env.reset(to_numpy=False)
    env.rollout(warm, want=("reward",), action_seed=7)
    out = {"obs": torch.empty((T, n, 1, 84, 84), dtype=torch.uint8, device="cuda")}
    for _ in range(3): env.rollout(T, out=out, action_seed=7)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record(); env.rollout(T, out=out, action_seed=7); e.record(); torch.cuda.synchronize(); ms.append(s.elapsed_time(e))
    env.close()
    return np.array(ms)
res = []
for gt, n, T, reps, k in (("autoturn", 4096, 20, 9, 1), ("autoturn", 4096, 1, 60, 1), ("autoturn", 4096, 64, 3, 1), ("youturn", 65536, 16, 3, 1),
                         ("youturn", 16384, 16, 5, 4)):
    ms = run(gt, n, T, reps, k=k)
    res.append("%s/%d/T%d%s: med %.1f us (min %.1f) = %.1f M/s" % (gt[:4], n, T, "/k%d" % k if k > 1 else "", 1e3 * np.median(ms), 1e3 * ms.min(),
                                                              n * T / np.median(ms) / 1e3))
def run_state(gt, n, T, reps, obs_type="image"):
    env = SFVecEnv(gt, num_envs=n, device=0, render=False, obs_type=obs_type); env.reset(to_numpy=False)
    env.rollout(300, want=("reward",), action_seed=7)
    out = {"reward": torch.empty((T, n), dtype=torch.int32, device="cuda"), "done": torch.empty((T, n), dtype=torch.uint8, device="cuda")}
    if obs_type != "image":
        out["obs"] = torch.empty((T, n) + env.obs_shape, dtype=torch.float32, device="cuda")
    for _ in range(3): env.rollout(T, out=out, action_seed=7)
    torch.cuda.synchronize()
    s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps): env.rollout(T, out=out, action_seed=7)
    e.record(); torch.cuda.synchronize()
    env.close()
    return s.elapsed_time(e) / reps
if os.environ.get("SF_AB_STATE", "1") == "1":
    for gt, n, T, reps, obs_type in (("youturn", 65536, 1, 2000, "image"), ("autoturn", 65536, 1, 2000, "image"), ("youturn", 65536, 64, 50, "image"),
                                     ("autoturn", 65536, 64, 50, "image"), ("youturn", 131072, 64, 30, "features")):
        ms = run_state(gt, n, T, reps, obs_type)
        res.append("state %s/%d/T%d%s: %.1f us = %.2f G/s" % (gt[:4], n, T, "/" + obs_type if obs_type != "image" else "", 1e3 * ms, n * T / ms / 1e6))
print(os.path.basename(os.environ.get("SF_B200_LIB", "product")), " | ".join(res), flush=True)
'''
libs = sys.argv[1:]
# the card and its clock / power limit as read during the session (read only)
subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv"])
for rnd in range(int(os.environ.get("SF_AB_ROUNDS", "2"))):
    for lib in libs:
        env = dict(os.environ)
        if lib != "product":
            env["SF_B200_LIB"] = os.path.abspath(lib)
        subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT)
