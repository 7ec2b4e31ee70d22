"""Cycles the warps spend at the block barriers (-DSF_BARRIER_TIMING probe, csrc/sf_probe.cuh: one clock pair + one global
atomic per warp and barrier, nothing else). Builds the probe as build_variants/libsf_bt.so and runs it; the product library
is not touched. usage: python tools/gpu_barrier_timing.py [n] [gametype]"""
import os, sys, ctypes as C
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
VARIANT = os.path.join(ROOT, "build_variants", "libsf_bt.so")
os.environ["SF_B200_LIB"] = VARIANT  # read when the package is imported
from spacefortress_b200 import build
build.build(out=VARIANT, defs="-DSF_BARRIER_TIMING")
import torch
from spacefortress_b200 import SFVecEnv, _lib
n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
gt = sys.argv[2] if len(sys.argv) > 2 else "autoturn"
T = 64
env = SFVecEnv(gt, num_envs=n, device=0); env.reset(to_numpy=False)
env.rollout(300, want=("reward",))
out = {"obs": torch.empty((T, n, 1, 84, 84), dtype=torch.uint8, device="cuda")}
env.rollout(T, out=out); torch.cuda.synchronize()
L = _lib.lib(); buf = (C.c_ulonglong * 16)()
L.sf_barrier_cycles.restype = C.c_int; L.sf_barrier_cycles.argtypes = [C.c_void_p, C.c_int]
L.sf_barrier_cycles(buf, 1)
s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
s.record(); env.rollout(T, out=out); e.record(); torch.cuda.synchronize()
L.sf_barrier_cycles(buf, 1)
ms = s.elapsed_time(e); v = list(buf)
blocks = min(148, (n + 31) // 32 if n > 148 * 32 else 147)
cyc = ms * 1e-3 * 1.965e9
W = 24
print("%s n=%d: launch %.3f ms = %.0f cycles; %.3e steps/s" % (gt, n, ms, cyc, n * T / ms * 1e3))
print("per drawing warp: waiting for a prepared stage (full barriers) %.1f %%, drawing-warp barriers %.1f %% of the launch; stepping warp waiting for a free ring slot (empty barriers) %.1f %%"
      % (100 * v[0] / (blocks * (W - 1)) / cyc, 100 * v[1] / (blocks * (W - 1)) / cyc, 100 * v[2] / blocks / cyc))
print("stepping warp, share of the launch: steps %.1f %%, memo state %.1f %%, round scans %.1f %%, stroke gathering %.1f %%, stage control words %.1f %%"
      % tuple(100 * v[k] / blocks / cyc for k in (3, 4, 5, 6, 7)))
print("step sections, cycles per tick and block: load %.0f | keys + respawn %.0f | ship %.0f | fortress %.0f | shells %.0f | missiles %.0f | timers + shaping %.0f | outputs + store + record %.0f"
      % tuple(v[k] / blocks / T for k in (8, 9, 10, 11, 12, 13, 14, 15)))
