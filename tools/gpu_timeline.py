"""Wall-clock timeline of the fused rollout (-DSF_TIMELINE probe, csrc/sf_probe.cuh; built here as build_variants/libsf_tl.so):
marks of warp 0 (stepper) and warp 1 (a drawing warp) of every block: kernel entry, tables loaded, first stage prepared,
arrival at / release from every stage hand-over (warp 0: wait for a free ring slot, warp 1: wait for a prepared stage), end.
usage: python tools/gpu_timeline.py [n] [T] [gametype]"""
import os, sys, ctypes as C
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
VARIANT = os.path.join(ROOT, "build_variants", "libsf_tl.so")
os.environ["SF_B200_LIB"] = VARIANT  # read when the package is imported
from spacefortress_b200 import build
build.build(out=VARIANT, defs="-DSF_TIMELINE")
import numpy as np, torch
from spacefortress_b200 import SFVecEnv, _lib
n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
T = int(sys.argv[2]) if len(sys.argv) > 2 else 20
gt = sys.argv[3] if len(sys.argv) > 3 else "autoturn"
env = SFVecEnv(gt, num_envs=n, device=0); env.reset(to_numpy=False)
env.rollout(400, want=("reward",))
out = {"obs": torch.empty((T, n, 1, 84, 84), dtype=torch.uint8, device="cuda")}
L = _lib.lib()
L.sf_timeline.restype = C.c_int; L.sf_timeline.argtypes = [C.c_void_p]
buf = np.zeros(160 * 2 * 96, np.uint64)
for rep in range(3):
    env.rollout(T, out=out); torch.cuda.synchronize()
    L.sf_timeline(buf.ctypes.data)
s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
s.record(); env.rollout(T, out=out); e.record(); torch.cuda.synchronize()
ms = s.elapsed_time(e)
tl = L.sf_timeline(buf.ctypes.data)
a = buf.reshape(160, 2, tl)
t = (a >> np.uint64(8)).astype(np.int64); tag = (a & np.uint64(255)).astype(np.int64)
used = [b for b in range(160) if tag[b, 0, 0] == 1]
t0 = min(t[b, w, 0] for b in used for w in (0, 1))
print("%s n=%d T=%d: launch %.1f us (events), %d blocks" % (gt, n, T, ms * 1e3, len(used)))
end = np.array([max(t[b, w][tag[b, w] == 7].max() for w in (0, 1)) - t0 for b in used]) / 1e3
start = np.array([t[b, 0, 0] - t0 for b in used]) / 1e3
init = np.array([t[b, 1][tag[b, 1] == 2][0] - t[b, 0, 0] for b in used]) / 1e3
first = np.array([t[b, 0][tag[b, 0] == 3][0] - t[b, 0, 0] for b in used]) / 1e3
print("block start (us after the first): min %.1f median %.1f max %.1f" % (start.min(), np.median(start), start.max()))
print("tables loaded after: median %.1f max %.1f us; first stage prepared after (from block start): median %.1f max %.1f us" % (np.median(init), init.max(), np.median(first), first.max()))
print("block end (us): min %.1f median %.1f max %.1f" % (end.min(), np.median(end), end.max()))
def stages(b, w):
    tt, gg = t[b, w], tag[b, w]
    arr = tt[gg == 4]; rel = tt[gg == 5]
    return arr, rel
for b in (used[0], used[len(used) // 2], used[int(np.argmax(end))]):
    a0, r0 = stages(b, 0); a1, r1 = stages(b, 1)
    print("block %d: stage barriers released at (us): %s" % (b, " ".join("%.1f" % ((x - t0) / 1e3) for x in r1)))
    print("   stepper busy per stage (us): %s" % " ".join("%.1f" % ((a0[k + 1] - r0[k]) / 1e3) for k in range(len(a0) - 1)))
    print("   drawer  busy per stage (us): %s" % " ".join("%.1f" % ((a1[k + 1] - r1[k]) / 1e3) for k in range(len(a1) - 1)))
    print("   drawer last stage %.1f us; stepper waits %.1f us, drawer waits %.1f us in total"
          % ((t[b, 1][tag[b, 1] == 7][-1] - r1[-1]) / 1e3, sum(r0[:len(a0)] - a0[:len(r0)]) / 1e3, sum(r1[:len(a1)] - a1[:len(r1)]) / 1e3))
durs = []
for b in used:
    a1, r1 = stages(b, 1)
    durs.append(np.diff(r1) / 1e3)
m = min(len(d) for d in durs)
D = np.array([d[:m] for d in durs])
print("stage duration over blocks (us): per stage median %s" % " ".join("%.1f" % x for x in np.median(D, 0)))
print("   per stage max    %s" % " ".join("%.1f" % x for x in D.max(0)))
print("   sum over stages: min %.1f median %.1f max %.1f" % (D.sum(1).min(), np.median(D.sum(1)), D.sum(1).max()))
