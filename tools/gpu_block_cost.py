"""How well does the state of a block's envs predict the block's time in a T-step launch? (-DSF_TIMELINE probe, built
here as build_variants/libsf_tl.so.) Least-squares fit of the per-block duration on per-block sums of env features taken
BEFORE the launch. usage: python tools/gpu_block_cost.py [n] [T] [gametype]"""
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
EB = (n + 147) // 148 if n <= 148 * 32 else 32
X, Y = [], []
for rep in range(6):
    env.rollout(T, out=out); torch.cuda.synchronize()
    L.sf_timeline(buf.ctypes.data)
    st = env.get_state()
    feats = np.array([[1.0, 0.0 if r.ship_alive else 1.0, bin(r.missile_mask).count("1"), bin(r.shell_mask).count("1"), 1.0 if r.points >= 1 else 0.0,
                       1.0 if not r.fortress_alive else 0.0, (1.0 if (not r.ship_alive and r.ship_death_timer < 500) else 0.0)] for r in st])
    env.rollout(T, out=out); torch.cuda.synchronize()
    tl = L.sf_timeline(buf.ctypes.data)
    a = buf.reshape(160, 2, tl)
    t = (a >> np.uint64(8)).astype(np.int64); tag = (a & np.uint64(255)).astype(np.int64)
    nb = (n + EB - 1) // EB
    for b in range(min(nb, 148)):
        if n > 148 * 32:
            continue
        e0, e1 = b * EB, min((b + 1) * EB, n)
        if e1 - e0 < EB:
            continue
        dur = (t[b, 1][tag[b, 1] == 7][0] - t[b, 1][tag[b, 1] == 2][0]) / 1e3
        X.append(feats[e0:e1].sum(0)); Y.append(dur)
X, Y = np.array(X), np.array(Y)
names = ["envs", "dead", "missiles", "shells", "score>0", "fort dead", "freshly dead"]
print("%s n=%d T=%d: %d blocks; duration mean %.1f us, std %.1f us (%.1f %%), max/mean %.3f" % (gt, n, T, len(Y), Y.mean(), Y.std(), 100 * Y.std() / Y.mean(), Y.max() / Y.mean()))
Xc = X[:, 1:]
A = np.c_[np.ones(len(Y)), Xc]
coef, res, rk, sv = np.linalg.lstsq(A, Y, rcond=None)
pred = A @ coef
print("fit: const %.1f" % coef[0], " ".join("%s %.2f" % (nm, c) for nm, c in zip(names[1:], coef[1:])))
print("R^2 = %.3f; residual std %.1f us (%.1f %%)" % (1 - ((Y - pred) ** 2).sum() / ((Y - Y.mean()) ** 2).sum(), (Y - pred).std(), 100 * (Y - pred).std() / Y.mean()))
for k in range(1, X.shape[1]):
    print("   corr(duration, %s) = %.3f   (per-block mean %.2f, std %.2f)" % (names[k], np.corrcoef(X[:, k], Y)[0, 1], X[:, k].mean(), X[:, k].std()))
