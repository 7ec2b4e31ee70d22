"""Env blobs: time sf_save_envs / sf_load_envs against a device copy of the same bytes and against the host record path.
usage: python tools/gpu_env_blob_bench.py OUT_DIR   -> OUT_DIR/env_blob_bench.json

Per size (4096, 65 536 and 262 144 envs, youturn, 300 random steps first so that projectiles are in flight and
ships are dead): save and load with contiguous indices (None) and with a random permutation, timed with CUDA
events over >= 0.2 s of back-to-back calls after warm-up; `copy` is torch's device copy of the blob's bytes (read
+ write of k x 832 B, the same traffic as a save or a load moves on the blob side); `host` is get_state + set_state of
the same envs (synchronous, wall time, fewer repetitions). At 4096 envs blob and state sit in L2; at 262 144 envs
the blob (218 MB) and the state rows exceed the 126 MB L2."""
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

L2_BYTES = 126 * 2 ** 20


def timed(fn, min_s=0.2, min_calls=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    calls = min_calls
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= min_s * 1e3:
            return ms * 1e3 / calls, calls  # us per call
        calls *= max(2, int(min_s * 1e3 / max(ms, 1e-3)) + 1)


def where(touched):
    """blob + the state rows a call touches (about the blob's size again; the render caches are not touched)"""
    if touched < L2_BYTES / 2:
        return "L2 (blob + touched state %.0f MB)" % (touched / 2 ** 20)
    if touched < L2_BYTES:
        return "partly L2 (blob + touched state %.0f MB, L2 126 MB)" % (touched / 2 ** 20)
    return "HBM (blob + touched state %.0f MB exceed the 126 MB L2)" % (touched / 2 ** 20)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")[0]
    return q


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    res = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=gpu_info(), blob_bytes=_lib.ENV_BLOB_BYTES, sizes=[])
    print(res["nvidia_smi"])
    for n in (4096, 65536, 262144):
        env = SFVecEnv("youturn", num_envs=n, device=0, seeds=np.arange(1, n + 1), render=False)
        env.reset()
        rng = np.random.RandomState(0)
        acts = torch.from_numpy(rng.randint(env.num_actions, size=(300, n)).astype(np.int32)).cuda()
        env.rollout(300, actions=acts, want=("done",))
        torch.cuda.synchronize()
        perm = torch.from_numpy(rng.permutation(n).astype(np.int32)).cuda()
        blob = env.save_envs()
        blob2 = torch.empty_like(blob)
        ref = blob.clone()
        row = dict(n=n, blob_mb=blob.numel() / 1e6, state_mb=env.state_bytes() / 1e6,
                   where=where(2 * blob.numel()))
        h = env.h
        rej = torch.zeros(1, dtype=torch.int32, device="cuda")
        bp, b2p, pp, rp = blob.data_ptr(), blob2.data_ptr(), perm.data_ptr(), rej.data_ptr()
        Lb = env.L
        calls = {
            "save_contiguous": lambda: Lb.sf_save_envs(h, None, n, C.c_void_p(b2p), None),
            "save_permuted": lambda: Lb.sf_save_envs(h, C.c_void_p(pp), n, C.c_void_p(b2p), None),
            "load_contiguous": lambda: Lb.sf_load_envs(h, C.c_void_p(bp), None, n, C.c_void_p(rp), None),
            "load_permuted": lambda: Lb.sf_load_envs(h, C.c_void_p(bp), C.c_void_p(pp), n, C.c_void_p(rp), None),
            "copy": lambda: blob2.copy_(blob),
        }
        for k, fn in calls.items():
            if k != "copy":
                _lib.check(fn())
            us, c = timed(fn)
            row[k + "_us"] = round(us, 2)
            row[k + "_calls"] = c
            row[k + "_gbps"] = round(2 * blob.numel() / us / 1e3, 1)  # blob bytes once each way
        assert int(rej.item()) == 0
        env.load_envs(ref)
        assert torch.equal(env.save_envs(), ref)
        for k in ("save_contiguous", "save_permuted", "load_contiguous", "load_permuted"):
            row[k + "_over_copy"] = round(row[k + "_us"] / row["copy_us"], 3)
        # host record path of the same envs (synchronous; fewer envs timed at the largest size would change nothing)
        reps = 3 if n <= 65536 else 1
        t0 = time.perf_counter()
        for _ in range(reps):
            recs = env.get_state()
            env.set_state(recs)
        row["host_get_set_us"] = round((time.perf_counter() - t0) * 1e6 / reps, 1)
        row["host_over_save_plus_load"] = round(row["host_get_set_us"] / (row["save_contiguous_us"] + row["load_contiguous_us"]), 1)
        print(json.dumps(row))
        res["sizes"].append(row)
        env.close()
        del blob, blob2, ref
        torch.cuda.empty_cache()
    with open(os.path.join(out_dir, "env_blob_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1])
