"""Host-buffer steps with every rank of a torchrun launch stepping at once (the host side of the box is shared):
per granule size of the delta updates, us per step (max over ranks) and env-steps/s of the whole box.
The granule is fixed when the library is built: each one is a variant build (-DSF_DELTA_GRANULE, build_variants/
libsf_granule<bytes>.so) that every rank measures in a child process of its own, which loads it through SF_B200_LIB.
usage: python [-m torch.distributed.run --nproc-per-node N] tools/gpu_host_step_ranks.py [granules ...]"""
import os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
if sys.argv[1:2] != ["--measure"]:
    from spacefortress_b200 import build
    for k, gran in enumerate(sys.argv[1:] or ["32"]):
        variant = os.path.join(ROOT, "build_variants", "libsf_granule%s.so" % gran)
        if local == 0:
            build.build(out=variant, defs="-DSF_DELTA_GRANULE=%s" % gran)
        # the children of one granule form their own process group (a store of their own on a port of their own); the
        # other ranks' children wait in it until the local rank 0 has built the variant
        env = dict(os.environ, SF_B200_LIB=variant)
        if world > 1:
            env.update(MASTER_PORT=str(int(os.environ["MASTER_PORT"]) + 1 + k), TORCHELASTIC_USE_AGENT_STORE="False")
        subprocess.run([sys.executable, os.path.abspath(__file__), "--measure", gran], env=env, check=True)
    sys.exit(0)

gran = sys.argv[2]
import numpy as np, torch, torch.distributed as dist
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dist.barrier()
from spacefortress_b200 import SFVecEnv
n, steps = 4096, 300
for gt in ("autoturn", "youturn"):
    env = SFVecEnv(gt, num_envs=n, device=local, first_global_env=rank * n)
    env.reset(); env.rollout(400, want=("reward",), action_seed=7); torch.cuda.synchronize()
    acts = np.random.RandomState(rank).randint(0, env.num_actions, size=(steps + 5, n)).astype(np.int32)
    for t in range(5):
        env.step(acts[t])
    s0 = env.host_delta_stats()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for t in range(steps):
        env.step(acts[5 + t])
    dt = time.perf_counter() - t0
    s1 = env.host_delta_stats()
    tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("granule %s B, %s, %d ranks: %.1f us/step (max over ranks), %.1f M env-steps/s, %.0f obs bytes/env-step"
              % (gran, gt, world, 1e6 * tt.item() / steps, n * world * steps / tt.item() / 1e6, (s1[0] - s0[0]) / steps / n), flush=True)
    env.close()
if world > 1:
    dist.destroy_process_group()
