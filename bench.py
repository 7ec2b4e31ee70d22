#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (env step + 84x84 render + auto-reset).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--envs-per-gpu E] [--skip-configs]
                  [--dump-outputs DIR]

Metric (BASELINE.json): env-steps/sec with 84x84 obs; headline workload = configs[1]: autoturn, 4096 batched envs per
GPU, 84x84 grayscale obs, random actions (weak scaling: every rank owns its own slab of 4096 envs; no data-path
collective).

One "step" = one pass of the hot path over the whole batch (one env-step of every env). The K timed steps (--steps K)
run as back-to-back launches of the fused multi-step kernel (sf_rollout, up to LAUNCH_STEPS steps per launch, one output
buffer reused; actions come from the on-device counter-hash policy, so inputs are resident). The whole run of K steps is
bracketed by barrier + synchronize and timed with CUDA events on the launching stream, max over ranks; the default K
covers about 0.35 s on a B200. Before it run `--presteps` state-only ticks and W warm-up steps, none of them timed.
Env seeds and actions are fixed by --seed, so the same arguments give the same inputs in every run, and
`--dump-outputs DIR` writes what the last timed step returned (see dump_outputs) to compare two builds output for output.
`e2e` is the same metric through the numpy drop-in API (SFVecEnv.step(np.ndarray) -> sf_step_host):
host actions in, host observations out, transfers inside the timed region: `e2e.value` with the delta updates of the
page-locked observation buffer (SF_FLAG_HOST_DELTA, the default), `e2e.drop_in_ring` with the fresh-array contract of the
SubprocVecEnv look-alike, `e2e.full_copy` with whole frames copied every step, next to a plain pinned device->host
copy probe run by every rank at the same time. `roofline` is for the dominant (only) kernel. `configs` holds the other
BASELINE.json configs measured in the same run (C3: 65 536-env on-device rollout with the SF-GRU policy, C4: 131 072
envs/GPU state-only with both game types, C5: 262 144 envs/GPU with staggered episode ends and the episode-stat
all-reduce inside the timed loop). `cpu_baseline` / `--impl reference` time the reference's own CPU implementation on
the host cores (see cpu_arm / cpu_pipe_arm).
"""
import argparse
import atexit
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
GAMETYPE = "autoturn"
METRIC = "env-steps/sec with 84x84 obs"
B_RENDER = 84 * 84 + 10 + 2 * 648  # SURVEY.md §8(d): obs + action/reward/done/info + state read+write = 8362 B
B_STATE = 10 + 2 * 648             # render off: 1306 B
WORKLOAD = "autoturn, 4096 batched envs per GPU, 84x84 grayscale obs, random actions (BASELINE.json configs[1])"
LAUNCH_STEPS = 64                  # steps per launch of the fused kernel in the timed run
DUMP_ENVS = 2048                   # env rows kept by --dump-outputs: 2048 x (7056 + 3) float32 = 57.8 MB, under 64 MB


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU implementation of the path on the host cores
# ------------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    kind, gametype, seed, steps, render = args
    import numpy as np
    from oracle.oracle import OracleEnv, RefEnv
    helper = OracleEnv(gametype, 1)
    rng = np.random.RandomState(seed)
    km = np.array([helper.keymask(a) for a in rng.randint(0, helper.num_actions(1), steps)], np.uint8)
    env = RefEnv(gametype, 1) if kind == "reference" else OracleEnv(gametype, 1)
    t0 = time.perf_counter()
    env.run(km, render=render)
    return time.perf_counter() - t0


def cpu_arm(steps_per_core, cores=None, render=True):
    """One process per host core (the SubprocVecEnv layout of rl/train.py:30-34, WITHOUT the per-step pipe round
    trip: every worker free-runs), each running `steps_per_core` env steps of: the UNMODIFIED reference core compiled
    from /root/reference (oracle/_ref: key events, Game::stepOneTick, shaping, auto-reset) + a frame per step.
    libcairo cannot be built offline, so the frame is drawn by the restated renderer (oracle/sf_draw_oracle.c, with
    the static background and glyph masks cached like cairo's own caches) + INTER_AREA 84x84. render=False: the
    core alone (no frame)."""
    from oracle.oracle import ref_available
    kind = "reference" if ref_available() else "port"
    cores = cores or os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(kind, GAMETYPE, 0, 64, render)] * cores)  # warm-up: page in the libraries
        t0 = time.perf_counter()
        pool.map(_cpu_worker, [(kind, GAMETYPE, 100 + i, steps_per_core, render) for i in range(cores)])
        wall = time.perf_counter() - t0
    what = "frame by the restated renderer (no cairo offline) + INTER_AREA" if render else "no frame (core only)"
    return dict(value=steps_per_core * cores / wall, unit="env-steps/s", cores=cores, kind=kind,
                sample="%d procs x %d steps of %s, tick by the %s, %s; no per-step pipe; %.1f s wall"
                       % (cores, steps_per_core, GAMETYPE, "compiled reference core" if kind == "reference" else "oracle port", what, wall)), wall


def _pipe_worker(remote, kind, gametype, nenv, seed0):
    """gym_vecenv's worker loop (SURVEY.md §3.4) for a GROUP of envs: recv ('step', actions) -> step every env, auto-reset
    the finished ones, send (obs, rews, dones, infos) back through the pipe."""
    import ctypes as C
    import numpy as np
    from oracle.oracle import OracleEnv, RefEnv, oracle_lib
    helper = OracleEnv(gametype, 1)
    envs = [(RefEnv(gametype, 1) if kind == "reference" else OracleEnv(gametype, 1)) for _ in range(nenv)]
    obs = np.zeros((nenv, 1, 84, 84), np.uint8)
    rews, dones, infos = np.zeros(nenv, np.int64), np.zeros(nenv, bool), [False] * nenv
    draw = oracle_lib().sfo_draw_obs
    try:
        while True:
            cmd, data = remote.recv()
            if cmd == "step":
                for i, e in enumerate(envs):
                    r, d, k, _ = e.step(helper.keymask(int(data[i])))
                    if d:
                        e.reset()
                    st = e.get_state()
                    draw(C.byref(st), obs[i].ctypes.data)
                    rews[i], dones[i], infos[i] = r, d, k
                remote.send((obs, rews, dones, tuple(infos)))
            elif cmd == "reset":
                for i, e in enumerate(envs):
                    e.reset()
                    st = e.get_state()
                    draw(C.byref(st), obs[i].ctypes.data)
                remote.send(obs)
            else:
                remote.close()
                break
    except (EOFError, KeyboardInterrupt):
        pass


def cpu_pipe_arm(n_envs, steps, cores=None):
    """The CPU baseline as north_star words it: a gym_vecenv SubprocVecEnv across the box's host cores (rl/train.py:30-34,80):
    one worker process per env group, a multiprocessing.Pipe round trip per step (actions out, observations / rewards /
    dones / infos back, np.stack in the parent), auto-reset inside the worker. The reference spawns one process PER ENV;
    with n_envs >> cores that only adds context switches, so the envs are grouped one group per core (faster: the
    conservative choice). Tick by the compiled reference core, frame as in cpu_arm."""
    import numpy as np
    from oracle.oracle import OracleEnv, ref_available
    kind = "reference" if ref_available() else "port"
    cores = cores or os.cpu_count() or 1
    groups = [n_envs // cores + (1 if i < n_envs % cores else 0) for i in range(cores)]
    groups = [g for g in groups if g > 0]
    ctx = mp.get_context("spawn")
    pipes = [ctx.Pipe() for _ in groups]
    procs = [ctx.Process(target=_pipe_worker, args=(w, kind, GAMETYPE, g, 1), daemon=True) for (p, w), g in zip(pipes, groups)]
    for p in procs:
        p.start()
    remotes = [p for p, w in pipes]
    na = OracleEnv(GAMETYPE, 1).num_actions(1)
    rng = np.random.RandomState(0)

    def step(actions):
        o = 0
        for r, g in zip(remotes, groups):
            r.send(("step", actions[o:o + g]))
            o += g
        res = [r.recv() for r in remotes]
        return np.concatenate([x[0] for x in res]), np.concatenate([x[1] for x in res]), np.concatenate([x[2] for x in res]), sum((x[3] for x in res), ())
    for r in remotes:
        r.send(("reset", None))
    np.concatenate([r.recv() for r in remotes])
    for _ in range(2):
        step(rng.randint(0, na, n_envs))
    t0 = time.perf_counter()
    for _ in range(steps):
        obs, rew, done, info = step(rng.randint(0, na, n_envs))
    wall = time.perf_counter() - t0
    for r in remotes:
        r.send(("close", None))
    for p in procs:
        p.join(timeout=5)
    return dict(value=n_envs * steps / wall, unit="env-steps/s", cores=cores, kind=kind,
                sample="SubprocVecEnv protocol: %d worker procs x %d envs, %d steps of %s with a Pipe round trip per step "
                       "(obs %d B/env back), tick by the %s, frame by the restated renderer + INTER_AREA; %.1f s wall"
                       % (len(groups), groups[0], steps, GAMETYPE, 84 * 84, "compiled reference core" if kind == "reference" else "oracle port", wall))


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    # each "step" is a bounded sample of the workload: `per_core` env-steps per core-process
    per_core = 3000
    vals = []
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_arm(200, cores)
    t_all = time.perf_counter()
    for _ in range(max(1, min(args.steps, 3))):
        b, wall = cpu_arm(per_core, cores)
        vals.append(b)
    best = max(vals, key=lambda b: b["value"])
    extra = {}
    try:
        extra["subproc_pipe_protocol"] = cpu_pipe_arm(ENVS_PER_GPU, 12, cores)       # what north_star names; slower than `value`
        extra["core_only_no_frame"], _ = cpu_arm(40000, cores, render=False)
    except Exception as ex:
        extra["error"] = repr(ex)
    line = {
        "impl": "reference", "metric": METRIC, "value": best["value"], "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * ENVS_PER_GPU * args.gpus / best["value"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs": ENVS_PER_GPU * args.gpus, "gametype": GAMETYPE,
                   "note": "value = the FASTER of the CPU arms (free-running workers, no per-step pipe): the conservative denominator; "
                           "the SubprocVecEnv-protocol arm and the core-only number are under cpu_arms"},
        "cpu_baseline": best, "cpu_arms": extra,
        "e2e": {"value": best["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "wall_s": time.perf_counter() - t_all,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """Samples the SM clock and throttle reasons of one GPU every 50 ms (nvidia-smi queries) while a measurement runs.
    The samples go to an anonymous temporary file: the tree may be read-only."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.f = tempfile.TemporaryFile(mode="w+")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self._end)  # a measurement that raises before stop() must not leave the sampler running
        except Exception:
            self.proc = None
        return self

    def _end(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self._end()
        atexit.unregister(self._end)
        self.proc = None
        self.f.seek(0)
        lines = self.f.read().splitlines()
        self.f.close()
        sm, reasons, smmax = [], set(), None
        for ln in lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); smmax = float(p[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=smmax, reasons=sorted(reasons), samples=len(sm))
        return out


def _stats(ms):
    s = sorted(ms)
    return {"median": s[len(s) // 2], "min": s[0], "max": s[-1], "n": len(s)}


def dump_outputs(path, last):
    """--dump-outputs: writes `last` (what sf_rollout returned for the last timed step: obs [N,1,84,84], reward / done /
    kill [N]) to path/<name>.npy as float32, which holds every value exactly. Above DUMP_ENVS envs only a fixed, seeded
    sample of env rows is kept, the same rows in every file."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    n = next(iter(last.values())).shape[0]
    rows = np.arange(n) if n <= DUMP_ENVS else np.sort(np.random.RandomState(0).choice(n, DUMP_ENVS, replace=False))
    for name, t in last.items():
        keep = t[torch.from_numpy(rows).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), keep.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------------
# the other BASELINE.json configs, measured in the same run
# ------------------------------------------------------------------------------------------------------
def config_c3(torch, dist, rank, local, world, args, peak):
    """configs[2]: youturn, 65 536 envs, frame-stack 4, fully on-device 128-step rollout with the SF-GRU policy."""
    from spacefortress_b200 import SFVecEnv
    from spacefortress_b200.rollout import OnDeviceRollout, SFGRUPolicy
    from spacefortress_b200.ppo import PPOLearner
    n, T = args.c3_envs, args.c3_steps
    dev = torch.device("cuda", local)
    res = {"workload": "youturn, %d envs/GPU, frame-stack 4, %d-step on-device rollout, SF-GRU policy (BASELINE.json configs[2])" % (n, T)}
    clocks = ClockSampler(local).start()
    env = SFVecEnv("youturn", num_envs=n, device=local, first_global_env=rank * n)
    policy = SFGRUPolicy(env.num_actions).to(dev).eval().bfloat16().to(memory_format=torch.channels_last)
    ro = OnDeviceRollout(env, policy, num_steps=T, graph=True)
    ro.collect(); torch.cuda.synchronize()           # warm-up + graph capture
    # env only: the fused rollout kernel replaying the recorded actions into the same frame buffer (one launch of T steps)
    obs = ro.frames[ro.S:ro.S + T].unsqueeze(2)
    ms = []
    for _ in range(max(3, int(0.35 / 0.06))):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        env.rollout(T, actions=ro.actions, out={"obs": obs})
        e1.record(); torch.cuda.synchronize(); ms.append(e0.elapsed_time(e1))
    st = _stats(ms)
    res["env_only"] = {"value": n * world * T / (st["median"] * 1e-3), "unit": "env-steps/s", "launch_ms": st,
                       "roofline_frac": n * T * B_RENDER / (st["median"] * 1e-3) / 1e9 / peak}
    # env + policy: the captured per-step graphs (policy input kernel -> cuDNN/cuBLAS policy -> sf_step -> bookkeeping)
    ms = []
    for _ in range(2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(); ro.collect(); e1.record(); torch.cuda.synchronize(); ms.append(e0.elapsed_time(e1))
    st = _stats(ms)
    res["env_plus_policy_bf16"] = {"value": n * world * T / (st["min"] * 1e-3), "unit": "env-steps/s", "rollout_ms": st, "cuda_graphs": True,
                                   "policy": "SF-GRU bf16 channels_last, first layer fed by sf_policy_input"}
    # the learner on the same rollout: a bounded sample (one epoch over `c3_update_envs` envs x T steps, chunked)
    try:
        sub = min(args.c3_update_envs, n)
        fp32 = SFGRUPolicy(env.num_actions).to(dev)
        fp32.load_state_dict({k: v.float() for k, v in policy.state_dict().items()})

        class Slice(object):  # the first `sub` envs of the rollout
            rewards, dones, values, logps, actions = ro.rewards[:, :sub], ro.dones[:, :sub], ro.values[:, :sub], ro.logps[:, :sub], ro.actions[:, :sub]
            state0, mask0, state, mask = ro.state0[:sub].float(), ro.mask0[:sub].float(), ro.state[:sub].float(), ro.mask[:sub].float()
            states_hist = ro.states_hist[:, :sub].float()
            stack = staticmethod(lambda t: ro.stack(t)[:sub])
        learner = PPOLearner(fp32, ppo_epoch=1, num_mini_batch=4)
        torch.backends.cudnn.allow_tf32 = True; torch.backends.cuda.matmul.allow_tf32 = True
        learner.update(Slice, env_chunk=256)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(); learner.update(Slice, env_chunk=256); e1.record(); torch.cuda.synchronize()
        ums = e0.elapsed_time(e1)
        res["ppo_update_tf32"] = {"value": sub * T / (ums * 1e-3), "unit": "samples/s (one epoch, 4 minibatches, forward + backward + Adam)",
                                  "sample": "%d envs x %d steps of the rollout above, evaluated in chunks of 256 envs" % (sub, T), "ms": ums}
    except Exception as ex:
        res["ppo_update_tf32"] = {"error": repr(ex)}
    del ro
    # fp32 (TF32 matmul/conv) policy beside bf16: the reference's ACNet is fp32 (rl/networks.py:20-49)
    try:
        env2 = SFVecEnv("youturn", num_envs=n, device=local, first_global_env=rank * n)
        p32 = SFGRUPolicy(env2.num_actions).to(dev).eval()
        ro2 = OnDeviceRollout(env2, p32, num_steps=args.c3_fp32_steps, graph=True)
        ro2.collect(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); ro2.collect(); e1.record(); torch.cuda.synchronize()
        res["env_plus_policy_tf32"] = {"value": n * world * args.c3_fp32_steps / (e0.elapsed_time(e1) * 1e-3), "unit": "env-steps/s",
                                       "rollout_ms": e0.elapsed_time(e1), "steps": args.c3_fp32_steps, "policy": "SF-GRU fp32 weights, TF32 conv / matmul"}
        del ro2
        env2.close()
    except Exception as ex:
        res["env_plus_policy_tf32"] = {"error": repr(ex)}
    env.close()
    torch.cuda.empty_cache()
    res["clocks"] = clocks.stop()
    return res


def config_c4(torch, dist, rank, local, world, args, peak):
    """configs[3]: autoturn + youturn, 131 072 envs/GPU (half / half), state-only (render off)."""
    from spacefortress_b200 import SFVecEnv
    n = args.c4_envs // 2
    res = {"workload": "autoturn + youturn, %d envs/GPU (half / half), state-only step (BASELINE.json configs[3]; 1M envs at 8 GPUs)" % (2 * n)}
    clocks = ClockSampler(local).start()
    envs = [SFVecEnv(gt, num_envs=n, device=local, render=False, first_global_env=(2 * rank + k) * n) for k, gt in enumerate(("autoturn", "youturn"))]
    for e in envs:
        e.reset(to_numpy=False)
        e.rollout(300, want=("reward",))
    outs = [{"reward": torch.empty((64, n), dtype=torch.int32, device=torch.device("cuda", local)),
             "done": torch.empty((64, n), dtype=torch.uint8, device=torch.device("cuda", local))} for _ in envs]
    for T, reps in ((1, 4000), (64, 100)):
        o = [{k: v[:T] for k, v in d.items()} for d in outs]
        for e, oo in zip(envs, o):
            e.rollout(T, out=oo)
        # T = 1 launches take ~10 us each: replayed from a CUDA graph of 50 launch pairs so that the host's launch rate
        # does not bound the number (the state-only kernel is what is measured)
        graph, per_graph = None, 1
        if T == 1:
            try:
                torch.cuda.synchronize()
                side = torch.cuda.Stream(device=torch.device("cuda", local))
                side.wait_stream(torch.cuda.current_stream())
                graph, per_graph = torch.cuda.CUDAGraph(), 50
                t_env = [e._t for e in envs]
                with torch.cuda.graph(graph, stream=side):
                    for _ in range(per_graph):
                        for e, oo in zip(envs, o):
                            e.rollout(T, out=oo)
                for e, t0 in zip(envs, t_env):
                    e._t = t0
                torch.cuda.synchronize()
            except Exception:
                graph, per_graph = None, 1
        ms = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(); e0.record()
            for _ in range(reps // per_graph):
                if graph is not None:
                    graph.replay()
                else:
                    for e, oo in zip(envs, o):
                        e.rollout(T, out=oo)
            e1.record(); torch.cuda.synchronize(); ms.append(e0.elapsed_time(e1))
        st = _stats(ms)
        if world > 1:
            t = torch.tensor([st["median"]], dtype=torch.float64, device=torch.device("cuda", local)); dist.all_reduce(t, op=dist.ReduceOp.MAX); st["median"] = float(t.item())
        steps = 2 * n * T * reps
        ent = {"value": steps * world / (st["median"] * 1e-3), "unit": "env-steps/s", "region_ms": st, "launches_per_region": 2 * reps,
               "launched_from": "a CUDA graph of %d launch pairs" % per_graph if graph is not None else "the host, one call per launch"}
        if T == 1:  # the per-step byte model (state read + write every step) only describes T = 1
            ent["roofline_frac"] = steps * B_STATE / (st["median"] * 1e-3) / 1e9 / peak
            ent["note"] = "the %.0f MB of state of this config stay resident in the 126 MB L2, so a fraction of the HBM peak above 1 is possible" % (2 * n * 648 / 1e6)
        else:
            ent["note"] = "the state stays in registers across the 64 ticks of a launch: SURVEY \u00a78(d)'s 1306 B/step model does not describe it"
        res["T%d" % T] = ent
        del graph
    for e in envs:
        e.close()
    res["clocks"] = clocks.stop()
    return res


def config_c5(torch, dist, rank, local, world, args, peak):
    """configs[4]: youturn, 262 144 envs/GPU, render + auto-reset under episode-length variance (staggered clocks), with
    the episode-stat all-reduce (NCCL when world > 1) INSIDE the timed loop, once per rollout."""
    import numpy as np
    from spacefortress_b200 import SFVecEnv
    n, T = args.c5_envs, args.c5_steps
    dev = torch.device("cuda", local)
    res = {"workload": "youturn, %d envs/GPU, render + auto-reset, episode clocks staggered over the whole episode, %d-step rollouts, "
                       "episode_stats() all-reduce after every rollout inside the timed loop (BASELINE.json configs[4])" % (n, T)}
    clocks = ClockSampler(local).start()
    env = SFVecEnv("youturn", num_envs=n, device=local, first_global_env=rank * n)
    env.reset(to_numpy=False)
    env.rollout(300, want=("reward",))
    env.set_ticks(np.random.RandomState(rank).randint(300, 5295, size=n))
    out = {"obs": torch.empty((T, n, 1, 84, 84), dtype=torch.uint8, device=dev), "done": torch.empty((T, n), dtype=torch.uint8, device=dev)}
    env.rollout(T, out=out); env.episode_stats()
    reps = max(3, int(0.4 / (n * T / 1.5e8)))
    ms, episodes = [], 0
    for _ in range(2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(); e0.record()
        for _ in range(reps):
            env.rollout(T, out=out)
            st = env.episode_stats()      # device reduction -> all-reduce over the ranks -> host
            episodes += st["episodes"]
        e1.record(); torch.cuda.synchronize(); ms.append(e0.elapsed_time(e1))
    st_ms = _stats(ms)
    if world > 1:
        t = torch.tensor([st_ms["median"]], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); st_ms["median"] = float(t.item())
    res.update({"value": n * world * T * reps / (st_ms["median"] * 1e-3), "unit": "env-steps/s", "region_ms": st_ms, "rollouts_per_region": reps,
                "episodes_finished_all_ranks": int(episodes), "roofline_frac": n * T * reps * B_RENDER / (st_ms["median"] * 1e-3) / 1e9 / peak,
                "collective": "torch.distributed all_reduce (NCCL) of the 24 x int64 episode-stat vector, once per rollout" if world > 1 else "none (1 rank)"})
    env.close()
    torch.cuda.empty_cache()
    res["clocks"] = clocks.stop()
    return res


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def ours(args):
    import numpy as np
    import torch
    from spacefortress_b200 import SFVecEnv
    from spacefortress_b200 import dist as sfdist
    import torch.distributed as dist

    # Native libraries print to stdout (NCCL's version banner at init, for one): stdout is for the ONE JSON line, so
    # everything else goes to stderr until the line is printed
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    rank, local, world = sfdist.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    n = args.envs_per_gpu
    K, Wm = args.steps, max(args.warmup, 3)
    first = rank * n
    env = SFVecEnv(GAMETYPE, num_envs=n, device=local, first_global_env=first)
    env.reset(to_numpy=False)
    # All envs start an episode together; the first ticks after a reset (no dead ships, no missiles in flight)
    # are cheaper than the long-run mix. Advance the state (render off) so the timed steps see a
    # representative mid-episode population. Not part of W or K.
    if args.presteps > 0:
        env.rollout(args.presteps, want=("reward",), action_seed=args.seed + 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput: K timed steps as back-to-back fused launches of up to T steps -----------
    T = min(K, LAUNCH_STEPS)
    obs_buf = torch.empty((T, n, 1, 84, 84), dtype=torch.uint8, device=dev)  # T * 28.9 MB >> L2 for T >= 8
    out = {"obs": obs_buf, "reward": torch.empty((T, n), dtype=torch.int32, device=dev),
           "done": torch.empty((T, n), dtype=torch.uint8, device=dev), "kill": torch.empty((T, n), dtype=torch.uint8, device=dev)}

    def run_steps(count):
        """`count` steps as launches of up to T steps into `out`; returns the outputs of the last step"""
        left = count
        while left > 0:
            t = min(T, left)
            env.rollout(t, out={k: v[:t] for k, v in out.items()}, action_seed=args.seed)
            left -= t
        return {k: v[t - 1] for k, v in out.items()}

    run_steps(Wm)  # W untimed warm-up steps
    clocks = ClockSampler(local).start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = run_steps(K)  # exactly K steps
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = n * world * K / (ms * 1e-3)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)

    # ---- e2e through the numpy drop-in API (host actions -> host observations) ------------------------
    rng = np.random.RandomState(1 + rank)
    acts = rng.randint(0, env.num_actions, size=(args.e2e_steps + 3, n)).astype(np.int32)

    calls = []

    def e2e_run(delta, copy_outputs=False):
        """steps of SFVecEnv.step(np.ndarray); delta: frames reach the host buffer as SF_FLAG_HOST_DELTA updates (the
        default of SFVecEnv) or as whole-frame copies. Returns (env-steps/s over all ranks, s, observation bytes per step)."""
        env.host_delta = delta
        env.copy_outputs = copy_outputs
        for t in range(3):
            o, r, d, info = env.step(acts[t])
        b0 = env.host_delta_stats()
        barrier()
        t0 = time.perf_counter()
        for t in range(args.e2e_steps):
            o, r, d, info = env.step(acts[3 + t])
        torch.cuda.synchronize()
        s_ = time.perf_counter() - t0
        b1 = env.host_delta_stats()
        calls.append({"delta_updates": b1[1] - b0[1], "whole_frame_steps": b1[2] - b0[2]})  # counted by the library
        if world > 1:
            t = torch.tensor([s_], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            s_ = float(t.item())
        obs_b = ((b1[0] - b0[0]) + (b1[2] - b0[2]) * n * 7056) / args.e2e_steps
        return n * world * args.e2e_steps / s_, s_, obs_b

    full_value, full_s, full_obs_b = e2e_run(False)
    ring_value, ring_s, ring_obs_b = e2e_run(True, "ring")
    e2e_value, e2e_s, obs_b = e2e_run(True)
    d2h_bytes = obs_b + n * (4 + 1 + 1 + 4)
    full_d2h = full_obs_b + n * (4 + 1 + 1 + 4)
    # what bounds it: a plain device->host copy of one step's frames into pinned memory, all ranks at the same time,
    # and the T = 1 kernel alone
    pin = torch.empty(n * 7056, dtype=torch.uint8, pin_memory=True)
    src = obs_buf.view(-1)[:n * 7056]
    pin.copy_(src, non_blocking=True); barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        pin.copy_(src, non_blocking=True)
    e1.record(); torch.cuda.synchronize()
    probe_ms = e0.elapsed_time(e1) / 20
    if world > 1:
        t = torch.tensor([probe_ms], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); probe_ms = float(t.item())
    barrier()
    a_dev = torch.from_numpy(acts[0]).to(dev)
    env.step(a_dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        env.step(a_dev)
    e1.record(); torch.cuda.synchronize()
    kern1_ms = e0.elapsed_time(e1) / 20
    step_ms = 1e3 * e2e_s / args.e2e_steps

    stats = env.episode_stats(reset=False)  # the one collective of the path (NCCL all-reduce when world > 1)
    peak, peak_src = measured_peak_gbs()
    achieved = n * K * B_RENDER / (ms * 1e-3) / 1e9  # this rank's kernel: algorithmic bytes of the timed steps / their duration
    traffic = None  # dram__bytes_read.sum + dram__bytes_write.sum per env-step of the committed `ncu --set full` capture, x the timed env-steps
    traffic_src = None
    try:
        import glob
        traffic_src = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_traffic.json")))[-1]  # latest capture
        prof = json.load(open(traffic_src))
        traffic = prof["dram_bytes_per_env_step"] * n * K
    except Exception:
        pass
    line = {
        "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs_per_gpu": n, "envs": n * world, "gametype": GAMETYPE, "kernel": "sf_rollout_kernel, %d launches of up to %d steps (one block of 24 warps per SM: a stepping warp up to two ticks ahead + 23 drawing warps in a block-cooperative frame pipeline)" % (-(-K // T), T), "presteps": args.presteps,
                   "l2": "obs output %.1f MB/step streams into a %d-step buffer (%.0f MB) larger than L2; env state (%.1f MB) is intentionally cache resident"
                         % (n * 7056 / 1e6, T, T * n * 7056 / 1e6, env.state_bytes() / 1e6),
                   "timing": "the K timed steps as back-to-back launches, CUDA events on the launching stream, barrier + synchronize around them, max over ranks",
                   "region_ms": ms},
        "clocks": {"sm_mhz": clk["sm_mhz"], "sm_max_mhz": clk["sm_max_mhz"], "reasons": clk["reasons"], "samples": clk["samples"]},
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": n * 4, "d2h_bytes_per_step": d2h_bytes,
                "api": "SFVecEnv.step(np.ndarray) -> sf_step_host, actions from and results into page-locked numpy buffers, %d steps" % args.e2e_steps,
                "transfer": "SF_FLAG_HOST_DELTA (SFVecEnv's default): every frame is rendered on the device every step; the GPU writes the 64-byte granules "
                            "that differ from the previous step's frame straight into the page-locked host buffer, which then holds exactly the full frames "
                            "(tests/test_gpu_surface.py::test_host_delta_*). d2h_bytes_per_step is what was written, counted on the device",
                "ms_per_step": step_ms, "steps_by_kind": calls[2],
                "drop_in_ring": {"value": ring_value, "ms_per_step": 1e3 * ring_s / args.e2e_steps, "d2h_bytes_per_step": ring_obs_b + n * (4 + 1 + 1 + 4),
                                 "note": "the same loop with copy_outputs='ring', which is what the SubprocVecEnv / DummyVecEnv look-alikes do: every step returns a fresh read-only observation array "
                                         "(a rotation of page-locked buffers, each updated in place; never one the caller still holds), int64 rewards, bool dones and a tuple of N bools"},
                "full_copy": {"value": full_value, "ms_per_step": 1e3 * full_s / args.e2e_steps, "d2h_bytes_per_step": full_d2h,
                              "note": "the same loop with SFVecEnv(host_delta=False): whole frames copied device -> host every step (4 slices, copy of slice k under the kernel of slice k + 1)"},
                "bound": {"pinned_d2h_probe_ms": probe_ms, "pinned_d2h_probe_gbs_per_rank": n * 7056 / (probe_ms * 1e-3) / 1e9, "kernel_T1_ms": kern1_ms,
                          "full_copy_gbs_per_rank": full_d2h / (full_s / args.e2e_steps) / 1e9,
                          "full_copy_frac_of_pcie_probe": (full_d2h / (full_s / args.e2e_steps)) / (n * 7056 / (probe_ms * 1e-3)),
                          "delta_frac_of_kernel_T1": kern1_ms / step_ms,
                          "note": "probe = 20 back-to-back copies of one step's frames (%.1f MB) device -> pinned host, every rank at once, max over ranks" % (n * 7056 / 1e6)}},
        "gpu_launches": -(-K // T),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": "not measured in this run: dram bytes per env-step of the committed ncu capture %s x the timed env-steps" % (os.path.basename(traffic_src) if traffic_src else None),
                     "peak_source": peak_src, "bytes_per_env_step": B_RENDER, "timed_env_steps": n * K, "region_ms": ms},
        "episode_stats": {k: stats[k] for k in ("episodes", "sum_return", "fort_kills")},
    }
    env.close()
    del obs_buf, out, last
    torch.cuda.empty_cache()
    if not args.skip_configs:
        cfgs = {}
        for name, fn in (("C3", config_c3), ("C4", config_c4), ("C5", config_c5)):
            try:
                cfgs[name] = fn(torch, dist, rank, local, world, args, peak)
            except Exception as ex:  # a config that fails must not take the headline down
                cfgs[name] = {"error": repr(ex)}
                torch.cuda.empty_cache()
        line["configs"] = cfgs
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            b, _ = cpu_arm(args.cpu_steps_per_core)
            line["cpu_baseline"] = b
        except Exception as ex:  # the baseline must never take the GPU number down with it
            line["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": os.cpu_count(), "kind": "port", "sample": "failed: %r" % (ex,)}
    sys.stdout.flush()
    os.dup2(json_fd, 1)
    if rank == 0:
        print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16384, help="timed steps, run as launches of up to %d steps" % LAUNCH_STEPS)
    ap.add_argument("--warmup", type=int, default=8, help="untimed warm-up steps before them (at least 3)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (float32)")
    ap.add_argument("--e2e-steps", type=int, default=60)
    ap.add_argument("--cpu-steps-per-core", type=int, default=40000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="headline only (no C3 / C4 / C5 block)")
    ap.add_argument("--c3-envs", type=int, default=65536)
    ap.add_argument("--c3-steps", type=int, default=128)
    ap.add_argument("--c3-fp32-steps", type=int, default=16)
    ap.add_argument("--c3-update-envs", type=int, default=2048)
    ap.add_argument("--c4-envs", type=int, default=131072)
    ap.add_argument("--c5-envs", type=int, default=262144)
    ap.add_argument("--c5-steps", type=int, default=8)
    ap.add_argument("--seed", type=int, default=12345)
    ap.add_argument("--presteps", type=int, default=400, help="untimed state-only ticks before W and K (mid-episode mix)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return reference_arm(args)
    return ours(args)


if __name__ == "__main__":
    sys.exit(main())
