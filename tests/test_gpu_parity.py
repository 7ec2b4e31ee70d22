"""GPU (-m gpu): parity of the CUDA path, called through the C-ABI, against the oracle on the same seeded
inputs. Bars: integer state / events / episode boundaries bit-exact; continuous kinematics bit-exact except the
shells, which carry the device fp64 atan2 / cos / sin and stay within 1e-9 absolute (gpu_helpers.SHELL_ABS_TOL); frames bit-exact (gpu_helpers.assert_frame_close)."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import scripted_kill_policy
from gpu_helpers import END_TICK, GAMETYPES, assert_frame_close, assert_state_close, make, stagger, to_oracle_record, torch_cuda
from oracle.oracle import OracleEnv, Record, draw_native, draw_obs

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("gametype", GAMETYPES)
def test_free_running_trace_parity(gametype):
    n, T = 48, 700
    seeds = np.arange(1, n + 1)
    env = make(gametype, n, seeds=seeds, reset=False)
    obs = env.reset()
    orc = [OracleEnv(gametype, int(s)) for s in seeds]
    for i in range(n):
        assert np.array_equal(orc[i].obs(), obs[i, 0]), "first frame env %d" % i
    rng = np.random.RandomState(11)
    for t in range(T):
        a = rng.randint(0, env.num_actions, size=n)
        obs, rew, done, info = env.step(a)
        ev = env.last_events
        for i in range(n):
            r, d, k, e = orc[i].step(orc[i].keymask(int(a[i])))
            assert (r, d, k, e) == (int(rew[i]), bool(done[i]), bool(info[i]), int(ev[i])), (gametype, t, i)
        if t % 50 == 49:
            recs = env.get_state()
            for i in range(n):
                assert_state_close(orc[i].get_state(), recs[i], (gametype, t, i))
            for i in range(0, n, 5):
                assert_frame_close(orc[i].obs(), obs[i, 0], (gametype, t, i))
    env.close()


def test_config1_youturn_single_env_10k_steps_with_frames():
    """BASELINE.json configs[0]: youturn, 1 env, seeded random-action rollout of 10k steps (crosses the
    episode boundary at tick 5295), state trace + 84x84 frames, through the on-device rollout path."""
    torch = torch_cuda()
    T = 10000
    env = make("youturn", 1)
    o = OracleEnv("youturn", 1)
    rng = np.random.RandomState(2)
    actions = rng.randint(0, 5, size=(T, 1)).astype(np.int32)
    out = env.rollout(T, actions=torch.from_numpy(actions))
    obs = out["obs"].cpu().numpy(); rew = out["reward"].cpu().numpy(); done = out["done"].cpu().numpy(); kill = out["kill"].cpu().numpy()
    ndone = 0
    for t in range(T):
        r, d, k, _ = o.step(o.keymask(int(actions[t, 0])))
        assert (r, d, k) == (int(rew[t, 0]), bool(done[t, 0]), bool(kill[t, 0])), t
        if d:
            ndone += 1
            assert t == 5294
            o.reset()
        if t % 7 == 0 or d or 5290 <= t <= 5300:
            assert_frame_close(o.obs(), obs[t, 0, 0], t)
    assert ndone == 1
    assert_state_close(o.get_state(), env.get_state()[0], "final")
    env.close()


def test_golden_fixtures_replayed_on_gpu():
    torch = torch_cuda()
    for name in ("youturn", "autoturn", "test-youturn", "test-autoturn", "autoturn_kill"):
        z = np.load(os.path.join(GOLD, "trace_%s.npz" % name))
        gametype = "autoturn" if name == "autoturn_kill" else name
        from spacefortress_b200 import _lib
        env = make(gametype, 1, render=False, reset=False)
        env._flags |= _lib.FLAG_ACTIONS_ARE_KEYMASKS
        env.reset()
        T = len(z["keymask"])
        km = torch.from_numpy(z["keymask"].astype(np.int32).reshape(T, 1))
        recs = {int(t): z["records"][k] for k, t in enumerate(z["record_t"])}
        pos = 0
        while pos < T:  # replay in chunks of 100 so the stored records can be compared
            out = env.rollout(100, actions=km[pos:pos + 100])
            assert np.array_equal(out["reward"].cpu().numpy()[:, 0], z["reward"][pos:pos + 100]), (name, pos)
            assert np.array_equal(out["done"].cpu().numpy()[:, 0], z["done"][pos:pos + 100]), (name, pos)
            assert np.array_equal(out["kill"].cpu().numpy()[:, 0], z["fort_kill"][pos:pos + 100]), (name, pos)
            pos += 100
            ref = Record(); C.memmove(C.byref(ref), bytes(recs[pos]), C.sizeof(Record))
            assert_state_close(ref, env.get_state()[0], (name, pos))
        env.close()


def test_kill_path_and_events():
    env = make("autoturn", 4, render=False, reset=False)
    from spacefortress_b200 import _lib
    env._flags |= _lib.FLAG_ACTIONS_ARE_KEYMASKS
    env.reset()
    orc = [OracleEnv("autoturn", 1) for _ in range(4)]
    kills = 0
    for t in range(3000):
        km = np.array([scripted_kill_policy(t + 3 * i, orc[i].get_state().vulnerability) for i in range(4)], np.int32)
        _, rew, done, info = env.step(km)
        for i in range(4):
            r, d, k, e = orc[i].step(int(km[i]))
            assert (r, d, k, e) == (int(rew[i]), bool(done[i]), bool(info[i]), int(env.last_events[i])), (t, i)
            kills += k
    assert kills >= 8
    for i, g in enumerate(env.get_state()):
        assert_state_close(orc[i].get_state(), g, i)
    env.close()


def test_teacher_forced_single_steps():
    """load state -> one step -> compare (shells within 1e-9 absolute, everything else exact)."""
    n = 64
    for gametype in ("youturn", "autoturn"):
        env = make(gametype, n, render=False, reset=False)
        from spacefortress_b200 import _lib
        env._flags |= _lib.FLAG_ACTIONS_ARE_KEYMASKS
        env.reset()
        src = [OracleEnv(gametype, 100 + i) for i in range(n)]
        rng = np.random.RandomState(3)
        for rnd in range(12):
            for s in src:
                for _ in range(int(rng.randint(1, 60))):
                    s.step(int(rng.randint(16)))
            recs = [s.get_state() for s in src]
            env.set_state([to_gpu_record(r) for r in recs])
            back = env.get_state()
            for i in range(n):
                assert_state_close(recs[i], back[i], ("roundtrip", rnd, i))
            km = rng.randint(0, 16, size=n).astype(np.int32)
            _, rew, done, info = env.step(km)
            after = env.get_state()
            for i in range(n):
                r, d, k, e = src[i].step(int(km[i]))
                assert (r, d, k, e) == (int(rew[i]), bool(done[i]), bool(info[i]), int(env.last_events[i])), (gametype, rnd, i)
                assert_state_close(src[i].get_state(), after[i], (gametype, rnd, i))
        env.close()


def to_gpu_record(r):
    from spacefortress_b200 import _lib
    g = _lib.StateRecord()
    C.memmove(C.byref(g), C.byref(r), C.sizeof(Record))
    g.ep_return = 0
    return g


def test_frames_from_crafted_states():
    """Edge cases of the renderer: dead ship (explosion) near the border, dead fortress, objects partly or
    fully off the 90x92 surface, many missiles, a shell inside/outside the 21-unit hide radius, score digits,
    all vulnerability bar states."""
    n = 40
    env = make("youturn", n)
    rng = np.random.RandomState(4)
    recs = []
    for i in range(n):
        r = OracleEnv("youturn", 1).get_state()
        r.ship_x = float(rng.uniform(120, 600)); r.ship_y = float(rng.uniform(60, 560)); r.ship_angle = float(rng.randint(360))
        r.ship_alive = int(i % 3 != 0)
        r.fortress_alive = int(i % 4 != 1)
        r.fortress_angle = float(10 * rng.randint(36)); r.fortress_last_angle = r.fortress_angle
        nm = int(rng.randint(0, 21)) if i % 5 == 0 else int(rng.randint(0, 4))
        for s in rng.choice(20, nm, replace=False):
            r.missile_mask |= 1 << int(s)
            r.missile_x[s] = float(rng.uniform(100, 620)); r.missile_y[s] = float(rng.uniform(50, 580)); r.missile_angle[s] = float(rng.randint(360))
        for s in range(int(rng.randint(0, 4))):
            r.shell_mask |= 1 << s
            rad = 15 + 12 * s if i % 2 else float(rng.uniform(22, 250))
            ang = float(rng.uniform(0, 360))
            r.shell_x[s] = 355 + rad * np.cos(np.deg2rad(ang)); r.shell_y[s] = 315 + rad * np.sin(np.deg2rad(ang)); r.shell_angle[s] = ang
        r.points = float([0, 7, 42, 1234567, 9999999, 30.95][i % 6])
        r.vulnerability = int(i % 14); r.fortress_vuln_timer = int([0, 249, 250, 1000][i % 4])
        recs.append(r)
    env.set_state([to_gpu_record(r) for r in recs])
    nat = env.render_frames(native=True)
    obs = env.render_frames(native=False)
    for i, r in enumerate(recs):
        assert_frame_close(draw_native(r), nat[i], ("native", i))
        assert_frame_close(draw_obs(r), obs[i], ("obs", i))
    # rendering twice (explosion sprite memo path) gives the same frames
    assert np.array_equal(env.render_frames(native=True), nat)
    env.close()


def test_explosion_all_phases_and_box_cache():
    """The ship explosion is scan-converted from per-y-phase span tables (csrc/sf_tables.h SfExpPhase): put a dead
    ship at every one of the 256 sub-pixel y phases (x phases spread over 0..255), with and without wireframes
    reaching into the explosion box, and compare with the oracle. Rendering the same state again takes the sprite
    and resampled-box memo paths and must give the same frames."""
    n = 512
    env = make("autoturn", n)
    rng = np.random.RandomState(11)
    recs = []
    for i in range(n):
        r = OracleEnv("autoturn", 1).get_state()
        phy, phx = i % 256, (i * 37 + 11) % 256
        cx, cy = int(rng.randint(8, 82)) * 256 + phx, int(rng.randint(14, 80)) * 256 + phy   # 24.8 device centre
        r.ship_x = 5.0 * (cx / 256.0 + 26.0); r.ship_y = 5.0 * (cy / 256.0 + 16.0)           # inverse of the base CTM
        r.ship_alive = 0; r.ship_angle = float(rng.randint(360))
        r.fortress_alive = int(i % 7 != 3)
        r.fortress_angle = float(10 * rng.randint(36)); r.fortress_last_angle = r.fortress_angle
        if i >= 256:  # missiles flying through the explosion box
            for s in range(int(rng.randint(1, 4))):
                r.missile_mask |= 1 << s
                r.missile_x[s] = r.ship_x + float(rng.uniform(-70, 70)); r.missile_y[s] = r.ship_y + float(rng.uniform(-70, 70)); r.missile_angle[s] = float(rng.randint(360))
        r.points = float([0, 3][i % 2]); r.vulnerability = int(i % 12)
        recs.append(r)
    env.set_state([to_gpu_record(r) for r in recs])
    obs = env.render_frames(native=False)
    for i, r in enumerate(recs):
        assert_frame_close(draw_obs(r), obs[i], ("obs", i, "phase", i % 256))
    assert np.array_equal(env.render_frames(native=False), obs)   # cached sprite; quarters without wireframes copied
    assert np.array_equal(env.render_frames(native=False), obs)
    nat = env.render_frames(native=True)
    for i in range(0, n, 5):
        assert_frame_close(draw_native(recs[i]), nat[i], ("native", i))
    env.close()


def test_rollout_equals_stepwise_and_synthetic_stream():
    torch = torch_cuda()
    n, T = 96, 64
    a = make("youturn", n, reset=False); b = make("youturn", n, reset=False)
    a.reset(); b.reset()
    acts = a.synthetic_actions(T, action_seed=5)
    out = a.rollout(T, action_seed=5)  # device-side hash policy
    for t in range(T):
        obs, rew, done, info = b.step(torch.from_numpy(acts[t]).cuda())
        assert torch.equal(out["obs"][t], obs) and torch.equal(out["reward"][t], rew)
        assert torch.equal(out["done"][t].bool(), done) and torch.equal(out["kill"][t].bool(), info)
    ra, rb = a.get_state(), b.get_state()
    assert bytes(ra) == bytes(rb)
    a.close(); b.close()


def test_rollout_with_many_strokes_and_odd_lengths_equals_stepwise():
    """The fused rollout draws two consecutive ticks per stage and splits a stage into rounds when the stroke or
    cell pools are full; a single step draws one tick per stage. From crowded states (up to 20 missiles and 3 shells
    per env, a third of the ships dead: several rounds per stage) both must give the same frames, for even and odd
    numbers of ticks."""
    torch = torch_cuda()
    n = 64
    rng = np.random.RandomState(21)
    recs = []
    for i in range(n):
        r = OracleEnv("youturn", 1).get_state()
        r.ship_x = float(rng.uniform(250, 460)); r.ship_y = float(rng.uniform(200, 430)); r.ship_angle = float(rng.randint(360))
        r.ship_alive = int(i % 3 != 0)
        for s in rng.choice(20, int(rng.randint(8, 21)), replace=False):
            r.missile_mask |= 1 << int(s)
            r.missile_x[s] = float(rng.uniform(200, 520)); r.missile_y[s] = float(rng.uniform(150, 480)); r.missile_angle[s] = float(rng.randint(360))
        for s in range(int(rng.randint(0, 4))):
            r.shell_mask |= 1 << s
            ang = float(rng.uniform(0, 360)); rad = float(rng.uniform(30, 150))
            r.shell_x[s] = 355 + rad * np.cos(np.deg2rad(ang)); r.shell_y[s] = 315 + rad * np.sin(np.deg2rad(ang)); r.shell_angle[s] = ang
            r.shell_vx[s] = 6 * np.cos(np.deg2rad(ang)); r.shell_vy[s] = 6 * np.sin(np.deg2rad(ang))
        recs.append(to_gpu_record(r))
    for T in (1, 2, 5, 8):
        a = make("youturn", n, reset=False); b = make("youturn", n, reset=False)
        a.reset(); b.reset()
        a.set_state(recs); b.set_state(recs)
        acts = a.synthetic_actions(T, action_seed=9)
        out = a.rollout(T, action_seed=9)
        for t in range(T):
            obs, rew, done, info = b.step(torch.from_numpy(acts[t]).cuda())
            assert torch.equal(out["obs"][t], obs), (T, t)
            assert torch.equal(out["reward"][t], rew), (T, t)
        assert bytes(a.get_state()) == bytes(b.get_state())
        a.close(); b.close()
    # and the first frames against the oracle
    a = make("youturn", n); a.set_state(recs)
    obs = a.render_frames(native=False)
    for i in range(0, n, 7):
        assert_frame_close(draw_obs(to_oracle_record(recs[i])), obs[i], ("crowded", i))
    a.close()


def test_soak_fused_rollout_equals_single_steps_many_envs():
    """Every block of the GPU busy (4096 envs, the bench workload), 192 ticks into the steady state: the pipelined
    multi-tick kernel and single steps must agree on every frame (a race between the stepping warp and the
    drawing warps, or between two stages, would show up as a sporadic mismatch). tools/gpu_soak.py runs longer."""
    torch = torch_cuda()
    n, T = 4096, 64
    a = make("autoturn", n, reset=False); b = make("autoturn", n, reset=False)
    a.reset(to_numpy=False); b.reset(to_numpy=False)
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    for chunk in range(3):
        acts = torch.randint(0, a.num_actions, (T, n), generator=g, device="cuda", dtype=torch.int32)
        out = a.rollout(T, actions=acts)
        for t in range(T):
            obs, rew, done, info = b.step(acts[t])
            assert torch.equal(out["obs"][t], obs), (chunk, t)
            assert torch.equal(out["reward"][t], rew) and torch.equal(out["done"][t].bool(), done), (chunk, t)
    assert bytes(a.get_state()) == bytes(b.get_state())
    a.close(); b.close()


def test_shard_invariance_two_slabs_equal_one():
    """N envs in one slab == the same envs split over two slabs (what two ranks would own), bitwise;
    episode statistics add up."""
    n, T = 64, 150
    seeds = np.arange(1, n + 1)
    whole = make("autoturn", n, seeds=seeds, reset=False)
    lo = make("autoturn", n // 2, seeds=seeds[:n // 2], first_global_env=0, reset=False)
    hi = make("autoturn", n // 2, seeds=seeds[n // 2:], first_global_env=n // 2, reset=False)
    for e in (whole, lo, hi):
        e.reset()
    ow = whole.rollout(T, action_seed=9); ol = lo.rollout(T, action_seed=9); oh = hi.rollout(T, action_seed=9)
    import torch
    assert torch.equal(ow["obs"][:, :n // 2], ol["obs"]) and torch.equal(ow["obs"][:, n // 2:], oh["obs"])
    assert torch.equal(ow["reward"][:, :n // 2], ol["reward"]) and torch.equal(ow["reward"][:, n // 2:], oh["reward"])
    assert bytes(whole.get_state(0, n // 2)) == bytes(lo.get_state()) and bytes(whole.get_state(n // 2, n // 2)) == bytes(hi.get_state())
    for e in (whole, lo, hi):
        e.close()


def test_auto_reset_and_episode_stats():
    """All envs finish at tick 5295; the returned obs is the first frame of the next episode, prev_vlner
    survives (quirk Q7), and the device-side episode statistics equal the host sums."""
    torch = torch_cuda()
    n = 8
    env = make("autoturn", n, seeds=np.arange(1, n + 1))
    orc = [OracleEnv("autoturn", s) for s in range(1, n + 1)]
    T = 5295
    acts = env.synthetic_actions(T, action_seed=1)
    out = env.rollout(T, action_seed=1, want=("reward", "done", "kill"))
    done = out["done"].cpu().numpy(); rew = out["reward"].cpu().numpy()
    assert done[:-1].sum() == 0 and done[-1].all()
    exp = dict(episodes=0, sum_return=0, sum_length=0, shipDeaths=0, totalShots=0, fort_kills=0)
    for i in range(n):
        ret = 0
        for t in range(T):
            r, d, k, _ = orc[i].step(orc[i].keymask(int(acts[t, i])))
            assert r == int(rew[t, i])
            ret += r
        assert d
        s = orc[i].get_state()
        exp["episodes"] += 1; exp["sum_return"] += ret; exp["sum_length"] += s.tick
        exp["shipDeaths"] += s.stats[3]; exp["totalShots"] += s.stats[7]; exp["fort_kills"] += s.stats[5]
        orc[i].reset()
    st = env.episode_stats()
    for k, v in exp.items():
        assert st[k] == v, (k, st[k], v)
    frames = env.render_frames()
    recs = env.get_state()
    for i in range(n):
        assert_state_close(orc[i].get_state(), recs[i], ("after auto-reset", i))
        assert_frame_close(orc[i].obs(), frames[i], ("first frame of next episode", i))
    assert env.episode_stats()["episodes"] == 0  # accumulators were reset
    env.close()


def test_staggered_episode_ends_auto_reset_and_stats():
    """BASELINE.json configs[4]: auto-reset under episode-length variance. The clocks of the envs are staggered
    (sf_set_ticks), so they finish at different steps; done flags, rewards, the first frames of the new episodes and
    the episode statistics must equal the oracle's, step by step."""
    torch = torch_cuda()
    n, T = 24, 48
    env = make("youturn", n, seeds=np.arange(1, n + 1))
    ticks = stagger(env, 1 + np.random.RandomState(3).randint(0, 40, size=n))
    orc = [OracleEnv("youturn", s) for s in range(1, n + 1)]
    for i in range(n):
        r = orc[i].get_state(); r.tick = int(ticks[i]); r.time = int(ticks[i]) * 34; orc[i].set_state(r)
    acts = env.synthetic_actions(T, action_seed=2)
    out = env.rollout(T, action_seed=2)
    done = out["done"].cpu().numpy(); rew = out["reward"].cpu().numpy(); obs = out["obs"].cpu().numpy()
    episodes, sum_len = 0, 0
    for i in range(n):
        for t in range(T):
            r, d, k, _ = orc[i].step(orc[i].keymask(int(acts[t, i])))
            assert r == int(rew[t, i]) and bool(d) == bool(done[t, i]), (i, t)
            if d:
                assert t == END_TICK - 1 - int(ticks[i]), (i, t)
                episodes += 1; sum_len += orc[i].get_state().tick
                orc[i].reset()
            if d or t % 11 == 0:
                assert_frame_close(orc[i].obs(), obs[t, i, 0], ("frame", i, t))
    assert len(set(int(np.argmax(done[:, i])) for i in range(n))) > 5  # the ends really are spread
    st = env.episode_stats()
    assert st["episodes"] == episodes == n and st["sum_length"] == sum_len
    env.close()


def test_vecenv_numpy_api_matches_reference_usage():
    """rl/train.py:30-41,60,80-85 usage pattern with the drop-in classes."""
    torch_cuda()
    from spacefortress_b200 import SubprocVecEnv, make_env
    envs = SubprocVecEnv([make_env("SpaceFortress-autoturn-image-v0", 0, i) for i in range(6)])
    assert envs.observation_space.shape == (1, 84, 84) and envs.action_space.n == 3 and envs.num_envs == 6
    obs = envs.reset()
    assert obs.shape == (6, 1, 84, 84) and obs.dtype == np.uint8
    obs, rew, done, infos = envs.step(np.array([0, 1, 2, 0, 1, 2]))
    assert obs.shape == (6, 1, 84, 84) and rew.shape == (6,) and done.dtype == bool and len(infos) == 6 and isinstance(infos[0], bool)
    assert sum(infos) == 0
    envs.step_async(np.zeros(6, np.int64)); envs.step_wait()
    envs.close()
    with pytest.raises(Exception):
        SubprocVecEnv([make_env("SpaceFortress-nonsense-v0", 0, 0)])


def test_single_env_facade_matches_oracle():
    """SSF_Env facade: native (92,90) frames, python-int rewards, bool info, no auto-reset, reset keeps prev_vlner."""
    torch_cuda()
    from spacefortress_b200.gym import make as gym_make
    env = gym_make("SpaceFortress-youturn-image-v0")
    o = OracleEnv("youturn", 1)  # == SSF_Env.__init__ (constructs the first Game)
    first = env.reset()
    o.reset()
    assert first.shape == (92, 90) and np.array_equal(first, o.native_frame())
    rng = np.random.RandomState(8)
    for t in range(120):
        a = int(rng.randint(5))
        obs, r, d, k = env.step(a)
        ro, do, ko, _ = o.step(o.keymask(a))
        assert (r, d, k) == (ro, do, ko) and isinstance(k, bool)
        if t % 15 == 0:
            assert np.array_equal(obs, o.native_frame())
            assert env.g.dump().split(",[")[0] == o.dump().split(",[")[0]
    assert env.g.stats[:13] == tuple(o.get_state().stats)
    env.close()


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_policy_input_kernel_matches_the_torch_stack(dtype):
    """sf_policy_input / sf_policy_input_f32 (stack + zero the frames from before a reset + 1/255 + space-to-depth, one
    kernel) against the plain torch formulation, bit for bit; and conv1 on it against conv1 on the NCHW stack."""
    torch = torch_cuda()
    from spacefortress_b200.rollout import OnDeviceRollout, SFGRUPolicy
    n = 300
    dt = torch.bfloat16 if dtype == "bf16" else torch.float32
    tol = 0.06 if dtype == "bf16" else 2e-3
    tf = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
    env = make("youturn", n, reset=False)
    policy = SFGRUPolicy(env.num_actions).cuda().eval().to(dt)
    ro = OnDeviceRollout(env, policy, num_steps=6)
    assert ro.fused_input
    ro.collect()
    for t in (0, 3, 5):
        ro.valid_hist[t][::7] = 1; ro.valid_hist[t][3::7] = 2; ro.valid_hist[t][5::7] = 3   # resets of different ages
        stack = ro.stack(t)                                           # [N,4,84,84] u8, masked
        ref = (stack.to(dt) / 255.0).view(n, 4, 21, 4, 21, 4).permute(0, 1, 3, 5, 2, 4).reshape(n, 64, 21, 21)
        got = ro.policy_input(t)
        assert got.shape == ref.shape and got.dtype == dt and torch.equal(got.float(), ref.float()), t
        a = torch.nn.functional.conv2d(got, policy.conv1_s2d_weight(), policy.conv1.bias).float()
        b = policy.conv1(stack.to(dt) / 255.0).float()
        assert (a - b).abs().max().item() <= tol * max(1.0, b.abs().max().item()), t
        # the whole feature path (fused conv + bias + relu, NHWC fc1) against the generic one
        st = torch.zeros(n, 256, device="cuda", dtype=dt); mk = torch.ones(n, 1, device="cuda", dtype=dt)
        with torch.no_grad():
            fa, _ = policy.features(got, st, mk, s2d=True)
            fb, _ = policy.features(stack, st, mk)
        assert (fa.float() - fb.float()).abs().max().item() <= tol * max(1.0, fb.float().abs().max().item()), t
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf
    env.close()


def test_on_device_rollout_frame_stack_matches_reference_loop():
    """OnDeviceRollout (config 3 plumbing): the 4-frame window over the single-frame buffer equals the
    reference's running `current_obs` (rl/train.py:51-56,92-97: zero the stack on done, shift, append)."""
    torch = torch_cuda()
    from spacefortress_b200.rollout import OnDeviceRollout, SFGRUPolicy
    n, T = 6, 24
    env = make("youturn", n)
    recs = env.get_state()
    for i in range(n):  # stagger the episode ends so that dones fall inside the rollout
        recs[i].tick = END_TICK - 3 - 2 * i
        recs[i].time = recs[i].tick * 34
    env.set_state(recs)
    torch.manual_seed(0)

    class Recording(SFGRUPolicy):  # remembers every input it acted on
        def act(self, obs, state, mask, **kw):
            self.seen.append(obs.clone())
            return SFGRUPolicy.act(self, obs, state, mask, **kw)
    policy = Recording(env.num_actions).cuda().eval()
    policy.seen = []
    ro = OnDeviceRollout(env, policy, num_steps=T, fused_input=False)   # the policy sees the plain u8 stack here
    env.set_state(recs)  # OnDeviceRollout reset the envs: restore the staggered clocks and re-render the first frame
    ro.frames[ro.S - 1].copy_(torch.from_numpy(env.render_frames()).cuda())
    cur = torch.zeros((n, 4, 84, 84), device="cuda")
    cur[:, -1] = ro.frames[ro.S - 1].float()
    for rollout in range(2):  # the second one starts from the carried-over history of the first
        policy.seen = []
        ro.collect()
        assert len(policy.seen) == T
        for t in range(T):
            # what the learner replays (PPOLearner.update uses ro.stack(t)) is what the policy acted on ...
            assert torch.equal(ro.stack(t), policy.seen[t]), (rollout, t)
            # ... and that is the reference's running current_obs (rl/train.py:51-56,92-97)
            assert torch.equal(policy.seen[t].float(), cur), (rollout, t)
            mask = (~ro.dones[t]).float()
            cur *= mask.view(-1, 1, 1, 1)
            cur[:, :-1] = cur[:, 1:].clone()
            cur[:, -1] = ro.frames[t + ro.S].float()
        assert torch.equal(ro.stack(T).float(), cur)
        if rollout == 0:
            assert int(ro.dones.sum()) == n, "every env should have finished its episode inside the first rollout"
            assert int((ro.valid_hist[:T] < ro.S).sum()) > 0
    env.close()


def test_graphed_rollout_equals_the_eager_one():
    """OnDeviceRollout(graph=True) replays one CUDA graph per step index: with a deterministic policy it produces the
    same actions, frames, rewards and values as the eager loop, over two consecutive rollouts (history carry-over)."""
    torch = torch_cuda()
    from spacefortress_b200.rollout import OnDeviceRollout, SFGRUPolicy

    class Greedy(SFGRUPolicy):
        def act(self, obs, state, mask, **kw):
            kw["deterministic"] = True
            return SFGRUPolicy.act(self, obs, state, mask, **kw)
    n, T = 96, 6
    outs = []
    for graph in (False, True):
        env = make("youturn", n, reset=False)
        torch.manual_seed(3)
        ro = OnDeviceRollout(env, Greedy(env.num_actions).cuda().eval(), num_steps=T, graph=graph)
        got = []
        for _ in range(2):
            ro.collect()
            torch.cuda.synchronize()
            got.append([x.clone() for x in (ro.actions, ro.frames, ro.rewards, ro.dones, ro.values, ro.valid_hist)])
        outs.append(got)
        env.close()
    for r in range(2):
        for a, b in zip(outs[0][r], outs[1][r]):
            assert torch.equal(a, b), r


def test_ppo_update_on_an_on_device_rollout():
    """Collect a rollout on the device and update on it without leaving the device (rl/train.py:73-146)."""
    torch = torch_cuda()
    from spacefortress_b200.rollout import OnDeviceRollout, SFGRUPolicy
    from spacefortress_b200.ppo import PPOLearner
    n, T = 64, 8
    env = make("youturn", n, reset=False)
    policy = SFGRUPolicy(env.num_actions).cuda()
    ro = OnDeviceRollout(env, policy, num_steps=T)
    ro.collect()
    before = [p.detach().clone() for p in policy.parameters()]
    stats = PPOLearner(policy, ppo_epoch=2, num_mini_batch=4).update(ro, env_chunk=8)
    assert len(stats) == 8 and all(np.isfinite(s).all() for s in stats)
    assert any(not torch.equal(a, b) for a, b in zip(before, policy.parameters()))
    env.close()

