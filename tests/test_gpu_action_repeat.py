"""GPU (-m gpu): action repeat (sf_set_action_repeat, SFVecEnv(action_repeat=k)). One agent step with action a is the
gym wrapper loop around SSF_Env: up to k ticks with the same key mask, stopping on the tick the episode ends; the reward
is the sum, done / kill / events the OR, the observation that of the state after the step. The CPU oracle runs that loop;
every stepping entry point must give the same bits."""
import ctypes as C

import numpy as np
import pytest

from gpu_helpers import (END_TICK, GAMETYPES, KINDS, STEP_OUTPUTS, assert_state_close, hp, make, outputs, ptrs, rollout,
                         rollout_features, single_steps, stagger, step_host, to_oracle_record, torch_cuda, vp)
from oracle.oracle import OracleEnv, draw_native, draw_obs

pytestmark = pytest.mark.gpu


def oracle_agent_step(o, km, k, autoreset=True):
    """The wrapper loop: (reward sum, done, kill, events OR, ticks run, the record at the episode end or None)."""
    from spacefortress_b200 import _lib
    R, D, K, EV, end = 0, False, False, 0, None
    for j in range(k):
        r, d, kl, e = o.step(km)
        R += r; K |= kl; EV |= e
        if d:
            D = True
            if autoreset:
                EV |= _lib.EV_EPISODE_RESET
                end = o.get_state()
                o.reset()
            return R, D, K, EV, j + 1, end
    return R, D, K, EV, k, end


def oracles(gametype, recs):
    """one OracleEnv per record, set to it"""
    orc = []
    for r in recs:
        o = OracleEnv(gametype, 1)
        o.set_state(to_oracle_record(r))
        orc.append(o)
    return orc


# ------------------------------------------------------------------------------------------------ 1 + 4: the oracle
def run_against_oracle(gametype, k, n=48, T=160, flags=0, frame_every=4):
    """sf_rollout with 84x84 and with native frames (two handles in the same state) against OracleEnvs started from the
    handle's state records, given actions. Returns the per-env episode-end records and returns for the statistics."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    a = make(gametype, n, seeds=7, action_repeat=k, warm=30)
    b = make(gametype, n, seeds=7, action_repeat=k, warm=30, native_obs=True)
    stagger(a, 1 + 5 * np.arange(n)); stagger(b, 1 + 5 * np.arange(n))  # env i ends at tick position (5 * i) % k of a step
    assert torch.equal(a.save_envs(), b.save_envs())
    a.episode_stats(reset=True, all_reduce=False)
    recs = a.get_state()
    orc = oracles(gametype, recs)
    ret0 = [int(recs[i].ep_return) for i in range(n)]
    acts = np.random.RandomState(k * 100 + len(gametype)).randint(a.num_actions, size=(T, n)).astype(np.int32)
    da = torch.from_numpy(acts).cuda()
    ga, gb = [{key: v.cpu().numpy() for key, v in rollout(env, T, da, flags=env._flags | flags).items()} for env in (a, b)]
    for key in ("reward", "done", "kill"):
        assert np.array_equal(ga[key], gb[key]), key
    ends, positions = [], set()
    autoreset = not (flags & _lib.FLAG_NO_AUTORESET)
    ret = list(ret0)
    for t in range(T):
        for i in range(n):
            R, D, K, EV, ran, end = oracle_agent_step(orc[i], orc[i].keymask(int(acts[t, i])), k, autoreset)
            assert (R, D, K) == (int(ga["reward"][t, i]), bool(ga["done"][t, i]), bool(ga["kill"][t, i])), (gametype, k, t, i)
            ret[i] += R
            if D:
                positions.add(ran - 1)
            if end is not None:
                ends.append((end, ret[i]))
                ret[i] = 0
            if D or t % frame_every == 0 or t == T - 1:
                s = orc[i].get_state()
                assert np.array_equal(draw_obs(s), ga["obs"][t, i]), ("84x84", gametype, k, t, i)
                assert np.array_equal(draw_native(s), gb["obs"][t, i]), ("native", gametype, k, t, i)
    assert positions == set(range(k)), positions  # the episodes ended at every tick position inside an agent step
    recs = a.get_state()
    for i in range(n):
        assert_state_close(orc[i].get_state(), recs[i], (gametype, k, "final", i))
    assert bytes(recs) == bytes(b.get_state())
    stats = a.episode_stats(reset=True, all_reduce=False)
    a.close(); b.close()
    return ends, stats, orc


@pytest.mark.parametrize("k", [2, 3, 4])
@pytest.mark.parametrize("gametype", GAMETYPES)
def test_repeat_equals_the_oracle_wrapper_loop(gametype, k):
    """Reward sums, done, kill, the final state and every 4th frame (and every frame of an episode end), 84x84 and native,
    against the oracle running the wrapper loop, with episode ends at every tick position of an agent step."""
    ends, _, _ = run_against_oracle(gametype, k)
    assert len(ends) == 48


def test_repeat_events_equal_the_oracle():
    """The events OR of every agent step (sf_step, which returns them) against the oracle, episode resets included."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, k, T = 48, 3, 80
    env = make("youturn", n, seeds=7, action_repeat=k, warm=40, render=False)
    stagger(env, 1 + 5 * np.arange(n))
    orc = oracles("youturn", env.get_state())
    acts = np.random.RandomState(5).randint(env.num_actions, size=(T, n)).astype(np.int32)
    out = single_steps(env, torch.from_numpy(acts).cuda(), want=("reward", "events"))
    rew, ev = out["reward"].cpu().numpy(), out["events"].cpu().numpy().view(np.uint32)
    seen = 0
    for t in range(T):
        for i in range(n):
            R, D, K, EV, _, _ = oracle_agent_step(orc[i], orc[i].keymask(int(acts[t, i])), k)
            assert (R, EV) == (int(rew[t, i]), int(ev[t, i])), (t, i)
            seen |= EV
    assert seen & _lib.EV_EPISODE_RESET and seen & _lib.EVENT_BITS["missile-fired"]
    env.close()


def test_episode_statistics_equal_the_oracle_sums():
    """sf_episode_stats over the episodes that ended inside the repeated steps: the oracle's sums (lengths in ticks)."""
    ends, st, _ = run_against_oracle("autoturn", 4, n=40, T=90, frame_every=1000)
    assert len(ends) == 40
    exp = dict(episodes=len(ends), sum_return=0, sum_return_sq=0, sum_length=0, maxVlner_max=0, sum_points_int=0, sum_raw_points_milli=0)
    names = ["bigHexDeaths", "smallHexDeaths", "shellDeaths", "shipDeaths", "resets", "destroyedFortresses", "missedShots",
             "totalShots", "totalThrusts", "totalLefts", "totalRights", "vlnerIncs", "maxVlner_sum"]
    for nm in names:
        exp[nm] = 0
    exp["fort_kills"] = 0
    for rec, ret in ends:
        exp["sum_return"] += ret; exp["sum_return_sq"] += ret * ret; exp["sum_length"] += rec.tick
        for j, nm in enumerate(names):
            exp[nm] += int(rec.stats[j])
        exp["fort_kills"] += int(rec.stats[5])
        exp["maxVlner_max"] = max(exp["maxVlner_max"], int(rec.stats[12]))
        exp["sum_points_int"] += int(np.float32(rec.points))
        exp["sum_raw_points_milli"] += int(np.rint(np.float64(np.float32(rec.raw_points)) * 1000.0))
    assert exp["sum_length"] == END_TICK * len(ends)
    for key, v in exp.items():
        assert st[key] == v, (key, st[key], v)


def test_no_autoreset_stops_at_done_and_stays_finished():
    """SF_FLAG_NO_AUTORESET: the repeat stops at the tick the episode ends; after that every agent step is one tick of a
    finished env that reports done again (the oracle's loop without a reset), and no step sets SF_EV_EPISODE_RESET."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, k, T = 24, 3, 40
    env = make("youturn", n, seeds=7, action_repeat=k, warm=20)
    ticks = stagger(env, 1 + 2 * np.arange(n))
    orc = oracles("youturn", env.get_state())
    acts = np.random.RandomState(4).randint(env.num_actions, size=(T, n)).astype(np.int32)
    out = rollout(env, T, torch.from_numpy(acts).cuda(), flags=env._flags | _lib.FLAG_NO_AUTORESET, want=("obs", "reward", "done"))
    obs, rew, done = [out[name].cpu().numpy() for name in ("obs", "reward", "done")]
    for i in range(n):
        first = (END_TICK - int(ticks[i]) - 1) // k  # the agent step in which the episode ends
        for t in range(T):
            R, D, _, EV, ran, _ = oracle_agent_step(orc[i], orc[i].keymask(int(acts[t, i])), k, autoreset=False)
            assert (R, D) == (int(rew[t, i]), bool(done[t, i])), (t, i)
            assert not EV & _lib.EV_EPISODE_RESET
            assert D == (t >= first), (t, i, first)
            if t > first:
                assert ran == 1
            if t % 5 == 0 or t == first:
                assert np.array_equal(draw_obs(orc[i].get_state()), obs[t, i]), (t, i)
        assert orc[i].get_state().tick == END_TICK + (T - 1 - first), i
    recs = env.get_state()
    for i in range(n):
        assert_state_close(orc[i].get_state(), recs[i], ("final", i))
    env.close()


# ------------------------------------------------------------------------------------------------ 2: entry points
@pytest.mark.parametrize("k", [2, 4])
@pytest.mark.parametrize("n", [1, 33, 4096, 4737])
def test_entry_points_agree(n, k):
    """From one start state (clocks staggered so that episodes end inside the run): sf_rollout with and without frames
    (synthetic and given actions), T x sf_step, sf_step_host (page-locked with and without delta updates, pageable),
    sf_rollout_features (3 kinds) and sf_step_host_features give the same rewards, dones, kills, events and final state;
    frame t is sf_render after agent step t, feature row t is sf_features after it."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    T, seed, t0 = 10, 3, 17
    env = make("youturn", n, seeds=n, action_repeat=k, warm=12, ends=(1, T * k + 4))
    L, h = env.L, env.h
    start = env.save_envs()
    acts = env.synthetic_actions(T, action_seed=seed, t0=t0)
    da = torch.from_numpy(acts).cuda()

    def restart():
        env.load_envs(start)
        torch.cuda.synchronize()

    def same(a, b, ctx):
        assert torch.equal(a, b), ctx

    # the reference: T x (sf_step, sf_render, sf_features of every kind)
    restart()
    ref = outputs(env, T, ("obs",) + STEP_OUTPUTS + tuple(KINDS))
    render = torch.empty((n, 84, 84), dtype=torch.uint8, device="cuda")
    for t in range(T):
        _lib.check(L.sf_step(h, vp(da[t]), *ptrs(ref, ("obs",) + STEP_OUTPUTS, t), _lib.FLAG_RENDER, None))
        _lib.check(L.sf_render(h, vp(render), 0, None))
        torch.cuda.synchronize()
        same(render, ref["obs"][t], ("sf_step frame == sf_render", t))
        for kind in KINDS:
            _lib.check(L.sf_features(h, _lib.OBS_TYPES[kind], vp(ref[kind][t]), None))
    torch.cuda.synchronize()
    end = env.save_envs()
    assert int(ref["done"].sum()) > 0 and bool((ref["events"] & _lib.EV_EPISODE_RESET).any())

    def check(got, ctx):
        """every output equals the reference's byte for byte (feature rows bit for bit), and so does the final state"""
        for name, x in got.items():
            same(torch.as_tensor(x, device="cuda").view(torch.uint8), ref[name].view(torch.uint8), (ctx, name))
        same(env.save_envs(), end, (ctx, "final state"))

    # sf_rollout: synthetic and given actions, with frames and without
    for actions, case in ((None, "synthetic"), (da, "given")):
        for frames in (True, False):
            restart()
            got = rollout(env, T, actions, seed, t0, _lib.FLAG_RENDER if frames else 0, want=("obs",) * frames + ("reward", "done", "kill"))
            check(got, ("sf_rollout", case, frames))

    # sf_step_host: page-locked with delta updates, page-locked whole frames, pageable whole frames
    for pinned, delta in ((True, True), (True, False), (False, False)):
        restart()
        stats0 = env.host_delta_stats()
        check(step_host(env, acts, _lib.FLAG_RENDER | (_lib.FLAG_HOST_DELTA if delta else 0), pinned), ("sf_step_host", pinned, delta))
        stats1 = env.host_delta_stats()
        if delta:  # the first call sends whole frames, the others delta updates, which are counted
            assert stats1[1] - stats0[1] == T - 1 and stats1[2] - stats0[2] == 1 and stats1[0] > stats0[0]
        else:
            assert stats1[2] - stats0[2] == T and stats1[1] == stats0[1]

    # sf_rollout_features: every kind, synthetic actions
    for kind in KINDS:
        restart()
        check(rollout_features(env, kind, T, None, seed, t0), ("sf_rollout_features", kind))

    # sf_step_host_features: page-locked and pageable rows
    for pinned, kind in ((True, "normalized-features"), (False, "monitors")):
        restart()
        check(step_host(env, acts, 0, pinned, want=(kind,) + STEP_OUTPUTS), ("sf_step_host_features", kind))
    env.close()


def test_native_frames_host_step_with_delta():
    """Native 92x90 frames (8280 B, not a multiple of 16) through sf_step_host with delta updates, whole-frame copies and
    the device path: the host buffer holds exactly sf_render's frames after every agent step."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, k, T = 333, 3, 12
    env = make("autoturn", n, seeds=7, action_repeat=k, warm=10, native_obs=True)
    stagger(env, np.random.RandomState(1).randint(1, T * k, size=n))
    L, h = env.L, env.h
    flags = _lib.FLAG_RENDER | _lib.FLAG_NATIVE_OBS
    rng = np.random.RandomState(6)
    buf = _lib.pinned_array((n, 92, 90), np.uint8)  # one buffer for all steps: the delta updates build on its contents
    act = _lib.pinned_array((n,), np.int32)
    done = _lib.pinned_array((n,), np.uint8)
    render = torch.empty((n, 92, 90), dtype=torch.uint8, device="cuda")
    ends = 0
    for t in range(T):
        act[:] = rng.randint(env.num_actions, size=n)
        before = env.save_envs()
        _lib.check(L.sf_step_host(h, hp(act), hp(buf), None, hp(done), None, None, flags | _lib.FLAG_HOST_DELTA))
        _lib.check(L.sf_render(h, vp(render), _lib.FLAG_NATIVE_OBS, None))
        torch.cuda.synchronize()
        exp = render.cpu().numpy()
        assert np.array_equal(buf, exp), ("delta", t)
        after = env.save_envs()
        env.load_envs(before)
        assert np.array_equal(step_host(env, act[None], flags, pinned=False, want=("obs",))["obs"][0], exp), ("whole", t)
        assert torch.equal(env.save_envs(), after), ("whole", t)
        env.load_envs(before)
        assert torch.equal(single_steps(env, torch.from_numpy(act[None].copy()).cuda(), flags, want=("obs",))["obs"][0], render), ("device", t)
        assert torch.equal(env.save_envs(), after), ("device", t)
        ends += int(done.sum())
    assert ends > 0
    assert env.host_delta_stats()[1] == T - 1
    L.sf_host_forget(h, None)
    env.close()


# ------------------------------------------------------------------------------------------------ 5: k == 1
def test_repeat_one_is_the_plain_step():
    """A handle set to 1 (after 3) gives byte-identical outputs and state to a handle that was never set, on every
    stepping entry point."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv, _lib
    n, T = 300, 6
    envs = []
    for k in (None, 1):
        e = SFVecEnv("youturn", num_envs=n, device=0, seeds=2)
        if k is None:  # undo the constructor's call: a handle that has never been set
            e.L.sf_destroy(e.h)
            h = C.c_void_p()
            _lib.check(e.L.sf_create(b"youturn", 1, n, 0, C.byref(h)))
            e.h = h
            e.seed_streams(2)
            assert e.L.sf_action_repeat(e.h) == 1
        else:
            _lib.check(e.L.sf_set_action_repeat(e.h, 3))
            _lib.check(e.L.sf_set_action_repeat(e.h, 1))
        e.reset()
        stagger(e, 3 + np.arange(n) % 7)
        envs.append(e)
    outs = []
    acts = torch.from_numpy(np.random.RandomState(0).randint(5, size=(T, n)).astype(np.int32)).cuda()
    for e in envs:
        o = {}
        o["roll"] = e.rollout(T, action_seed=4)
        o["step"] = [x.clone() for x in e.step(acts[0])]
        o["host"] = [np.array(x) for x in e.step(acts[1].cpu().numpy())]
        o["feat"] = rollout_features(e, "features", T, acts, want=())["features"]
        o["state"] = e.save_envs()
        outs.append(o)
    a, b = outs
    for key in ("obs", "reward", "done", "kill"):
        assert torch.equal(a["roll"][key], b["roll"][key]), key
    assert all(torch.equal(x, y) for x, y in zip(a["step"], b["step"]))
    assert all(np.array_equal(x, y) for x, y in zip(a["host"], b["host"]))
    assert torch.equal(a["feat"].view(torch.int32), b["feat"].view(torch.int32))
    assert torch.equal(a["state"], b["state"])
    for e in envs:
        e.close()


# ------------------------------------------------------------------------------------------------ 6: arguments
def test_rejected_arguments():
    torch_cuda()
    from spacefortress_b200 import SFVecEnv, _lib
    env = SFVecEnv("youturn", num_envs=4, device=0, action_repeat=3)
    L, h = env.L, env.h
    assert env.action_repeat == 3 and L.sf_action_repeat(h) == 3
    for k in (0, -1, -5295, _lib.MAX_ACTION_REPEAT + 1, 1 << 30):
        assert L.sf_set_action_repeat(h, k) == _lib.SF_ERR_INVALID, k
        assert L.sf_action_repeat(h) == 3, k
    assert L.sf_set_action_repeat(h, _lib.MAX_ACTION_REPEAT) == _lib.SF_OK and L.sf_action_repeat(h) == _lib.MAX_ACTION_REPEAT
    assert L.sf_set_action_repeat(None, 2) == _lib.SF_ERR_INVALID and L.sf_action_repeat(None) == -1
    env.close()
    for k in (0, _lib.MAX_ACTION_REPEAT + 1):
        with pytest.raises(ValueError):
            SFVecEnv("youturn", num_envs=4, device=0, action_repeat=k)


# ------------------------------------------------------------------------------------------------ 7: SFVecEnv
def test_vec_env_contract():
    """Shapes and dtypes of step (numpy, torch) and rollout with action_repeat=2; SubprocVecEnv passes it through; a
    repeat-2 step equals two one-tick steps when no episode ends."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv, SubprocVecEnv, make_env
    n = 20
    env = SFVecEnv("autoturn", num_envs=n, device=0, action_repeat=2)
    one = SFVecEnv("autoturn", num_envs=n, device=0)
    assert env.action_repeat == 2 and one.action_repeat == 1
    o0, o1 = env.reset(), one.reset()
    assert np.array_equal(o0, o1)
    a = np.random.RandomState(0).randint(env.num_actions, size=n)
    obs, rew, done, info = env.step(a)
    assert obs.shape == (n, 1, 84, 84) and obs.dtype == np.uint8 and rew.shape == (n,) and done.dtype == np.bool_
    r1 = np.zeros(n, np.int64)
    for _ in range(2):
        obs1, rew1, d1, _k1 = one.step(a)
        r1 += rew1
    assert np.array_equal(obs, obs1) and np.array_equal(rew.astype(np.int64), r1) and not done.any()
    ot, rt, dt, kt = env.step(torch.zeros(n, dtype=torch.int32, device="cuda"))
    assert ot.is_cuda and tuple(ot.shape) == (n, 1, 84, 84) and ot.dtype == torch.uint8 and rt.dtype == torch.int32 and dt.dtype == torch.bool
    out = env.rollout(5)
    assert tuple(out["obs"].shape) == (5, n, 1, 84, 84) and tuple(out["reward"].shape) == (5, n)
    assert env._t == 7
    assert env.get_state()[0].tick == 14
    env.close(); one.close()
    envs = SubprocVecEnv([make_env("SpaceFortress-youturn-image-v0", 0, i) for i in range(6)], action_repeat=2)
    assert envs.action_repeat == 2 and envs.L.sf_action_repeat(envs.h) == 2
    obs = envs.reset()
    obs, rew, done, infos = envs.step(np.zeros(6, np.int64))
    assert obs.shape == (6, 1, 84, 84) and len(infos) == 6 and isinstance(infos[0], bool)
    assert envs.get_state()[0].tick == 2
    envs.close()
    f = SFVecEnv("youturn", num_envs=n, device=0, obs_type="features", action_repeat=3)
    f.reset()
    x, _, _, _ = f.step(np.zeros(n, np.int32))
    assert x.shape == (n, f.num_features) and x.dtype == np.float32 and f.get_state()[0].tick == 3
    assert tuple(f.rollout(4)["obs"].shape) == (4, n, f.num_features) and f.get_state()[0].tick == 15
    f.close()


def test_graphed_rollout_equals_the_eager_one_with_repeat():
    """OnDeviceRollout(graph=True) captures the two launches of a repeated step with frames and replays them: the same
    actions, frames, rewards and values as the eager loop, action_repeat=2."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    from spacefortress_b200.rollout import OnDeviceRollout, SFGRUPolicy

    class Greedy(SFGRUPolicy):
        def act(self, obs, state, mask, **kw):
            kw["deterministic"] = True
            return SFGRUPolicy.act(self, obs, state, mask, **kw)
    n, T = 96, 6
    outs = []
    for graph in (False, True):
        env = SFVecEnv("youturn", num_envs=n, device=0, action_repeat=2)
        torch.manual_seed(3)
        ro = OnDeviceRollout(env, Greedy(env.num_actions).cuda().eval(), num_steps=T, graph=graph)
        got = []
        for _ in range(2):
            ro.collect()
            torch.cuda.synchronize()
            got.append([x.clone() for x in (ro.actions, ro.frames, ro.rewards, ro.dones, ro.values, ro.valid_hist)])
        assert env.get_state()[0].tick == 2 * 2 * T
        outs.append(got)
        env.close()
    for r in range(2):
        for a, b in zip(outs[0][r], outs[1][r]):
            assert torch.equal(a, b), r
