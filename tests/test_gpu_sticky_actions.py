"""GPU (-m gpu): sticky actions (sf_set_sticky_actions, SFVecEnv(repeat_action_probability=p, sticky_seed=s)). Before every
executed tick an env draws sf_sticky_draw(seed, global_env, rng_count, tick, p) from its pre-tick state; on "stick" the
tick runs with the keys the env holds instead of the action's, and the agent step reports SF_EV_STICKY. The CPU oracle,
drawing with the host form of the same function, must give the same bits on every stepping entry point."""
import ctypes as C

import numpy as np
import pytest

from gpu_helpers import (GAMETYPES, KINDS, STEP_OUTPUTS, assert_state_close, make, outputs, ptrs, rollout,
                         rollout_features, stagger, step_host, to_oracle_record, torch_cuda, vp)
from oracle.oracle import OracleEnv, draw_native, draw_obs

pytestmark = pytest.mark.gpu


def held_keys(s):
    """the key mask an env holds (its FIRE / THRUST / LEFT / RIGHT flags)"""
    from spacefortress_b200 import _lib
    return ((_lib.KEY_FIRE if s.fire_flag else 0) | (_lib.KEY_THRUST if s.thrust_flag else 0) |
            (_lib.KEY_LEFT if s.left_flag else 0) | (_lib.KEY_RIGHT if s.right_flag else 0))


def oracle_sticky_step(o, km, k, p, seed, genv, autoreset=True):
    """One agent step of the oracle: up to k ticks, each drawing from the pre-tick state whether it keeps the held keys,
    stopping on the tick the episode ends. (reward sum, done, kill, events OR, ticks run, the record at the episode end)"""
    from spacefortress_b200 import _lib
    L = _lib.lib()
    R, D, K, EV, end = 0, False, False, 0, None
    for j in range(k):
        s = o.state
        keys = km
        if L.sf_sticky_draw(seed, genv, s.rng_count, s.tick, p):
            keys = held_keys(s)
            EV |= _lib.EV_STICKY
        r, d, kl, e = o.step(keys)
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
    orc = []
    for r in recs:
        o = OracleEnv(gametype, 1)
        o.set_state(to_oracle_record(r))
        orc.append(o)
    return orc


# ------------------------------------------------------------------------------------------------ the oracle
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("p", [0.25, 0.75, 1.0])
@pytest.mark.parametrize("gametype", GAMETYPES)
def test_sticky_steps_equal_the_oracle(gametype, p, k):
    """sf_rollout with 84x84 frames, with native frames and sf_rollout_features (for the events) from one state, given
    actions, against OracleEnvs drawing with sf_sticky_draw: rewards, done, kill, events (SF_EV_STICKY included), every
    4th frame and every frame of an episode end, and the final records, bit for bit. Episodes end at every tick position
    of an agent step."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T, seed = 48, 160, 11
    kw = dict(seeds=7, action_repeat=k, warm=30, repeat_action_probability=p, sticky_seed=seed)
    a = make(gametype, n, **kw)
    b = make(gametype, n, native_obs=True, **kw)
    c = make(gametype, n, render=False, **kw)
    for env in (a, b, c):
        stagger(env, 1 + (5 if k > 1 else 3) * np.arange(n))
    assert torch.equal(a.save_envs(), b.save_envs()) and torch.equal(a.save_envs(), c.save_envs())
    orc = oracles(gametype, a.get_state())
    acts = np.random.RandomState(int(p * 100) + k * 7 + len(gametype)).randint(a.num_actions, size=(T, n)).astype(np.int32)
    da = torch.from_numpy(acts).cuda()
    ga, gb = [{key: v.cpu().numpy() for key, v in rollout(env, T, da, flags=env._flags).items()} for env in (a, b)]
    gc = {key: v.cpu().numpy() for key, v in rollout_features(c, "features", T, da).items()}
    for key in ("reward", "done", "kill"):
        assert np.array_equal(ga[key], gb[key]) and np.array_equal(ga[key], gc[key]), key
    ev = gc["events"].view(np.uint32)
    positions, sticky = set(), 0
    for t in range(T):
        for i in range(n):
            R, D, K, EV, ran, _ = oracle_sticky_step(orc[i], orc[i].keymask(int(acts[t, i])), k, p, seed, i)
            assert (R, D, K, EV) == (int(ga["reward"][t, i]), bool(ga["done"][t, i]), bool(ga["kill"][t, i]), int(ev[t, i])), (gametype, p, k, t, i)
            sticky += bool(EV & _lib.EV_STICKY)
            if D:
                positions.add(ran - 1)
            if D or t % 4 == 0 or t == T - 1:
                s = orc[i].get_state()
                assert np.array_equal(draw_obs(s), ga["obs"][t, i]), ("84x84", gametype, p, k, t, i)
                assert np.array_equal(draw_native(s), gb["obs"][t, i]), ("native", gametype, p, k, t, i)
    assert positions == set(range(k)), positions
    assert 0 < sticky and (p < 1.0 or sticky == T * n)
    recs = a.get_state()
    for i in range(n):
        assert_state_close(orc[i].get_state(), recs[i], (gametype, p, k, "final", i))
    assert bytes(recs) == bytes(b.get_state()) and bytes(recs) == bytes(c.get_state())
    for env in (a, b, c):
        env.close()


# ------------------------------------------------------------------------------------------------ p = 0 and p = 1
def test_p_zero_is_the_plain_step_on_every_entry_point():
    """A handle set to p = 0 (after 0.5) gives byte-identical outputs and state to a handle that was never set, on
    sf_rollout, sf_step, sf_step_host, sf_rollout_features and sf_step_host_features."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv, _lib
    n, T = 300, 6
    envs = []
    for p in (None, 0.0):
        e = SFVecEnv("youturn", num_envs=n, device=0, seeds=2)
        if p is None:  # undo the constructor's call: a handle that has never been set
            e.L.sf_destroy(e.h)
            h = C.c_void_p()
            _lib.check(e.L.sf_create(b"youturn", 1, n, 0, C.byref(h)))
            e.h = h
            e.seed_streams(2)
            assert e.L.sf_sticky_actions(e.h) == 0.0
        else:
            _lib.check(e.L.sf_set_sticky_actions(e.h, 0.5, 3))
            _lib.check(e.L.sf_set_sticky_actions(e.h, p, 3))
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
        o["feat"] = rollout_features(e, "features", T, acts)
        o["hostfeat"] = step_host(e, acts.cpu().numpy(), 0, want=("monitors",) + STEP_OUTPUTS)
        o["state"] = e.save_envs()
        outs.append(o)
    a, b = outs
    for key in ("obs", "reward", "done", "kill"):
        assert torch.equal(a["roll"][key], b["roll"][key]), key
    assert all(torch.equal(x, y) for x, y in zip(a["step"], b["step"]))
    assert all(np.array_equal(x, y) for x, y in zip(a["host"], b["host"]))
    for key, x in a["feat"].items():
        assert torch.equal(x.view(torch.uint8), b["feat"][key].view(torch.uint8)), key
    for key, x in a["hostfeat"].items():
        assert np.array_equal(x.view(np.uint8), b["hostfeat"][key].view(np.uint8)), key
    assert not (a["feat"]["events"] & _lib.EV_STICKY).any()
    assert torch.equal(a["state"], b["state"])
    for e in envs:
        e.close()


@pytest.mark.parametrize("k", [1, 2])
def test_p_one_from_a_fresh_reset_holds_no_keys(k):
    """From a reset every env holds no keys, so at p = 1 every tick is a tick of the all-zero key mask, whatever the
    actions, through auto-resets too: the outputs (SF_EV_STICKY aside, which every agent step sets), frames, feature rows
    and final state of a p = 0 handle stepping key mask 0."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T = 200, 12
    ends = 1 + np.arange(n) % (T * k)
    s = make("youturn", n, seeds=5, action_repeat=k, repeat_action_probability=1.0, sticky_seed=9)
    z = make("youturn", n, seeds=5, action_repeat=k)
    stagger(s, ends); stagger(z, ends)
    start = s.save_envs()
    acts = torch.from_numpy(np.random.RandomState(1).randint(1, 5, size=(T, n)).astype(np.int32)).cuda()
    zero = torch.zeros((T, n), dtype=torch.int32, device="cuda")
    km = _lib.FLAG_ACTIONS_ARE_KEYMASKS
    gs = rollout(s, T, acts, flags=_lib.FLAG_RENDER)
    gz = rollout(z, T, zero, flags=_lib.FLAG_RENDER | km)
    for key in ("obs", "reward", "done", "kill"):
        assert torch.equal(gs[key], gz[key]), key
    assert int(gs["done"].sum()) > 0
    assert torch.equal(s.save_envs(), z.save_envs())
    s.load_envs(start); z.load_envs(start)
    fs = rollout_features(s, "features", T, acts)
    fz = rollout_features(z, "features", T, zero, flags=km)
    assert bool((fs["events"] & _lib.EV_STICKY == _lib.EV_STICKY).all())
    fs["events"] &= ~_lib.EV_STICKY
    for key in fs:
        assert torch.equal(fs[key].view(torch.uint8), fz[key].view(torch.uint8)), key
    s.close(); z.close()


# ------------------------------------------------------------------------------------------------ entry points
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("n", [1, 33, 4096, 4737])
def test_entry_points_agree(n, k):
    """From one start state with p = 0.25 (clocks staggered so that episodes end inside the run): sf_rollout with and
    without frames (synthetic and given actions), T x sf_step, sf_step_host (page-locked with and without delta updates,
    pageable; 84x84 and native), sf_rollout_features (3 kinds) and sf_step_host_features give the same rewards, dones,
    kills, events and final state; frame t is sf_render after agent step t, feature row t is sf_features after it."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    T, seed, t0 = 10, 3, 17
    env = make("youturn", n, seeds=n, action_repeat=k, warm=12, ends=(1, T * k + 4), repeat_action_probability=0.25,
               sticky_seed=seed)
    L, h = env.L, env.h
    start = env.save_envs()
    acts = env.synthetic_actions(T, action_seed=seed, t0=t0)
    da = torch.from_numpy(acts).cuda()

    nat = make("youturn", n, seeds=n, action_repeat=k, warm=12, ends=(1, T * k + 4), repeat_action_probability=0.25,
               sticky_seed=seed, native_obs=True)  # for the host step's native frame buffers

    def restart():
        env.load_envs(start)
        nat.load_envs(start)
        torch.cuda.synchronize()

    def same(a, b, ctx):
        assert torch.equal(a, b), ctx

    # the reference: T x (sf_step, sf_render, sf_features of every kind), and the same with native frames
    ref = {}
    for native in (False, True):
        restart()
        fl = _lib.FLAG_NATIVE_OBS if native else 0
        shape = (92, 90) if native else (84, 84)
        r = outputs(env, T, STEP_OUTPUTS + tuple(KINDS))
        r["obs"] = torch.empty((T, n) + shape, dtype=torch.uint8, device="cuda")
        render = torch.empty((n,) + shape, dtype=torch.uint8, device="cuda")
        for t in range(T):
            _lib.check(L.sf_step(h, vp(da[t]), *ptrs(r, ("obs",) + STEP_OUTPUTS, t), _lib.FLAG_RENDER | fl, None))
            _lib.check(L.sf_render(h, vp(render), fl, None))
            torch.cuda.synchronize()
            same(render, r["obs"][t], ("sf_step frame == sf_render", native, t))
            for kind in KINDS:
                _lib.check(L.sf_features(h, _lib.OBS_TYPES[kind], vp(r[kind][t]), None))
        torch.cuda.synchronize()
        ref[native] = r
    end = env.save_envs()
    for key in STEP_OUTPUTS + tuple(KINDS):
        same(ref[False][key].view(torch.uint8), ref[True][key].view(torch.uint8), ("native", key))
    r0 = ref[False]
    assert int(r0["done"].sum()) > 0 and bool((r0["events"] & _lib.EV_EPISODE_RESET).any())
    assert bool((r0["events"] & _lib.EV_STICKY).any()) and not bool((r0["events"] & _lib.EV_STICKY).all())

    def check(got, ctx, native=False):
        """every output equals the reference's byte for byte (feature rows bit for bit), and so does the final state"""
        for name, x in got.items():
            same(torch.as_tensor(x, device="cuda").view(torch.uint8), ref[native][name].view(torch.uint8), (ctx, name))
        same((nat if native else env).save_envs(), end, (ctx, "final state"))

    for actions, case in ((None, "synthetic"), (da, "given")):
        for frames in (True, False):
            restart()
            got = rollout(env, T, actions, seed, t0, _lib.FLAG_RENDER if frames else 0, want=("obs",) * frames + ("reward", "done", "kill"))
            check(got, ("sf_rollout", case, frames))

    # sf_step_host: page-locked with delta updates, page-locked whole frames, pageable whole frames; 84x84 and native
    for native, e in ((False, env), (True, nat)):
        fl = _lib.FLAG_RENDER | (_lib.FLAG_NATIVE_OBS if native else 0)
        for pinned, delta in ((True, True), (True, False), (False, False)):
            restart()
            stats0 = e.host_delta_stats()
            check(step_host(e, acts, fl | (_lib.FLAG_HOST_DELTA if delta else 0), pinned), ("sf_step_host", native, pinned, delta), native)
            stats1 = e.host_delta_stats()
            if delta:  # the first call sends whole frames, the others delta updates, which are counted
                assert stats1[1] - stats0[1] == T - 1 and stats1[2] - stats0[2] == 1 and stats1[0] > stats0[0]
            else:
                assert stats1[2] - stats0[2] == T and stats1[1] == stats0[1]

    for kind in KINDS:
        for actions in (None, da):
            restart()
            check(rollout_features(env, kind, T, actions, seed, t0), ("sf_rollout_features", kind, actions is None))

    for pinned, kind in ((True, "normalized-features"), (False, "monitors")):
        restart()
        check(step_host(env, acts, 0, pinned, want=(kind,) + STEP_OUTPUTS), ("sf_step_host_features", kind))
    env.close(); nat.close()


# ------------------------------------------------------------------------------------------------ reproducibility
def test_restored_envs_continue_with_the_same_draws():
    """Save, step m agent steps; load the rows into a second handle with the same setting and label, step m: the same
    outputs and final state. Loaded into other slots (another label) the draws differ."""
    torch = torch_cuda()
    n, m = 256, 24
    kw = dict(action_repeat=2, repeat_action_probability=0.5, sticky_seed=21)
    a = make("autoturn", n, seeds=3, warm=20, ends=(1, 40), **kw)
    b = make("autoturn", n, seeds=99, **kw)
    blob = a.save_envs()
    acts = torch.from_numpy(np.random.RandomState(2).randint(a.num_actions, size=(m, n)).astype(np.int32)).cuda()
    ga = rollout(a, m, acts, flags=a._flags)
    b.load_envs(blob)
    gb = rollout(b, m, acts, flags=b._flags)
    for key in ga:
        assert torch.equal(ga[key], gb[key]), key
    assert torch.equal(a.save_envs(), b.save_envs())
    from spacefortress_b200 import _lib
    b.load_envs(blob)
    gq = rollout_features(b, "features", m, acts)
    perm = torch.roll(torch.arange(n, dtype=torch.int32, device="cuda"), 1)  # env i -> slot i + 1
    b.load_envs(blob, perm)
    gp = rollout_features(b, "features", m, torch.roll(acts, 1, dims=1))
    assert not torch.equal(torch.roll(gq["events"], 1, dims=1) & _lib.EV_STICKY, gp["events"] & _lib.EV_STICKY)
    a.close(); b.close()


def test_graphed_rollout_equals_the_eager_one_with_sticky_actions():
    """OnDeviceRollout(graph=True) captures the repeat-kernel and draw launches of a sticky step and replays them: graph
    replays draw afresh from the envs' state, so two collects give the eager loop's actions, frames, rewards and values."""
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
        env = SFVecEnv("youturn", num_envs=n, device=0, repeat_action_probability=0.25, sticky_seed=5)
        torch.manual_seed(3)
        ro = OnDeviceRollout(env, Greedy(env.num_actions).cuda().eval(), num_steps=T, graph=graph)
        got = []
        for _ in range(2):
            ro.collect()
            torch.cuda.synchronize()
            got.append([x.clone() for x in (ro.actions, ro.frames, ro.rewards, ro.dones, ro.values, ro.valid_hist)])
        got.append(env.save_envs())
        outs.append(got)
        env.close()
    for r in range(2):
        for a, b in zip(outs[0][r], outs[1][r]):
            assert torch.equal(a, b), r
    assert torch.equal(outs[0][2], outs[1][2])


def test_sharded_handles_equal_one_handle():
    """Two handles labelled first_global_env 0 and n/2, loaded with the halves of one handle's envs, step exactly as that
    handle does (synthetic actions, frames, sticky draws)."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    n, T, h2 = 512, 16, 256
    kw = dict(action_repeat=2, repeat_action_probability=0.25, sticky_seed=8)
    one = make("youturn", n, seeds=4, warm=10, ends=(1, 2 * T), **kw)
    blob = one.save_envs()
    halves = []
    for lo in (0, h2):
        e = SFVecEnv("youturn", num_envs=h2, device=0, first_global_env=lo, **kw)
        e.reset()
        e.load_envs(blob[lo:lo + h2].contiguous())
        halves.append(e)
    g = rollout(one, T, None, action_seed=6, flags=one._flags)
    parts = [rollout(e, T, None, action_seed=6, flags=e._flags) for e in halves]
    for key in g:
        assert torch.equal(g[key], torch.cat([p[key] for p in parts], dim=1)), key
    assert torch.equal(one.save_envs(), torch.cat([e.save_envs() for e in halves]))
    for e in [one] + halves:
        e.close()


# ------------------------------------------------------------------------------------------------ statistics
def test_sticky_rate_is_p():
    """4096 envs x 256 one-tick steps at p = 0.25: the rate of SF_EV_STICKY is within 5 sigma of p, and with
    sticky_seed == action_seed so is the rate among the ticks of each synthetic action value."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T, p, seed = 4096, 256, 0.25, 13
    env = make("youturn", n, seeds=1, ends=(1, 5000), render=False, repeat_action_probability=p, sticky_seed=seed)
    g = rollout_features(env, "features", T, None, seed, 0)
    st = ((g["events"] & _lib.EV_STICKY) != 0).cpu().numpy()
    acts = env.synthetic_actions(T, action_seed=seed, t0=0)

    def near(x, m):
        assert abs(x - p) < 5 * np.sqrt(p * (1 - p) / m), (x, m)
    near(st.mean(), st.size)
    for v in range(env.num_actions):
        sel = acts == v
        near(st[sel].mean(), int(sel.sum()))
    env.close()


# ------------------------------------------------------------------------------------------------ contract
def test_rejected_arguments_leave_the_setting():
    torch_cuda()
    from spacefortress_b200 import SFVecEnv, SubprocVecEnv, make_env, _lib
    env = SFVecEnv("youturn", num_envs=4, device=0, repeat_action_probability=0.3, sticky_seed=7)
    L, h = env.L, env.h
    assert env.repeat_action_probability == 0.3 and env.sticky_seed == 7 and L.sf_sticky_actions(h) == 0.3
    for p in (-0.1, -1e-300, 1.0000001, 2.0, float("nan"), float("inf"), float("-inf")):
        assert L.sf_set_sticky_actions(h, p, 1) == _lib.SF_ERR_INVALID, p
        assert L.sf_sticky_actions(h) == 0.3, p
    for p in (0.0, 1.0, 0.25):
        assert L.sf_set_sticky_actions(h, p, 1) == _lib.SF_OK and L.sf_sticky_actions(h) == p
    assert L.sf_set_sticky_actions(None, 0.1, 1) == _lib.SF_ERR_INVALID and L.sf_sticky_actions(None) == -1.0
    env.close()
    for p in (-0.5, 1.5, float("nan")):
        with pytest.raises(ValueError):
            SFVecEnv("youturn", num_envs=4, device=0, repeat_action_probability=p)
        with pytest.raises(ValueError):
            SubprocVecEnv([make_env("SpaceFortress-youturn-image-v0", 0, i) for i in range(3)], repeat_action_probability=p)
    for seed in (-1, 1 << 32):  # a uint32 on the handle: no silent aliasing of another seed
        with pytest.raises(ValueError):
            SFVecEnv("youturn", num_envs=4, device=0, repeat_action_probability=0.25, sticky_seed=seed)
    top = SFVecEnv("youturn", num_envs=4, device=0, repeat_action_probability=0.25, sticky_seed=(1 << 32) - 1)
    assert top.sticky_seed == (1 << 32) - 1
    top.close()


def test_vec_env_contract():
    """SFVecEnv with p = 1 from a reset holds no keys, so its steps equal a p = 0 env's no-op steps on the numpy, torch
    and rollout() paths, with the usual shapes and dtypes; SubprocVecEnv / DummyVecEnv pass the setting through."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv, SubprocVecEnv, DummyVecEnv, make_env
    n = 20
    s = SFVecEnv("autoturn", num_envs=n, device=0, repeat_action_probability=1.0, sticky_seed=2, action_repeat=2)
    z = SFVecEnv("autoturn", num_envs=n, device=0, action_repeat=2)
    assert s.repeat_action_probability == 1.0 and s.sticky_seed == 2 and z.repeat_action_probability == 0.0
    assert np.array_equal(s.reset(), z.reset())
    a = np.random.RandomState(0).randint(1, s.num_actions, size=n)
    so, sr, sd, si = s.step(a)
    zo, zr, zd, zi = z.step(np.zeros(n, np.int64))
    assert so.shape == (n, 1, 84, 84) and so.dtype == np.uint8 and sr.shape == (n,) and sd.dtype == np.bool_
    assert np.array_equal(so, zo) and np.array_equal(sr, zr) and np.array_equal(sd, zd)
    to, tr, td, tk = s.step(torch.ones(n, dtype=torch.int32, device="cuda"))
    uo, ur, ud, uk = z.step(torch.zeros(n, dtype=torch.int32, device="cuda"))
    assert to.is_cuda and tuple(to.shape) == (n, 1, 84, 84) and tr.dtype == torch.int32 and td.dtype == torch.bool
    assert torch.equal(to, uo) and torch.equal(tr, ur) and torch.equal(td, ud)
    rs, rz = s.rollout(5, action_seed=1), z.rollout(5, torch.zeros((5, n), dtype=torch.int32, device="cuda"))
    assert tuple(rs["obs"].shape) == (5, n, 1, 84, 84)
    for key in ("obs", "reward", "done", "kill"):
        assert torch.equal(rs[key], rz[key]), key
    assert s.get_state()[0].tick == 14
    s.close(); z.close()
    for cls in (SubprocVecEnv, DummyVecEnv):
        envs = cls([make_env("SpaceFortress-youturn-image-v0", 0, i) for i in range(6)], repeat_action_probability=0.25, sticky_seed=4)
        assert envs.repeat_action_probability == 0.25 and envs.sticky_seed == 4 and envs.L.sf_sticky_actions(envs.h) == 0.25
        envs.reset()
        obs, rew, done, infos = envs.step(np.zeros(6, np.int64))
        assert obs.shape == (6, 1, 84, 84) and len(infos) == 6 and isinstance(infos[0], bool)
        envs.close()
