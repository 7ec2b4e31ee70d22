"""GPU (-m gpu): final observations at auto-reset (sf_set_final_obs, SFVecEnv(final_obs=True)). While the setting is
enabled every stepping call writes final_step[i] (the agent step whose events carry SF_EV_EPISODE_RESET, or -1) and, for
the envs that ended, the frame / feature row of the state after the ending tick and before the new game. The finished
state is checked against the CPU oracle and bit for bit against sf_render / sf_features of the same state reached under
SF_FLAG_NO_AUTORESET; everything else a call returns or leaves behind must equal the disabled run."""
import ctypes as C

import numpy as np
import pytest

from gpu_helpers import (GAMETYPES, KINDS, STEP_OUTPUTS, assert_state_close, make, oracle_agent_step, oracle_features, oracles,
                         outputs, ptrs, rollout, rollout_features, stagger, step_host, torch_cuda, vp)
from oracle.oracle import draw_native, draw_obs

pytestmark = pytest.mark.gpu

NAT = 92 * 90  # bytes of the largest frame: one frame slot per env covers both layouts
ROWS = 19      # floats of the widest feature row
SENTINEL_U8, SENTINEL_F32, SENTINEL_STEP = 0xA5, 12345.5, -7


def register(env):
    """device final buffers filled with sentinels, registered on env's handle: {"frames" [n, NAT] u8, "rows" [n, ROWS]
    f32, "step" [n] i32}"""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n = env.num_envs
    fin = dict(frames=torch.full((n, NAT), SENTINEL_U8, dtype=torch.uint8, device="cuda"),
               rows=torch.full((n, ROWS), SENTINEL_F32, dtype=torch.float32, device="cuda"),
               step=torch.full((n,), SENTINEL_STEP, dtype=torch.int32, device="cuda"))
    _lib.check(env.L.sf_set_final_obs(env.h, vp(fin["frames"]), vp(fin["rows"]), vp(fin["step"])))
    assert env.L.sf_final_obs_enabled(env.h) == 1
    return fin


def frames_of(fin, per):
    """the frame slots of the registered buffer as [n, per] (env i's slot starts at i * per)"""
    return fin["frames"].view(-1)[:fin["frames"].shape[0] * per].view(-1, per)


def rows_of(fin, nf):
    return fin["rows"].view(-1)[:fin["rows"].shape[0] * nf].view(-1, nf)


def kill_some(env, every=3):
    """ships of every `every`-th env dead from now (death timer 0: they respawn 30 ticks later), so that episodes end
    with dead ships and the explosion caches are in play"""
    recs = env.get_state()
    for i in range(0, env.num_envs, every):
        recs[i].ship_alive = 0
        recs[i].ship_death_timer = 0
    env.set_state(recs)


# ------------------------------------------------------------------------------------------------ the oracle
@pytest.mark.parametrize("p", [0.0, 0.25])
@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("gametype", GAMETYPES)
def test_final_observations_equal_the_oracle(gametype, k, p):
    """One sf_rollout with 84x84 frames, one with native frames and one sf_rollout_features per kind, from one state with
    the episode ends staggered over every tick position of an agent step: final_step is the agent step of
    SF_EV_EPISODE_RESET, the final frames are the oracle's frames of the finished state, the final rows its features."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, seed = 40, 11
    ends = 1 + (5 if k > 1 else 3) * np.arange(n)
    T = int(ends.max()) // k + 2
    kw = dict(seeds=7, action_repeat=k, warm=30, repeat_action_probability=p, sticky_seed=seed)
    a = make(gametype, n, **kw)
    b = make(gametype, n, native_obs=True, **kw)
    c = make(gametype, n, render=False, **kw)
    for env in (a, b, c):
        kill_some(env)
        stagger(env, ends)
    start = a.save_envs()
    fa, fb, fc = register(a), register(b), register(c)
    orc = oracles(gametype, a.get_state())
    acts = np.random.RandomState(k * 7 + len(gametype)).randint(a.num_actions, size=(T, n)).astype(np.int32)
    da = torch.from_numpy(acts).cuda()
    ga = {key: v.cpu().numpy() for key, v in rollout(a, T, da, flags=a._flags).items()}
    rollout(b, T, da, flags=b._flags)
    gc = {}
    for kind in KINDS:
        c.load_envs(start)
        gc[kind] = rollout_features(c, kind, T, da)
        torch.cuda.synchronize()
        gc[kind]["final_rows"] = rows_of(fc, c.L.sf_num_features(c.h, _lib.OBS_TYPES[kind])).cpu().numpy()
        gc[kind]["final_step"] = fc["step"].cpu().numpy()
    ev = gc["features"]["events"].cpu().numpy().view(np.uint32)
    fra, frb = frames_of(fa, 84 * 84).cpu().numpy(), frames_of(fb, NAT).cpu().numpy()
    youturn = gametype in ("youturn", "test-youturn")
    features_of = lambda o: {kind: oracle_features(o, kind, youturn) for kind in KINDS}  # noqa: E731
    positions, dead = set(), 0
    for i in range(n):
        end_t = -1
        for t in range(T):
            R, D, K, EV, ran, end = oracle_agent_step(orc[i], orc[i].keymask(int(acts[t, i])), k, p, seed, i, features_of=features_of)
            assert (R, D, K, EV) == (int(ga["reward"][t, i]), bool(ga["done"][t, i]), bool(ga["kill"][t, i]), int(ev[t, i])), (t, i)
            if D:
                end_t = t
                positions.add(ran - 1)
                s, feats = end
                dead += not s.ship_alive
                assert np.array_equal(draw_obs(s).reshape(-1), fra[i]), ("84x84", t, i)
                assert np.array_equal(draw_native(s).reshape(-1), frb[i]), ("native", t, i)
                for kind in KINDS:
                    got = gc[kind]["final_rows"][i]
                    if kind == "monitors":
                        assert (got != feats[kind].astype(np.float32)).mean() <= 0.1, (kind, t, i, got, feats[kind])
                    else:
                        assert np.allclose(got, feats[kind].astype(np.float32), rtol=1e-6, atol=1e-6), (kind, t, i, got, feats[kind])
        assert end_t >= 0, i
        assert int(fa["step"][i]) == end_t and int(fb["step"][i]) == end_t, i
        for kind in KINDS:
            assert gc[kind]["final_step"][i] == end_t, (kind, i)
        assert bool(ev[end_t, i] & _lib.EV_EPISODE_RESET) and not (np.delete(ev[:, i], end_t) & _lib.EV_EPISODE_RESET).any()
    assert positions == set(range(k)), positions
    assert dead > 0
    recs = a.get_state()
    for i in range(n):
        assert_state_close(orc[i].get_state(), recs[i], ("final", i))
    for env in (a, b, c):
        env.close()


# ------------------------------------------------------------------------------------------------ bit for bit
def reference_finals(env, ref, probe, start, acts, flags, kind=None):
    """final_step, final frames [n, per] and final rows of one T-step run from `start`, built without the setting: `ref`
    steps one agent step at a time (saving the envs before each step); for the envs that end at step t, `probe` loads the
    saved rows and steps them under SF_FLAG_NO_AUTORESET, then sf_render / sf_features shows the finished state."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T = env.num_envs, len(acts)
    native = bool(flags & _lib.FLAG_NATIVE_OBS)
    per = NAT if native else 84 * 84
    ref.load_envs(start)
    step = np.full(n, -1, np.int32)
    frames = np.zeros((n, per), np.uint8)
    nf = env.L.sf_num_features(env.h, _lib.OBS_TYPES[kind or "features"])
    rows = np.zeros((n, nf), np.float32)
    done = torch.empty(n, dtype=torch.uint8, device="cuda")
    render = torch.empty((n, per), dtype=torch.uint8, device="cuda")
    feat = torch.empty((n, nf), dtype=torch.float32, device="cuda")
    for t in range(T):
        blob = ref.save_envs()
        _lib.check(ref.L.sf_step(ref.h, vp(acts[t]), None, None, vp(done), None, None, 0, None))
        ended = done.cpu().numpy().astype(bool)
        if not ended.any():
            continue
        step[ended] = t
        probe.load_envs(blob)
        _lib.check(probe.L.sf_step(probe.h, vp(acts[t]), None, None, None, None, None, _lib.FLAG_NO_AUTORESET, None))
        _lib.check(probe.L.sf_render(probe.h, vp(render), flags & _lib.FLAG_NATIVE_OBS, None))
        _lib.check(probe.L.sf_features(probe.h, _lib.OBS_TYPES[kind or "features"], vp(feat), None))
        torch.cuda.synchronize()
        frames[ended] = render.cpu().numpy()[ended]
        rows[ended] = feat.cpu().numpy()[ended]
    return step, frames, rows


@pytest.mark.parametrize("k,p", [(1, 0.0), (3, 0.25)])
def test_final_observations_equal_sf_render_and_sf_features_of_the_finished_state(k, p):
    """sf_rollout (84x84 and native), T x sf_step, T x sf_step_host (delta updates), sf_rollout_features (3 kinds) and
    T x sf_step_host_features: final_step, the final frames and rows equal sf_render / sf_features of the finished state,
    bit for bit; the slots of envs that did not end keep their sentinels."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T = 300, 8
    kw = dict(seeds=3, action_repeat=k, warm=20, ends=(1, T * k + 12), repeat_action_probability=p, sticky_seed=5)
    env = make("youturn", n, **kw)
    kill_some(env)
    nat = make("youturn", n, native_obs=True, reset=False, **dict(kw, warm=0, ends=None))
    ref = make("youturn", n, reset=False, **dict(kw, warm=0, ends=None))
    probe = make("youturn", n, reset=False, **dict(kw, warm=0, ends=None))
    start = env.save_envs()
    acts = torch.from_numpy(np.random.RandomState(1).randint(env.num_actions, size=(T, n)).astype(np.int32)).cuda()
    L = env.L
    fin, fin_nat = register(env), register(nat)

    def check(e, f, got_step, got_frames, got_rows, flags, kind, ctx):
        want_step, want_frames, want_rows = reference_finals(e, ref, probe, start, acts, flags, kind)
        assert (want_step >= 0).any() and not (want_step >= 0).all(), ctx
        assert np.array_equal(got_step, want_step), ctx
        ended = want_step >= 0
        if got_frames is not None:
            assert np.array_equal(got_frames[ended], want_frames[ended]), ctx
            assert (got_frames[~ended] == SENTINEL_U8).all(), ctx
        if got_rows is not None:
            assert np.array_equal(got_rows[ended].view(np.uint32), want_rows[ended].view(np.uint32)), ctx
            assert (got_rows[~ended] == SENTINEL_F32).all(), ctx

    def reset_sentinels(f):
        f["frames"].fill_(SENTINEL_U8); f["rows"].fill_(SENTINEL_F32); f["step"].fill_(SENTINEL_STEP)

    def gather(f, per, nf, calls):
        """T single-step calls: the final_step of call t becomes t, and the final slots are read after each call"""
        step = np.full(n, -1, np.int32)
        frames = np.full((n, per), SENTINEL_U8, np.uint8) if per else None
        rows = np.full((n, nf), SENTINEL_F32, np.float32) if nf else None
        for t in range(T):
            calls(t)
            torch.cuda.synchronize()
            s = f["step"].cpu().numpy()
            assert set(np.unique(s)) <= {-1, 0}, s
            ended = s == 0
            step[ended] = t
            if per:
                frames[ended] = frames_of(f, per).cpu().numpy()[ended]
            if nf:
                rows[ended] = rows_of(f, nf).cpu().numpy()[ended]
        return step, frames, rows

    # sf_rollout, 84x84 and native
    for e, f, per in ((env, fin, 84 * 84), (nat, fin_nat, NAT)):
        e.load_envs(start); reset_sentinels(f)
        rollout(e, T, acts, flags=e._flags)
        check(e, f, f["step"].cpu().numpy(), frames_of(f, per).cpu().numpy(), None, e._flags, None, ("sf_rollout", per))
        assert (f["rows"] == SENTINEL_F32).all()

    # T x sf_step
    env.load_envs(start); reset_sentinels(fin)
    obs = torch.empty((n, 84 * 84), dtype=torch.uint8, device="cuda")
    got = gather(fin, 84 * 84, 0, lambda t: _lib.check(L.sf_step(env.h, vp(acts[t]), vp(obs), None, None, None, None, _lib.FLAG_RENDER, None)))
    check(env, fin, got[0], got[1], None, env._flags, None, "sf_step")

    # T x sf_step_host with delta updates (page-locked buffers)
    env.load_envs(start); reset_sentinels(fin)
    hacts = acts.cpu().numpy()
    hobs = _lib.pinned_array((n, 84 * 84), np.uint8)
    got = gather(fin, 84 * 84, 0, lambda t: _lib.check(L.sf_step_host(env.h, C.c_void_p(np.ascontiguousarray(hacts[t]).ctypes.data), C.c_void_p(hobs.ctypes.data),
                                                                       None, None, None, None, _lib.FLAG_RENDER | _lib.FLAG_HOST_DELTA)))
    _lib.check(L.sf_host_forget(env.h, C.c_void_p(hobs.ctypes.data)))
    check(env, fin, got[0], got[1], None, env._flags, None, "sf_step_host")

    # sf_rollout_features, every kind; T x sf_step_host_features
    for kind in KINDS:
        nf = L.sf_num_features(env.h, _lib.OBS_TYPES[kind])
        env.load_envs(start); reset_sentinels(fin)
        rollout_features(env, kind, T, acts)
        check(env, fin, fin["step"].cpu().numpy(), None, rows_of(fin, nf).cpu().numpy(), 0, kind, ("sf_rollout_features", kind))
        assert (fin["frames"] == SENTINEL_U8).all()
    nf = L.sf_num_features(env.h, _lib.OBS_TYPES["monitors"])
    env.load_envs(start); reset_sentinels(fin)
    got = gather(fin, 0, nf, lambda t: step_host(env, hacts[t:t + 1], 0, want=("monitors",)))
    check(env, fin, got[0], None, got[2], 0, "monitors", "sf_step_host_features")
    for e in (env, nat, ref, probe):
        e.close()


# ------------------------------------------------------------------------------------------------ no change
@pytest.mark.parametrize("p", [0.0, 0.25])
@pytest.mark.parametrize("k", [1, 4])
@pytest.mark.parametrize("n", [1, 33, 4096, 4737])
def test_enabled_changes_nothing_else(n, k, p):
    """A handle with the setting enabled and one without, from one state with episode ends inside the run: every entry
    point gives the same observations, rewards, dones, kills, events, env state after each call and episode statistics;
    the host step's page-locked buffers hold the same bytes, with and without delta updates."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    T = 6
    kw = dict(seeds=n, action_repeat=k, warm=10, ends=(1, T * k + 4), repeat_action_probability=p, sticky_seed=2)
    on, off = make("autoturn", n, **kw), make("autoturn", n, **kw)
    for e in (on, off):
        kill_some(e, 4)
    start = on.save_envs()
    assert torch.equal(start, off.save_envs())
    fin = register(on)  # the buffers must outlive the registration
    acts = torch.from_numpy(np.random.RandomState(n + k).randint(on.num_actions, size=(T, n)).astype(np.int32)).cuda()
    hacts = acts.cpu().numpy()
    stats = []

    def run(e):
        e.load_envs(start)
        e.episode_stats(reset=True, all_reduce=False)
        o = {}
        o["roll"] = rollout(e, T, acts, flags=_lib.FLAG_RENDER)
        o["roll_state"] = e.save_envs()
        o["roll_syn"] = rollout(e, T, None, action_seed=4, t0=9, flags=0, want=("reward", "done", "kill"))
        o["steps"] = []
        out = outputs(e, T, ("obs",) + STEP_OUTPUTS)
        for t in range(T):
            _lib.check(e.L.sf_step(e.h, vp(acts[t]), *ptrs(out, ("obs",) + STEP_OUTPUTS, t), _lib.FLAG_RENDER, None))
        torch.cuda.synchronize()
        o["steps"] = out
        o["step_state"] = e.save_envs()
        for delta in (True, False):
            o["host", delta] = step_host(e, hacts, _lib.FLAG_RENDER | (_lib.FLAG_HOST_DELTA if delta else 0))
            o["host_state", delta] = e.save_envs()
        o["feat"] = rollout_features(e, "normalized-features", T, acts)
        o["hostfeat"] = step_host(e, hacts, 0, want=("features",) + STEP_OUTPUTS)
        o["state"] = e.save_envs()
        stats.append(e.episode_stats(reset=True, all_reduce=False))
        return o
    a, b = run(on), run(off)
    assert stats[0] == stats[1] and stats[0]["episodes"] > 0
    for key, x in a.items():
        y = b[key]
        if isinstance(x, dict):
            for name, v in x.items():
                if isinstance(v, np.ndarray):
                    assert np.array_equal(v.view(np.uint8), y[name].view(np.uint8)), (key, name)
                else:
                    assert torch.equal(v.view(torch.uint8), y[name].view(torch.uint8)), (key, name)
        else:
            assert torch.equal(x, y), key
    assert bool((fin["step"] >= -1).all())  # the last call wrote final_step
    on.close(); off.close()


def test_graphed_rollout_equals_the_eager_one_with_final_observations():
    """OnDeviceRollout(graph=True) captures the launches of a step with final frames (the memset of final_step, the
    deferred-reset step, the masked draw, the reset kernel and the draw) and replays them: two collects give the eager
    loop's actions, frames, rewards and values, and the same final buffers, state and episode statistics; the eager loop
    without the setting gives the same too."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    from spacefortress_b200.rollout import OnDeviceRollout, SFGRUPolicy

    class Greedy(SFGRUPolicy):
        def act(self, obs, state, mask, **kw):
            kw["deterministic"] = True
            return SFGRUPolicy.act(self, obs, state, mask, **kw)
    n, T = 96, 6
    outs = []
    for graph, final in ((False, True), (True, True), (False, False)):
        env = SFVecEnv("youturn", num_envs=n, device=0, action_repeat=2, final_obs=final)
        torch.manual_seed(3)
        ro = OnDeviceRollout(env, Greedy(env.num_actions).cuda().eval(), num_steps=T, graph=graph)
        stagger(env, 1 + np.arange(n) % (4 * T))
        got = []
        for _ in range(2):
            ro.collect()
            torch.cuda.synchronize()
            got.append([x.clone() for x in (ro.actions, ro.frames, ro.rewards, ro.dones, ro.values, ro.valid_hist)])
            if final:
                got.append([env.final_obs_buf.clone(), env.final_step_buf.clone()])
        got.append(env.save_envs())
        got.append(torch.tensor(list(env.episode_stats(all_reduce=False).values())))
        outs.append(got)
        env.close()
    assert int(outs[0][1][1].max()) >= 0 and int(outs[0][3][1].max()) >= 0  # episodes ended in the last step of a collect
    for x, y in zip(outs[0], outs[1]):
        for u, v in zip(x if isinstance(x, list) else [x], y if isinstance(y, list) else [y]):
            assert torch.equal(u, v)
    plain = [outs[0][0], outs[0][2], outs[0][4], outs[0][5]]
    for x, y in zip(plain, outs[2]):
        for u, v in zip(x if isinstance(x, list) else [x], y if isinstance(y, list) else [y]):
            assert torch.equal(u, v)


# ------------------------------------------------------------------------------------------------ edges
def test_no_autoreset_writes_only_minus_one():
    """Under SF_FLAG_NO_AUTORESET there is no auto-reset: final_step is all -1 and the frame and row slots keep their
    sentinels, on the frame route and the feature route."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T = 64, 10
    env = make("youturn", n, seeds=2, warm=5, ends=(1, T))
    fin = register(env)
    g = rollout(env, T, None, flags=_lib.FLAG_RENDER | _lib.FLAG_NO_AUTORESET)
    assert int(g["done"].sum()) > 0
    assert bool((fin["step"] == -1).all()) and bool((fin["frames"] == SENTINEL_U8).all()) and bool((fin["rows"] == SENTINEL_F32).all())
    fin["step"].fill_(SENTINEL_STEP)
    rollout_features(env, "features", T, None, flags=_lib.FLAG_NO_AUTORESET)
    assert bool((fin["step"] == -1).all()) and bool((fin["rows"] == SENTINEL_F32).all())
    env.close()


def test_a_call_longer_than_an_episode_is_rejected():
    """T * k > 5295 with the setting enabled: SF_ERR_INVALID before any launch, state and buffers unchanged; at
    T * k == 5295 the call runs."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n = 32
    env = make("autoturn", n, seeds=1, action_repeat=3, warm=3)
    fin = register(env)
    before = env.save_envs()
    L, h = env.L, env.h
    assert L.sf_rollout(h, 1766, None, 0, 0, None, None, None, None, 0, None) == _lib.SF_ERR_INVALID
    feats = torch.empty((1766, n, 17), dtype=torch.float32, device="cuda")
    assert L.sf_rollout_features(h, _lib.OBS_TYPES["features"], 1766, None, 0, 0, vp(feats), None, None, None, None, 0, None) == _lib.SF_ERR_INVALID
    torch.cuda.synchronize()
    assert torch.equal(env.save_envs(), before)
    assert bool((fin["step"] == SENTINEL_STEP).all())
    _lib.check(L.sf_rollout(h, 1765, None, 0, 0, None, None, None, None, 0, None))
    torch.cuda.synchronize()
    assert bool((fin["step"] >= -1).all())
    _lib.check(L.sf_set_final_obs(h, None, None, None))
    _lib.check(L.sf_rollout(h, 1766, None, 0, 0, None, None, None, None, 0, None))  # disabled: any T
    env.close()


def test_buffers_without_final_step_are_rejected():
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    env = make("youturn", 8, reset=False)
    L, h = env.L, env.h
    buf = torch.zeros((8, NAT), dtype=torch.uint8, device="cuda")
    assert L.sf_final_obs_enabled(h) == 0
    assert L.sf_set_final_obs(h, vp(buf), None, None) == _lib.SF_ERR_INVALID
    assert L.sf_set_final_obs(h, None, vp(buf), None) == _lib.SF_ERR_INVALID
    assert L.sf_final_obs_enabled(h) == 0
    fin = register(env)
    assert L.sf_set_final_obs(h, vp(buf), None, None) == _lib.SF_ERR_INVALID
    assert L.sf_final_obs_enabled(h) == 1  # unchanged
    _lib.check(L.sf_set_final_obs(h, None, None, vp(fin["step"])))  # final_step alone
    assert L.sf_final_obs_enabled(h) == 1
    _lib.check(L.sf_set_final_obs(h, None, None, None))
    assert L.sf_final_obs_enabled(h) == 0
    env.close()


def test_disabling_restores_the_plain_route():
    """A handle enabled, stepped and disabled again gives the bits of a handle that was never set (fused rollout frames,
    host step with delta updates, feature rollout, state)."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T = 200, 6
    a, b = make("youturn", n, seeds=4, warm=8, ends=(1, 3 * T)), make("youturn", n, seeds=4, warm=8, ends=(1, 3 * T))
    fin = register(a)
    rollout(a, 2, None, flags=_lib.FLAG_RENDER)
    rollout(b, 2, None, flags=_lib.FLAG_RENDER)
    _lib.check(a.L.sf_set_final_obs(a.h, None, None, None))
    assert a.L.sf_final_obs_enabled(a.h) == 0
    fin["step"].fill_(SENTINEL_STEP)
    acts = np.random.RandomState(0).randint(a.num_actions, size=(T, n)).astype(np.int32)
    ga, gb = [rollout(e, T, torch.from_numpy(acts).cuda(), flags=_lib.FLAG_RENDER) for e in (a, b)]
    for key in ga:
        assert torch.equal(ga[key], gb[key]), key
    ha, hb = [step_host(e, acts, _lib.FLAG_RENDER | _lib.FLAG_HOST_DELTA) for e in (a, b)]
    for key in ha:
        assert np.array_equal(ha[key], hb[key]), key
    assert a.host_delta_stats()[:2] == b.host_delta_stats()[:2]
    fa, fb = [rollout_features(e, "features", T, torch.from_numpy(acts).cuda()) for e in (a, b)]
    for key in fa:
        assert torch.equal(fa[key].view(torch.uint8), fb[key].view(torch.uint8)), key
    assert torch.equal(a.save_envs(), b.save_envs())
    assert bool((fin["step"] == SENTINEL_STEP).all())
    a.close(); b.close()


# ------------------------------------------------------------------------------------------------ Python contract
@pytest.mark.parametrize("obs_type,native", [("image", False), ("image", True), ("features", False), ("monitors", False)])
def test_vec_env_final_observations(obs_type, native):
    """SFVecEnv(final_obs=True): buffers of (N,) + obs_shape (uint8 frames / float32 rows) and final_step int32 [N];
    rollout() adds them to its dict; final_observations() gives the envs whose `done` is set and their rows; step()'s
    infos are unchanged. Without the option the rollout dict has its usual keys."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    n = 24
    env = SFVecEnv("autoturn", num_envs=n, device=0, obs_type=obs_type, native_obs=native, final_obs=True, copy_outputs=True)
    plain = SFVecEnv("autoturn", num_envs=n, device=0, obs_type=obs_type, native_obs=native, copy_outputs=True)
    features = obs_type != "image"
    assert env.final_obs and env.L.sf_final_obs_enabled(env.h) == 1 and plain.L.sf_final_obs_enabled(plain.h) == 0
    assert tuple(env.final_obs_buf.shape) == (n,) + env.obs_shape and env.final_obs_buf.is_cuda
    assert env.final_obs_buf.dtype == (torch.float32 if features else torch.uint8)
    assert tuple(env.final_obs_buf.shape[1:]) == ((env.num_features,) if features else ((1, 92, 90) if native else (1, 84, 84)))
    assert env.final_step_buf.dtype == torch.int32 and tuple(env.final_step_buf.shape) == (n,)
    for e in (env, plain):
        e.reset()
        stagger(e, 1 + np.arange(n) % 5)
    seen = 0
    for t in range(6):
        a = np.random.RandomState(t).randint(env.num_actions, size=n)
        obs, rew, done, infos = env.step(a)
        obs2, rew2, done2, infos2 = plain.step(a)
        assert isinstance(infos, tuple) and isinstance(infos[0], bool) and infos == infos2
        assert np.array_equal(obs, obs2) and np.array_equal(rew, rew2) and np.array_equal(done, done2)
        idx, fobs = env.final_observations()
        assert np.array_equal(idx, np.nonzero(done)[0]), t
        assert fobs.shape == (len(idx),) + env.obs_shape
        assert np.array_equal(fobs, env.final_obs_buf.cpu().numpy()[idx])
        seen += len(idx)
    assert seen > 0
    stagger(env, 1 + np.arange(n) % 6)
    out, out2 = env.rollout(4), plain.rollout(4)
    assert set(out2) == {"obs", "reward", "done", "kill"}
    assert set(out) == set(out2) | {"final_obs", "final_step"}
    step = out["final_step"].cpu().numpy()
    d = out["done"].cpu().numpy()
    for i in range(n):
        assert step[i] == (np.nonzero(d[:, i])[0][0] if d[:, i].any() else -1), i
    env.close(); plain.close()
    with pytest.raises(RuntimeError):
        SFVecEnv("youturn", num_envs=2, device=0).final_observations()


def test_subproc_vec_env_passes_the_option_through():
    torch_cuda()
    from spacefortress_b200 import SubprocVecEnv, DummyVecEnv, make_env
    for cls in (SubprocVecEnv, DummyVecEnv):
        envs = cls([make_env("SpaceFortress-youturn-image-v0", 0, i) for i in range(6)], final_obs=True)
        assert envs.final_obs and envs.L.sf_final_obs_enabled(envs.h) == 1
        envs.reset()
        stagger(envs, [1, 2, 1, 3, 1, 2])
        obs, rew, done, infos = envs.step(np.zeros(6, np.int64))
        assert obs.shape == (6, 1, 84, 84) and len(infos) == 6 and isinstance(infos[0], bool)
        idx, fobs = envs.final_observations()
        assert list(idx) == [0, 2, 4] and fobs.shape == (3, 1, 84, 84) and fobs.dtype == np.uint8
        envs.close()
