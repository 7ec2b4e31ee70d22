"""GPU (-m gpu): the rest of the reference-facing surface, through the C-ABI, against the oracle / the compiled
reference core: feature observations (ssf_env.py:95-157, S8 computeExtra incl. quirk Q11), chorded action sets 0 / -1
(ssf_env.py:65-90), the `events` / `collisions` string getters (pymodule.cpp:136-143,182-197), the drop-in VecEnv's
output ownership, and the BASELINE.json configs at their own sizes (65 536-env soak, mixed game types, config-5
episode statistics)."""
import numpy as np
import pytest

from gpu_helpers import END_TICK, stagger, to_oracle_record, torch_cuda
from oracle.oracle import OracleEnv, RefEnv, ref_available

pytestmark = pytest.mark.gpu


def oracle_features(o, kind, youturn):
    """ssf_env.py:95-157 restated over the oracle's state and computeExtra (vdir, fdist, ndist, aim). Documented
    divergences of the product are followed: len(shells) counts shells and the vulnerability timer is the real one (the
    reference's getters for them are broken, pymodule.cpp:44-45,131-134)."""
    s = o.get_state()
    vdir, _fdist, ndist, aim = o.extra()
    nm, ns = bin(s.missile_mask).count("1"), bin(s.shell_mask).count("1")
    kill = 1 if s.vulnerability > 10 and s.fortress_vuln_timer < 250 else 0
    timers = [s.fire_timer, s.thrust_timer, s.left_timer, s.right_timer]
    timers = timers if youturn else timers[:2]
    if kind == "monitors":
        return np.array([0.5 if nm > 0 else -0.5, 0.5 if s.fortress_alive else -0.5, 0.5 if s.vulnerability > 10 else -0.5,
                         0.5 if kill else -0.5, 0.5 if aim < 3 else -0.5, 0.5 if aim > 3 else -0.5, 0.5 if ndist > .75 else -0.5,
                         0.5 if ndist > .25 else -0.5, 0.5 if ndist < -.25 else -0.5, 0.5 if ndist < -.75 else -0.5])
    if kind == "normalized-features":
        max_ticks = np.floor(180000 / 34)
        f = [1 if s.ship_alive else 0, s.ship_x / 90, s.ship_y / 92, s.ship_vx / 10, s.ship_vy / 10, s.ship_angle / 360, aim / 180,
             vdir % 360 / 360, ndist, 1 if s.fortress_alive else 0, s.fortress_angle / 360, max(s.vulnerability, 10) / 10, kill,
             nm / 20, ns / 20] + [x / max_ticks for x in timers]
        return np.clip(f, -1, 1)
    return np.array([bool(s.ship_alive), s.ship_x, s.ship_y, s.ship_vx, s.ship_vy, s.ship_angle, aim, vdir, ndist, bool(s.fortress_alive),
                     s.fortress_angle, s.vulnerability, kill, nm, ns] + timers, dtype=np.float64)


@pytest.mark.parametrize("gametype", ["youturn", "autoturn"])
@pytest.mark.parametrize("kind", ["features", "normalized-features", "monitors"])
def test_ssf_env_feature_observations_match_the_oracle(gametype, kind):
    """SSF_Env(obs_type=...) (single-env facade, float64 like np.array(f)) step by step against the oracle's state +
    computeExtra. fp64 atan2 on the device is within 2 ulp of libm's, hence the 1e-9 absolute bar; the monitors are
    thresholds of the same numbers (compared exactly unless a value sits within 1e-9 of its threshold)."""
    torch_cuda()
    from spacefortress_b200.gym.envs import SSF_Env
    youturn = gametype == "youturn"
    env = SSF_Env(gametype=gametype, obs_type=kind)
    o = OracleEnv(gametype, 1)
    f0 = env.reset(); o.reset()
    assert f0.dtype == np.float64 and f0.shape == ((10,) if kind == "monitors" else (19 if youturn else 17,))
    assert np.allclose(f0, oracle_features(o, kind, youturn), rtol=0, atol=1e-9)  # tick 0: vdir = aim = ndist = 0
    rng = np.random.RandomState(5)
    saw_dead = saw_q11 = False
    for t in range(900):
        a = int(rng.randint(env.action_space.n))
        f, r, d, k = env.step(a)
        ro, do, ko, _ = o.step(o.keymask(a))
        assert (r, d, k) == (ro, do, ko), t
        exp = oracle_features(o, kind, youturn)
        if kind == "monitors":
            _, _, ndist, aim = o.extra()
            near = min(abs(aim - 3), abs(abs(ndist) - .75), abs(abs(ndist) - .25)) < 1e-9
            assert near or np.array_equal(f, exp), (t, f, exp)
        else:
            assert np.allclose(f, exp, rtol=0, atol=1e-9), (t, f - exp)
        s = o.get_state()
        saw_dead |= not s.ship_alive
        # Q11: fdist ignores the y distance, so ndist is NOT the true normalised distance when the ship is above / below the fortress
        true_nd = -1 + (np.hypot(s.ship_x - 355, s.ship_y - 315) - 40) / 80
        saw_q11 |= abs(true_nd - o.extra()[2]) > 0.2
    assert saw_dead and saw_q11
    env.close()


@pytest.mark.parametrize("gametype", ["youturn", "autoturn"])
def test_batched_feature_observations(gametype):
    """SFVecEnv(obs_type=...) returns the [N, F] float32 matrix of sf_features; rows equal the oracle's features of the
    same env (float32 of the fp64 values, 1e-6 relative)."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    n, youturn = 96, gametype == "youturn"
    for kind in ("features", "normalized-features", "monitors"):
        env = SFVecEnv(gametype, num_envs=n, device=0, obs_type=kind, seeds=11)
        oracles = [OracleEnv(gametype, 11 + i) for i in range(n)]
        f = env.reset()
        assert f.dtype == np.float32 and f.shape == (n, 10 if kind == "monitors" else (19 if youturn else 17))
        assert env.observation_space.shape == f.shape[1:]
        rng = np.random.RandomState(3)
        for t in range(120):
            a = rng.randint(env.num_actions, size=n)
            f, r, d, k = env.step(a)
            for i in range(n):
                oracles[i].step(oracles[i].keymask(int(a[i])))
            if t % 10 == 9 or t < 3:
                exp = np.stack([oracle_features(oracles[i], kind, youturn) for i in range(n)])
                if kind == "monitors":
                    assert (f != exp.astype(np.float32)).mean() < 0.002, t
                else:
                    assert np.allclose(f, exp.astype(np.float32), rtol=1e-6, atol=1e-6), (kind, t, np.abs(f - exp).max())
        # the same numbers from the device path (torch actions in, torch features out)
        ft, _, _, _ = env.step(torch.zeros(n, dtype=torch.int32, device="cuda"))
        assert ft.is_cuda and tuple(ft.shape) == f.shape
        env.close()


@pytest.mark.parametrize("gametype,action_set,ncols", [("youturn", 0, 4), ("youturn", -1, 4), ("autoturn", 0, 2), ("autoturn", -1, 4),
                                                       ("test-youturn", -1, 4), ("test-autoturn", 0, 2)])
def test_chorded_action_sets_through_the_product(gametype, action_set, ncols):
    """action_set 0 / -1 (ssf_env.py:65-90): the product's action -> key table (sf_action_keymask) is the reference's
    np.meshgrid(...).T.reshape table, and stepping with action a equals the oracle stepped with that row's keys."""
    torch_cuda()
    from spacefortress_b200 import SFVecEnv, _lib
    table = np.array(np.meshgrid(*([[0, 1]] * ncols))).T.reshape(-1, ncols)
    youturn = gametype in ("youturn", "test-youturn")
    n = len(table)
    env = SFVecEnv(gametype, num_envs=n, device=0, action_set=action_set)
    assert env.num_actions == n == env.action_space.n
    bits = (_lib.KEY_FIRE, _lib.KEY_THRUST, _lib.KEY_LEFT, _lib.KEY_RIGHT)
    for a in range(n):
        km = env.L.sf_action_keymask(env.h, a)
        keys = [int(bool(km & bits[c])) for c in range(ncols)]
        expect = table[a].tolist() if youturn else table[a].tolist()[:2] + [0] * (ncols - 2)  # autoturn reads keystate[0:2] only
        assert keys == expect, (a, km)
    # env i always plays action i: the chord held down
    env.reset()
    oracles = [OracleEnv(gametype, 1) for _ in range(n)]
    acts = np.arange(n)
    for t in range(150):
        # alternate with NOOP (row 0) so that fire has press edges
        cur = acts if t % 3 else np.zeros(n, np.int64)
        obs, r, d, k = env.step(cur)
        for i in range(n):
            row = table[int(cur[i])]
            km = sum(bits[c] for c in range(ncols) if row[c])
            ro, do, ko, _ = oracles[i].step(km if youturn else km & 3)
            assert (int(r[i]), bool(d[i]), bool(k[i])) == (ro, do, ko), (t, i)
        if t % 50 == 49:
            for i in (0, n // 2, n - 1):
                assert np.array_equal(obs[i, 0], oracles[i].obs()), (t, i)
    env.close()


@pytest.mark.skipif(not ref_available(), reason="oracle/_ref/libsfref.so not built (needs /root/reference)")
@pytest.mark.parametrize("gametype", ["youturn", "autoturn"])
def test_event_and_collision_strings_match_the_reference(gametype):
    """Game.events / Game.collisions (pymodule.cpp:136-143,182-197) against the compiled reference core, tick by tick,
    with the key calls of SSF_Env.step (ssf_env.py:213-229). The device keeps one bit per event kind: ticks in which
    the reference logs a kind twice (two missiles hitting) are compared as sets."""
    torch_cuda()
    from spacefortress_b200.core import Game
    youturn = gametype == "youturn"
    g = Game(gametype, width=90, height=92, viewport=(130, 80, 450, 460), lw=3, grayscale=True)
    ref = RefEnv(gametype, 1)
    rng = np.random.RandomState(2)
    seen, repeats = set(), 0
    for t in range(2500):
        km = int(rng.randint(16)) if t % 7 else 1   # plenty of fire edges
        (g.press_key if km & 1 else g.release_key)(1)
        (g.press_key if km & 2 else g.release_key)(2)
        if youturn:
            (g.press_key if km & 4 else g.release_key)(3)
            (g.press_key if km & 8 else g.release_key)(4)
        r = g.step_one_tick(34)
        assert r == ref.core_step(km), t
        ev_ref, ev = ref.events(), g.events
        if len(set(ev_ref)) == len(ev_ref):
            assert ev == ev_ref, (t, ev, ev_ref)
        else:
            repeats += 1
            assert set(ev) == set(ev_ref), (t, ev, ev_ref)
        assert g.collisions == ref.collisions(), (t, g.collisions, ref.collisions())
        seen.update(ev_ref)
    need = ["missile-fired", "ship-respawn", "press-fire", "release-thrust"]
    need += ["press-left", "release-right"] if youturn else ["fortress-fired", "shell-hit-ship"]  # (a random youturn ship flies out first)
    for name in need:
        assert name in seen, name
    assert ("explode-bighex" in seen) or ("explode-smallhex" in seen)


def test_kill_events_and_collisions_on_the_scripted_kill_path():
    """The same getters on the double-shot kill path (hit-fortress, vlner-increased, fortress-destroyed, fortress-respawn,
    the 'missile' collision) against the reference core."""
    if not ref_available():
        pytest.skip("oracle/_ref/libsfref.so not built")
    torch_cuda()
    from conftest import scripted_kill_policy
    from spacefortress_b200.core import Game
    g = Game("autoturn", width=90, height=92, viewport=(130, 80, 450, 460), lw=3, grayscale=True)
    ref = RefEnv("autoturn", 1)
    seen = set()
    for t in range(3000):
        km = scripted_kill_policy(t, ref.get_state().vulnerability)
        (g.press_key if km & 1 else g.release_key)(1)
        (g.press_key if km & 2 else g.release_key)(2)
        assert g.step_one_tick(34) == ref.core_step(km), t
        ev_ref = ref.events()
        if len(set(ev_ref)) == len(ev_ref):
            assert g.events == ev_ref, (t, g.events, ev_ref)
        else:
            assert set(g.events) == set(ev_ref), t
        assert g.collisions == ref.collisions(), t
        seen.update(ev_ref)
    for name in ("hit-fortress", "vlner-increased", "fortress-destroyed", "fortress-respawn", "hit-dead-fortress"):
        assert name in seen, name


def test_drop_in_vec_env_returns_fresh_arrays_and_fast_path_aliases():
    """SubprocVecEnv (the literal gym_vecenv drop-in) returns fresh arrays and a tuple of bools every step; SFVecEnv's
    default numpy path returns views of its page-locked buffers, which stay readable after close()."""
    torch_cuda()
    from spacefortress_b200 import SFVecEnv, SubprocVecEnv, make_env
    env = SubprocVecEnv([make_env("SpaceFortress-autoturn-image-v0", 0, i) for i in range(8)])
    env.reset()
    o1, r1, d1, i1 = env.step(np.ones(8, np.int64))
    keep = o1.copy()
    o2, r2, d2, i2 = env.step(np.zeros(8, np.int64))
    assert o1 is not o2 and np.array_equal(o1, keep) and not np.shares_memory(o1, o2)
    assert isinstance(i1, tuple) and all(isinstance(x, bool) for x in i1) and r1.dtype == np.int64 and d1.dtype == np.bool_
    env.close()
    fast = SFVecEnv("autoturn", num_envs=8, device=0)
    fast.reset()
    oa, ra, da, ia = fast.step(np.ones(8, np.int64))
    ob, rb, db, ib = fast.step(np.zeros(8, np.int64))
    assert np.shares_memory(oa, ob) and ia.dtype == np.bool_ and int(sum(ia)) == int(ia.sum())
    snap = ob.copy()
    fast.close()
    del fast
    import gc
    gc.collect()
    assert np.array_equal(ob, snap)  # the pinned block lives as long as the array that was handed out


@pytest.mark.parametrize("gametype,native,n", [("youturn", False, 2500), ("autoturn", False, 6001), ("autoturn", True, 301)])
def test_host_delta_updates_equal_whole_frame_copies(gametype, native, n):
    """SF_FLAG_HOST_DELTA (SFVecEnv's default numpy path): the page-locked observation buffer, updated with only the
    64-byte granules that changed, equals the whole-frame copy at every step — across auto-resets (staggered clocks),
    an explicit reset(), device-path steps taken in between, with more groups than blocks (6001 envs: the blocks of the step
    kernel send the changes of several groups each) and for a frame size that is not a multiple of 16 bytes."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    a = SFVecEnv(gametype, num_envs=n, device=0, native_obs=native)                      # delta
    b = SFVecEnv(gametype, num_envs=n, device=0, native_obs=native, host_delta=False)    # whole frames
    rng = np.random.RandomState(3)
    for e in (a, b):
        e.reset()
        stagger(e, 1 + np.arange(n) % 37)
    per = a.obs_shape[1] * a.obs_shape[2]
    resets = 0
    for t in range(60):
        act = rng.randint(0, a.num_actions, size=n)
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert np.array_equal(oa, ob), (t, int((oa != ob).sum()))
        assert np.array_equal(ra, rb) and np.array_equal(da, db) and np.array_equal(ia, ib)
        resets += int(da.sum())
        if t == 20:   # the env's history changes under the buffer: the update is against the buffer's contents
            for e in (a, b):
                e.reset()
        if t == 30:
            dact = torch.from_numpy(act.astype(np.int32)).cuda()
            for e in (a, b):
                e.step(dact); e.step(dact)
    assert resets > n // 2  # the envs whose clocks ran out before the reset() at t = 20 crossed their episode end
    assert not oa.flags.writeable and ob.flags.writeable
    sent, calls, full = a.host_delta_stats()
    assert calls == 59 and full == 1 and b.host_delta_stats() == (0, 0, 60)
    assert sent / calls < 0.35 * n * per, sent / calls / n  # around a thousand bytes per env-step, not 7056 (resets included)
    a.close(); b.close()


@pytest.mark.parametrize("n", [1, 7, 33, 147, 149, 4737])
def test_host_delta_at_awkward_batch_sizes(n):
    """Delta updates at batch sizes around the group / block boundaries (one env, a partial warp, one more env than SMs,
    one more group than blocks): equal to whole-frame copies, and the device path sees the same frames."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    a = SFVecEnv("youturn", num_envs=n, device=0)
    b = SFVecEnv("youturn", num_envs=n, device=0, host_delta=False)
    a.reset(); b.reset()
    rng = np.random.RandomState(n)
    for t in range(12):
        act = rng.randint(0, a.num_actions, size=n)
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert np.array_equal(oa, ob), (n, t)
        assert np.array_equal(ra, rb) and np.array_equal(da, db) and np.array_equal(ia, ib)
    assert np.array_equal(a.render_frames(to_numpy=True).reshape(oa.shape), oa)
    a.close(); b.close()


def test_host_delta_needs_page_locked_memory():
    torch_cuda()
    import ctypes as C
    from spacefortress_b200 import SFVecEnv, _lib
    env = SFVecEnv("autoturn", num_envs=64, device=0)
    env.reset()
    act = np.zeros(64, np.int32); obs = np.zeros((64, 1, 84, 84), np.uint8); rew = np.zeros(64, np.int32); done = np.zeros(64, np.uint8)
    rc = env.L.sf_step_host(env.h, act.ctypes.data, obs.ctypes.data, rew.ctypes.data, done.ctypes.data, None, None, _lib.FLAG_RENDER | _lib.FLAG_HOST_DELTA)
    assert rc != 0 and b"page-locked" in env.L.sf_last_error()
    rc = env.L.sf_step_host(env.h, act.ctypes.data, obs.ctypes.data, rew.ctypes.data, done.ctypes.data, None, None, _lib.FLAG_RENDER)
    assert rc == 0 and obs.any()   # pageable memory is fine for whole-frame copies
    env.close()


def test_drop_in_ring_hands_out_fresh_observations_without_a_host_copy():
    """SubprocVecEnv's default (copy_outputs="ring"): the observations come from a rotation of page-locked buffers that the
    GPU updates in place; an array the caller still holds is never overwritten, a loop that drops the previous
    observation (rl/train.py:79-90) alternates between two buffers, and every frame equals the whole-frame copy."""
    torch_cuda()
    import gc
    from spacefortress_b200 import SFVecEnv, SubprocVecEnv, make_env
    n = 600
    env = SubprocVecEnv([make_env("SpaceFortress-youturn-image-v0", 0, i) for i in range(n)])
    ref = SFVecEnv("youturn", num_envs=n, device=0, host_delta=False)
    env.reset(); ref.reset()
    rng = np.random.RandomState(5)
    obs = None
    for t in range(40):                      # the training-loop pattern: the previous observation dies when the next is bound
        act = rng.randint(0, env.num_actions, size=n)
        obs, rew, done, info = env.step(act)
        want = ref.step(act)[0]
        assert np.array_equal(obs, want), t
        assert not obs.flags.writeable and isinstance(info, tuple) and rew.dtype == np.int64
    assert len(env._ring) == 2
    sent, calls, full = env.host_delta_stats()
    assert full == 2 and calls == 38         # one whole-frame copy per buffer, updates from then on
    held = []
    for t in range(7):                       # a caller that keeps everything: nothing it holds may change
        act = rng.randint(0, env.num_actions, size=n)
        o = env.step(act)[0]
        want = ref.step(act)[0]
        held.append((o, want.copy()))
        for a, b in held:
            assert np.array_equal(a, b)
    assert len(set(a.ctypes.data for a, _ in held)) == 7 and len(env._ring) <= 4
    del held, o, a, b
    gc.collect()
    import warnings
    import torch
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")       # torch warns once that the array is read-only (rl/train.py:86 does exactly this)
        kept = torch.from_numpy(env.step(act)[0])
    ref.step(act)
    snap = kept.clone()
    for t in range(4):                       # a tensor made from an observation keeps its buffer out of the rotation
        act = rng.randint(0, env.num_actions, size=n)
        assert np.array_equal(env.step(act)[0], ref.step(act)[0])
        assert torch.equal(kept, snap)
    del kept
    gc.collect()
    for t in range(12):                      # buffers come back (or new ones land on old addresses): still exact
        act = rng.randint(0, env.num_actions, size=n)
        obs = env.step(act)[0]
        assert np.array_equal(obs, ref.step(act)[0]), t
    env.close(); ref.close()


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs at their own sizes
# ---------------------------------------------------------------------------------------------------------------------
def test_soak_config3_size_rollout_equals_single_steps():
    """configs[2] size: 65 536 youturn envs; the pipelined multi-step kernel (persistent blocks, groups handed out first
    come first served) against the same ticks taken one launch at a time — frames, rewards, dones, kills bit for bit."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    n, T = 65536, 24
    a = SFVecEnv("youturn", num_envs=n, device=0, seeds=1)
    b = SFVecEnv("youturn", num_envs=n, device=0, seeds=1)
    a.reset(to_numpy=False); b.reset(to_numpy=False)
    for env in (a, b):
        env.rollout(150, want=("reward",), action_seed=9)   # mid-episode mix (state-only)
    out = a.rollout(T, action_seed=4)
    bad = 0
    for t in range(T):
        one = b.rollout(1, action_seed=4)   # the same synthetic action stream: hash(seed, global env, tick)
        bad += int((one["obs"][0] != out["obs"][t]).flatten(1).any(1).sum())
        assert torch.equal(one["reward"][0], out["reward"][t]) and torch.equal(one["done"][0], out["done"][t]) and torch.equal(one["kill"][0], out["kill"][t]), t
    assert bad == 0
    assert int((out["obs"][-1] != out["obs"][0]).flatten(1).any(1).sum()) > n // 2   # the frames do change
    a.close(); b.close()


def test_mixed_game_types_two_handles_share_a_device():
    """configs[3] shape: one autoturn and one youturn slab on the same GPU, stepped alternately on the same stream and
    state-only (render off), equal their oracles; the two handles do not disturb each other (tables, counters)."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    n, T = 2048, 40
    envs = {gt: SFVecEnv(gt, num_envs=n, device=0, render=False) for gt in ("autoturn", "youturn")}
    for e in envs.values():
        e.reset(to_numpy=False)
    acts = {gt: e.synthetic_actions(T, action_seed=5)[:, :16] for gt, e in envs.items()}
    outs = {gt: [] for gt in envs}
    for chunk in range(4):
        for gt, e in envs.items():
            outs[gt].append(e.rollout(T // 4, action_seed=5))
    for gt, e in envs.items():
        rew = torch.cat([o["reward"] for o in outs[gt]], 0).cpu().numpy()
        for i in range(16):
            o = OracleEnv(gt, 1)
            for t in range(T):
                r, d, k, _ = o.step(o.keymask(int(acts[gt][t, i])))
                assert r == int(rew[t, i]), (gt, t, i)
        e.close()


def test_config5_episode_stats_equal_host_sums():
    """configs[4] shape at 32 768 envs: staggered episode clocks (sf_set_ticks), render on, auto-reset; the device-side
    finished-episode accumulators (what the NCCL all-reduce carries) equal the sums recomputed on the host from the
    per-step done / reward / kill outputs."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    n, T = 32768, 48
    env = SFVecEnv("youturn", num_envs=n, device=0)
    env.reset(to_numpy=False)
    rng = np.random.RandomState(0)
    ticks = rng.randint(END_TICK - T - 8, END_TICK, size=n).astype(np.int32)   # most envs finish inside the rollout
    env.set_ticks(ticks)
    env.episode_stats(reset=True)
    out = env.rollout(T, action_seed=2)
    st = env.episode_stats(reset=True, all_reduce=False)
    done = out["done"].cpu().numpy().astype(bool)
    rew = out["reward"].cpu().numpy().astype(np.int64)
    kill = out["kill"].cpu().numpy().astype(np.int64)
    first_done = np.where(done.any(0), done.argmax(0), -1)
    fin = first_done >= 0
    assert fin.sum() > n // 2
    assert st["episodes"] == int(done.sum())
    # return / kills of the episode that ended at first_done: everything up to and including that step (the envs were
    # reset to return 0 by set_ticks? no: ep_return keeps running from the reset) -> compare sums over finished envs
    ret = np.array([rew[:first_done[i] + 1, i].sum() if fin[i] else 0 for i in range(n)])
    kl = np.array([kill[:first_done[i] + 1, i].sum() if fin[i] else 0 for i in range(n)])
    second = np.array([done[first_done[i] + 1:, i].any() if fin[i] else False for i in range(n)])
    assert not second.any()  # a second episode end would need 5295 more ticks
    assert st["sum_return"] == int(ret.sum())
    assert st["sum_return_sq"] == int((ret * ret).sum())
    assert st["fort_kills"] == int(kl.sum())
    assert st["sum_length"] == END_TICK * int(fin.sum())
    # frames of the step after a reset are first frames of a new episode (all envs share seed 1 -> the same spawn order
    # per env index): spot-check one finished env against its oracle
    env.close()


def test_one_ppo_minibatch_on_the_gpu_matches_the_reference_code():
    """The reference's first PPO minibatch (rl/train.py:105-132 evaluated by the reference's own ACNet / RolloutStorage on the
    CPU, tests/golden/make_ppo_minibatch_golden.py) against ppo.py on the GPU in fp32 (TF32 off): loss terms within 1e-4,
    every parameter's gradient within 2e-3 of its norm."""
    torch = torch_cuda()
    from test_ppo import check_minibatch
    tf = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
    try:
        check_minibatch(torch.device("cuda"), 1e-4, 2e-3)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf


def test_installed_glyph_masks_are_drawn_by_kernels_and_oracle_alike():
    """sf_set_glyph_masks: score digits from (here: synthetic) font masks in the format tools/dump_cairo_glyphs.py writes.
    With the same masks installed on both sides the frames stay bit-exact (static default observation with "0000000",
    the score window of a non-zero score, a dead ship's cached box under the strip); None restores the built-in face."""
    torch_cuda()
    from oracle import oracle as O
    from spacefortress_b200 import SFVecEnv
    rng = np.random.RandomState(12)
    slot = np.full(27, 255, np.uint8)
    for k in range(7):
        slot[4 * k:4 * k + 3] = k          # three columns per digit, one free column between digits
    alpha = np.zeros((10, 5, 27), np.uint8)
    for d in range(10):
        glyph = rng.randint(0, 256, (5, 3)).astype(np.uint8) * (rng.rand(5, 3) < 0.7)
        for k in range(7):
            alpha[d, :, 4 * k:4 * k + 3] = glyph
    n = 24
    env = SFVecEnv("youturn", num_envs=n, device=0)
    env.reset()
    recs = env.get_state()
    for i in range(n):
        recs[i].points = float([0, 5, 1234567, 9081726][i % 4])
        if i % 3 == 0:   # dead ship right under the score strip
            recs[i].ship_alive = 0; recs[i].ship_x = 330.0 + 5 * i; recs[i].ship_y = 120.0
    env.set_state(recs)
    try:
        env.set_glyph_masks(alpha, slot); O.set_glyph_masks(alpha, slot)
        for native in (True, False):
            frames = env.render_frames(native=native)
            frames2 = env.render_frames(native=native)   # second pass: explosion memo path
            for i in range(n):
                r = to_oracle_record(recs[i])
                exp = O.draw_native(r) if native else O.draw_obs(r)
                assert np.array_equal(frames[i], exp) and np.array_equal(frames2[i], exp), (native, i)
        assert env.render_frames(native=True)[1][1:6, 32:59].max() > 0
        # stepping (cached boxes, score windows) with the installed masks
        oracles = [O.OracleEnv("youturn", 1) for _ in range(n)]
        for i in range(n):
            oracles[i].set_state(to_oracle_record(recs[i]))
        for t in range(12):
            a = rng.randint(env.num_actions, size=n)
            obs, _, _, _ = env.step(a)
            for i in range(n):
                oracles[i].step(oracles[i].keymask(int(a[i])))
                assert np.array_equal(obs[i, 0], oracles[i].obs()), (t, i)
    finally:
        O.set_glyph_masks(None)
    env.set_glyph_masks(None)
    frames = env.render_frames(native=False)
    for i in range(n):
        assert np.array_equal(frames[i], oracles[i].obs()), i
    env.close()
