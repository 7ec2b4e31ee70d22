"""GPU (-m gpu): env blobs (sf_save_envs / sf_load_envs, SFVecEnv.save_envs / load_envs, Game / SSF_Env clone_state /
restore_state). A loaded env must continue exactly as the saved one did: observations (84x84 and native), rewards,
done, fort_kill and event bits are compared bit for bit, across auto-resets, forks, in-place resampling, handles,
devices and disk; the records after a load equal the source's, and the oracle started from them stays in parity."""
import pickle

import numpy as np
import pytest

from gpu_helpers import END_TICK, GAMETYPES, assert_frame_close, assert_state_close, make, stagger, to_oracle_record, torch_cuda
from oracle.oracle import OracleEnv

pytestmark = pytest.mark.gpu


def step(env, a):
    """numpy-path step -> [obs, reward, done, fort_kill, events] as fresh arrays"""
    obs, r, d, k = env.step(np.asarray(a, np.int32))
    return [np.array(obs), np.array(r), np.array(d), np.array(k), np.array(env.last_events)]


def run(env, acts):
    return [step(env, a) for a in acts]


def assert_same_outputs(x, y, ctx):
    for t, (a, b) in enumerate(zip(x, y)):
        for name, u, v in zip(("obs", "reward", "done", "kill", "events"), a, b):
            assert np.array_equal(u, v), (ctx, t, name)


def records_bytes(env):
    return [bytes(r) for r in env.get_state()]


@pytest.mark.parametrize("native", [False, True])
@pytest.mark.parametrize("gametype", GAMETYPES[:2])
def test_replay_from_a_saved_point(gametype, native):
    """64 envs, 300 random steps with staggered clocks (some ships dead, missiles and shells in flight), save, 200
    recorded steps, load, the same 200 steps again: identical outputs, auto-resets included."""
    n = 64
    rng = np.random.RandomState(1)
    env = make(gametype, n, seeds=np.arange(1, n + 1), native_obs=native, copy_outputs=True)
    stagger(env, rng.randint(250, 650, size=n))
    run(env, rng.randint(env.num_actions, size=(300, n)))
    recs = env.get_state()
    assert any(not r.ship_alive for r in recs) and any(r.missile_mask for r in recs) and any(r.shell_mask for r in recs)
    blob = env.save_envs()
    acts = rng.randint(env.num_actions, size=(200, n))
    first = run(env, acts)
    assert 0 < sum(o[2].sum() for o in first) < n  # some envs cross the episode end in the window, not all
    env.load_envs(blob)
    assert_same_outputs(first, run(env, acts), "replay")
    env.close()


@pytest.mark.parametrize("gametype", GAMETYPES[:2])
def test_loaded_records_equal_the_source_and_the_oracle_continues_them(gametype):
    """The records of the target envs equal the source envs' byte for byte (rng_count, stats and ep_return included);
    the oracle set to those records (it rebuilds the rand() ring from seed and count) stays in parity for 300 steps."""
    n = 16
    rng = np.random.RandomState(2)
    src = make(gametype, n, seeds=np.arange(1, n + 1), copy_outputs=True)
    run(src, rng.randint(src.num_actions, size=(300, n)))
    dst = make(gametype, n, seeds=np.arange(100, 100 + n), copy_outputs=True)
    run(dst, rng.randint(dst.num_actions, size=(40, n)))
    perm = rng.permutation(n)
    dst.load_envs(src.save_envs(), idx=perm)
    sr, dr = src.get_state(), dst.get_state()
    for k in range(n):
        assert bytes(dr[perm[k]]) == bytes(sr[k]), k
    assert len(set(r.rng_count for r in sr)) > 1 and any(r.ep_return for r in sr)
    orc = [OracleEnv(gametype, 1) for _ in range(n)]
    for i in range(n):
        orc[i].set_state(to_oracle_record(dr[i]))
    for t in range(300):
        a = rng.randint(dst.num_actions, size=n)
        obs, r, d, k, _ = step(dst, a)
        for i in range(n):
            ro, do, ko, _ = orc[i].step(orc[i].keymask(int(a[i])))
            assert (ro, do, ko) == (int(r[i]), bool(d[i]), bool(k[i])), (t, i)
            if t % 25 == 0:
                assert_frame_close(orc[i].obs(), obs[i, 0], ("frame", t, i))
        if t % 50 == 49:
            recs = dst.get_state()
            for i in range(n):
                assert_state_close(orc[i].get_state(), recs[i], ("state", t, i))
    dst.close(); src.close()


@pytest.mark.parametrize("gametype", GAMETYPES[:2])
def test_fork_one_env_into_all(gametype):
    """One env's row loaded into every env: under identical actions each env reproduces the source's own continuation,
    and they all save to the same row afterwards."""
    n, j = 32, 5
    rng = np.random.RandomState(3)
    env = make(gametype, n, seeds=np.arange(1, n + 1), copy_outputs=True)
    run(env, rng.randint(env.num_actions, size=(150, n)))
    blob = env.save_envs()
    acts = np.repeat(rng.randint(env.num_actions, size=(150, 1)), n, axis=1)
    own = [[x[j:j + 1] for x in o] for o in run(env, acts)]
    env.load_envs(blob[j:j + 1].expand(n, -1))
    forked = run(env, acts)
    for i in range(n):
        assert_same_outputs(own, [[x[i:i + 1] for x in o] for o in forked], ("fork", i))
    rows = env.save_envs()
    assert bool((rows == rows[0]).all())
    env.close()


def test_in_place_resampling_is_gather_then_scatter():
    """load_envs(save_envs()[perm]) on one handle, perm with cycles and fixed points: env i then continues as old
    env perm[i] did."""
    n = 12
    perm = np.array([0, 2, 3, 1, 4, 6, 5, 7, 9, 10, 11, 8])  # fixed points 0, 4, 7; cycles (1 2 3), (5 6), (8 9 10 11)
    rng = np.random.RandomState(4)
    env = make("youturn", n, seeds=np.arange(1, n + 1), copy_outputs=True)
    run(env, rng.randint(env.num_actions, size=(120, n)))
    blob = env.save_envs()
    acts = rng.randint(env.num_actions, size=(100, n))
    ref = run(env, acts)
    env.load_envs(blob)
    env.load_envs(env.save_envs()[perm])
    got = run(env, acts[:, perm])
    assert_same_outputs([[x[perm] for x in o] for o in ref], got, "resample")
    env.close()


def test_loaded_dead_ship_is_not_drawn_with_the_destination_explosion_cache():
    """Two envs of the same seed, both ships dead with equal rng_count (= the key of the cached explosion) at different
    positions: after loading one into the other, its frames equal the source's for the rest of the explosion."""
    n = 256
    rng = np.random.RandomState(5)
    env = make("youturn", n, copy_outputs=True)  # every env seed 1
    pair = None
    for t in range(600):
        step(env, rng.randint(env.num_actions, size=n))
        recs = env.get_state()
        dead = {}
        for i, r in enumerate(recs):
            if not r.ship_alive:
                dead.setdefault(r.rng_count, []).append(i)
        for idx in dead.values():
            for a in idx:
                for b in idx:
                    if (recs[a].ship_x, recs[a].ship_y) != (recs[b].ship_x, recs[b].ship_y):
                        pair = (a, b)
            if pair:
                break
        if pair:
            break
    assert pair, "no two dead ships with equal rand() counts found"
    src, dst = pair
    ra, rb = recs[src], recs[dst]
    assert not ra.ship_alive and not rb.ship_alive and ra.rng_count == rb.rng_count and ra.rng_seed == rb.rng_seed
    assert (ra.ship_x, ra.ship_y) != (rb.ship_x, rb.ship_y)
    env.load_envs(env.save_envs([src]), idx=[dst])
    for native in (False, True):
        f = env.render_frames(native=native)
        assert np.array_equal(f[dst], f[src]), ("first frame", native)
    a = np.zeros(n, np.int32)
    respawned = False
    for t in range(60):
        obs = step(env, a)[0]
        assert np.array_equal(obs[dst], obs[src]), ("explosion", t)
        respawned |= bool(env.get_state()[src].ship_alive)
    assert respawned
    env.close()


@pytest.mark.parametrize("gametype", GAMETYPES[:2])
def test_rows_are_canonical(gametype):
    """save(load(b)) == b byte for byte; dead missile / shell slots and the padding of a row are zero."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n = 64
    rng = np.random.RandomState(6)
    env = make(gametype, n, seeds=np.arange(1, n + 1), copy_outputs=True)
    run(env, rng.randint(env.num_actions, size=(250, n)))
    b = env.save_envs()
    other = make(gametype, n, seeds=np.arange(7, 7 + n), copy_outputs=True)
    run(other, rng.randint(other.num_actions, size=(90, n)))  # stale projectile slots in the destination
    other.load_envs(b)
    assert torch.equal(other.save_envs(), b)
    rows = b.cpu().numpy()
    hdr = rows[:, :16].view(np.uint32)
    assert (hdr[:, 0] == 0x42465353).all() and (hdr[:, 1] == _lib.ENV_BLOB_VERSION).all() and (hdr[:, 3] == 0).all()
    assert (hdr[:, 2] == GAMETYPES.index(gametype)).all()
    pmask = rows[:, 52:56].copy().view(np.uint32)[:, 0]
    saw_dead = False
    for i in range(n):
        for s in range(20):
            if not (pmask[i] >> s) & 1:
                saw_dead = True
                assert not rows[i, 176 + 16 * s:192 + 16 * s].any() and not rows[i, 656 + 2 * s:658 + 2 * s].any(), (i, s)
        for s in range(4):
            if not (pmask[i] >> (20 + s)) & 1:
                assert not rows[i, 496 + 16 * s:512 + 16 * s].any() and not rows[i, 560 + 16 * s:576 + 16 * s].any(), (i, s)
                assert not rows[i, 624 + 8 * s:632 + 8 * s].any(), (i, s)
    assert saw_dead and (pmask & 0xFFFFF).any() and not rows[:, 820:].any()
    other.close(); env.close()


def test_across_handles_and_disk(tmp_path):
    """Save from a 48-env handle, torch.save / torch.load, load into chosen envs of a 100-env handle with another
    first_global_env: records equal and the continuations match."""
    torch = torch_cuda()
    rng = np.random.RandomState(7)
    a = make("autoturn", 48, seeds=np.arange(1, 49), copy_outputs=True)
    run(a, rng.randint(a.num_actions, size=(200, 48)))
    torch.save(a.save_envs(), str(tmp_path / "envs.pt"))
    blob = torch.load(str(tmp_path / "envs.pt"))
    b = make("autoturn", 100, seeds=np.arange(500, 600), first_global_env=4096, copy_outputs=True)
    run(b, rng.randint(b.num_actions, size=(30, 100)))
    idx = rng.choice(100, size=48, replace=False)
    b.load_envs(blob, idx=torch.from_numpy(idx).cuda())
    rb = b.get_state()
    assert [bytes(rb[i]) for i in idx] == records_bytes(a)
    acts_a = rng.randint(a.num_actions, size=(150, 48))
    acts_b = rng.randint(b.num_actions, size=(150, 100))
    acts_b[:, idx] = acts_a
    ra, rb = run(a, acts_a), run(b, acts_b)
    assert_same_outputs(ra, [[x[idx] for x in o] for o in rb], "across handles")
    b.close(); a.close()


def test_onto_a_second_gpu():
    torch = torch_cuda()
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    rng = np.random.RandomState(8)
    a = make("youturn", 32, seeds=np.arange(1, 33), copy_outputs=True)
    run(a, rng.randint(a.num_actions, size=(150, 32)))
    b = make("youturn", 32, device=1, copy_outputs=True)
    b.load_envs(a.save_envs().to("cuda:1"))
    assert records_bytes(b) == records_bytes(a)
    acts = rng.randint(a.num_actions, size=(100, 32))
    assert_same_outputs(run(a, acts), run(b, acts), "cuda:1")
    b.close(); a.close()


def test_rejected_rows_and_indices():
    """A youturn row into an autoturn handle, a corrupted magic and an out-of-range index raise SFError and leave the
    targets untouched; repeated target indices raise ValueError."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    rng = np.random.RandomState(9)
    y = make("youturn", 8, seeds=np.arange(1, 9), copy_outputs=True)
    a = make("autoturn", 8, seeds=np.arange(1, 9), copy_outputs=True)
    run(y, rng.randint(y.num_actions, size=(60, 8)))
    run(a, rng.randint(a.num_actions, size=(60, 8)))
    before = records_bytes(a)
    with pytest.raises(_lib.SFError):
        a.load_envs(y.save_envs([1, 2]), idx=[3, 4])
    good = a.save_envs([1, 2])
    bad = good.clone()
    bad[1, 0] ^= 0xFF
    with pytest.raises(_lib.SFError):
        a.load_envs(bad[1:], idx=[5])
    with pytest.raises(_lib.SFError):
        a.load_envs(good[:1], idx=[8])
    with pytest.raises(_lib.SFError):
        a.load_envs(good[:1], idx=torch.tensor([-1], device="cuda"))  # a device index is checked by the kernel
    assert records_bytes(a) == before
    with pytest.raises(_lib.SFError):  # the good row of a call is loaded, the bad one is counted
        a.load_envs(bad, idx=[6, 7])
    after = records_bytes(a)
    assert after[6] == before[1] and after[7] == before[7]
    with pytest.raises(ValueError):
        a.load_envs(good, idx=[3, 3])
    with pytest.raises(ValueError):
        a.load_envs(good)  # two rows for eight envs
    assert not a.save_envs(torch.tensor([200], device="cuda")).any()  # no such env: an all-zero row
    y.close(); a.close()


def test_host_delta_buffers_after_a_load():
    """After load_envs a host_delta numpy-path env's observations equal a whole-frame (host_delta=False) env's."""
    n = 32
    rng = np.random.RandomState(10)
    hd = make("youturn", n, seeds=np.arange(1, n + 1), copy_outputs=False, host_delta=True)
    full = make("youturn", n, seeds=np.arange(1, n + 1), copy_outputs=False, host_delta=False)
    src = make("youturn", n, seeds=np.arange(40, 40 + n), copy_outputs=True)
    run(src, rng.randint(src.num_actions, size=(100, n)))
    for t in range(20):
        a = rng.randint(hd.num_actions, size=n)
        assert np.array_equal(hd.step(a)[0], full.step(a)[0]), t
    blob = src.save_envs()
    hd.load_envs(blob); full.load_envs(blob)
    for t in range(80):
        a = rng.randint(hd.num_actions, size=n)
        o1, o2, o3 = hd.step(a)[0], full.step(a)[0], step(src, a)[0]
        assert np.array_equal(o1, o2) and np.array_equal(o1, o3), t
    for e in (hd, full, src):
        e.close()


@pytest.mark.parametrize("gametype", GAMETYPES[:2])
def test_rollout_from_a_loaded_state_equals_single_steps(gametype):
    torch = torch_cuda()
    n, T = 64, 24
    rng = np.random.RandomState(11)
    env = make(gametype, n, seeds=np.arange(1, n + 1), copy_outputs=True)
    stagger(env, rng.randint(150, 180, size=n))
    run(env, rng.randint(env.num_actions, size=(160, n)))
    blob = env.save_envs()
    acts = rng.randint(env.num_actions, size=(T, n)).astype(np.int32)
    env.load_envs(blob)
    out = env.rollout(T, actions=torch.from_numpy(acts).cuda())
    roll = {k: v.cpu().numpy() for k, v in out.items()}
    env.load_envs(blob)
    single = run(env, acts)
    assert roll["done"].any()
    for t in range(T):
        assert np.array_equal(roll["obs"][t], single[t][0]), t
        assert np.array_equal(roll["reward"][t], single[t][1]) and np.array_equal(roll["done"][t], single[t][2]), t
        assert np.array_equal(roll["kill"][t].astype(bool), single[t][3].astype(bool)), t
    env.close()


def test_episode_stats_count_the_restored_return():
    """A restored env that finishes its episode adds its full return (the part before the save included) once."""
    n = 16
    rng = np.random.RandomState(12)
    src = make("youturn", n, seeds=np.arange(1, n + 1), copy_outputs=True)
    stagger(src, np.full(n, 400))
    run(src, rng.randint(src.num_actions, size=(300, n)))
    ret0 = np.array([r.ep_return for r in src.get_state()])
    assert ret0.any()
    dst = make("youturn", n, seeds=np.arange(50, 50 + n), copy_outputs=True)
    dst.load_envs(src.save_envs())
    dst.episode_stats(reset=True)
    rew = np.zeros(n, np.int64)
    for t in range(100):
        _, r, d, _, _ = step(dst, rng.randint(dst.num_actions, size=n))
        rew += r
        assert d.all() == (t == 99) and d.any() == (t == 99), t
    st = dst.episode_stats()
    assert st["episodes"] == n and st["sum_return"] == int((ret0 + rew).sum()) and st["sum_length"] == n * END_TICK
    dst.close(); src.close()


@pytest.mark.parametrize("gametype", GAMETYPES[:2])
def test_game_clone_and_restore(gametype):
    """Game: clone after 500 ticks, 100 ticks, restore (a pickled copy), the same 100 ticks: rewards, frames, features and
    dump() identical."""
    torch_cuda()
    from spacefortress_b200 import _lib
    from spacefortress_b200.core import Game
    g = Game(gametype, lw=3, grayscale=True, width=90, height=92, viewport=(130, 80, 450, 460))
    rng = np.random.RandomState(13)
    keys = rng.randint(0, 2, size=(700, 4))

    def tick(k):
        for sym in range(1, 5):
            (g.press_key if k[sym - 1] else g.release_key)(sym)
        return (g.step_one_tick(34), g.gray_frame(), g.obs84(), g.features("features"), g.dump(), g.stats)

    for t in range(500):
        tick(keys[t])
    blob = g.clone_state()
    assert blob.dtype == np.uint8 and blob.shape == (_lib.ENV_BLOB_BYTES,)
    first = [tick(k) for k in keys[500:600]]
    g.press_key(1)  # a pending key press is dropped by the restore
    g.restore_state(pickle.loads(pickle.dumps(blob)))
    again = [tick(k) for k in keys[500:600]]
    for t, (x, y) in enumerate(zip(first, again)):
        assert x[0] == y[0] and x[4] == y[4] and x[5] == y[5], t
        for u, v in zip(x[1:4], y[1:4]):
            assert np.array_equal(u, v), t
    other = Game("autoturn" if gametype == "youturn" else "youturn", lw=3, grayscale=True, width=90, height=92, viewport=(130, 80, 450, 460))
    with pytest.raises(_lib.SFError):
        other.restore_state(blob)


@pytest.mark.parametrize("obs_type", ["image", "features"])
def test_ssf_env_clone_and_restore(obs_type):
    torch_cuda()
    from spacefortress_b200.gym.envs import SSF_Env
    env = SSF_Env(gametype="youturn", obs_type=obs_type)
    rng = np.random.RandomState(14)
    acts = rng.randint(env.action_space.n, size=600)
    for a in acts[:500]:
        env.step(int(a))
    blob = env.clone_state()
    frame = env.render("rgb_array").copy()
    first = [env.step(int(a)) for a in acts[500:]]
    env.restore_state(blob)
    assert np.array_equal(env.render("rgb_array"), frame)
    again = [env.step(int(a)) for a in acts[500:]]
    for t, (x, y) in enumerate(zip(first, again)):
        assert np.array_equal(x[0], y[0]) and x[1:] == y[1:], t
    env.close()
