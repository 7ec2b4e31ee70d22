"""GPU (-m gpu): feature observations as outputs of the state-only step kernel (sf_rollout_features,
sf_step_host_features, SFVecEnv(obs_type != 'image')). The reference is the two-launch path on a second handle in the
same state: sf_step (render off) followed by sf_features, once per tick. Feature rows are compared as raw bits."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GAMETYPES = ["youturn", "autoturn", "test-youturn", "test-autoturn"]
KINDS = ["features", "normalized-features", "monitors"]
END_TICK = 5295  # fixed episode length (game.cpp:487-489)


def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def vp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def make(gametype, n, seed=7, warm=20, end_lo=1, end_hi=60):
    """A state-only env with seeds seed + i, `warm` synthetic steps behind it (ships, missiles and shells in flight) and
    clocks staggered so that the episodes end end_lo..end_hi steps from now. Deterministic: two calls give equal states."""
    torch_cuda()
    from spacefortress_b200 import SFVecEnv
    env = SFVecEnv(gametype, num_envs=n, device=0, render=False, seeds=seed)
    env.reset()
    if warm:
        env.rollout(warm, action_seed=seed, want=("reward",))
    rng = np.random.RandomState(seed)
    env.set_ticks((END_TICK - rng.randint(end_lo, end_hi, size=n)).astype(np.int32))
    return env


def outputs(torch, T, n, nf, offset=0):
    """time-major outputs; `offset` floats in front of the feature rows (a base address that is not 16-byte aligned)"""
    dev = "cuda"
    feat = torch.full((T * n * nf + offset,), float("nan"), dtype=torch.float32, device=dev)
    return dict(feat=feat[offset:].view(T, n, nf), reward=torch.empty((T, n), dtype=torch.int32, device=dev),
                done=torch.empty((T, n), dtype=torch.uint8, device=dev), kill=torch.empty((T, n), dtype=torch.uint8, device=dev),
                events=torch.empty((T, n), dtype=torch.int32, device=dev))


def rollout_features(env, kind, T, actions=None, action_seed=0, t0=0, flags=0, offset=0):
    from spacefortress_b200 import _lib
    torch = torch_cuda()
    nf = env.L.sf_num_features(env.h, _lib.OBS_TYPES[kind])
    o = outputs(torch, T, env.num_envs, nf, offset)
    _lib.check(env.L.sf_rollout_features(env.h, _lib.OBS_TYPES[kind], T, vp(actions), action_seed, t0, vp(o["feat"]), vp(o["reward"]),
                                         vp(o["done"]), vp(o["kill"]), vp(o["events"]), flags, None))
    torch.cuda.synchronize()
    return o


def two_launch(env, kind, actions, flags=0):
    """the reference: T x (sf_step without frames, then sf_features of the state it left)"""
    from spacefortress_b200 import _lib
    torch = torch_cuda()
    T, n = actions.shape
    nf = env.L.sf_num_features(env.h, _lib.OBS_TYPES[kind])
    o = outputs(torch, T, n, nf)
    for t in range(T):
        _lib.check(env.L.sf_step(env.h, vp(actions[t]), None, vp(o["reward"][t]), vp(o["done"][t]), vp(o["kill"][t]), vp(o["events"][t]),
                                 flags, None))
        _lib.check(env.L.sf_features(env.h, _lib.OBS_TYPES[kind], vp(o["feat"][t]), None))
    torch.cuda.synchronize()
    return o


def assert_same(a, b, ctx):
    torch = torch_cuda()
    fa, fb = a["feat"].contiguous().view(torch.int32), b["feat"].contiguous().view(torch.int32)
    if not torch.equal(fa, fb):
        t, i, k = [int(x) for x in (fa != fb).nonzero()[0]]
        raise AssertionError("%s: feature rows differ first at tick %d env %d column %d: %r vs %r"
                             % (ctx, t, i, k, float(a["feat"][t, i, k]), float(b["feat"][t, i, k])))
    for name in ("reward", "done", "kill", "events"):
        assert torch.equal(a[name], b[name]), (ctx, name)


def synthetic(env, T, action_seed, t0):
    torch = torch_cuda()
    return torch.from_numpy(env.synthetic_actions(T, action_seed=action_seed, t0=t0)).cuda()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("gametype", GAMETYPES)
def test_rollout_features_equal_the_two_launch_path(gametype, kind):
    """1000 envs, T = 48 with auto-resets inside the launch: rows, rewards, dones, kills, events and the final state equal
    T x (sf_step + sf_features); rewards and dones also equal a plain state-only sf_rollout (the rows change nothing)."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T = 1000, 48
    a, b = make(gametype, n), make(gametype, n)
    start = a.save_envs()
    assert torch.equal(start, b.save_envs())
    rng = np.random.RandomState(3)
    given = torch.from_numpy(rng.randint(a.num_actions, size=(T, n)).astype(np.int32)).cuda()
    for case, acts in (("synthetic", None), ("given", given)):
        if case == "synthetic":
            got = rollout_features(a, kind, T, action_seed=5, t0=100)
            ref_acts = synthetic(b, T, 5, 100)
        else:
            got = rollout_features(a, kind, T, actions=acts)
            ref_acts = acts
        ref = two_launch(b, kind, ref_acts)
        assert_same(got, ref, (gametype, kind, case))
        assert 0 < int(got["done"].sum()) and bool((got["events"] & _lib.EV_EPISODE_RESET).any())
        assert torch.equal(a.save_envs(), b.save_envs()), (gametype, kind, case, "final state")
        # no perturbation: the state-only rollout of the same start gives the same rewards and dones
        end = b.save_envs()
        b.load_envs(start)
        r = b.rollout(T, actions=ref_acts, want=("reward", "done"))
        assert torch.equal(r["reward"], got["reward"]) and torch.equal(r["done"], got["done"]), (gametype, kind, case)
        b.load_envs(end)
        start = end
    a.close(); b.close()


@pytest.mark.parametrize("T", [1, 7, 9, 64])
@pytest.mark.parametrize("n", [1, 7, 33, 129, 4737])
def test_awkward_shapes(n, T):
    """A partial block, odd n (ticks that start off a 16-byte boundary), T past the 8-tick Stats flush; F = 19 and F = 10,
    with the output base 16-byte aligned and 4 bytes past that."""
    torch = torch_cuda()
    for gametype, kind, offset in (("youturn", "features", 0), ("autoturn", "monitors", 1), ("youturn", "normalized-features", 1)):
        a, b = make(gametype, n, seed=n + T), make(gametype, n, seed=n + T)
        acts = torch.from_numpy(np.random.RandomState(T).randint(a.num_actions, size=(T, n)).astype(np.int32)).cuda()
        got = rollout_features(a, kind, T, actions=acts, offset=offset)
        assert not torch.isnan(got["feat"]).any()
        assert_same(got, two_launch(b, kind, acts), (n, T, gametype, kind, offset))
        assert torch.equal(a.save_envs(), b.save_envs())
        a.close(); b.close()


def test_no_autoreset_rows_are_the_finished_state():
    """SF_FLAG_NO_AUTORESET: a finished env's rows are its finished state, as sf_features shows it."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T = 129, 24
    a, b = make("youturn", n, end_lo=1, end_hi=12), make("youturn", n, end_lo=1, end_hi=12)
    acts = torch.from_numpy(np.random.RandomState(2).randint(a.num_actions, size=(T, n)).astype(np.int32)).cuda()
    got = rollout_features(a, "features", T, actions=acts, flags=_lib.FLAG_NO_AUTORESET)
    assert_same(got, two_launch(b, "features", acts, flags=_lib.FLAG_NO_AUTORESET), "no-autoreset")
    assert int(got["done"].any(0).sum()) == n  # every env reached the end of its episode inside the launch
    a.close(); b.close()


@pytest.mark.parametrize("gametype,kind", [("youturn", "features"), ("autoturn", "normalized-features"), ("test-youturn", "monitors")])
def test_host_step_features(gametype, kind):
    """sf_step_host_features into a page-locked buffer (written in place by the kernel), into a pageable one (copied
    back) and the device path (sf_rollout_features, T = 1): identical rows over 40 steps with staggered episode ends,
    and the two-launch path agrees. No frames are sent: sf_host_delta_stats does not move."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, steps = 333, 40
    envs = [make(gametype, n, end_lo=1, end_hi=steps) for _ in range(4)]
    pinned, pageable, device, ref = envs
    kid = _lib.OBS_TYPES[kind]
    nf = pinned.L.sf_num_features(pinned.h, kid)
    stats0 = [e.host_delta_stats() for e in envs[:2]]
    pin = {k: _lib.pinned_array(s, d) for k, s, d in (("feat", (n, nf), np.float32), ("actions", (n,), np.int32), ("reward", (n,), np.int32),
                                                      ("done", (n,), np.uint8), ("kill", (n,), np.uint8), ("events", (n,), np.uint32))}
    pag = {k: np.zeros_like(v) for k, v in pin.items()}
    rng = np.random.RandomState(9)
    ends = 0
    for t in range(steps):
        a = rng.randint(pinned.num_actions, size=n).astype(np.int32)
        for env, buf in ((pinned, pin), (pageable, pag)):
            buf["actions"][:] = a
            buf["feat"][:] = np.nan
            p = {k: C.c_void_p(v.ctypes.data) for k, v in buf.items()}
            _lib.check(env.L.sf_step_host_features(env.h, kid, p["actions"], p["feat"], p["reward"], p["done"], p["kill"], p["events"], 0))
        da = torch.from_numpy(a).cuda()
        got = rollout_features(device, kind, 1, actions=da[None])
        exp = two_launch(ref, kind, da[None])
        assert_same(got, exp, (gametype, kind, t, "device"))
        for name, buf in (("page-locked", pin), ("pageable", pag)):
            assert np.array_equal(buf["feat"].view(np.int32), exp["feat"][0].cpu().numpy().view(np.int32)), (name, t)
            for k in ("reward", "done", "kill"):
                assert np.array_equal(buf[k], exp[k][0].cpu().numpy()), (name, t, k)
            assert np.array_equal(buf["events"].view(np.int32), exp["events"][0].cpu().numpy()), (name, t)
        ends += int(pin["done"].sum())
    assert ends > 0
    assert [e.host_delta_stats() for e in envs[:2]] == stats0
    for e in envs:
        e.close()


@pytest.mark.parametrize("kind", KINDS)
def test_vec_env_feature_contract(kind):
    """step(np) returns a new writable float32 [n, F] array that equals features() read after the step and is not
    changed by later steps; step(torch) returns a new CUDA tensor; rollout(T)["obs"] equals T single steps."""
    torch = torch_cuda()
    from spacefortress_b200 import SFVecEnv
    n, T = 77, 30
    mk = lambda: SFVecEnv("youturn", num_envs=n, device=0, obs_type=kind, seeds=3)
    env = mk()
    env.reset()
    env.set_ticks(np.full(n, END_TICK - 12, np.int32))
    rng = np.random.RandomState(1)
    kept = []
    for t in range(T):
        f, r, d, k = env.step(rng.randint(env.num_actions, size=n))
        assert isinstance(f, np.ndarray) and f.dtype == np.float32 and f.shape == (n, env.num_features) and f.flags.writeable
        assert all(f is not g and not np.shares_memory(f, g) for g, _ in kept)
        assert np.array_equal(f.view(np.int32), env.features(to_numpy=True).view(np.int32)), t
        kept.append((f, f.copy()))
    assert all(np.array_equal(f, c) for f, c in kept)
    prev = None
    for t in range(3):
        ft, _, _, _ = env.step(torch.zeros(n, dtype=torch.int32, device="cuda"))
        assert ft.is_cuda and ft.dtype == torch.float32 and tuple(ft.shape) == (n, env.num_features)
        assert prev is None or ft.data_ptr() != prev.data_ptr()
        assert torch.equal(ft.view(torch.int32), env.features().view(torch.int32))
        prev = ft
    env.close()
    # rollout(T)["obs"] == T single device steps, from equal states
    a, b = mk(), mk()
    for e in (a, b):
        e.reset()
        e.set_ticks(np.full(n, END_TICK - 20, np.int32))
    acts = torch.from_numpy(rng.randint(a.num_actions, size=(T, n)).astype(np.int32)).cuda()
    out = a.rollout(T, actions=acts)
    assert out["obs"].dtype == torch.float32 and tuple(out["obs"].shape) == (T, n, a.num_features)
    for t in range(T):
        f, r, d, _ = b.step(acts[t])
        assert torch.equal(out["obs"][t].view(torch.int32), f.view(torch.int32)), t
        assert torch.equal(out["reward"][t], r) and torch.equal(out["done"][t].bool(), d), t
    a.close(); b.close()


def test_rejected_arguments():
    """Frame flags, a bad obs_type, NULL outputs or actions and T <= 0 give SF_ERR_INVALID; the handle keeps working."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n = 40
    env, ref = make("autoturn", n), make("autoturn", n)
    L, h = env.L, env.h
    nf = L.sf_num_features(h, _lib.OBS_TYPES["features"])
    feat = torch.zeros((4, n, nf), dtype=torch.float32, device="cuda")
    acts = torch.zeros((4, n), dtype=torch.int32, device="cuda")
    h_feat = _lib.pinned_array((n, nf), np.float32)
    h_act = _lib.pinned_array((n,), np.int32)
    h_act[:] = 0
    FEAT = _lib.OBS_TYPES["features"]

    def roll(kind=FEAT, T=1, out=vp(feat), flags=0):
        return L.sf_rollout_features(h, kind, T, vp(acts), 0, 0, out, None, None, None, None, flags, None)

    def host(kind=FEAT, a=C.c_void_p(h_act.ctypes.data), out=C.c_void_p(h_feat.ctypes.data), flags=0):
        return L.sf_step_host_features(h, kind, a, out, None, None, None, None, flags)

    for flag in (_lib.FLAG_RENDER, _lib.FLAG_NATIVE_OBS, _lib.FLAG_HOST_DELTA):
        assert roll(flags=flag) == _lib.SF_ERR_INVALID and host(flags=flag) == _lib.SF_ERR_INVALID, flag
    for kind in (_lib.OBS_TYPES["image"], 4, -1):
        assert roll(kind=kind) == _lib.SF_ERR_INVALID and host(kind=kind) == _lib.SF_ERR_INVALID, kind
    assert roll(out=None) == _lib.SF_ERR_INVALID and host(out=None) == _lib.SF_ERR_INVALID
    assert host(a=None) == _lib.SF_ERR_INVALID
    for T in (0, -1):
        assert roll(T=T) == _lib.SF_ERR_INVALID
    assert L.sf_rollout_features(None, FEAT, 1, vp(acts), 0, 0, vp(feat), None, None, None, None, 0, None) == _lib.SF_ERR_INVALID
    torch.cuda.synchronize()
    assert torch.equal(env.save_envs(), ref.save_envs())  # nothing was stepped
    # and the handle still steps
    _lib.check(roll(T=4))
    _lib.check(host())
    exp = two_launch(ref, "features", torch.zeros((5, n), dtype=torch.int32, device="cuda"))
    assert torch.equal(feat.view(torch.int32), exp["feat"][:4].view(torch.int32))
    assert np.array_equal(h_feat.view(np.int32), exp["feat"][4].cpu().numpy().view(np.int32))
    env.close(); ref.close()
