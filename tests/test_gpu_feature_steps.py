"""GPU (-m gpu): feature observations as outputs of the state-only step kernel (sf_rollout_features,
sf_step_host_features, SFVecEnv(obs_type != 'image')). The reference is the two-launch path on a second handle in the
same state: sf_step (render off) followed by sf_features, once per tick. Feature rows are compared as raw bits."""
import numpy as np
import pytest

from gpu_helpers import (GAMETYPES, KINDS, STEP_OUTPUTS, hp, make, outputs, ptrs, rollout_features, single_steps, stagger, step_host,
                         torch_cuda, vp)

pytestmark = pytest.mark.gpu


def assert_same(a, b, ctx):
    """every output of a equals b's; feature rows as raw bits, with the first difference reported"""
    torch = torch_cuda()
    for name, x in a.items():
        if name not in KINDS:
            assert torch.equal(x, b[name]), (ctx, name)
            continue
        fa, fb = x.contiguous().view(torch.int32), b[name].contiguous().view(torch.int32)
        if not torch.equal(fa, fb):
            t, i, k = [int(v) for v in (fa != fb).nonzero()[0]]
            raise AssertionError("%s: feature rows differ first at tick %d env %d column %d: %r vs %r"
                                 % (ctx, t, i, k, float(x[t, i, k]), float(b[name][t, i, k])))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("gametype", GAMETYPES)
def test_rollout_features_equal_the_two_launch_path(gametype, kind):
    """1000 envs, T = 48 with auto-resets inside the launch: rows, rewards, dones, kills, events and the final state equal
    T x (sf_step + sf_features); rewards and dones also equal a plain state-only sf_rollout (the rows change nothing)."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T = 1000, 48
    a, b = [make(gametype, n, seeds=7, render=False, warm=20, ends=(1, 60)) for _ in range(2)]
    start = a.save_envs()
    assert torch.equal(start, b.save_envs())
    rng = np.random.RandomState(3)
    given = torch.from_numpy(rng.randint(a.num_actions, size=(T, n)).astype(np.int32)).cuda()
    for case, acts in (("synthetic", None), ("given", given)):
        if case == "synthetic":
            got = rollout_features(a, kind, T, action_seed=5, t0=100)
            ref_acts = torch.from_numpy(b.synthetic_actions(T, action_seed=5, t0=100)).cuda()
        else:
            got = rollout_features(a, kind, T, actions=acts)
            ref_acts = acts
        ref = single_steps(b, ref_acts, want=(kind,) + STEP_OUTPUTS)
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
    from spacefortress_b200 import _lib
    for gametype, kind, offset in (("youturn", "features", 0), ("autoturn", "monitors", 1), ("youturn", "normalized-features", 1)):
        a, b = [make(gametype, n, seeds=n + T, render=False, warm=20, ends=(1, 60)) for _ in range(2)]
        acts = torch.from_numpy(np.random.RandomState(T).randint(a.num_actions, size=(T, n)).astype(np.int32)).cuda()
        got = outputs(a, T, STEP_OUTPUTS)
        nf = a.L.sf_num_features(a.h, _lib.OBS_TYPES[kind])  # `offset` floats in front of the rows
        got[kind] = torch.full((T * n * nf + offset,), float("nan"), dtype=torch.float32, device="cuda")[offset:].view(T, n, nf)
        _lib.check(a.L.sf_rollout_features(a.h, _lib.OBS_TYPES[kind], T, vp(acts), 0, 0, vp(got[kind]), *ptrs(got, STEP_OUTPUTS), 0, None))
        torch.cuda.synchronize()
        assert not torch.isnan(got[kind]).any()
        assert_same(got, single_steps(b, acts, want=(kind,) + STEP_OUTPUTS), (n, T, gametype, kind, offset))
        assert torch.equal(a.save_envs(), b.save_envs())
        a.close(); b.close()


def test_no_autoreset_rows_are_the_finished_state():
    """SF_FLAG_NO_AUTORESET: a finished env's rows are its finished state, as sf_features shows it."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    n, T = 129, 24
    a, b = [make("youturn", n, seeds=7, render=False, warm=20, ends=(1, 12)) for _ in range(2)]
    acts = torch.from_numpy(np.random.RandomState(2).randint(a.num_actions, size=(T, n)).astype(np.int32)).cuda()
    got = rollout_features(a, "features", T, actions=acts, flags=_lib.FLAG_NO_AUTORESET)
    assert_same(got, single_steps(b, acts, _lib.FLAG_NO_AUTORESET, want=("features",) + STEP_OUTPUTS), "no-autoreset")
    assert int(got["done"].any(0).sum()) == n  # every env reached the end of its episode inside the launch
    a.close(); b.close()


@pytest.mark.parametrize("gametype,kind", [("youturn", "features"), ("autoturn", "normalized-features"), ("test-youturn", "monitors")])
def test_host_step_features(gametype, kind):
    """sf_step_host_features into a page-locked buffer (written in place by the kernel), into a pageable one (copied
    back) and the device path (sf_rollout_features, T = 1): identical rows over 40 steps with staggered episode ends,
    and the two-launch path agrees. No frames are sent: sf_host_delta_stats does not move."""
    torch = torch_cuda()
    n, steps = 333, 40
    envs = [make(gametype, n, seeds=7, render=False, warm=20, ends=(1, steps)) for _ in range(4)]
    pinned, pageable, device, ref = envs
    stats0 = [e.host_delta_stats() for e in envs[:2]]
    want = (kind,) + STEP_OUTPUTS
    rng = np.random.RandomState(9)
    ends = 0
    for t in range(steps):
        a = rng.randint(pinned.num_actions, size=n).astype(np.int32)
        host = {name: step_host(env, a[None], pinned=p, want=want)
                for name, env, p in (("page-locked", pinned, True), ("pageable", pageable, False))}
        da = torch.from_numpy(a).cuda()
        got = rollout_features(device, kind, 1, actions=da[None])
        exp = single_steps(ref, da[None], want=want)
        assert_same(got, exp, (gametype, kind, t, "device"))
        for name, out in host.items():
            assert_same({k: torch.from_numpy(v).cuda() for k, v in out.items()}, exp, (gametype, kind, t, name))
        ends += int(host["page-locked"]["done"].sum())
    assert ends > 0
    assert [e.host_delta_stats() for e in envs[:2]] == stats0
    for e in envs:
        e.close()


@pytest.mark.parametrize("kind", KINDS)
def test_vec_env_feature_contract(kind):
    """step(np) returns a new writable float32 [n, F] array that equals features() read after the step and is not
    changed by later steps; step(torch) returns a new CUDA tensor; rollout(T)["obs"] equals T single steps."""
    torch = torch_cuda()
    n, T = 77, 30
    env = make("youturn", n, seeds=3, obs_type=kind)
    stagger(env, np.full(n, 12))
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
    a, b = [make("youturn", n, seeds=3, obs_type=kind, reset=False) for _ in range(2)]
    for e in (a, b):
        e.reset()
        stagger(e, np.full(n, 20))
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
    env, ref = [make("autoturn", n, seeds=7, render=False, warm=20, ends=(1, 60)) for _ in range(2)]
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

    def host(kind=FEAT, a=hp(h_act), out=hp(h_feat), flags=0):
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
    exp = single_steps(ref, torch.zeros((5, n), dtype=torch.int32, device="cuda"), want=("features",) + STEP_OUTPUTS)
    assert torch.equal(feat.view(torch.int32), exp["features"][:4].view(torch.int32))
    assert np.array_equal(h_feat.view(np.int32), exp["features"][4].cpu().numpy().view(np.int32))
    env.close(); ref.close()
