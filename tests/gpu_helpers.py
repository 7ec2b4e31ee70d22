"""The harness of the GPU tests (-m gpu): the env constructor, staggered episode clocks, thin callers of the stepping
entry points of the C-ABI (they allocate time-major outputs and pass the pointers) and the comparisons against the
oracle. A plain module: the tests import it as `from gpu_helpers import ...`."""
import ctypes as C

import numpy as np
import pytest

from oracle.oracle import Record

GAMETYPES = ["youturn", "autoturn", "test-youturn", "test-autoturn"]
KINDS = ["features", "normalized-features", "monitors"]
END_TICK = 5295  # fixed episode length (game.cpp:487-489)
FLOAT_REL_TOL = 1e-5  # north_star: continuous kinematics within 1e-5 relative per step
FRAME_MATCH_FRACTION = 0.999
FRAME_MAX_DELTA = 2
STEP_OUTPUTS = ("reward", "done", "kill", "events")  # the per-env outputs of the stepping entry points, in argument order


def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def vp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def hp(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def to_oracle_record(g):
    r = Record()
    C.memmove(C.byref(r), C.byref(g), C.sizeof(Record))
    return r


def assert_state_close(o, g, ctx):
    """int_state() (stats included) exact; the shells within FLOAT_REL_TOL (device cos/sin), every other float bit-exact"""
    assert o.int_state() == to_oracle_record(g).int_state(), ctx
    fo, fg = o.float_state(), to_oracle_record(g).float_state()
    for key in fo:
        a, b = np.atleast_1d(np.array(fo[key], dtype=np.float64)), np.atleast_1d(np.array(fg[key], dtype=np.float64))
        if key.startswith("shell_"):
            assert np.all(np.abs(a - b) <= FLOAT_REL_TOL * np.maximum(1.0, np.abs(a))), (ctx, key, a, b)
        else:
            assert np.array_equal(a, b), (ctx, key, a, b)


def assert_frame_close(expected, got, ctx):
    d = np.abs(expected.astype(np.int32) - got.astype(np.int32))
    assert d.max() <= FRAME_MAX_DELTA, (ctx, int(d.max()))
    assert (d == 0).mean() >= FRAME_MATCH_FRACTION, (ctx, float((d == 0).mean()))


def make(gametype, n, seeds=None, reset=True, warm=0, ends=None, device=0, **kw):
    """SFVecEnv(gametype, num_envs=n, device=device, seeds=seeds, **kw) (kw: render, native_obs, copy_outputs,
    action_repeat, ...), then in this order: reset() unless reset=False; `warm` synthetic steps of one tick each whatever
    the action repeat (action seed `seeds`, an int), which leave ships, missiles and shells in flight; with ends=(lo, hi),
    clocks staggered so that the episodes end lo..hi-1 ticks from now, drawn from RandomState(seeds). Deterministic: two
    calls with the same arguments give equal states."""
    torch_cuda()
    from spacefortress_b200 import SFVecEnv, _lib
    env = SFVecEnv(gametype, num_envs=n, device=device, seeds=seeds, **kw)
    k = env.action_repeat
    assert k == 1 or env.L.sf_action_repeat(env.h) == k
    if reset:
        env.reset()
    if warm:
        if k != 1:
            _lib.check(env.L.sf_set_action_repeat(env.h, 1))
        env.rollout(warm, action_seed=seeds, want=("reward",))
        if k != 1:
            _lib.check(env.L.sf_set_action_repeat(env.h, k))
    if ends:
        stagger(env, np.random.RandomState(seeds).randint(*ends, size=n))
    return env


def stagger(env, ends_in):
    """Clocks (sf_set_ticks) so that env i's episode ends ends_in[i] ticks from now. Returns the ticks."""
    ticks = (END_TICK - np.asarray(ends_in)).astype(np.int32)
    env.set_ticks(ticks)
    return ticks


def spec(env, name):
    """(per-env shape, numpy dtype) of an output: "obs" (a frame of the env's size), a feature kind (its row),
    "actions" or one of STEP_OUTPUTS"""
    from spacefortress_b200 import _lib
    if name == "obs":
        return env.obs_shape[1:], np.uint8
    if name in KINDS:
        return (env.L.sf_num_features(env.h, _lib.OBS_TYPES[name]),), np.float32
    return (), np.int32 if name in ("actions", "reward", "events") else np.uint8


def outputs(env, T, want):
    """time-major CUDA outputs [T, n, ...] of the names in `want` (see spec); feature rows are NaN until written"""
    torch = torch_cuda()
    out = {}
    for name in want:
        shape, dt = spec(env, name)
        out[name] = torch.empty((T, env.num_envs) + shape, dtype=getattr(torch, np.dtype(dt).name), device="cuda")
        if name in KINDS:
            out[name].fill_(float("nan"))
    return out


def ptrs(out, names, t=None):
    """pointers to the outputs `names` (of step t if given); None for a name not in `out`"""
    return [vp(out[k] if t is None else out[k][t]) if k in out else None for k in names]


def rollout(env, T, actions=None, action_seed=0, t0=0, flags=0, want=("obs", "reward", "done", "kill")):
    """sf_rollout: T agent steps in one launch, of the given actions (CUDA [T, n]) or the synthetic ones"""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    out = outputs(env, T, want)
    _lib.check(env.L.sf_rollout(env.h, T, vp(actions), action_seed, t0, *ptrs(out, ("obs", "reward", "done", "kill")), flags, None))
    torch.cuda.synchronize()
    return out


def single_steps(env, actions, flags=0, want=STEP_OUTPUTS):
    """T x sf_step, one launch per agent step of actions (CUDA [T, n]), each followed by sf_features of the state it left
    for every feature kind in `want`"""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    out = outputs(env, len(actions), want)
    for t in range(len(actions)):
        _lib.check(env.L.sf_step(env.h, vp(actions[t]), *ptrs(out, ("obs",) + STEP_OUTPUTS, t), flags, None))
        for kind in want:
            if kind in KINDS:
                _lib.check(env.L.sf_features(env.h, _lib.OBS_TYPES[kind], vp(out[kind][t]), None))
    torch.cuda.synchronize()
    return out


def rollout_features(env, kind, T, actions=None, action_seed=0, t0=0, flags=0, want=STEP_OUTPUTS):
    """sf_rollout_features: T agent steps in one launch; the feature rows of step t are out[kind][t]"""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    out = outputs(env, T, (kind,) + tuple(want))
    _lib.check(env.L.sf_rollout_features(env.h, _lib.OBS_TYPES[kind], T, vp(actions), action_seed, t0,
                                         *ptrs(out, (kind,) + STEP_OUTPUTS), flags, None))
    torch.cuda.synchronize()
    return out


def step_host(env, actions, flags=0, pinned=True, want=("obs",) + STEP_OUTPUTS):
    """T x sf_step_host, or T x sf_step_host_features when `want` names a feature kind instead of "obs", with the host
    actions [T, n], through page-locked (pinned) or pageable buffers that live for the T steps. Returns what the buffers
    held after every step, time-major (numpy). Feature rows are set to NaN before each step."""
    from spacefortress_b200 import _lib
    new = _lib.pinned_array if pinned else np.zeros
    buf = {}
    for name in ("actions",) + tuple(want):
        shape, dt = spec(env, name)
        buf[name] = new((env.num_envs,) + shape, dt)
    out = {name: np.empty((len(actions),) + b.shape, b.dtype) for name, b in buf.items() if name != "actions"}
    kind = next((k for k in want if k in KINDS), None)
    for t in range(len(actions)):
        buf["actions"][:] = actions[t]
        if kind is None:
            _lib.check(env.L.sf_step_host(env.h, hp(buf["actions"]), *[hp(buf.get(k)) for k in ("obs",) + STEP_OUTPUTS], flags))
        else:
            buf[kind][:] = np.nan
            _lib.check(env.L.sf_step_host_features(env.h, _lib.OBS_TYPES[kind], hp(buf["actions"]),
                                                   *[hp(buf.get(k)) for k in (kind,) + STEP_OUTPUTS], flags))
        for name in out:
            out[name][t] = buf[name]
    if pinned and "obs" in buf:
        _lib.check(env.L.sf_host_forget(env.h, hp(buf["obs"])))  # the library may remember it for delta updates
    return out
