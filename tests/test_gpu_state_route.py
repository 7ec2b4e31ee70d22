"""GPU (-m gpu): the state-only step (render off: sf_rollout without frames, sf_rollout_features) against the fused step +
render kernel (sf_rollout and sf_step with frames). Both run the same game step in different kernels; from equal states
with episodes ending inside the call they must return the same bits and leave the same states and episode statistics."""
import numpy as np
import pytest

from gpu_helpers import END_TICK, STEP_OUTPUTS, make, rollout, rollout_features, single_steps, stagger, torch_cuda

pytestmark = pytest.mark.gpu


def run(env, start, call):
    """load `start`, run `call` (returns the outputs as CUDA tensors), then (outputs as numpy, env blobs, episode stats)"""
    env.load_envs(start)
    env.episode_stats(reset=True, all_reduce=False)
    out = {key: v.cpu().numpy() for key, v in call().items()}
    return out, env.save_envs().cpu().numpy(), env.episode_stats(reset=True, all_reduce=False)


@pytest.mark.parametrize("T", [1, 7, 64])
@pytest.mark.parametrize("n", [1, 33, 4096, 4737])
@pytest.mark.parametrize("gametype", ["youturn", "autoturn"])
def test_state_only_steps_equal_the_fused_kernel(gametype, n, T):
    """Given actions from one state whose episodes end 1..T+1 ticks from now (most of them inside the call): the
    render-off sf_rollout and sf_rollout_features equal the frame sf_rollout in reward, done and kill; the events of
    sf_rollout_features equal those of T x sf_step with frames; the saved env blobs and sf_episode_stats after every
    call are equal."""
    torch = torch_cuda()
    from spacefortress_b200 import _lib
    env = make(gametype, n, seeds=n + T, warm=20)
    ends = np.random.RandomState(n + T).randint(1, T + 2, size=n)
    ends[0] = 1  # at least one episode ends, whatever n
    stagger(env, ends)
    start = env.save_envs()
    acts = torch.from_numpy(np.random.RandomState(T).randint(env.num_actions, size=(T, n)).astype(np.int32)).cuda()
    runs = {
        "fused sf_rollout": run(env, start, lambda: rollout(env, T, acts, flags=env._flags)),
        "fused sf_step": run(env, start, lambda: single_steps(env, acts, flags=env._flags, want=("obs",) + STEP_OUTPUTS)),
        "state-only sf_rollout": run(env, start, lambda: rollout(env, T, acts, want=("reward", "done", "kill"))),
        "sf_rollout_features": run(env, start, lambda: rollout_features(env, "features", T, acts)),
    }
    ref, ref_blob, ref_stats = runs["fused sf_rollout"]
    assert ref["done"].any() and ref_stats["episodes"] > 0
    for name, (out, blob, stats) in runs.items():
        for key in ("reward", "done", "kill"):
            assert np.array_equal(out[key], ref[key]), (gametype, n, T, name, key)
        assert np.array_equal(blob, ref_blob), (gametype, n, T, name, "env blobs")
        assert stats == ref_stats, (gametype, n, T, name, stats, ref_stats)
    ev, ev_ref = runs["sf_rollout_features"][0]["events"], runs["fused sf_step"][0]["events"]
    assert np.array_equal(ev, ev_ref), (gametype, n, T, "events")
    assert (ev.view(np.uint32) & _lib.EV_EPISODE_RESET).any()
    assert ref_stats["sum_length"] == END_TICK * ref_stats["episodes"]
    env.close()
