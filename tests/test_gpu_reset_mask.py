"""GPU (-m gpu): sf_reset with an env mask. The Python layer always resets every env, so this calls the C-ABI directly.
A masked-in env starts a new game and its first frame is drawn; a masked-out env keeps its state and its frame bytes are
not written. The batch is large enough that blocks own more than one group of envs."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5


@pytest.mark.parametrize("native", [False, True])
def test_reset_mask_draws_only_masked_envs(native):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from spacefortress_b200 import SFVecEnv, _lib
    n = 5000  # > 148 SMs x 32 envs: more groups than blocks
    env = SFVecEnv("youturn", num_envs=n, device=0, native_obs=native)
    try:
        env.reset(to_numpy=False)
        env.rollout(300, action_seed=7, want=("reward",))  # states far from a new game: moved ships, dead ships, shells
        torch.cuda.synchronize()
        mask = np.arange(n) % 3 == 0
        before = env.get_state()
        assert all(before[i].tick > 0 for i in np.flatnonzero(mask))
        before = [bytes(r) for r in before]

        d_mask = torch.from_numpy(mask.astype(np.uint8)).cuda()
        h, w = (_lib.NATIVE_H, _lib.NATIVE_W) if native else (_lib.OBS_H, _lib.OBS_W)
        obs = torch.full((n, h, w), SENTINEL, dtype=torch.uint8, device="cuda")
        flags = _lib.FLAG_NATIVE_OBS if native else 0
        _lib.check(env.L.sf_reset(env.h, C.c_void_p(d_mask.data_ptr()), 1, C.c_void_p(obs.data_ptr()), flags,
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        torch.cuda.synchronize()
        got = obs.cpu().numpy()
        ref = env.render_frames(native=native)
        after = env.get_state()

        on = np.flatnonzero(mask)
        off = np.flatnonzero(~mask)
        assert np.array_equal(got[on], ref[on]), "a masked-in env's reset frame differs from sf_render of its state"
        assert all(after[i].tick == 0 for i in on), "a masked-in env did not start a new game"
        assert (got[off] == SENTINEL).all(), "sf_reset wrote into the frame of a masked-out env"
        changed = [i for i in off if bytes(after[i]) != before[i]]
        assert not changed, "masked-out envs changed state: %r" % changed[:8]
    finally:
        env.close()
