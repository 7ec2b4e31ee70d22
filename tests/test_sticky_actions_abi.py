"""CPU: the sticky-action calls of the C-ABI without a device: the NULL handle, the event bit, and the host form of the
per-tick draw (sf_sticky_draw), which is the function the repeat kernel evaluates."""
import numpy as np

from spacefortress_b200 import _lib


def test_sticky_calls_reject_a_null_handle():
    L = _lib.lib()
    assert L.sf_set_sticky_actions(None, 0.25, 1) == _lib.SF_ERR_INVALID
    assert b"handle" in L.sf_last_error()
    assert L.sf_sticky_actions(None) == -1.0


def test_the_event_bit_matches_the_header():
    src = open(_lib.os.path.join(_lib.HERE, "..", "include", "sf_b200.h")).read()
    assert "SF_EV_STICKY = 1 << 22" in src
    assert _lib.EV_STICKY == 1 << 22 and not _lib.EV_STICKY & _lib.EV_EPISODE_RESET


def test_the_draw_at_the_ends_of_the_range():
    L = _lib.lib()
    rng = np.random.RandomState(0)
    for _ in range(2000):
        seed, env, cnt, tick = int(rng.randint(1 << 32, dtype=np.uint64)), int(rng.randint(1 << 40)), int(rng.randint(1 << 32, dtype=np.uint64)), int(rng.randint(-2, 6000))
        assert L.sf_sticky_draw(seed, env, cnt, tick, 0.0) == 0
        assert L.sf_sticky_draw(seed, env, cnt, tick, 1.0) == 1
    for p in (-0.01, 1.01, float("nan"), float("inf")):
        assert L.sf_sticky_draw(1, 0, 0, 0, p) == -1, p


def test_the_draw_rate_is_p():
    """10^6 (rng_count, tick) counters of a few envs: the stick rate is within 5 sigma of p, and a draw is monotone in p
    (the keys that stick at p stick at every larger p)."""
    L = _lib.lib()
    draw = L.sf_sticky_draw
    m = 10 ** 6
    for p in (0.25, 0.75):
        hits = 0
        for i in range(m):
            hits += draw(7, i & 3, 120 + (i >> 2) // 5295, (i >> 2) % 5295, p)
        sigma = np.sqrt(p * (1 - p) / m)
        assert abs(hits / m - p) < 5 * sigma, (p, hits / m)
    for i in range(20000):
        if draw(3, 5, 200, i, 0.3):
            assert draw(3, 5, 200, i, 0.6) == 1, i


M64 = (1 << 64) - 1


def header_draw(seed, env, rng_count, tick):
    """u of include/sf_b200.h, written out independently of the library"""
    c = (rng_count << 32) | (tick & 0xFFFFFFFF)
    z = ((env * 0x9E3779B97F4A7C15) & M64) ^ ((c * 0xC2B2AE3D27D4EB4F) & M64) ^ ((seed << 32) | 0x57)
    z ^= z >> 30
    z = (z * 0xBF58476D1CE4E5B9) & M64
    z ^= z >> 27
    z = (z * 0x94D049BB133111EB) & M64
    z ^= z >> 31
    return z >> 32


# (seed, global_env, rng_count, tick) -> u, from header_draw
KNOWN = [((0, 0, 0, 0), 3474303030), ((1, 0, 120, 1), 1556794415), ((11, 47, 3000, 5294), 12928952),
         ((0xFFFFFFFF, (1 << 40) + 3, 0xFFFFFFFF, -1), 2943730514), ((13, 4095, 77, 2500), 3837237623)]


def test_the_draw_is_the_header_formula():
    """The library's draw sticks at threshold u + 1 and not at u, i.e. it computes exactly the header's u: for fixed
    vectors (which pin the salt and the packing of the counter) and for random inputs against header_draw."""
    L = _lib.lib()
    rng = np.random.RandomState(5)
    cases = [v for v, _ in KNOWN] + [(int(rng.randint(1 << 32, dtype=np.uint64)), int(rng.randint(1 << 40)),
                                      int(rng.randint(1 << 32, dtype=np.uint64)), int(rng.randint(-5, 6000))) for _ in range(500)]
    for v, u in KNOWN:
        assert header_draw(*v) == u, v
    for v in cases:
        u = header_draw(*v)
        assert L.sf_sticky_draw(*v, u / 2.0 ** 32) == 0, v
        assert L.sf_sticky_draw(*v, (u + 1) / 2.0 ** 32) == 1, v
