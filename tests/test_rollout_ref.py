"""The fp64 references of tests/_rollout_ref.py that need no device: the numpy Philox port against the C mirror's draws."""
import numpy as np
from _rollout_ref import philox, u53


def test_philox_port_matches_the_reset_draws(fonet):
    """The numpy port against oracle.c_mirror.draw_random, whose philox4x32_10 draws are bit-matched to the GPU's resets:
    seeds and env ids past 2^32 included (all four counter words and both key words are live)."""
    from oracle import c_mirror
    for seed in (0, 1234, (7 << 32) + 5, 2 ** 64 - 1):
        for gid in (0, 3, 1000, (1 << 32) + 17):
            for episode in (0, 9):
                _, _, a0 = c_mirror.draw_random(fonet, seed, gid, episode, 1000)
                b = np.arange(10, dtype=np.uint32)
                c = philox(np.full(10, gid & 0xFFFFFFFF, np.uint32), np.full(10, gid >> 32, np.uint32),
                           np.full(10, episode, np.uint32), b, seed & 0xFFFFFFFF, seed >> 32)
                v0, v1 = u53(c[0], c[1]), u53(c[2], c[3])
                want = np.empty((5, 4)); want[:, 0] = v0[0::2]; want[:, 1] = v1[0::2]; want[:, 2] = v0[1::2]; want[:, 3] = v1[1::2]
                assert np.array_equal(a0.reshape(5, 4), want), (seed, gid, episode)
