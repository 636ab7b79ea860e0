"""CPU: the device-side observation-history reference (tests/_obs_ref.py) against the per-env list model of the window
(the last H pushes since the env's last reset, oldest first, zero-padded in front) over random push / reset sequences."""
import numpy as np
import pytest
import torch

from _obs_ref import ObsRef

H, NA = 24, 5


@pytest.mark.parametrize("n,seed", [(7, 0), (33, 1), (70, 2)])
def test_obs_ref_matches_list_model(n, seed, monkeypatch):
    import _obs_ref
    monkeypatch.setattr(_obs_ref, "CHUNK", 16)                        # several chunks even at these sizes
    rng = np.random.default_rng(seed)
    ref = ObsRef(n, NA, H, "cpu")
    lists = [[] for _ in range(n)]
    slot = H - 1                                                      # env-minor ring slot of the newest push

    def window(e, extra=None):
        h = (lists[e] + ([extra] if extra is not None else []))[-H:]
        w = np.zeros((NA, H, 6))
        for k, x in enumerate(h):
            w[:, H - len(h) + k, :] = x
        return w.reshape(NA, 6 * H)

    for t in range(90):
        cur = rng.normal(size=(n, NA, 6))
        op = rng.uniform()
        if op < 0.2:                                                  # masked reset, with or without its own push
            m = rng.uniform(size=n) < 0.4
            ref.reset(m)
            for e in np.nonzero(m)[0]:
                lists[e] = []
            if rng.uniform() < 0.5:
                ref.push(cur, m)
                for e in np.nonzero(m)[0]:
                    lists[e].append(cur[e])
        elif op < 0.3:                                                # masked push (a masked step's generic push)
            m = rng.uniform(size=n) < 0.6
            ref.push(cur, m)
            for e in np.nonzero(m)[0]:
                lists[e].append(cur[e])
        else:                                                         # every env pushes: the ring slot advances
            ref.push(cur)
            slot = (slot + 1) % H
            for e in range(n):
                lists[e].append(cur[e])
        want = np.stack([window(e) for e in range(n)])
        got = torch.cat([ref.window(lo, hi) for lo, hi in ref.chunks()]).numpy()
        assert np.array_equal(got, want), t
        peek_cur = rng.normal(size=(n, NA, 6))
        got = torch.cat([ref.window(lo, hi, cur=peek_cur) for lo, hi in ref.chunks()]).numpy()
        assert np.array_equal(got, np.stack([window(e, peek_cur[e]) for e in range(n)])), t
        ring = torch.cat([ref.ring(slot, lo, hi) for lo, hi in ref.chunks()], dim=3).numpy()
        w = want.reshape(n, NA, H, 6).astype(np.float32)
        for s in range(H):
            assert np.array_equal(ring[(slot - H + 1 + s) % H].transpose(2, 0, 1), w[:, :, s, :]), (t, s)
        for lo, hi in ref.chunks():
            hist, live = ref.history(lo, hi)
            hist = hist.view(hi - lo, H, 32).numpy(); live = live.view(hi - lo, H, 32).numpy()
            for e in range(lo, hi):
                cnt = len(lists[e])
                assert int(ref.count_word()[e]) == cnt
                for k in range(max(0, cnt - H), cnt):
                    assert live[e - lo, k % H].all()
                    assert np.array_equal(hist[e - lo, k % H, :6 * NA], lists[e][k].reshape(-1))
                    assert not hist[e - lo, k % H, 6 * NA:].any()
                assert live[e - lo].all(axis=1).sum() == min(cnt, H) and not (live[e - lo].any(axis=1) & ~live[e - lo].all(axis=1)).any()


def test_obs_ref_round_f32():
    ref = ObsRef(3, NA, H, "cpu")
    x = np.full((3, NA, 6), 0.1)
    ref.push(x)
    ref.round_f32()
    assert torch.equal(ref.window(0, 3)[:, :, -6:], torch.full((3, NA, 6), float(np.float32(0.1)), dtype=torch.float64))
