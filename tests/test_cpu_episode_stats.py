"""EpisodeStats without a GPU: the ring-to-deque step (episode_stats.ring_entries) against a brute-force deque, the
argument checks of the constructor and of record(), and the C entry point's refusals.

The ring rule restated here is the one hl_episode_stats applies: the j-th done env of a step (ascending env id) is entry
total + j and goes to slot (total + j) mod maxlen, and of a step with m > maxlen done envs only ranks j >= m - maxlen
write."""
import random
from collections import deque

import pytest
import torch

from isaacgymloco_b200 import _lib as L
from isaacgymloco_b200.episode_stats import EpisodeStats, check_step_args, ring_entries


def _write_step(ring, total, values):
    size, m = len(ring), len(values)
    for j, v in enumerate(values):
        if j >= m - size:
            ring[(total + j) % size] = v
    return total + m


@pytest.mark.parametrize("maxlen", [1, 2, 7, 100, 5000])
def test_ring_entries_equal_a_deque(maxlen):
    """Random per-step counts (none, a few, more than maxlen in one step) and irregular collection cadences: the deque
    extended from the ring at each collection equals the deque extended at every step."""
    rng = random.Random(maxlen)
    for trial in range(20):
        ring, total, seen = [float("nan")] * maxlen, 0, 0
        want, got = deque(maxlen=maxlen), deque(maxlen=maxlen)
        next_value = 0
        for step in range(rng.randrange(1, 60)):
            kind = rng.random()
            m = 0 if kind < 0.25 else rng.randrange(1, 4) if kind < 0.6 else rng.randrange(maxlen, 3 * maxlen + 2)
            values = [float(next_value + j) for j in range(m)]
            next_value += m
            want.extend(values)
            total = _write_step(ring, total, values)
            if rng.random() < [1.0, 0.3, 1 / 7][trial % 3]:
                got.extend(ring_entries(seen, total, ring))
                seen = total
                assert list(got) == list(want), (maxlen, trial, step)
        got.extend(ring_entries(seen, total, ring))
        assert list(got) == list(want), (maxlen, trial)


def test_ring_entries_edges():
    ring = [10.0, 11.0, 12.0]                      # entries 0..5 written: slots hold entries 3, 4, 5 as 10, 11, 12
    assert ring_entries(6, 6, ring) == []
    assert ring_entries(5, 6, ring) == [12.0]
    assert ring_entries(0, 6, ring) == [10.0, 11.0, 12.0]
    assert ring_entries(4, 7, ring) == [11.0, 12.0, 10.0]
    with pytest.raises(ValueError):
        ring_entries(7, 6, ring)
    with pytest.raises(ValueError):
        ring_entries(-1, 6, ring)


def test_constructor_rejects_bad_arguments():
    with pytest.raises(ValueError, match="num_envs"):
        EpisodeStats(0, "cuda:0")
    with pytest.raises(ValueError, match="maxlen"):
        EpisodeStats(16, "cuda:0", maxlen=0)
    with pytest.raises(ValueError, match="CPU fallback"):
        EpisodeStats(16, "cpu")


def test_record_arguments():
    n, dev = 16, torch.device("cuda", 0)
    rew, done = torch.zeros(n), torch.zeros(n, dtype=torch.bool)
    ids, cnt = torch.zeros(n, dtype=torch.long), torch.zeros(1, dtype=torch.int32)
    for args in ((rew, done, ids), (rew, done.view(torch.uint8), ids[:3]), (rew, done, ids, cnt)):
        with pytest.raises(RuntimeError, match="CPU fallback"):
            check_step_args(n, dev, *args)
    bad = [(rew.double(), done, ids), (rew[:-1], done, ids), (rew, done.int(), ids), (rew, done[:-1], ids),
           (rew, done, ids.int()), (rew, done, torch.zeros(n + 1, dtype=torch.long)), (rew, done, ids, cnt.long()),
           (rew, done, ids, torch.zeros(2, dtype=torch.int32))]
    for args in bad:
        with pytest.raises(ValueError):
            check_step_args(n, dev, *args)
    with pytest.raises(TypeError):
        check_step_args(n, dev, rew, done, [0, 1])


def test_c_entry_point_refuses_bad_arguments():
    """Refused before anything is launched (the pointers below are never dereferenced)."""
    p = [0x1000 * (k + 1) for k in range(9)]

    def call(rew=p[0], dones=p[1], ids=p[2], cnt=p[3], cur_r=p[4], cur_l=p[5], ring_r=p[6], ring_l=p[7], ring_size=4,
             cursor=p[8], n=16):
        return L.lib.hl_episode_stats(rew, dones, ids, cnt, cur_r, cur_l, ring_r, ring_l, ring_size, cursor, n, None)

    for kw in (dict(rew=None), dict(dones=None), dict(ids=None), dict(cnt=None), dict(cur_r=None), dict(cur_l=None),
               dict(ring_r=None), dict(ring_l=None), dict(cursor=None), dict(ring_size=0), dict(ring_size=-3), dict(n=0),
               dict(n=-1)):
        assert call(**kw) == 1, kw                  # HL_E_INVALID
        assert b"hl_episode_stats" in L.lib.hl_last_error(), kw
