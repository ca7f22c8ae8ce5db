"""The host mirror of the AMP replay-ring cursor (amp_rollout.advance_cursor) against a brute-force loop of
ReplayBuffer.insert's bookkeeping (replay_buffer.py: num_samples = min(size, max(step + n, num_samples)),
step = (step + n) % size per insert)."""
import itertools
import random

from isaacgymloco_b200.amp_rollout import advance_cursor


def _brute(step, num_samples, size, n, inserts):
    for _ in range(inserts):
        num_samples = min(size, max(step + n, num_samples))
        step = (step + n) % size
    return step, num_samples


def _starts(size, n):
    """Reachable cursors: the state after k inserts of n rows into an empty ring, and after eager inserts of other
    sizes (the runner may insert between rollouts)."""
    out = {(0, 0)}
    for k in range(1, 2 * size // max(n, 1) + 3):
        out.add(_brute(0, 0, size, n, k))
    for m in (1, n - 1, n + 1, size // 2, size):
        if 0 < m <= size:
            out.add(_brute(0, 0, size, m, 1))
            out.add(_brute(*_brute(0, 0, size, m, 1), size, n, 1))
    return out


def test_advance_cursor_small_exhaustive():
    for size in range(1, 24):
        for n in range(1, size + 1):
            for (s0, ns0) in _starts(size, n):
                for inserts in range(0, 3 * size // n + 3):
                    assert advance_cursor(s0, ns0, size, n, inserts) == _brute(s0, ns0, size, n, inserts), \
                        (size, n, s0, ns0, inserts)


def test_advance_cursor_training_sizes():
    """Ring sizes of a training run (1,000,000 rows, and sizes that are not a multiple of N) with the env counts the
    project runs, over up to several wraps."""
    rng = random.Random(5)
    for size, n in itertools.product((1_000_000, 150_001, 65_536, 49_153), (4096, 16385, 65536)):
        if n > size:
            continue
        starts = [(0, 0), (size - 1, size), (rng.randrange(size), size)] + [_brute(0, 0, size, n, k) for k in (1, 7, 30)]
        for (s0, ns0) in starts:
            for inserts in (0, 1, 2, 24, 100, 251):
                assert advance_cursor(s0, ns0, size, n, inserts) == _brute(s0, ns0, size, n, inserts), \
                    (size, n, s0, ns0, inserts)


def test_advance_cursor_composes():
    """Windows of any split advance the same as one window: run() may advance by one pass of `body` at a time."""
    size, n = 10_007, 97
    s, ns = 0, 0
    for k in (3, 1, 0, 40, 2, 250):
        s, ns = advance_cursor(s, ns, size, n, k)
    assert (s, ns) == _brute(0, 0, size, n, 296)
