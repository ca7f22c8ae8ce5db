"""CPU: RolloutGraph(capture_schedule=True)'s host side -- the window key when push and command-curriculum steps are
captured too (rollout_window(..., in_graph=True)), and the per-step max_command_x rebuilt from the ranges the device
curriculum logged -- against brute-force walks over the steps of a window."""
import random

import pytest

from isaacgymloco_b200.rollout_graph import max_command_x_per_step, rollout_window


def _brute(counter, T, dist, push, cur):
    """Step k of the window runs with common_step_counter == counter + k + 1: the steps that disturb, push, decide."""
    at = lambda m: tuple(k for k in range(T) if m > 0 and (counter + k + 1) % m == 0)
    return (at(dist), at(push), at(cur)), None


@pytest.mark.parametrize("T", [1, 2, 7, 8, 24, 25])
def test_in_graph_window_matches_brute_force(T):
    intervals = [0, 1, 3, 8, 24, 25, 250]
    n = 0
    for counter in range(0, 520, 7):
        for dist in intervals:
            for push in intervals:
                for cur in (0, 1, 8, 24, 1000):
                    got = rollout_window(counter, T, disturbance_interval=dist, push_interval=push, curriculum_interval=cur,
                                         in_graph=True)
                    assert got == _brute(counter, T, dist, push, cur), (counter, T, dist, push, cur)
                    assert got[0] is not None and got[1] is None          # never eager
                    n += 1
    assert n > 10000


def test_in_graph_window_examples():
    # the reference schedule: T = 100, a disturbance every 8 steps, a push every 800, the curriculum every 1000
    sched = dict(disturbance_interval=8, push_interval=800, curriculum_interval=1000)
    keys = [rollout_window(c, 100, **sched, in_graph=True)[0] for c in range(0, 4000, 100)]
    assert sum(1 for k in keys if k[1]) == 5 and sum(1 for k in keys if k[2]) == 4
    assert keys[0] == (tuple(range(7, 100, 8)), (), ())
    assert keys[7] == (tuple(range(3, 100, 8)), (99,), ())                # counter 800 is step 99 of the window at 700
    assert keys[9] == (tuple(range(3, 100, 8)), (), (99,))                # counter 1000
    assert keys[39] == (tuple(range(3, 100, 8)), (99,), (99,))            # counter 4000: both
    assert len(set(keys)) == 5                                            # the graphs one 4,000-step cycle needs
    # without in_graph the same windows still run eagerly
    assert rollout_window(700, 100, **sched) == (None, "push step at counter 800")
    assert rollout_window(900, 100, **sched) == (None, "command-curriculum step at counter 1000")


def _walk(start, T, cur_steps, moves):
    """Brute force: the host value after each step of a rollout in which step k of `cur_steps` moved the ranges to
    moves[k] (None = the decision left them alone)."""
    val, out = start, []
    for k in range(T):
        if k in cur_steps and moves[k] is not None:
            val = moves[k]
        out.append(val)
    return out


@pytest.mark.parametrize("n_cur", [0, 1, 2])
def test_max_command_x_from_logged_rows(n_cur):
    rng = random.Random(n_cur)
    for trial in range(200):
        T = rng.choice([1, 5, 20, 100])
        cur_steps = sorted(rng.sample(range(T), min(n_cur, T)))
        start = rng.choice([0.5, 1.0, 1.4999999999999998])
        moves, rows, val = {}, [[float("nan")] * 8 for _ in range(T)], start   # rows the device never wrote stay NaN
        for k in cur_steps:
            widen = rng.random() < 0.5
            moves[k] = min(val + 0.1, 1.5) if widen else None
            val = moves[k] if widen else val
            rows[k] = [-val, val, -0.3, 0.3, -1.0, 1.0, -3.14, 3.14]   # the ranges after step k's decision
        assert max_command_x_per_step(start, cur_steps, rows, T) == _walk(start, T, set(cur_steps), moves), (trial, cur_steps)


def test_max_command_x_examples():
    rows = [[0.0] * 8 for _ in range(6)]
    rows[2][1], rows[4][1] = 1.1, 1.2
    assert max_command_x_per_step(1.0, (), rows, 6) == [1.0] * 6
    assert max_command_x_per_step(1.0, (2,), rows, 6) == [1.0, 1.0, 1.1, 1.1, 1.1, 1.1]
    assert max_command_x_per_step(1.0, (2, 4), rows, 6) == [1.0, 1.0, 1.1, 1.1, 1.2, 1.2]
