"""CPU: the per-window decision of RolloutGraph.run() -- replay a captured rollout (and which cached graph), or run it
eagerly and why -- against a brute-force walk over the steps of the window, and the intervals it reads off an env."""
from types import SimpleNamespace

import pytest

from isaacgymloco_b200.rollout_graph import env_schedule, rollout_window


def _brute(counter, T, dist, push, cur):
    """Step k of the window runs with common_step_counter == counter + k + 1: what post_physics_step_device decides."""
    pushes, curs, dists = [], [], []
    for k in range(T):
        s = counter + k + 1
        if push > 0 and s % push == 0:
            pushes.append(s)
        if cur > 0 and s % cur == 0:
            curs.append(s)
        if dist > 0 and s % dist == 0:
            dists.append(k)
    if pushes:
        return None, f"push step at counter {pushes[0]}"
    if curs:
        return None, f"command-curriculum step at counter {curs[0]}"
    return tuple(dists), None


@pytest.mark.parametrize("T", [1, 2, 7, 8, 24, 25])
def test_window_decision_matches_brute_force(T):
    intervals = [0, 1, 3, 8, 24, 25, 250]
    n = 0
    for counter in range(0, 520, 7):
        for dist in intervals:
            for push in intervals:
                for cur in (0, 1, 8, 24, 1000):
                    got = rollout_window(counter, T, disturbance_interval=dist, push_interval=push, curriculum_interval=cur)
                    assert got == _brute(counter, T, dist, push, cur), (counter, T, dist, push, cur)
                    n += 1
    assert n > 10000


def test_window_examples():
    # disturbances every 8 steps, T = 24: every window has the same three disturbance steps, one graph serves all
    keys = {rollout_window(c, 24, disturbance_interval=8)[0] for c in range(0, 24 * 50, 24)}
    assert keys == {(7, 15, 23)}
    # T = 20 is out of step with the interval: the positions cycle through two keys
    keys = {rollout_window(c, 20, disturbance_interval=8)[0] for c in range(0, 20 * 50, 20)}
    assert keys == {(7, 15), (3, 11, 19)}
    assert rollout_window(990, 24, disturbance_interval=8, curriculum_interval=1000) == (None, "command-curriculum step at counter 1000")
    assert rollout_window(1000, 24, disturbance_interval=8, curriculum_interval=1000)[1] is None
    assert rollout_window(0, 24, push_interval=750) == ((), None)
    assert rollout_window(740, 24, push_interval=750) == (None, "push step at counter 750")


def test_env_schedule_follows_the_config_switches():
    reset = SimpleNamespace(disturbance=True, push_robots=True, commands_curriculum=True)
    env = SimpleNamespace(cfg_hot=SimpleNamespace(reset=reset, disturbance_interval=8), push_interval=750, max_episode_length=1001)
    assert env_schedule(env) == dict(disturbance_interval=8, push_interval=750, curriculum_interval=1001)
    reset.disturbance = reset.push_robots = reset.commands_curriculum = False
    assert env_schedule(env) == dict(disturbance_interval=0, push_interval=0, curriculum_interval=0)
