"""Replay a captured rollout every PPO iteration (FusedLeggedRobot.capture_rollout).

A CUDA graph repeats what was true when it was captured.  Two things make a replayed rollout equal to the same
rollout run eagerly:

* the kernels' randomness (observation noise, terminal-observation noise, pre-step command resampling, reset
  re-draws: Philox streams 0-3) is keyed by the step index.  While a rollout is captured the env passes step k as
  philox_offset = k relative to a device counter (HlEnvBuffers.step_base), and the last captured op advances that
  counter by T; a replay that starts at host counter c therefore draws the keys c .. c+T-1, as T eager steps do.
* the host's own per-step decisions -- a disturbance every `disturbance_interval` steps, a push every
  `push_interval` steps (the staged path), the command curriculum every `max_episode_length` steps (an .item()) --
  and everything copied into the launches (command and reset ranges) are frozen in a graph.  `rollout_window()`
  decides per window whether a captured graph fits; `RolloutGraph.run()` replays one when it does and runs the same
  `body` eagerly when it does not.

torch-RNG hooks inside `body` (_delay_actions, _disturbance_robots, the policy's action sampling) stay torch: PyTorch's
graph-safe Philox gives them fresh draws on every replay.  A live Isaac Gym sim cannot be captured (gym.simulate is
a host call); this mode is for standalone, replayed or otherwise capturable physics (physics_step_fn).
"""
from collections import OrderedDict
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np
import torch


def _first_multiple(lo: int, m: int) -> int:
    """Smallest multiple of m that is >= lo (m > 0)."""
    return -(-lo // m) * m


def rollout_window(counter: int, num_steps: int, disturbance_interval: int = 0, push_interval: int = 0,
                   curriculum_interval: int = 0) -> Tuple[Optional[Tuple[int, ...]], Optional[str]]:
    """Can the `num_steps` env steps that start at common_step_counter `counter` replay a captured graph?

    Step k of the window runs with the counter at counter + k + 1 (post_physics_step increments it first) and the
    host decides on that value: a disturbance when it is a multiple of `disturbance_interval`, a push when it is a
    multiple of `push_interval`, the command curriculum when it is a multiple of `curriculum_interval`; 0 = never.
    Returns (key, None), key = the window's steps k that apply a disturbance (graphs are cached by it), or
    (None, reason) when the window has to run eagerly."""
    lo, hi = counter + 1, counter + num_steps
    for name, m in (("push", push_interval), ("command-curriculum", curriculum_interval)):
        if m > 0 and _first_multiple(lo, m) <= hi:
            return None, f"{name} step at counter {_first_multiple(lo, m)}"
    if disturbance_interval <= 0:
        return (), None
    first = _first_multiple(lo, disturbance_interval)
    return tuple(range(first - lo, num_steps, disturbance_interval)), None


def env_schedule(env) -> Dict[str, int]:
    """The intervals rollout_window() needs, as the env's post_physics_step_device() applies them."""
    R = env.cfg_hot.reset
    return dict(disturbance_interval=int(env.cfg_hot.disturbance_interval) if R.disturbance else 0,
                push_interval=int(env.push_interval) if R.push_robots else 0,
                curriculum_interval=int(env.max_episode_length) if R.commands_curriculum else 0)


class EpisodeTables:
    """reset_idx's episode logging (LR:344-359) of every step of one rollout, kept on the device so the rollout needs
    no host sync: the reset launch of step k writes its means to row k (HlReset.means_out), and the step adds its reset
    count and the sum of terrain_levels (one reduction launch, only with the terrain curriculum)."""

    def __init__(self, env, num_steps: int):
        dev = env.device
        self.means = torch.zeros(num_steps, max(env._episode_sums_buf.shape[0], 1), device=dev)
        self.counts = torch.zeros(num_steps, dtype=torch.int32, device=dev)
        self.terrain_sum = torch.zeros(num_steps, dtype=torch.long, device=dev)
        self.max_command_x = [0.0] * num_steps
        pin = dict(device="cpu", pin_memory=True)
        self._host = (torch.zeros(self.means.shape, **pin), torch.zeros(num_steps, dtype=torch.int32, **pin),
                      torch.zeros(num_steps, dtype=torch.long, **pin))

    @staticmethod
    def logs_terrain(env) -> bool:
        return bool(env.cfg_hot.reset.terrain_curriculum and env.terrain_origins is not None)

    def record(self, env, k: int):
        """After the reset launch of step k (called by post_physics_step_device)."""
        self.counts[k:k + 1].copy_(env._n_reset)
        if self.logs_terrain(env):
            torch.sum(env.terrain_levels, dim=0, out=self.terrain_sum[k])
        self.max_command_x[k] = float(env.command_ranges["lin_vel_x"][1])

    def episode_infos(self, env) -> List[Dict]:
        """One dict per step that had resets, with _log_episode's keys and values (as Python floats: the tables come
        to the host in one go, the one host sync of a rollout)."""
        for h, d in zip(self._host, (self.means, self.counts, self.terrain_sum)):
            h.copy_(d, non_blocking=True)
        torch.cuda.current_stream(env.device).synchronize()
        means, counts, tsum = (h.tolist() for h in self._host)
        terrain = self.logs_terrain(env)
        names = list(env.episode_sums.keys())
        infos = []
        for k, cnt in enumerate(counts):
            if cnt <= 0:
                continue
            ep = {"rew_" + key: means[k][j] for j, key in enumerate(names)}
            if terrain:      # torch.mean(terrain_levels.float()) of LR:352-353: the float32 quotient of the exact sum
                ep["terrain_level"] = float(np.float32(tsum[k]) / np.float32(env.num_envs))
            if env.cfg_hot.reset.commands_curriculum:
                ep["max_command_x"] = self.max_command_x[k]
            infos.append(ep)
        return infos


class RolloutGraph:
    """`body(0) .. body(T-1)`, then `finish()`, as one CUDA graph replayed on every rollout whose window allows it
    (rollout_window), and run eagerly otherwise.  Graphs are cached by the positions of the window's disturbance
    steps (at most `max_graphs`) and recaptured when something the launches copy has changed since the capture
    (command / reset ranges, parity tensors, the storage slot the rollout starts from).  The first `warmup` rollouts
    run eagerly, so lazily initialised libraries (cuBLAS handles, allocator pools) are set up before any capture.

    Host-side effects of `body` happen only when it runs (eagerly or while capturing); after a replay run() restores
    what T eager steps leave on the host: common_step_counter += T, storage.step, the env's rollout-slot binding and
    extras.  run() returns the reference's per-step `ep_infos`."""

    def __init__(self, env, body: Callable[[int], None], num_steps: int, storage=None,
                 finish: Optional[Callable[[], None]] = None, max_graphs: int = 8, warmup: int = 1):
        if not env._kernel_reset_ok():
            raise ValueError("capture_rollout needs the in-kernel reset (a torch reset hook syncs on the host every step)")
        if getattr(env, "gym", None) is not None:
            raise ValueError("capture_rollout needs standalone physics: gym.simulate cannot be captured")
        if num_steps <= 0:
            raise ValueError("num_steps must be positive")
        self.env, self.body, self.num_steps, self.storage, self.finish = env, body, int(num_steps), storage, finish
        self.max_graphs, self.warmup = max(int(max_graphs), 1), int(warmup)
        self.tables = EpisodeTables(env, self.num_steps)
        self._graphs = OrderedDict()           # key -> (graph, signature, host state after the rollout)
        self._device_counter = None            # what env._step_base holds, when known
        self.stats = {"replays": 0, "captures": 0, "eager": 0}
        self.last_mode, self.last_reason = None, None

    # ------------------------------------------------------------------ pieces
    def _signature(self):
        """What the captured launches copied from the host, besides the schedule: the HlReset ranges / flags / pointers,
        the parity tensors, the slots the rollout reads its first observation from and the storage step."""
        env, st = self.env, self.storage
        noise = tuple(None if t is None else t.data_ptr() for t in env._noise.values())
        return (bytes(env._reset_struct()), noise, env.obs_buf.data_ptr(), env.privileged_obs_buf.data_ptr(),
                st.step if st is not None else None, env.resample_interval)

    def _host_state(self):
        env, st = self.env, self.storage
        return dict(counter=env.common_step_counter, step=st.step if st is not None else None, obs=env.obs_buf,
                    priv=env.privileged_obs_buf, extras=dict(env.extras))

    def _set_host_state(self, h):
        env, st = self.env, self.storage
        env.common_step_counter = h["counter"]
        if st is not None:
            st.step = h["step"]
        env.obs_buf, env.privileged_obs_buf = h["obs"], h["priv"]
        env.extras.clear()
        env.extras.update(h["extras"])

    def _steps(self):
        env = self.env
        try:
            for k in range(self.num_steps):
                env._ep_log = (self.tables, k)
                self.body(k)
        finally:
            env._ep_log = None
        if self.finish is not None:
            self.finish()

    def _capture(self):
        env = self.env
        before = self._host_state()
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream(device=env.device)
        s.wait_stream(torch.cuda.current_stream(env.device))
        env._capture_base = env.common_step_counter
        try:
            with torch.cuda.graph(g, stream=s):
                self._steps()
                env._step_base.add_(self.num_steps)
            after = self._host_state()
        finally:
            env._capture_base = None
            self._set_host_state(before)          # the capture executed nothing
        torch.cuda.current_stream(env.device).wait_stream(s)
        self.stats["captures"] += 1
        return g, after

    # ------------------------------------------------------------------ the rollout
    def run(self) -> List[Dict]:
        env, T = self.env, self.num_steps
        c = env.common_step_counter
        key, reason = rollout_window(c, T, **env_schedule(env))
        if key is not None and self.warmup > 0:
            key, reason = None, "warm-up"
            self.warmup -= 1
        if key is None:
            self._steps()
            env._step_base.fill_(env.common_step_counter)
            self._device_counter = env.common_step_counter
            self.stats["eager"] += 1
            self.last_mode, self.last_reason = "eager", reason
        else:
            sig = self._signature()
            entry = self._graphs.get(key)
            mode = "replay"
            if entry is None or entry[1] != sig:
                self._graphs.pop(key, None)
                g, after = self._capture()
                entry = self._graphs[key] = (g, sig, after)
                while len(self._graphs) > self.max_graphs:
                    self._graphs.popitem(last=False)
                mode = "capture+replay"
            self._graphs.move_to_end(key)
            g, _, after = entry
            if self._device_counter != c:
                env._step_base.fill_(c)
            g.replay()
            self._device_counter = c + T
            self._set_host_state(after)
            env.common_step_counter = c + T
            self.stats["replays"] += 1
            self.last_mode, self.last_reason = mode, None
        infos = self.tables.episode_infos(env)
        env.extras["time_outs"] = env.time_out_buf
        if infos:
            env.extras["episode"] = infos[-1]
        return infos
