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
  `body` eagerly when it does not.  With capture_schedule=True the push step (staged launches + torch RNG, no host
  sync) is captured as is, and the command ranges and the curriculum decision move to the device (HlReset.cmd_ranges,
  hl_command_curriculum), so windows with either step replay too; graphs are then cached by all three step positions.

torch-RNG hooks inside `body` (_delay_actions, _disturbance_robots, the policy's action sampling) stay torch: PyTorch's
graph-safe Philox gives them fresh draws on every replay.  A live Isaac Gym sim cannot be captured (gym.simulate is
a host call); this mode is for standalone, replayed or otherwise capturable physics (physics_step_fn).

amp=AMPRolloutStep (amp_rollout.py): the hybrid runner's AMP step inside `body` (hl_amp_transition, the discriminator
MLP, hl_amp_reward).  Its replay-ring cursor and normaliser snapshot live on the device; run() refreshes them from the
host objects at the start of every rollout and, after a replay, moves the replay buffer's host step / num_samples on by
the inserts the window made.

episode_stats=EpisodeStats (episode_stats.py): the runner's rewbuffer / lenbuffer bookkeeping inside `body`
(hl_episode_stats, one launch per step).  Its ring and entry count come back in the same copy batch as the episode
tables, before the one sync, and run() extends the host deques from them.
"""
from collections import OrderedDict
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np
import torch


def _first_multiple(lo: int, m: int) -> int:
    """Smallest multiple of m that is >= lo (m > 0)."""
    return -(-lo // m) * m


def rollout_window(counter: int, num_steps: int, disturbance_interval: int = 0, push_interval: int = 0,
                   curriculum_interval: int = 0, in_graph: bool = False) -> Tuple[Optional[tuple], Optional[str]]:
    """Can the `num_steps` env steps that start at common_step_counter `counter` replay a captured graph?

    Step k of the window runs with the counter at counter + k + 1 (post_physics_step increments it first) and the
    host decides on that value: a disturbance when it is a multiple of `disturbance_interval`, a push when it is a
    multiple of `push_interval`, the command curriculum when it is a multiple of `curriculum_interval`; 0 = never.
    Returns (key, None), key = the window's steps k that apply a disturbance (graphs are cached by it), or
    (None, reason) when the window has to run eagerly.

    in_graph=True (push and curriculum steps captured too, RolloutGraph(capture_schedule=True)): every window
    replays, and key = (disturbance steps, push steps, curriculum steps)."""
    lo, hi = counter + 1, counter + num_steps
    if in_graph:
        at = lambda m: tuple(range(_first_multiple(lo, m) - lo, num_steps, m)) if m > 0 else ()
        return (at(disturbance_interval), at(push_interval), at(curriculum_interval)), None
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


def max_command_x_per_step(start: float, curriculum_steps, logged_rows, num_steps: int) -> List[float]:
    """The per-step max_command_x of a rollout whose curriculum ran on the device: the value at the start of the rollout,
    carried forward and switched at each curriculum step k to lin_vel_x[1] of the ranges that step logged (row k of
    `logged_rows`, HlReset.cmd_ranges order)."""
    steps, cur, out = set(curriculum_steps), float(start), []
    for k in range(num_steps):
        if k in steps:
            cur = float(logged_rows[k][1])
        out.append(cur)
    return out


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
        # device-schedule mode: row k = the command ranges after the curriculum decision of step k (written by that
        # step's hl_command_curriculum launch only), and the device ranges after the rollout
        self.ranges_log = torch.zeros(num_steps, 8, dtype=torch.float64, device=dev)
        pin = dict(device="cpu", pin_memory=True)
        self._host = (torch.zeros(self.means.shape, **pin), torch.zeros(num_steps, dtype=torch.int32, **pin),
                      torch.zeros(num_steps, dtype=torch.long, **pin))
        self._host_ranges = (torch.zeros(num_steps, 8, dtype=torch.float64, **pin), torch.zeros(8, dtype=torch.float64, **pin))

    @staticmethod
    def logs_terrain(env) -> bool:
        return bool(env.cfg_hot.reset.terrain_curriculum and env.terrain_origins is not None)

    def record(self, env, k: int):
        """After the reset launch of step k (called by post_physics_step_device)."""
        self.counts[k:k + 1].copy_(env._n_reset)
        if self.logs_terrain(env):
            torch.sum(env.terrain_levels, dim=0, out=self.terrain_sum[k])
        self.max_command_x[k] = float(env.command_ranges["lin_vel_x"][1])

    def episode_infos(self, env, schedule=None) -> List[Dict]:
        """One dict per step that had resets, with _log_episode's keys and values (as Python floats: the tables come
        to the host in one go, the one host sync of a rollout).  schedule = (max_command_x at the start, the steps that
        ran the device curriculum) when the rollout ran in the device-schedule mode: the device ranges come back in the
        same batch, command_ranges takes them, and max_command_x is rebuilt from the logged rows."""
        for h, d in zip(self._host, (self.means, self.counts, self.terrain_sum)):
            h.copy_(d, non_blocking=True)
        if schedule is not None:
            for h, d in zip(self._host_ranges, (self.ranges_log, env._cmd_ranges_dev)):
                h.copy_(d, non_blocking=True)
        torch.cuda.current_stream(env.device).synchronize()
        means, counts, tsum = (h.tolist() for h in self._host)
        if schedule is not None:
            rows, now = (h.tolist() for h in self._host_ranges)
            env.set_command_ranges_flat(now)
            env._cmd_ranges_mirror = tuple(now)
            self.max_command_x = max_command_x_per_step(schedule[0], schedule[1], rows, len(counts))
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
    extras.  run() returns the reference's per-step `ep_infos`.

    amp (an AMPRolloutStep whose step() `body` calls): its discriminator parameters, ring tensors and buffers join the
    graph signature (rebinding any of them recaptures; in-place optimizer steps and load_state_dict do not), run()
    refreshes its normaliser snapshot and device cursor first, and after a replay the replay buffer's host step /
    num_samples advance by (amp.step() calls in one pass of `body`) x N inserts, as the eager window leaves them.

    episode_stats (an EpisodeStats whose record() `body` calls): its buffer addresses and ring size join the graph
    signature, and after every window, eager or replayed, run() extends its rewbuffer / lenbuffer by the episodes the
    window finished, with no sync beyond its one.

    capture_schedule=True: push and command-curriculum steps are captured too (graphs are cached by the positions of
    the window's disturbance, push and curriculum steps), so after the warm-up every window replays.  For every window
    run() executes, eager or replayed, the env is in its device-schedule mode: the kernels read the command ranges
    from the env's device copy and the curriculum decides on the device (hl_command_curriculum).  run() uploads
    command_ranges when the host values changed since the last rollout and copies the device ranges back with the
    episode tables.  A subclass that overrides update_command_curriculum keeps its curriculum windows eager, on the
    host ranges."""

    def __init__(self, env, body: Callable[[int], None], num_steps: int, storage=None,
                 finish: Optional[Callable[[], None]] = None, max_graphs: int = 8, warmup: int = 1,
                 capture_schedule: bool = False, amp=None, episode_stats=None):
        if not env._kernel_reset_ok():
            raise ValueError("capture_rollout needs the in-kernel reset (a torch reset hook syncs on the host every step)")
        if getattr(env, "gym", None) is not None:
            raise ValueError("capture_rollout needs standalone physics: gym.simulate cannot be captured")
        if num_steps <= 0:
            raise ValueError("num_steps must be positive")
        if episode_stats is not None and episode_stats.num_envs != env.num_envs:
            raise ValueError(f"episode_stats keeps {episode_stats.num_envs} envs, the env has {env.num_envs}")
        self.env, self.body, self.num_steps, self.storage, self.finish = env, body, int(num_steps), storage, finish
        self.max_graphs, self.warmup = max(int(max_graphs), 1), int(warmup)
        self.capture_schedule = bool(capture_schedule)
        self.amp = amp
        self.episode_stats = episode_stats
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
                st.step if st is not None else None, env.resample_interval,
                self.amp.signature() if self.amp is not None else None,
                self.episode_stats.signature() if self.episode_stats is not None else None)

    def _host_state(self):
        env, st = self.env, self.storage
        return dict(counter=env.common_step_counter, step=st.step if st is not None else None, obs=env.obs_buf,
                    priv=env.privileged_obs_buf, extras=dict(env.extras),
                    amp=self.amp.host_state() if self.amp is not None else None)

    def _set_host_state(self, h):
        env, st = self.env, self.storage
        env.common_step_counter = h["counter"]
        if st is not None:
            st.step = h["step"]
        env.obs_buf, env.privileged_obs_buf = h["obs"], h["priv"]
        env.extras.clear()
        env.extras.update(h["extras"])
        if self.amp is not None:
            self.amp.set_host_state(h["amp"])

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
            after["amp_calls"] = after["amp"][3] - before["amp"][3] if self.amp is not None else 0
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
        device_schedule, schedule = self.capture_schedule, None
        if device_schedule:
            key, reason = rollout_window(c, T, **env_schedule(env), in_graph=True)
            cur = key[2]
            if cur and not env._device_curriculum_ok():      # the host decides: this window runs eagerly on the host ranges
                key, reason = None, f"update_command_curriculum is overridden: command-curriculum step at counter {c + 1 + cur[0]}"
                device_schedule = False
            else:
                env._upload_command_ranges()
                schedule = (env.command_ranges["lin_vel_x"][1], cur if "tracking_lin_vel" in env.episode_sums else ())
        else:
            key, reason = rollout_window(c, T, **env_schedule(env))
        if key is not None and self.warmup > 0:
            key, reason = None, "warm-up"
            self.warmup -= 1
        env._device_schedule = device_schedule
        if self.amp is not None:
            self.amp.refresh()
        try:
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
                amp_before = self.amp.host_state() if self.amp is not None else None
                g.replay()
                self._device_counter = c + T
                self._set_host_state(after)
                if self.amp is not None:      # the inserts of the replayed window, counted while it was captured
                    self.amp.set_host_state(amp_before)
                    self.amp.advance(after["amp_calls"])
                    self.amp.calls += after["amp_calls"]
                env.common_step_counter = c + T
                self.stats["replays"] += 1
                self.last_mode, self.last_reason = mode, None
        finally:
            env._device_schedule = False
        if self.episode_stats is not None:
            self.episode_stats._enqueue_copies()     # completed by the sync in episode_infos
        infos = self.tables.episode_infos(env, schedule)
        if self.episode_stats is not None:
            self.episode_stats._extend()
        env.extras["time_outs"] = env.time_out_buf
        if infos:
            env.extras["episode"] = infos[-1]
        return infos
