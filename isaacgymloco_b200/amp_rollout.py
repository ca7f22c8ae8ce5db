"""The AMP part of a HybridPolicyRunner env-step as capturable device work (AMPRolloutStep).

Each AMP env-step of the reference runner (hybrid_runner.py:184-195, hybrid_ppo.py:144) is

    next_amp_obs = env.get_amp_observations()
    next_amp_obs_with_term = next_amp_obs.clone(); next_amp_obs_with_term[reset_env_ids] = terminal_amp_states
    rewards = disc.predict_amp_reward(amp_obs, next_amp_obs_with_term, rewards, normalizer)[0]
    amp_storage.insert(amp_obs, next_amp_obs_with_term)          # inside alg.process_env_step
    amp_obs = next_amp_obs.clone()

AMPRolloutStep.step() runs it as hl_amp_transition (everything but the MLP, one launch), the discriminator MLP (cuBLAS)
and hl_amp_reward, with no host sync and no allocation, so a RolloutGraph can capture it
(capture_rollout(..., amp=step)).  What a graph cannot take by value lives on the device: the replay-ring cursor
(step, num_samples) and a pointer-stable float64 snapshot of the normaliser's mean / var (Normalizer rebinds its
tensors on every update).  refresh() brings both up to date from the host objects; RolloutGraph.run() calls it at the
start of every rollout.
"""
from typing import Tuple

import torch

from . import _lib as L


def advance_cursor(step: int, num_samples: int, size: int, n: int, inserts: int) -> Tuple[int, int]:
    """(step, num_samples) of a ReplayBuffer of `size` rows after `inserts` inserts of `n` rows each (n <= size), as
    ReplayBuffer.insert's bookkeeping leaves them: num_samples = min(size, max(step + n, num_samples)) and
    step = (step + n) % size per insert.  num_samples grows with the rows written until the ring has wrapped once and is
    `size` from then on, so the loop folds to one expression."""
    if inserts <= 0:
        return step, num_samples
    end = step + n * inserts
    return end % size, min(size, max(end, num_samples))


class AMPRolloutStep:
    """The runner's AMP state and per-step work on device buffers of fixed address.

    amp_obs (N, 30): the carried AMP observation (begin() fills it, step() advances it); x (N, 60): the discriminator
    input of the last step; reward (N,): the AMP reward step() returns.  The host mirror replay_buffer.step /
    num_samples always equals what the ring holds: step() advances it as it goes, and after a replayed window
    RolloutGraph.run() advances it by the inserts the window made."""

    def __init__(self, env, discriminator, normalizer, replay_buffer):
        n, dev = int(env.num_envs), env.device
        if n > replay_buffer.buffer_size:
            raise ValueError(f"AMPRolloutStep: {n} envs do not fit a {replay_buffer.buffer_size}-row replay buffer "
                             "(one step inserts one row per env)")
        if int(replay_buffer.states.shape[1]) != 30:
            raise ValueError("AMPRolloutStep: the replay buffer must hold 30-column AMP observations")
        if discriminator.input_dim != 60:
            raise ValueError(f"AMPRolloutStep: discriminator input_dim must be 60, is {discriminator.input_dim}")
        if normalizer is not None and int(normalizer.dim) != 30:
            raise ValueError("AMPRolloutStep: the normaliser must have 30 columns")
        self.env, self.discriminator, self.normalizer, self.replay_buffer = env, discriminator, normalizer, replay_buffer
        self.num_envs = n
        self.amp_obs = torch.zeros(n, 30, device=dev)
        self.x = torch.zeros(n, 60, device=dev)
        self.reward = torch.zeros(n, device=dev)
        self._cursor = torch.zeros(3, dtype=torch.long, device=dev)     # step, num_samples, the launch's CTA ticket
        self._cursor_mirror = None                                       # (step, num_samples) the device holds
        self._stats = torch.zeros(2, 30, dtype=torch.float64, device=dev) if normalizer is not None else None
        self.calls = 0                                                   # step() calls so far (host side)

    def begin(self):
        """The runner's `amp_obs = env.get_amp_observations()` before its first step."""
        L.check(L.lib.hl_amp_observations(L.ptr(self.env.dof_state), L.ptr(self.env.base_lin_vel),
                                          L.ptr(self.env.base_ang_vel), L.ptr(self.amp_obs), self.num_envs, L.stream()))
        return self.amp_obs

    def refresh(self):
        """Copy the normaliser's mean / var into the snapshot, and upload the cursor when the host values differ from
        what the device holds (an eager ReplayBuffer.insert, clear, or the first use).  No recapture follows either."""
        if self._stats is not None:
            self._stats[0].copy_(self.normalizer.mean)
            self._stats[1].copy_(self.normalizer.var)
        rb = self.replay_buffer
        host = (int(rb.step), int(rb.num_samples))
        if host != self._cursor_mirror:
            if not (0 <= host[0] < rb.buffer_size and 0 <= host[1] <= rb.buffer_size):
                raise ValueError(f"AMPRolloutStep: replay buffer cursor {host} is outside its {rb.buffer_size} rows")
            self._cursor.copy_(torch.tensor([host[0], host[1], 0], dtype=torch.long))
            self._cursor_mirror = host

    def step(self, task_rewards, reset_ids, n_reset, terminal_amp):
        """One AMP env-step after env.step_device(): reset_ids / terminal_amp with capacity N and the device count
        n_reset, as step_device returns them.  Returns the AMP reward (predict_amp_reward(...)[0]) in `reward`."""
        env, disc, norm, rb = self.env, self.discriminator, self.normalizer, self.replay_buffer
        if self._cursor_mirror is None:
            self.refresh()
        L.check(L.lib.hl_amp_transition(
            L.ptr(env.dof_state), L.ptr(env.base_lin_vel), L.ptr(env.base_ang_vel), L.ptr(env.reset_buf), L.ptr(reset_ids),
            L.ptr(n_reset), L.ptr(terminal_amp), L.ptr(self._stats), float(norm.epsilon) if norm is not None else 0.0,
            float(norm.clip_obs) if norm is not None else 0.0, L.ptr(self.amp_obs), L.ptr(self.x), L.ptr(rb.states),
            L.ptr(rb.next_states), rb.buffer_size, L.ptr(self._cursor), self.num_envs, L.stream()))
        with torch.no_grad():
            d = disc.amp_linear(disc.trunk(self.x))
        L.check(L.lib.hl_amp_reward(L.ptr(d), L.ptr(task_rewards), float(disc.amp_reward_coef), float(disc.task_reward_lerp),
                                    L.ptr(self.reward), self.num_envs, L.stream()))
        self.advance(1)
        self.calls += 1
        return self.reward

    def advance(self, inserts: int):
        """Move the host mirror (and what the device is known to hold) on by `inserts` N-row inserts."""
        rb = self.replay_buffer
        rb.step, rb.num_samples = advance_cursor(rb.step, rb.num_samples, rb.buffer_size, self.num_envs, inserts)
        self._cursor_mirror = (rb.step, rb.num_samples)

    # ------------------------------------------------------------------ RolloutGraph
    def signature(self):
        """What a captured step copies by value or by address besides its own buffers' contents: the discriminator's
        parameter pointers, the ring tensors, the buffers of this object and the launch constants."""
        disc, norm, rb = self.discriminator, self.normalizer, self.replay_buffer
        params = tuple(p.data_ptr() for m in (disc.trunk, disc.amp_linear) for p in m.parameters())
        consts = (float(disc.amp_reward_coef), float(disc.task_reward_lerp),
                  None if norm is None else (float(norm.epsilon), float(norm.clip_obs)))
        bufs = (self.amp_obs.data_ptr(), self.x.data_ptr(), self.reward.data_ptr(), self._cursor.data_ptr(),
                None if self._stats is None else self._stats.data_ptr())
        return params, rb.states.data_ptr(), rb.next_states.data_ptr(), rb.buffer_size, bufs, consts

    def host_state(self):
        rb = self.replay_buffer
        return rb.step, rb.num_samples, self._cursor_mirror, self.calls

    def set_host_state(self, s):
        rb = self.replay_buffer
        rb.step, rb.num_samples, self._cursor_mirror, self.calls = s
