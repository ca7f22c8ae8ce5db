"""HIMPPO.act's action sampling as one keyed launch (hl_policy_sample).

HIMPPO.act (him_ppo.py:90) builds `Normal(mean, mean*0. + std)` from the actor's mean, samples it, and stores the
sample, its summed log-probability, the mean and the sigma in the transition; add_transitions then copies the four
into the rollout slots.  `keyed_act` does all of that after the actor's mean in one launch with no host sync: the
standard normals come from the library's Philox stream 7, keyed by (seed, step, global env id) like every other
in-kernel draw, so an eager step, a captured step and a replayed step draw the same actions, and two shards draw
what one big env draws.  The actor MLP, the critic and the PPO update stay torch.

Differences from the torch composition:
* the log-probability sums its per-action terms in column order, where torch's `.sum(-1)` has its own reduction order;
  every other output is bit-equal for the same standard normals (see test_gpu_policy_sampling.py);
* sigma is not validated (as with `validate_args=False`): a NaN or non-positive std propagates instead of raising;
* the draw is a function of the step key, not of a generator state: two calls at the same common_step_counter (without
  a step() between them) draw the same standard normals.
"""
import ctypes
from typing import Optional

import torch

from . import _lib as L

MAX_ACT_DIM = 16


def _check(name, t, shapes, device):
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if t.dtype != torch.float32:
        raise ValueError(f"{name}: expected float32, got {t.dtype}")
    if tuple(t.shape) not in shapes:
        raise ValueError(f"{name}: expected shape {' or '.join(map(str, shapes))}, got {tuple(t.shape)}")
    if not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (there is no CPU fallback), got one on {t.device}")
    if t.device != device:
        raise ValueError(f"{name}: expected a tensor on {device}, got one on {t.device}")
    t = t.detach()
    return t if t.is_contiguous() else t.contiguous()


def keyed_act(env, mean: torch.Tensor, std: torch.Tensor, transition=None, storage=None,
              z: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Sample actions ~ Normal(mean, mean*0. + std) from Philox stream 7 and return them.

    env: the FusedLeggedRobot the actions are for.  The draw is keyed by its step key at call time (env._buffers():
    common_step_counter, or the device counter while capture_rollout captures), so call it before the step() /
    step_device() that takes the actions: it then shares the key of that step's action delay (stream 4).
    mean: (N, A) float32, the actor's mean (e.g. actor_critic.act_inference(obs)); std: (A,) or (N, A) float32 (e.g.
    actor_critic.std).  1 <= A <= 16.
    storage: a HIMRolloutStorage with storage.step < T: the outputs are its slots actions[s], actions_log_prob[s], mu[s]
    and sigma[s], so record_env_step / add_transitions copy none of the four.  Without it the outputs are new tensors.
    transition: filled as HIMPPO.act fills it -- actions, actions_log_prob ((N,), as get_actions_log_prob returns),
    action_mean and action_sigma.
    z: parity mode, (N, A) float32 standard normals used in place of the draw.

    Bad tensors raise ValueError; a full storage raises AssertionError("Rollout buffer overflow") as add_transitions
    does.  Nothing here synchronises with the device."""
    if storage is not None and storage.step >= storage.num_transitions_per_env:
        raise AssertionError("Rollout buffer overflow")
    dev = torch.device(env.device)
    if not isinstance(mean, torch.Tensor) or mean.dim() != 2:
        raise ValueError(f"mean: expected an (N, A) tensor, got {getattr(mean, 'shape', type(mean).__name__)}")
    n, a = env.num_envs, int(mean.shape[1])
    if not 1 <= a <= MAX_ACT_DIM:
        raise ValueError(f"mean: the action dimension must lie in [1, {MAX_ACT_DIM}], got {a}")
    mean = _check("mean", mean, [(n, a)], dev)
    std = _check("std", std, [(a,), (n, a)], dev)
    if z is not None:
        z = _check("z", z, [(n, a)], dev)
    if storage is not None:
        s = storage.step
        if tuple(storage.actions.shape[1:]) != (n, a):
            raise ValueError(f"storage: its action slots are {tuple(storage.actions.shape[1:])}, the mean is {(n, a)}")
        actions, log_prob = storage.actions[s], storage.actions_log_prob[s].view(n)
        mu, sigma = storage.mu[s], storage.sigma[s]
    else:
        actions, log_prob = torch.empty(n, a, device=dev), torch.empty(n, device=dev)
        mu, sigma = torch.empty(n, a, device=dev), torch.empty(n, a, device=dev)
    L.check(L.lib.hl_policy_sample(ctypes.byref(env._c), ctypes.byref(env._buffers()), L.ptr(mean), L.ptr(std),
                                   a if std.dim() == 2 else 0, L.ptr(z), a, L.ptr(actions), L.ptr(log_prob), L.ptr(mu),
                                   L.ptr(sigma), n, L.stream()))
    if transition is not None:
        transition.actions, transition.actions_log_prob = actions, log_prob
        transition.action_mean, transition.action_sigma = mu, sigma
    return actions
