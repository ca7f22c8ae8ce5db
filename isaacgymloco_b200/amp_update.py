"""The discriminator minibatches of HybridPPO.update drawn on the device (AMPUpdateSampler).

For every minibatch HybridPPO.update (hybrid_ppo.py:160-281) pulls one item from each of two generators and builds the
discriminator inputs from them:

    policy_state, policy_next_state = next(amp_storage.feed_forward_generator(...))   # ReplayBuffer, np.random.choice
    expert_state, expert_next_state = next(amp_data.feed_forward_generator(...))      # AMPLoader preload, np.random.choice
    policy_d = discriminator(torch.cat([normalize_torch(policy_state), normalize_torch(policy_next_state)], -1))
    expert_d = discriminator(torch.cat([normalize_torch(expert_state), normalize_torch(expert_next_state)], -1))

AMPUpdateSampler.sample() does all of that up to the discriminator in one launch (hl_amp_update_batch) with no host
sync: the rows come from the library's Philox stream 8, keyed by (seed, the sampler's draw counter, row_offset + row),
the gathers and the normalisation are bit-equal to the public composition on the same rows.  The draw counter lives on
the device and the launch advances it, so k eager calls, one captured call replayed k times and any mix of the two draw
the same k minibatches; two samplers with the same seed draw the same sequence.  The losses, the gradient penalty and
the normaliser update stay torch.

Differences from the two host generators: the rows are uniform draws from another generator (statistically, not
bitwise, np.random.choice), and the policy rows come from [0, num_samples) read at launch time -- from the host mirror
replay_buffer.num_samples, or, with ring_cursor, from the device cursor of an AMPRolloutStep.
"""
import ctypes
from collections import namedtuple
from typing import Optional

import torch

from . import _lib as L

AMPUpdateBatch = namedtuple("AMPUpdateBatch", ["policy_state", "policy_next_state", "expert_state", "expert_next_state",
                                               "x_policy", "x_expert"])
AMPUpdateBatchWithIndices = namedtuple("AMPUpdateBatchWithIndices", AMPUpdateBatch._fields + ("indices",))

U64 = 1 << 64


def _device_tensor(name, t, dtype, shape, device):
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if t.dtype != dtype:
        raise ValueError(f"{name}: expected {dtype}, got {t.dtype}")
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name}: expected shape {tuple(shape)}, got {tuple(t.shape)}")
    if not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (there is no CPU fallback), got one on {t.device}")
    if device is not None and t.device != device:
        raise ValueError(f"{name}: expected a tensor on {device}, got one on {t.device}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous tensor")
    return t


class AMPUpdateSampler:
    """Draws the policy and expert minibatches of the AMP update and their normalised discriminator inputs.

    amp_loader: an AMPLoader with preload_transitions=True (preloaded_s / preloaded_s_next, (n, 49)).
    replay_buffer: the ReplayBuffer of policy transitions (states / next_states, (rows, 30)).
    normalizer: the Normalizer (dim 30) or None.  Its mean / var are read at every call: Normalizer.update rebinds them.
    mini_batch_size: rows per minibatch (N*T / num_mini_batches in HybridPPO.update).
    seed: the Philox key (0 <= seed < 2**64).
    row_offset: global id of row 0; with envs sharded, rank * mini_batch_size, so ranks draw independent rows.
    ring_cursor: AMPRolloutStep._cursor, so the row count is read on the device at launch time (a graph captured after a
    replayed rollout then sees the current count); None: replay_buffer.num_samples on the host at call time."""

    def __init__(self, amp_loader, replay_buffer, normalizer, mini_batch_size: int, seed: int, row_offset: int = 0,
                 ring_cursor: Optional[torch.Tensor] = None):
        if not getattr(amp_loader, "preload_transitions", False):
            raise ValueError("AMPUpdateSampler: the AMP loader has no preloaded transitions (preload_transitions=False); "
                             "the lerp-frame branch of AMPLoader.feed_forward_generator is not drawn on the device")
        mb = int(mini_batch_size)
        if mb < 1:
            raise ValueError(f"AMPUpdateSampler: mini_batch_size must be >= 1, got {mini_batch_size}")
        if not 0 <= int(seed) < U64:
            raise ValueError(f"AMPUpdateSampler: seed must lie in [0, 2**64), got {seed}")
        if int(row_offset) < 0:
            raise ValueError(f"AMPUpdateSampler: row_offset must be >= 0, got {row_offset}")
        rb = replay_buffer
        for name, t in (("replay_buffer.states", rb.states), ("replay_buffer.next_states", rb.next_states)):
            if t.dim() != 2 or int(t.shape[1]) != 30:
                raise ValueError(f"AMPUpdateSampler: {name} must be (rows, 30), got {tuple(t.shape)}")
        for name, t in (("amp_loader.preloaded_s", amp_loader.preloaded_s),
                        ("amp_loader.preloaded_s_next", amp_loader.preloaded_s_next)):
            if t.dim() != 2 or int(t.shape[1]) != 49:
                raise ValueError(f"AMPUpdateSampler: {name} must be (n, 49), got {tuple(t.shape)}")
        if normalizer is not None and int(normalizer.dim) != 30:
            raise ValueError(f"AMPUpdateSampler: the normaliser must have 30 columns, has {normalizer.dim}")
        rows = int(rb.states.shape[0])
        _device_tensor("replay_buffer.states", rb.states, torch.float32, None, None)
        dev = rb.states.device
        _device_tensor("replay_buffer.next_states", rb.next_states, torch.float32, (rows, 30), dev)
        n_pre = int(amp_loader.preloaded_s.shape[0])
        _device_tensor("amp_loader.preloaded_s", amp_loader.preloaded_s, torch.float32, (n_pre, 49), dev)
        _device_tensor("amp_loader.preloaded_s_next", amp_loader.preloaded_s_next, torch.float32, (n_pre, 49), dev)
        if n_pre < 1 or rows < 1:
            raise ValueError("AMPUpdateSampler: the preload tables and the replay ring must have rows")
        if ring_cursor is not None:
            _device_tensor("ring_cursor", ring_cursor, torch.int64, (3,), dev)
        if normalizer is not None:
            self._norm_stats(normalizer, dev)
        self.amp_loader, self.replay_buffer, self.normalizer = amp_loader, rb, normalizer
        self.mini_batch_size, self.seed, self.row_offset = mb, int(seed), int(row_offset)
        self.ring_cursor = ring_cursor
        self.device = dev
        self.draw_counter = torch.zeros(2, dtype=torch.long, device=dev)      # {draws, the launch's CTA ticket}

    @staticmethod
    def _norm_stats(norm, dev):
        mean = _device_tensor("normalizer.mean", norm.mean, torch.float64, (30,), dev)
        var = _device_tensor("normalizer.var", norm.var, torch.float64, (30,), dev)
        return mean, var

    def sample(self, indices: Optional[torch.Tensor] = None, return_indices: bool = False):
        """One minibatch: (policy_state, policy_next_state, expert_state, expert_next_state, x_policy, x_expert
        [, indices]).  The states are (mb, 30) and the inputs (mb, 60) fresh tensors (inside a CUDA graph capture they
        come from the graph's pool); indices (mb, 2) int64 [policy row, expert row].
        indices: parity mode, (mb, 2) int64 rows used in place of the draw (the draw counter still advances).
        Nothing here synchronises with the device."""
        rb, norm, mb, dev = self.replay_buffer, self.normalizer, self.mini_batch_size, self.device
        if self.ring_cursor is None:
            n_s = int(rb.num_samples)
            if n_s < 1:
                raise ValueError("AMPUpdateSampler.sample: the replay buffer holds no samples (num_samples = 0)")
        else:
            n_s = 0
        if indices is not None:
            indices = _device_tensor("indices", indices, torch.int64, (mb, 2), dev)
        mean = var = None
        if norm is not None:
            mean, var = self._norm_stats(norm, dev)
        buf = torch.empty(240 * mb, device=dev)     # one allocation: four (mb, 30) states, two (mb, 60) inputs
        ps, psn, es, esn = (buf[k * 30 * mb:(k + 1) * 30 * mb].view(mb, 30) for k in range(4))
        xp, xe = buf[120 * mb:180 * mb].view(mb, 60), buf[180 * mb:].view(mb, 60)
        idx_out = torch.empty(mb, 2, dtype=torch.long, device=dev) if return_indices else None
        a = L.HlAmpUpdateBatch()
        a.struct_bytes = ctypes.sizeof(L.HlAmpUpdateBatch)
        a.clip = float(norm.clip_obs) if norm is not None else 0.0
        a.ring_states, a.ring_next, a.ring_rows = L.ptr(rb.states), L.ptr(rb.next_states), int(rb.states.shape[0])
        a.ring_cursor, a.num_samples = L.ptr(self.ring_cursor), n_s
        loader = self.amp_loader
        a.preloaded_s, a.preloaded_s_next = L.ptr(loader.preloaded_s), L.ptr(loader.preloaded_s_next)
        a.n_preloaded = int(loader.preloaded_s.shape[0])
        a.norm_mean, a.norm_var = L.ptr(mean), L.ptr(var)
        a.eps = float(norm.epsilon) if norm is not None else 0.0
        a.seed, a.draw_counter, a.row_offset = self.seed, L.ptr(self.draw_counter), self.row_offset
        a.idx_in, a.idx_out = L.ptr(indices), L.ptr(idx_out)
        a.policy_s, a.policy_sn, a.expert_s, a.expert_sn = L.ptr(ps), L.ptr(psn), L.ptr(es), L.ptr(esn)
        a.x_policy, a.x_expert, a.mb = L.ptr(xp), L.ptr(xe), mb
        L.check(L.lib.hl_amp_update_batch(ctypes.byref(a), L.stream()))
        if return_indices:
            return AMPUpdateBatchWithIndices(ps, psn, es, esn, xp, xe, idx_out)
        return AMPUpdateBatch(ps, psn, es, esn, xp, xe)

    def generator(self, num_mini_batch: int):
        """Yields sample() num_mini_batch times, lazily: zips with storage.mini_batch_generator as the two reference
        generators do."""
        for _ in range(int(num_mini_batch)):
            yield self.sample()
