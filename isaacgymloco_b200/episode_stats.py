"""The runners' episode statistics (`Mean reward`, `Mean episode length`) kept on the device (EpisodeStats).

HIMOnPolicyRunner.learn, and the hybrid runner after its AMP reward, keep these every env-step:

    cur_reward_sum += rewards
    cur_episode_length += 1
    new_ids = (dones > 0).nonzero(as_tuple=False)
    rewbuffer.extend(cur_reward_sum[new_ids][:, 0].cpu().numpy().tolist())
    lenbuffer.extend(cur_episode_length[new_ids][:, 0].cpu().numpy().tolist())
    cur_reward_sum[new_ids] = 0
    cur_episode_length[new_ids] = 0

The two `.cpu()` calls are host syncs, which a captured rollout cannot contain.  EpisodeStats.record() is the block as
one hl_episode_stats launch: the finished episodes go to a device ring of `maxlen` entries per buffer behind a device
cursor, and collect() -- or RolloutGraph.run(), with the copies it makes anyway -- brings them to the host deques
rewbuffer / lenbuffer in one sync.  A ring of `maxlen` entries loses nothing: deque(maxlen=maxlen) keeps only the last
`maxlen` entries too.  cur_episode_length is the runner's own float counter, not the env's episode_length_buf.
"""
from collections import deque
from typing import List, Optional, Sequence

import torch

from . import _lib as L


def ring_entries(seen: int, total: int, ring: Sequence[float]) -> List[float]:
    """The entries a deque(maxlen=len(ring)) takes at a collection.  `seen` and `total` count the entries written up to
    the previous and up to this collection; entry i is ring[i % len(ring)].  Returns the last min(total - seen,
    len(ring)) of the new entries, oldest first: older ones were overwritten in the ring, and the deque would have
    dropped them."""
    if not 0 <= seen <= total:
        raise ValueError(f"ring_entries: need 0 <= seen <= total, got seen={seen}, total={total}")
    size = len(ring)
    return [ring[i % size] for i in range(max(seen, total - size), total)]


def check_step_args(num_envs: int, device: torch.device, rewards, dones, ids, n_ids=None) -> None:
    """What EpisodeStats.record() accepts: (N,) fp32 rewards and bool / uint8 dones, int64 ids of the done envs in
    ascending order, all contiguous on `device`; n_ids=None means ids holds exactly the step's ids, otherwise ids is a
    buffer of capacity N and n_ids the (1,) int32 device count (step_device()'s form)."""
    named = dict(rewards=rewards, dones=dones, ids=ids)
    if n_ids is not None:
        named["n_ids"] = n_ids
    for name, t in named.items():
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"EpisodeStats.record: {name} must be a tensor")
    if rewards.dtype != torch.float32 or rewards.numel() != num_envs:
        raise ValueError(f"EpisodeStats.record: rewards must be {num_envs} float32 values, got {rewards.dtype} "
                         f"{tuple(rewards.shape)}")
    if dones.dtype not in (torch.bool, torch.uint8) or dones.numel() != num_envs:
        raise ValueError(f"EpisodeStats.record: dones must be {num_envs} bool / uint8 values, got {dones.dtype} "
                         f"{tuple(dones.shape)}")
    if ids.dtype != torch.int64 or ids.numel() > num_envs:
        raise ValueError(f"EpisodeStats.record: ids must be at most {num_envs} int64 env ids, got {ids.dtype} "
                         f"{tuple(ids.shape)}")
    if n_ids is not None and (n_ids.dtype != torch.int32 or n_ids.numel() != 1):
        raise ValueError(f"EpisodeStats.record: n_ids must be one int32 count, got {n_ids.dtype} {tuple(n_ids.shape)}")
    for name, t in named.items():
        if not t.is_cuda:
            raise RuntimeError(f"EpisodeStats.record: {name} is on {t.device}; the statistics need CUDA tensors "
                               "(there is no CPU fallback)")
        if t.device != device:
            raise ValueError(f"EpisodeStats.record: {name} is on {t.device}, the statistics on {device}")
        if not t.is_contiguous():
            raise ValueError(f"EpisodeStats.record: {name} must be contiguous")


class EpisodeStats:
    """The runner's rewbuffer / lenbuffer and running sums, with the per-step work on the device.

    cur_reward_sum, cur_episode_length: (N,) fp32 device tensors, as the runner names them.  rewbuffer, lenbuffer: host
    deque(maxlen=maxlen), filled by collect() or RolloutGraph.run(), so log() reads them unchanged.  record() never
    syncs or allocates and changes no host state, so a RolloutGraph can capture it: capture_rollout(...,
    episode_stats=stats)."""

    def __init__(self, num_envs: int, device, maxlen: int = 100):
        if int(num_envs) < 1:
            raise ValueError(f"EpisodeStats: num_envs must be at least 1, got {num_envs}")
        if int(maxlen) < 1:
            raise ValueError(f"EpisodeStats: maxlen must be at least 1, got {maxlen}")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise ValueError(f"EpisodeStats: the statistics live on a CUDA device, not {dev} (there is no CPU fallback)")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        n, m = int(num_envs), int(maxlen)
        self.num_envs, self.device, self.maxlen = n, dev, m
        self.cur_reward_sum = torch.zeros(n, dtype=torch.float, device=dev)
        self.cur_episode_length = torch.zeros(n, dtype=torch.float, device=dev)
        self.rewbuffer, self.lenbuffer = deque(maxlen=m), deque(maxlen=m)
        self._ring = torch.zeros(2, m, device=dev)                        # rewards, lengths; entry i in column i % m
        self._ring_reward, self._ring_length = self._ring[0], self._ring[1]
        self._cursor = torch.zeros(2, dtype=torch.long, device=dev)       # entries written so far, the launch's CTA ticket
        self._count = torch.zeros(1, dtype=torch.int32, device=dev)       # the count when record() gets exact ids
        self._host_ring = torch.zeros(2, m, pin_memory=True)
        self._host_total = torch.zeros(1, dtype=torch.long, pin_memory=True)
        self._seen = 0                                                    # the device total at the last collection

    def record(self, rewards, dones, ids, n_ids: Optional[torch.Tensor] = None):
        """The runner's per-step block, after env.step() (the hybrid runner: with the AMP reward).  With n_ids, ids and
        n_ids are step_device()'s capacity-N buffer and (1,) int32 device count; without it, ids are exactly the done
        envs, as step() returns them.  dones may be the env's bool reset_buf."""
        check_step_args(self.num_envs, self.device, rewards, dones, ids, n_ids)
        if n_ids is None:
            self._count.fill_(ids.numel())
            n_ids = self._count
        # an empty id tensor may have no storage at all; the kernel reads no id when the count is 0
        ids_ptr = ids.data_ptr() or self._count.data_ptr()
        L.check(L.lib.hl_episode_stats(L.ptr(rewards), L.ptr(dones), ids_ptr, L.ptr(n_ids), L.ptr(self.cur_reward_sum),
                                       L.ptr(self.cur_episode_length), L.ptr(self._ring_reward), L.ptr(self._ring_length),
                                       self.maxlen, L.ptr(self._cursor), self.num_envs, L.stream()))

    def collect(self):
        """Extend rewbuffer / lenbuffer by the episodes recorded since the last collection: one copy of the ring and the
        total to pinned memory and one sync.  The eager loop calls it once per iteration, before log()."""
        self._enqueue_copies()
        torch.cuda.current_stream(self.device).synchronize()
        self._extend()

    def _enqueue_copies(self):
        self._host_ring.copy_(self._ring, non_blocking=True)
        self._host_total.copy_(self._cursor[:1], non_blocking=True)

    def _extend(self):
        """After the copies of _enqueue_copies() have completed."""
        total = int(self._host_total[0])
        rewards, lengths = self._host_ring.tolist()
        self.rewbuffer.extend(ring_entries(self._seen, total, rewards))
        self.lenbuffer.extend(ring_entries(self._seen, total, lengths))
        self._seen = total

    def signature(self):
        """What a captured record() holds by address or value (RolloutGraph recaptures when it changes)."""
        return (self.cur_reward_sum.data_ptr(), self.cur_episode_length.data_ptr(), self._ring.data_ptr(),
                self._cursor.data_ptr(), self._count.data_ptr(), self.maxlen)
