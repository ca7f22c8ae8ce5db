"""Catch NaN and Inf in a rollout on the device (FiniteGuard, one hl_finite_scan launch per env-step).

The reference fails loudly when training diverges: HIMPPO.act's `Normal(mean, mean*0. + std)` validates its
arguments, and torch.clip passes NaN through, so a diverged policy or an exploded physics state shows up as NaN
everywhere.  Here nothing would surface it: keyed_act does not validate sigma, a replayed rollout runs no host code
between its one sync, and the kernels' clamps (fminf(fmaxf(x, lo), hi)) turn a NaN into the lower bound -- a NaN
action becomes a torque of -torque_limits, a NaN observation entry -clip_observations, a NaN reward 0 under
only_positive_rewards.  FiniteGuard scans the sources those clamps hide, on the device, and reports at the one sync
the loop already has:

* record(k), in `body(k)` after record_env_step: one launch that counts the flagged elements of every field, finds
  the first one and writes row k of a (num_steps, F, 3) device table.  No sync, no allocation, capturable.
* check(), once per iteration of an eager loop, or capture_rollout(..., finite_guard=guard), whose run() brings the
  table back with the episode tables: NonFiniteError when any row has a count.

Fields (resolved at record(k), so a captured step k holds the pointers of its own slot): the env's root_states,
dof_state and contact_forces, and rew_buf when there is no storage; with a HIMRolloutStorage, slot k's actions, mu,
sigma (flagged unless 0 < sigma < inf, Normal's scale constraint), values, actions_log_prob and rewards.  Observations
are not scanned by default: every entry passes the clip_observations clamp, which turns a NaN into -clip_observations,
so a NaN never shows there.
"""
import ctypes
import struct
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib as L

ENV_FIELDS = ("root_states", "dof_state", "contact_forces", "rew_buf")
STORAGE_FIELDS = ("actions", "mu", "sigma", "values", "actions_log_prob", "rewards")
POSITIVE_FIELDS = ("sigma",)


def default_fields(has_storage: bool) -> Tuple[str, ...]:
    env = ("root_states", "dof_state", "contact_forces")
    return env + STORAGE_FIELDS if has_storage else env + ("rew_buf",)


def bits_to_float(bits: int) -> float:
    """The fp32 value of raw bits (any int whose low 32 bits hold them); NaN payloads and signs survive the widening."""
    return struct.unpack("<f", struct.pack("<I", int(bits) & 0xFFFFFFFF))[0]


def table_events(table, fields: Sequence[str], widths: Sequence[int], env_id_offset: int = 0,
                 counters: Optional[Sequence[Optional[int]]] = None) -> List[Dict]:
    """The events of a (T, F, 3) table (nested lists or a tensor): one per step k and field with a count, in step then
    field order.  env = env_id_offset + index // width, column = index % width; common_step_counter = counters[k]."""
    rows = table.tolist() if isinstance(table, torch.Tensor) else table
    events = []
    for k, row in enumerate(rows):
        for f, (count, index, bits) in enumerate(row):
            if count <= 0:
                continue
            events.append(dict(k=k, common_step_counter=None if counters is None else counters[k], field=fields[f],
                               env=int(env_id_offset) + index // widths[f], column=index % widths[f],
                               value=bits_to_float(bits), count=count))
    return events


def describe(events: Sequence[Dict]) -> str:
    """The message of NonFiniteError: the earliest step and every field flagged at it."""
    if not events:
        return "no non-finite values"
    k = min(ev["k"] for ev in events)
    first = [ev for ev in events if ev["k"] == k]
    c = first[0]["common_step_counter"]
    at = f"rollout step {k}" + (f" (common_step_counter {c})" if c is not None else "")
    parts = [f"{ev['field']}: {ev['count']} element(s), first env {ev['env']} column {ev['column']} = {ev['value']}"
             for ev in first]
    later = len({ev["k"] for ev in events}) - 1
    tail = f"; {later} later step(s) flagged too" if later else ""
    return f"non-finite values at {at}: " + "; ".join(parts) + tail


class NonFiniteError(FloatingPointError):
    """A guarded rollout produced NaN / Inf (or a scale that is not positive).  `.events`: one dict per flagged step
    and field -- k, common_step_counter, field, env (global id), column, value (the first flagged element) and count."""

    def __init__(self, events: Sequence[Dict]):
        self.events = list(events)
        super().__init__(describe(self.events))


def rows_view(t: torch.Tensor, n_rows: int, name: str) -> Tuple[int, int]:
    """(row_stride, width) of an fp32 CUDA tensor whose dim 0 has n_rows rows and whose rows are contiguous."""
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if t.dtype != torch.float32:
        raise ValueError(f"{name}: expected float32, got {t.dtype}")
    if not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (there is no CPU fallback), got one on {t.device}")
    if t.dim() < 1 or t.shape[0] != n_rows:
        raise ValueError(f"{name}: expected {n_rows} rows, got shape {tuple(t.shape)}")
    width = int(t[0].numel()) if t.dim() > 1 else 1
    if width < 1 or (t.dim() > 1 and not t[0].is_contiguous()):
        raise ValueError(f"{name}: each row must be a non-empty contiguous block, got strides {t.stride()}")
    stride = int(t.stride(0))
    if stride < width:
        raise ValueError(f"{name}: rows overlap (row stride {stride} < width {width})")
    return stride, width


def fields_struct(sources: Sequence[Tuple[torch.Tensor, int]], n_rows: int, names: Sequence[str]) -> "L.HlFiniteFields":
    if not 1 <= len(sources) <= L.MAX_FINITE_FIELDS:
        raise ValueError(f"between 1 and {L.MAX_FINITE_FIELDS} fields, got {len(sources)}")
    s = L.HlFiniteFields()
    s.struct_bytes = ctypes.sizeof(L.HlFiniteFields)
    s.n_fields = len(sources)
    for f, ((t, kind), name) in enumerate(zip(sources, names)):
        stride, width = rows_view(t, n_rows, name)
        s.field[f].src, s.field[f].row_stride, s.field[f].width, s.field[f].kind = t.data_ptr(), stride, width, int(kind)
    return s


def new_workspace(device) -> torch.Tensor:
    """hl_finite_scan's workspace, armed: counts 0, first indices all-ones, ticket 0."""
    ws = torch.zeros(L.FINITE_WORKSPACE_WORDS, dtype=torch.int64, device=device)
    ws[L.MAX_FINITE_FIELDS:2 * L.MAX_FINITE_FIELDS] = -1
    return ws


def finite_scan(sources: Sequence[Tuple[torch.Tensor, int]], record: torch.Tensor, workspace: torch.Tensor,
                names: Optional[Sequence[str]] = None) -> None:
    """One hl_finite_scan launch: `sources` = (tensor, L.FINITE or L.FINITE_POSITIVE) pairs with equal row counts;
    record: a contiguous (F, 3) int64 device tensor; workspace: new_workspace()'s, re-armed by every launch."""
    names = names or [f"field {f}" for f in range(len(sources))]
    t0 = sources[0][0] if sources else None
    n = int(t0.shape[0]) if isinstance(t0, torch.Tensor) and t0.dim() else 0
    if n < 1:
        raise ValueError("finite_scan: the first field has no rows")
    s = fields_struct(sources, n, names)
    if record.dtype != torch.int64 or tuple(record.shape) != (len(sources), 3) or not record.is_contiguous():
        raise ValueError(f"record: expected a contiguous ({len(sources)}, 3) int64 tensor, got {record.dtype} "
                         f"{tuple(record.shape)}")
    if workspace.dtype != torch.int64 or workspace.numel() != L.FINITE_WORKSPACE_WORDS:
        raise ValueError(f"workspace: expected {L.FINITE_WORKSPACE_WORDS} int64 words")
    L.check(L.lib.hl_finite_scan(ctypes.byref(s), n, L.ptr(record), L.ptr(workspace), L.stream()))


class FiniteGuard:
    """Per-step NaN / Inf detection for a rollout of `num_steps` env-steps of `env` (a FusedLeggedRobot).

    storage: the HIMRolloutStorage the loop records into (its slots join the default fields); fields: a subset of
    ENV_FIELDS + STORAGE_FIELDS, for cost control.  table: the (num_steps, F, 3) int64 device table, row k field f =
    {count, first flagged index e*width + c or -1, its fp32 bits}; record(k) writes row k."""

    def __init__(self, env, num_steps: int, storage=None, fields: Optional[Sequence[str]] = None):
        if int(num_steps) < 1:
            raise ValueError(f"FiniteGuard: num_steps must be at least 1, got {num_steps}")
        names = default_fields(storage is not None) if fields is None else tuple(fields)
        if not names:
            raise ValueError("FiniteGuard: fields must name at least one field")
        for name in names:
            if name not in ENV_FIELDS + STORAGE_FIELDS:
                raise ValueError(f"FiniteGuard: unknown field {name!r} (known: {', '.join(ENV_FIELDS + STORAGE_FIELDS)})")
            if name in STORAGE_FIELDS and storage is None:
                raise ValueError(f"FiniteGuard: field {name!r} is a storage slot, and no storage was given")
        if len(set(names)) != len(names):
            raise ValueError(f"FiniteGuard: fields repeat a name: {names}")
        if len(names) > L.MAX_FINITE_FIELDS:
            raise ValueError(f"FiniteGuard: at most {L.MAX_FINITE_FIELDS} fields, got {len(names)}")
        if storage is not None:
            if storage.num_envs != env.num_envs:
                raise ValueError(f"FiniteGuard: the storage keeps {storage.num_envs} envs, the env has {env.num_envs}")
            if storage.num_transitions_per_env < int(num_steps):
                raise ValueError(f"FiniteGuard: the storage has {storage.num_transitions_per_env} slots, fewer than "
                                 f"num_steps = {num_steps}")
        dev = torch.device(env.device)
        if dev.type != "cuda":
            raise ValueError(f"FiniteGuard: the env is on {dev}; the guard needs CUDA (there is no CPU fallback)")
        self.env, self.storage, self.fields, self.num_steps = env, storage, names, int(num_steps)
        self.kinds = tuple(L.FINITE_POSITIVE if name in POSITIVE_FIELDS else L.FINITE for name in names)
        self.widths = tuple(rows_view(t, env.num_envs, name)[1] for t, name in zip(self._sources(0), names))
        self.table = torch.zeros(self.num_steps, len(names), 3, dtype=torch.int64, device=dev)
        self._workspace = new_workspace(dev)
        self._host = torch.zeros(self.table.shape, dtype=torch.int64, pin_memory=True)
        self._counters = [None] * self.num_steps

    def _sources(self, k: int) -> List[torch.Tensor]:
        env, st = self.env, self.storage
        # the env's tensors in rows of one env (dof_state is Isaac Gym's (N*12, 2)); a view, never a copy
        return [getattr(st, name)[k] if name in STORAGE_FIELDS else getattr(env, name).view(env.num_envs, -1)
                for name in self.fields]

    def record(self, k: int) -> None:
        """Scan step k's fields into row k: call in body(k) after record_env_step.  One launch; no sync, no
        allocation.  The host counter it sees is the common_step_counter check() reports for the step."""
        k = int(k)
        if not 0 <= k < self.num_steps:
            raise ValueError(f"FiniteGuard.record: step {k} outside [0, {self.num_steps})")
        finite_scan(list(zip(self._sources(k), self.kinds)), self.table[k], self._workspace, self.fields)
        self._counters[k] = self.env.common_step_counter

    def check(self) -> None:
        """For the eager loop, once per iteration: one copy of the table to pinned memory and one sync; the table is
        zeroed for the next iteration.  Raises NonFiniteError when anything was flagged."""
        self._enqueue_copy()
        self.table.zero_()
        torch.cuda.current_stream(self.table.device).synchronize()
        events = self._events(self._counters)
        self._counters = [None] * self.num_steps
        if events:
            raise NonFiniteError(events)

    def _enqueue_copy(self):
        self._host.copy_(self.table, non_blocking=True)

    def _events(self, counters) -> List[Dict]:
        """After _enqueue_copy() has completed."""
        offset = int(getattr(getattr(self.env, "cfg_hot", None), "env_id_offset", 0))
        return table_events(self._host.tolist(), self.fields, self.widths, offset, counters)

    def signature(self):
        """What a captured record() holds by address (RolloutGraph recaptures when it changes)."""
        bases = tuple(getattr(self.storage if name in STORAGE_FIELDS else self.env, name).data_ptr()
                      for name in self.fields)
        return (self.table.data_ptr(), self._workspace.data_ptr(), self.fields, bases)
