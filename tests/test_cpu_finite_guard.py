"""CPU (-m "not gpu"): the host side of the non-finite guard (hl_finite_scan, FiniteGuard) without a GPU.

* hl_finite_scan returns an error, before any launch, for a bad struct size, NULL struct / record / workspace /
  field, a field count outside [1, 16], n_rows < 1, width < 1, row_stride < width, an unknown kind and a field that is
  not 4-byte aligned;
* FiniteGuard raises ValueError for num_steps < 1, unknown, repeated or storage-only field names without a storage,
  more than 16 fields, a storage of another env count or with too few slots, and an env that is not on CUDA;
* table_events() builds the events of a synthetic table (NaN payloads of both signs, infinities, negative and zero
  scales, several fields and steps, a shard offset) as a brute-force walk does, and NonFiniteError names the earliest
  step and every field flagged at it.
"""
import ctypes
import math
import random
import struct
from types import SimpleNamespace as NS

import numpy as np
import pytest
import torch


def _args(n_fields=3):
    from isaacgymloco_b200 import _lib as L
    f = L.HlFiniteFields()
    f.struct_bytes = ctypes.sizeof(L.HlFiniteFields)
    f.n_fields = n_fields
    for k in range(L.MAX_FINITE_FIELDS):
        # fake device addresses: every case below is refused on the host, before a launch
        f.field[k].src, f.field[k].row_stride, f.field[k].width, f.field[k].kind = 4096 * (k + 1), 13, 13, L.FINITE
    return f


def _call(f, n_rows=64, record=8192 * 64, workspace=8192 * 65):
    from isaacgymloco_b200 import _lib as L
    return L.lib.hl_finite_scan(ctypes.byref(f) if f is not None else None, n_rows, record, workspace, None)


def test_the_c_entry_checks_its_arguments():
    from isaacgymloco_b200 import _lib as L
    assert L.lib.hl_sizeof_finite_fields() == ctypes.sizeof(L.HlFiniteFields) == 8 + 24 * L.MAX_FINITE_FIELDS
    cases = [(None, {}, "size mismatch")]
    f = _args()
    f.struct_bytes -= 8
    cases.append((f, {}, "size mismatch"))
    cases += [(_args(), dict(record=None), "null record"), (_args(), dict(workspace=None), "null record"),
              (_args(0), {}, "n_fields"), (_args(17), {}, "n_fields"), (_args(-1), {}, "n_fields"),
              (_args(), dict(n_rows=0), "n_rows"), (_args(), dict(n_rows=-5), "n_rows")]
    for field, value, msg in [("src", None, "null field"), ("src", 4096 + 2, "aligned"), ("width", 0, "width"),
                              ("width", -3, "width"), ("row_stride", 12, "row_stride"), ("kind", 2, "kind"),
                              ("kind", -1, "kind")]:
        for k in (0, 2):                   # the first and the last field of the launch
            f = _args()
            setattr(f.field[k], field, value)
            cases.append((f, {}, msg))
    for f, kw, msg in cases:
        assert _call(f, **kw) != 0, msg
        assert msg.encode() in L.lib.hl_last_error(), (msg, L.lib.hl_last_error())


def _env(n=8, device="cpu"):
    return NS(num_envs=n, device=torch.device(device), common_step_counter=0)


def test_guard_rejects_bad_arguments():
    from isaacgymloco_b200.finite_guard import FiniteGuard
    storage = NS(num_envs=8, num_transitions_per_env=24)
    bad = [
        (dict(num_steps=0), "num_steps"),
        (dict(num_steps=-3), "num_steps"),
        (dict(fields=()), "at least one"),
        (dict(fields=("root_states", "obs_buf")), "unknown field 'obs_buf'"),
        (dict(fields=("root_state",)), "unknown field"),
        (dict(fields=("sigma",)), "storage slot"),
        (dict(fields=("root_states", "actions")), "storage slot"),
        (dict(fields=("root_states", "root_states")), "repeat"),
        (dict(storage=storage, fields=("actions",) * 17), "repeat"),
        (dict(storage=NS(num_envs=4, num_transitions_per_env=24)), "4 envs"),
        (dict(storage=storage, num_steps=25), "24 slots"),
        (dict(), "CUDA"),                                            # no CPU fallback
        (dict(storage=storage), "CUDA"),
    ]
    for kw, match in bad:
        args = dict(num_steps=24)
        args.update(kw)
        with pytest.raises(ValueError, match=match):
            FiniteGuard(_env(), **args)


def _f32_bits(x):
    return struct.unpack("<i", struct.pack("<f", x))[0]


def test_events_of_a_synthetic_table_against_brute_force():
    from isaacgymloco_b200.finite_guard import NonFiniteError, table_events
    rng = random.Random(5)
    fields = ("root_states", "dof_state", "contact_forces", "actions", "sigma", "rewards")
    widths = (13, 24, 51, 12, 12, 1)
    n, t_len, offset = 4099, 9, 65536
    specials = [0x7FC00000, 0x7FC00001, -0x00400000, -0x003EDCBB, 0x7F800000, -0x00800000, _f32_bits(-1.0),
                _f32_bits(0.0), -0x80000000, _f32_bits(-1e-38)]       # NaNs (both signs, payloads), +-inf, -1, +-0, -1e-38
    table = np.zeros((t_len, len(fields), 3), dtype=np.int64)
    table[:, :, 1] = -1
    for k in range(t_len):
        for f in range(len(fields)):
            if k in (0, 4) or rng.random() < 0.3:
                continue                                             # clean rows: count 0, index -1
            table[k, f] = (rng.randint(1, 10 ** 6), rng.randrange(n * widths[f]), rng.choice(specials))
    counters = [1000 + k + 1 for k in range(t_len)]
    got = table_events(torch.from_numpy(table), fields, widths, offset, counters)
    want = []
    for k in range(t_len):
        for f in range(len(fields)):
            count, index, bits = (int(v) for v in table[k, f])
            if count:
                value = float(np.array([bits & 0xFFFFFFFF], dtype=np.uint32).view(np.float32)[0])
                want.append(dict(k=k, common_step_counter=1000 + k + 1, field=fields[f], env=offset + index // widths[f],
                                 column=index % widths[f], value=value, count=count))
    assert len(got) == len(want) > 10
    for g, w in zip(got, want):
        assert {x: g[x] for x in g if x != "value"} == {x: w[x] for x in w if x != "value"}
        assert struct.pack("<d", g["value"]) == struct.pack("<d", w["value"]), (g, w)   # NaN sign / payload, +-inf
    assert any(math.isnan(g["value"]) and math.copysign(1.0, g["value"]) < 0 for g in got)
    assert table_events(table.tolist(), fields, widths)[0]["common_step_counter"] is None
    err = NonFiniteError(got)
    assert isinstance(err, FloatingPointError) and err.events == got
    k0 = min(ev["k"] for ev in got)
    msg = str(err)
    assert f"rollout step {k0} (common_step_counter {1000 + k0 + 1})" in msg
    for ev in got:
        if ev["k"] == k0:
            assert f"{ev['field']}: {ev['count']} element(s), first env {ev['env']} column {ev['column']}" in msg
    assert table_events(np.zeros((3, 2, 3), dtype=np.int64).tolist(), fields[:2], widths[:2]) == []
