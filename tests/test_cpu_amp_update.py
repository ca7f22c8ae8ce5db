"""CPU (-m "not gpu"): the host side of the device-drawn AMP update minibatches checks its inputs before anything is
allocated or launched.

* hl_amp_update_batch returns an error for a bad struct size, NULL ring / preload / counter / outputs, a lone mean or
  var pointer and a negative row offset, and accepts mb = 0 without a launch;
* AMPUpdateSampler raises ValueError for a loader without preloaded transitions, widths other than 30 / 49, a
  normaliser whose dim is not 30, mini_batch_size < 1, a seed outside [0, 2**64), a negative row_offset and CPU tensors
  (there is no CPU fallback).
"""
import ctypes
from types import SimpleNamespace as NS

import pytest
import torch


def _args():
    from isaacgymloco_b200 import _lib as L
    a = L.HlAmpUpdateBatch()
    a.struct_bytes = ctypes.sizeof(L.HlAmpUpdateBatch)
    # fake device addresses: every check below refuses the call on the host, before a launch
    a.ring_states, a.ring_next, a.ring_rows = 256, 512, 100
    a.preloaded_s, a.preloaded_s_next, a.n_preloaded = 768, 1024, 200
    a.draw_counter = 1280
    a.policy_s, a.policy_sn, a.expert_s, a.expert_sn, a.x_policy, a.x_expert = 1536, 1792, 2048, 2304, 2560, 2816
    a.mb = 0
    return a


def _call(a):
    from isaacgymloco_b200 import _lib as L
    return L.lib.hl_amp_update_batch(ctypes.byref(a), None)


def test_the_c_entry_checks_its_arguments():
    from isaacgymloco_b200 import _lib as L
    assert _call(_args()) == 0                       # mb = 0: nothing to launch, accepted without a device
    assert L.lib.hl_amp_update_batch(None, None) != 0
    cases = []
    for field, value, msg in [("struct_bytes", ctypes.sizeof(L.HlAmpUpdateBatch) - 8, "layout"),
                              ("ring_states", None, "ring"), ("ring_next", None, "ring"), ("ring_rows", 0, "ring"),
                              ("preloaded_s", None, "preload"), ("preloaded_s_next", None, "preload"),
                              ("n_preloaded", 0, "preload"), ("norm_mean", 4096, "go together"),
                              ("norm_var", 4096, "go together"), ("draw_counter", None, "counter"),
                              ("policy_s", None, "output"), ("x_expert", None, "output"), ("row_offset", -1, "row_offset")]:
        a = _args()
        setattr(a, field, value)
        a.mb = 64
        cases.append((a, msg))
    for a, msg in cases:
        assert _call(a) != 0, msg
        assert msg.encode() in L.lib.hl_last_error(), (msg, L.lib.hl_last_error())


def _objects(rows=64, n_pre=128, obs=30, frame=49, preload=True, norm_dim=30):
    loader = NS(preload_transitions=preload, preloaded_s=torch.zeros(n_pre, frame), preloaded_s_next=torch.zeros(n_pre, frame))
    rb = NS(states=torch.zeros(rows, obs), next_states=torch.zeros(rows, obs), num_samples=rows, buffer_size=rows)
    norm = NS(dim=norm_dim, mean=torch.zeros(norm_dim, dtype=torch.float64), var=torch.ones(norm_dim, dtype=torch.float64),
              epsilon=1e-4, clip_obs=10.0)
    return loader, rb, norm


def test_sampler_rejects_bad_inputs():
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    bad = [
        (_objects(preload=False), dict(), "preload"),
        (_objects(obs=42), dict(), r"\(rows, 30\)"),
        (_objects(frame=42), dict(), r"\(n, 49\)"),
        (_objects(frame=30), dict(), r"\(n, 49\)"),
        (_objects(norm_dim=60), dict(), "30 columns"),
        (_objects(), dict(mini_batch_size=0), ">= 1"),
        (_objects(), dict(mini_batch_size=-4), ">= 1"),
        (_objects(), dict(seed=-1), "seed"),
        (_objects(), dict(seed=1 << 64), "seed"),
        (_objects(), dict(row_offset=-1), "row_offset"),
        (_objects(), dict(), "CUDA"),                                   # CPU tensors: no CPU fallback
        (_objects()[:2] + (None,), dict(), "CUDA"),
    ]
    for (loader, rb, norm), kw, match in bad:
        args = dict(mini_batch_size=16, seed=0)
        args.update(kw)
        with pytest.raises(ValueError, match=match):
            AMPUpdateSampler(loader, rb, norm, **args)
    loader = NS(preload_transitions=False)                              # no preload tables at all
    with pytest.raises(ValueError, match="preload"):
        AMPUpdateSampler(loader, _objects()[1], None, 16, 0)
