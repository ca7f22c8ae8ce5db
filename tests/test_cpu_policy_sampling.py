"""CPU (-m "not gpu"): the host side of the keyed policy sampling checks its inputs before anything is launched.

* hl_policy_sample returns an error for bad struct sizes, NULL tensors, act_dim outside 1..16, a std row stride other
  than 0 or act_dim and a negative env count;
* keyed_act raises ValueError for CPU tensors (there is no CPU fallback), wrong shapes and dtypes, an action dimension
  above 16 and a z of the wrong shape, and AssertionError("Rollout buffer overflow") for a full storage.
"""
import ctypes
from types import SimpleNamespace as NS

import pytest
import torch

from isaacgymloco_b200 import config as C


def _args(n=8, a=12):
    from isaacgymloco_b200 import _lib as L
    cfg = C.aliengo("flat", num_envs=n).to_c()
    b = L.HlEnvBuffers()
    b.struct_bytes = ctypes.sizeof(L.HlEnvBuffers)
    # fake device addresses: every check below refuses the call on the host, before a launch
    return dict(cfg=cfg, bufs=b, mean=256, std=512, stride=0, z=None, a=a, act=768, logp=1024, mu=None, sigma=None, n=n)


def _call(d):
    from isaacgymloco_b200 import _lib as L
    return L.lib.hl_policy_sample(ctypes.byref(d["cfg"]), ctypes.byref(d["bufs"]), d["mean"], d["std"], d["stride"], d["z"],
                                  d["a"], d["act"], d["logp"], d["mu"], d["sigma"], d["n"], None)


def test_the_c_entry_checks_its_arguments():
    from isaacgymloco_b200 import _lib as L
    assert _call(dict(_args(), n=0)) == 0            # nothing to launch: accepted without a device
    assert _call(dict(_args(a=5), stride=5, n=0)) == 0
    bad_cfg, bad_bufs = _args(), _args()
    bad_cfg["cfg"].struct_bytes += 4
    bad_bufs["bufs"].struct_bytes -= 8
    cases = [(bad_cfg, "HlCfg"), (bad_bufs, "HlEnvBuffers")]
    for key in ("mean", "std", "act", "logp"):
        cases.append((dict(_args(), **{key: None}), "null"))
    for a in (0, -1, 17, 64):
        cases.append((dict(_args(a=a)), "act_dim"))
    for stride in (1, 11, 13, -12, 24):
        cases.append((dict(_args(), stride=stride), "std_row_stride"))
    cases.append((dict(_args(), n=-1), "negative n_envs"))
    for d, msg in cases:
        assert _call(d) != 0, msg
        assert msg.encode() in L.lib.hl_last_error(), (msg, L.lib.hl_last_error())


class _Storage:
    """The host state keyed_act reads from a HIMRolloutStorage (no device needed for the checks)."""

    def __init__(self, t, step, n=6, a=12):
        self.num_transitions_per_env, self.step = t, step
        self.actions = torch.zeros(t, n, a)


def test_keyed_act_rejects_bad_inputs():
    from isaacgymloco_b200.policy_sampling import keyed_act
    n, a = 6, 12
    env = NS(num_envs=n, device=torch.device("cuda:0"))
    mean, std = torch.zeros(n, a), torch.ones(a)
    bad = [
        dict(mean=mean, std=std),                                               # CPU tensors: no CPU fallback
        dict(mean=mean, std=std, z=torch.zeros(n, a)),
        dict(mean=torch.zeros(n + 1, a), std=std),                              # shapes
        dict(mean=torch.zeros(n, a, 1), std=std),
        dict(mean=torch.zeros(n * a), std=std),
        dict(mean=mean, std=torch.ones(a + 1)),
        dict(mean=mean, std=torch.ones(n, a + 1)),
        dict(mean=mean, std=torch.ones(1, a)),
        dict(mean=torch.zeros(n, 17), std=torch.ones(17)),                     # A > 16
        dict(mean=torch.zeros(n, 0), std=torch.ones(0)),
        dict(mean=mean, std=std, z=torch.zeros(n, a - 1)),                      # z of the wrong shape
        dict(mean=mean, std=std, z=torch.zeros(a)),
        dict(mean=mean.double(), std=std),                                      # dtypes
        dict(mean=mean, std=std.half()),
        dict(mean=mean, std=std, z=torch.zeros(n, a, dtype=torch.float64)),
        dict(mean=mean.tolist(), std=std),                                      # not a tensor
        dict(mean=mean, std=1.0),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            keyed_act(env, **kw)
    with pytest.raises(ValueError, match="CUDA"):
        keyed_act(env, mean, std)
    for step in (4, 5):
        with pytest.raises(AssertionError, match="Rollout buffer overflow"):
            keyed_act(env, mean, std, storage=_Storage(4, step))
