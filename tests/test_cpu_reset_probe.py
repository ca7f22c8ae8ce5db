"""The reset probe (tests/reset_probe.py) checked without a GPU.

Coverage: every decision of reset_idx's re-draws, the command resampling and the terrain curriculum is taken on at
least 10 % and skipped on at least 10 % of the envs it applies to, clear of its threshold.  Calibration: the plain
fp32 oracle stays within the bound the GPU tests use, |got - ref64| <= 1e-5 |ref64| + 1e-6 max_e |ref64[:, col]|, on
every drawn field and every observation column of the reset envs, and meets every exactness claim those tests make.
"""
import pytest
import torch

import reset_probe as RP
from isaacgymloco_b200 import config as C

MIN_SHARE = 0.10
N = 4099
CPU = C.INDEX_MATH_TORCH_CPU


def _probe(task, variant, n=N, **kw):
    cfg = RP.reset_cfg(task, variant, n, CPU, **kw)
    return cfg, RP.make_reset_probe(cfg, n)


@pytest.mark.parametrize("task", RP.TASKS)
@pytest.mark.parametrize("variant", RP.VARIANTS)
def test_reset_probe_covers_every_gate(task, variant):
    """Each gate on and off for >= 10 % of the reset envs it applies to (printed with its share); no decided value
    within 1e-3 of its threshold unless fp32 computes it exactly; every uniform column at 0 and at 1 - 2^-24 on some
    reset envs; the step resets exactly the intended envs."""
    cfg, pr = _probe(task, variant)
    env = RP.reference64_reset(cfg, pr)
    assert torch.equal(env.ids, pr["ids"])
    shares = {k: float(v.double().mean()) for k, v in RP.gates(cfg, pr, env).items()}
    print(f"\n[{task} {variant}] {len(env.ids)} reset envs\n" + "\n".join(f"{k:42s} {v:6.1%}" for k, v in shares.items()))
    bad = [f"{k}: {v:.1%}" for k, v in shares.items() if not MIN_SHARE <= v <= 1 - MIN_SHARE]
    assert not bad, "gates outside [10 %, 90 %]:\n" + "\n".join(bad)
    expect = 5 if cfg.is_plane else 12
    expect += variant == "wide"
    assert len(shares) == expect, sorted(shares)
    close = RP.margins_ok(cfg, pr, env)
    assert not close, "values at their thresholds:\n" + "\n".join(close[:20])
    u = pr["u"][env.ids]
    assert ((u == 0).any(dim=0)).all() and ((u == RP.U_TOP).any(dim=0)).all() and (u < 1).all()
    if not cfg.is_plane:
        top_up = RP.gates(cfg, pr, env)["curriculum: top level + up (wraps)"]
        w = u[top_up, 43]
        assert (w == 0).any() and (w == RP.U_TOP).any() and ((w > 0) & (w < RP.U_TOP)).any()


@pytest.mark.parametrize("task", RP.TASKS)
@pytest.mark.parametrize("variant", RP.VARIANTS)
def test_fp32_oracle_reset_within_the_bound(task, variant):
    """The fp32 oracle's reset step (mark resampling, pre_reset, reset_idx_draw, apply_reset, post_reset) against the
    float64 reference: root_states, dof_state, commands, the three factors, obs_buf[:, :45] and privileged_obs_buf of
    the reset envs within the bound; the exactness claims of the GPU tests hold."""
    cfg, pr = _probe(task, variant)
    e32 = RP.reference32_reset(cfg, pr)
    e64 = RP.reference64_reset(cfg, pr, root32_after=e32.root_states)
    assert torch.equal(e32.ids, e64.ids)
    RP.check_reset_rows(e32, e64, e64.ids, f"{task} {variant}")
    bad = RP.exact_failures(cfg, pr, e32, e64)
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("n,num_envs,offset", [(4100, 4100, 0), (4099, 20000, 3000), (7, 7, 0)])
def test_fp32_oracle_reset_on_shards_within_the_bound(n, num_envs, offset):
    """The high-speed slice boundary: a multiple of 5, a shard with env_id_offset > 0 whose first 1,000 envs lie in
    the slice, and 7 envs (one in the slice); every env resets."""
    cfg = RP.reset_cfg("flat", "wide", n, CPU, num_envs=num_envs, env_id_offset=offset)
    pr = RP.make_reset_probe(cfg, n, reset_share=1.0)
    e32 = RP.reference32_reset(cfg, pr)
    e64 = RP.reference64_reset(cfg, pr, root32_after=e32.root_states)
    assert len(e64.ids) == n
    h = C.high_vel_env_count(num_envs) - offset
    assert 0 < h < n
    RP.check_reset_rows(e32, e64, e64.ids, f"shard {n}/{num_envs}+{offset}")
    assert not RP.exact_failures(cfg, pr, e32, e64)
    assert not RP.margins_ok(cfg, pr, e64)


def test_fp32_oracle_reset_idx_alone_within_the_bound():
    """reset_idx on a given id list without the step before it (the form of reset_idx_device)."""
    cfg, pr = _probe("stairs", "wide")
    e32 = RP.reference32_reset(cfg, pr, pre_step=False)
    e64 = RP.reference64_reset(cfg, pr, pre_step=False, root32_after=e32.root_states)
    RP.check_reset_rows(e32, e64, e64.ids, "reset_idx alone")
    assert not RP.exact_failures(cfg, pr, e32, e64)
