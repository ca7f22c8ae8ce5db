"""The termination probe (tests/termination_probe.py) checked without a GPU.

Coverage: every termination clause a config applies is on for at least 10 % of the envs, off for at least 10 % and
the only reason to reset for at least 5 %; each side of the border, the border strip, both signs of the velocity
violation, the wrong signs, a zero command and levels 3 and 4 among the violators all occur; every decided value stays
clear of its threshold unless fp32 computes it exactly.  Calibration: the plain fp32 oracle reaches the float64
reference's decisions on every env, and its frame and heading command stay within the bound the GPU tests use,
|got - ref64| <= 1e-5 |ref64| + 1e-6 max_e |ref64[:, col]|.
"""
import numpy as np
import pytest
import torch

import termination_probe as TP
from isaacgymloco_b200 import config as C

N = 4099
CPU = C.INDEX_MATH_TORCH_CPU
IDS = [f"{t}-{v}" for t, v in TP.CONFIGS]


def _probe(task, variant, n=N):
    cfg = TP.termination_cfg(task, variant, n, CPU)
    return cfg, TP.make_termination_probe(cfg, n)


@pytest.mark.parametrize("task,variant", TP.CONFIGS, ids=IDS)
def test_termination_probe_covers_every_gate(task, variant):
    """Every gate's share printed; each applied clause on / off for >= 10 % and the only reason for >= 5 % of the
    envs; the reset envs are exactly those of the clauses the config applies; the exact slices present; no value
    within the margin of its threshold."""
    cfg, pr = _probe(task, variant)
    env = TP.reference64_termination(cfg, pr)
    shares = {k: float(m[over].double().mean()) if over.any() else float("nan")
              for k, (m, over) in TP.gates(cfg, pr, env).items()}
    print(f"\n[{task} {variant}] clauses {TP.clauses(cfg)}, {len(env.ids)} of {N} envs reset\n"
          + "\n".join(f"{k:58s} {v:6.1%}" for k, v in shares.items()))
    dec = TP.clause_decisions(cfg, pr, env)
    assert sorted(dec) == sorted(TP.clauses(cfg))
    want = torch.zeros(N, dtype=torch.bool)
    for m in dec.values():
        want |= m
    assert torch.equal(env.reset_buf, want), "reset_buf is not the OR of the applied clauses"
    bad = []
    for c in dec:
        on, sole = shares[f"{c}: resets"], shares[f"{c}: the only reason"]
        if not 0.10 <= on <= 0.90:
            bad.append(f"{c}: on for {on:.1%}")
        if sole < 0.05:
            bad.append(f"{c}: the only reason for {sole:.1%}")
    for k in ("border: x < 0", "border: y < 0", "border: x >= x_limit", "border: y >= y_limit",
              "border: x in the strip [x_size, x_limit)", "border: y in the strip [y_size, y_limit)"):
        if shares[k] < 0.03:
            bad.append(f"{k}: {shares[k]:.1%}")
    keys = ["no reset", "on the resampling mark", "fall-down: v_z < -5", "upside down (projected gravity z > 0)",
            "foot Fz > 1 (per foot)", "last_contacts (per foot)"]
    if cfg.heading_command:
        keys += [k for k in shares if k.startswith("heading:")]
    if cfg.base_vel_violate_commands:
        keys += [k for k in shares if k.startswith("velocity: ")]
    if len(cfg.termination_contact_indices) > 1:
        keys += ["contact: one body only", "contact: the second body only"]
    for k in keys:
        if not 0.03 <= shares[k] <= 0.97:
            bad.append(f"{k}: {shares[k]:.1%}")
    for k in ("pre-step episode length max - 1", "pre-step episode length max"):
        if shares[k] == 0:
            bad.append(f"{k}: no env")
    if cfg.base_vel_violate_commands:
        for k in [k for k in shares if k.startswith("velocity violators") or k.startswith("mark:")]:
            if not shares[k] > 0.01:
                bad.append(f"{k}: {shares[k]:.1%}")
    assert not bad, "gates outside their shares:\n" + "\n".join(bad)
    for k, m in TP.exact_slices(cfg, pr).items():
        assert m.sum() >= 5, f"exact slice {k}: {int(m.sum())} envs"
    close = TP.margins_ok(cfg, pr, env)
    assert not close, "values at their thresholds:\n" + "\n".join(close[:20])


@pytest.mark.parametrize("task,variant", TP.CONFIGS, ids=IDS)
def test_fp32_oracle_termination_matches_float64(task, variant):
    """The fp32 oracle's step (mark resampling, pre_reset): reset_buf, time_out_buf, vel_violate, contact_filt,
    last_contacts and the reset ids equal the float64 reference's; the frame and commands[:, 2] within the bound."""
    cfg, pr = _probe(task, variant)
    e32 = TP.reference32_termination(cfg, pr)
    e64 = TP.reference64_termination(cfg, pr)
    for k in ("reset_buf", "time_out_buf", "vel_violate", "contact_filt", "last_contacts"):
        assert torch.equal(getattr(e32, k), getattr(e64, k)), k
    assert torch.equal(e32.ids, e64.ids)
    TP.check_frame(e32, e64, torch.ones(N, dtype=torch.bool), f"{task} {variant}")


@pytest.mark.parametrize("n,num_envs,offset", [(7, 7, 0), (4099, 20000, 3000)])
def test_termination_probe_small_and_sharded(n, num_envs, offset):
    """7 envs and a shard with env_id_offset > 0 (part of it in the high-speed slice): the fp32 oracle's decisions
    equal the float64 reference's and the probe stays clear of every threshold."""
    cfg = TP.termination_cfg("stairs", "default", n, CPU, num_envs=num_envs, env_id_offset=offset)
    pr = TP.make_termination_probe(cfg, n)
    e32, e64 = TP.reference32_termination(cfg, pr), TP.reference64_termination(cfg, pr)
    assert torch.equal(e32.reset_buf, e64.reset_buf) and torch.equal(e32.time_out_buf, e64.time_out_buf)
    assert not TP.margins_ok(cfg, pr, e64)


def test_exact_slices_are_exact_in_fp32():
    """The thresholds the exact slices sit on are fp32 numbers, and the slices land on the intended side in fp32."""
    for task in ("flat", "stairs"):
        cfg = TP.termination_cfg(task, "default", 8)
        xl, yl = TP.limits(cfg)
        assert (xl, yl) == {"flat": (87.5, 167.5), "stairs": (107.5, 207.5)}[task]
        assert float(np.float32(xl)) == xl and float(np.float32(yl)) == yl
        assert float(np.float32(cfg.x_size + cfg.border_size / 2)) == cfg.to_c().x_limit == xl
        assert cfg.to_c().y_limit == yl
        nx = np.nextafter(np.float32(xl), np.float32(-np.inf))
        assert nx < np.float32(xl) and not np.float32(xl) < np.float32(xl)
    one, up = np.float32(1.0), np.float32(TP.ONE_UP)
    assert up > one and np.sqrt(np.float32(up * up)) > one and np.sqrt(one * one) == one
    assert np.float32(TP.FIVE_DOWN) < np.float32(-5.0) and not np.float32(-5.0) < np.float32(-5.0)
    # the fresh c0 of a zero command: u = 0.5 gives exactly 0 in both command forms (columns 36 and 39)
    u = np.float32(0.5)
    assert np.float32(2.0) * u - np.float32(1.0) == 0.0
