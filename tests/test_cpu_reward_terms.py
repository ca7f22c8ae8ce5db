"""The reward probe state (tests/reward_probe.py) and its float64 reference, checked without a GPU.

Coverage: on the probe every reward term is clearly non-zero on a sizeable share of the envs and every gate the
terms branch on is on for at least 10 % of the envs and off for at least 10 %, so a kernel term that is wrong on
either side of a gate shows up in tests/test_gpu_reward_terms.py.  Calibration: the fp32 oracle stays within the
bound those tests use, |got - ref64| <= 1e-5 |ref64| + 1e-6 max_e |ref64[k]|, on every row, so the bound is
attainable in fp32."""
import pytest

import reward_probe as P
from isaacgymloco_b200 import config as C

MIN_SHARE = 0.10
CPU = C.INDEX_MATH_TORCH_CPU


def _case(task, n):
    cfg = P.probe_cfg(task, n, index_math=CPU)
    state, hf = P.make_probe(cfg, n)
    return cfg, state, hf, P.reference64(cfg, state, hf)


@pytest.mark.parametrize("task", ("allterms",) + P.TASKS)
def test_probe_covers_every_term_and_gate(task):
    """Each term's row is above 1e3 x the comparison floor on >= 10 % of envs.  With all 51 terms, each gate is on and
    off on >= 10 %.  With the stairs list (the one only_positive_rewards is tested with) the loop sum is negative on
    >= 10 % and positive on >= 10 %.  Run with -s for the table."""
    n = 4099
    cfg, state, hf, env = _case(task, n)
    rows = P.rows64(env)
    names = cfg.episode_sum_names()
    assert len(names) == (51 if task == "allterms" else len(rows))
    lines, bad = [], []
    for k, name in enumerate(names):
        share = float((rows[k].abs() > 1e3 * P.FLOOR * rows[k].abs().max()).double().mean())
        lines.append(f"term {name:28s} {share:6.1%}")
        if share < MIN_SHARE:
            bad.append(lines[-1])
    shares = {k: float(v.double().mean()) for k, v in P.gates(cfg, state, env).items()} if task == "allterms" else {}
    if task == "stairs":
        shares["loop sum < 0"] = float((P.loop_sum(env) < 0).double().mean())
    for k, share in shares.items():
        lines.append(f"gate {k:45s} {share:6.1%}")
        if not MIN_SHARE <= share <= 1 - MIN_SHARE:
            bad.append(lines[-1])
    print(f"\n[{task}, {n} envs]\n" + "\n".join(lines))
    assert not bad, "below 10 % (terms) or outside 10-90 % (gates):\n" + "\n".join(bad)


@pytest.mark.parametrize("task", ("allterms",) + P.TASKS)
@pytest.mark.parametrize("n", [4099, 65536])
def test_fp32_oracle_within_the_bound(task, n):
    """The fp32 oracle (torch-CPU arithmetic) against the float64 reference: every episode_sums row and rew_buf
    within the bound; feet_air_time and last_contacts equal the fp32 values the reference rounds to."""
    cfg, state, hf, env = _case(task, n)
    e32 = P.reference32(cfg, state, hf)
    names = cfg.episode_sum_names()
    P.check_bound(P.rows64(e32), P.rows64(env), names, f"{task} episode_sums")
    P.check_bound(e32.rew_buf, env.rew_buf, ["rew_buf"], f"{task} rew_buf")
    assert (e32.last_contacts == env.last_contacts).all()
    assert (e32.reset_buf == env.reset_buf).all() and (e32.time_out_buf == env.time_out_buf).all()
    P.check_bound(e32.feet_air_time.T, env.feet_air_time.T, [f"foot {f}" for f in range(4)], f"{task} feet_air_time")


def test_reference_cells_follow_the_fp32_index_arithmetic():
    """Oracle64 picks terrain cells as the fp32 reference does: its base-height cells equal those of the fp32 oracle
    (torch-CPU flavour), while a plain float64 scan picks other cells for some points."""
    import torch
    from oracle import torch_oracle as O
    n = 4099
    cfg, state, hf, env = _case("allterms", n)
    e32 = O.OracleEnv(cfg, {k: v.clone() for k, v in state.items()}, hf)
    want, wx, wy = e32._scan(e32.base_height_points)
    got, gx, gy = env._scan(env.base_height_points)
    assert torch.equal(gx, wx) and torch.equal(gy, wy) and torch.equal(got, want)
    with P.default_dtype(torch.float64):
        plain = O.OracleEnv(cfg, {k: (v.double() if v.is_floating_point() else v) for k, v in state.items()}, hf)
        _, px, py = plain._scan(plain.base_height_points)
    assert not (torch.equal(px, wx) and torch.equal(py, wy)), "the probe no longer has points whose cell depends on precision"
