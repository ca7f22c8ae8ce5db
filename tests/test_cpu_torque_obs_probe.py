"""The torque and observation probes (tests/torque_obs_probe.py) and the float64 references of the rollout
statistics, checked without a GPU.

Coverage: every clip and control branch the probes are built for is taken on at least 10 % of its entries on each
side.  Calibration: the plain fp32 oracle stays within the bound the GPU tests use,
|got - ref64| <= 1e-5 |ref64| + 1e-6 max_e |ref64[:, col]|, on every torque, observation, privileged, terminal-row
and AMP column, so the bound is attainable in fp32.  The references of tests/test_gpu_advantage_moments.py (the
oracle's GAE, and tests/stats_reference.py: advantage normalisation, column moments, the running mean/std merge) agree
with naive float64 loops."""
import numpy as np
import pytest
import torch

import torque_obs_probe as TP
from isaacgymloco_b200 import config as C

MIN_SHARE = 0.10
N = 4099
CPU = C.INDEX_MATH_TORCH_CPU


def _shares(gates):
    return {k: float(v.double().mean()) for k, v in gates.items()}


@pytest.mark.parametrize("ctl", TP.CONTROL_TYPES)
def test_torque_probe_covers_every_branch(ctl):
    """Per DOF the raw torque is above +limit, below -limit and inside on >= 10 % of the envs each, at least 4 % of the
    limit away from it; motor strengths, Kp and Kd factors are not 1; last_dof_vel differs from dof_vel; the hip
    columns see hip_reduction = 0.8."""
    cfg = TP.torque_cfg(ctl, N, CPU)
    state, hf = TP.make_torque_probe(cfg, N)
    _, _, raw = TP.reference64_torques(cfg, state, hf)
    bad = []
    for name, g in TP.torque_gates(cfg, raw).items():
        for d in range(12):
            share = float(g[:, d].double().mean())
            if share < MIN_SHARE:
                bad.append(f"{name} dof {d}: {share:.1%}")
    assert not bad, "below 10 %:\n" + "\n".join(bad)
    assert TP.torque_margin(cfg, raw) > 0.04
    assert cfg.hip_reduction == 0.8
    for k in ("motor_strength", "Kp_factors", "Kd_factors"):
        assert ((state[k] - 1).abs() > 0.02).all(), k
    vel = state["dof_state"].view(N, 12, 2)[..., 1]
    assert float((state["last_dof_vel"] != vel).double().mean()) > 0.99


@pytest.mark.parametrize("ctl", TP.CONTROL_TYPES)
@pytest.mark.parametrize("n", [N, 65539])
def test_fp32_oracle_torques_within_the_bound(ctl, n):
    """The fp32 oracle's torques and joint_pos_target against the float64 reference, per column."""
    cfg = TP.torque_cfg(ctl, n, CPU)
    state, hf = TP.make_torque_probe(cfg, n)
    tq64, tg64, _ = TP.reference64_torques(cfg, state, hf)
    from oracle import torch_oracle as O
    env = O.OracleEnv(cfg, {k: v.clone() for k, v in state.items()}, hf)
    tq = env._compute_torques(state["actions"].clone())
    cols = [f"dof {d}" for d in range(12)]
    TP.check_bound(tq.T, tq64.T, cols, f"{ctl} torques")
    TP.check_bound(env.joint_pos_target.T, tg64.T, cols, f"{ctl} joint_pos_target")


@pytest.mark.parametrize("task", TP.OBS_TASKS)
@pytest.mark.parametrize("variant", TP.OBS_VARIANTS)
def test_obs_probe_covers_every_clip(task, variant):
    """The +-1 height clip binds above and below on >= 10 % of the height entries each and is inactive on >= 10 %;
    with clip_observations = 3 that clip binds on both sides of the ang-vel, dof-vel and height groups on >= 10 %;
    noise draws sit at u = 0 and u = 1 - 2^-24 in all four tables; heading commands stay away from the wrap_to_pi
    discontinuity; the disturbance is non-zero; some envs reset."""
    cfg = TP.obs_cfg(task, variant, N, CPU)
    state, hf, noise = TP.make_obs_probe(cfg, N)
    env, ids, _, _ = TP.reference64_obs(cfg, state, hf, noise)
    shares = _shares(TP.obs_gates(cfg, env))
    assert len(shares) == (9 if variant == "clip" else 3)
    bad = [f"{k}: {v:.1%}" for k, v in shares.items() if v < MIN_SHARE]
    print(f"\n[{task} {variant}]\n" + "\n".join(f"{k:40s} {v:6.1%}" for k, v in shares.items()))
    assert not bad, "below 10 %:\n" + "\n".join(bad)
    for k, v in noise.items():
        assert float((v == 0).double().mean()) >= MIN_SHARE, k
        assert float((v == TP.U_TOP).double().mean()) >= MIN_SHARE, k
        assert (v < 1).all(), k
    from oracle import torch_oracle as O
    q = state["root_states"][:, 3:7].double()
    fwd = O.quat_apply(q, torch.tensor([[1.0, 0.0, 0.0]], dtype=torch.float64).expand(N, 3))
    w = O.wrap_to_pi(state["commands"][:, 3].double() - torch.atan2(fwd[:, 1], fwd[:, 0]))
    assert float((w.abs() - np.pi).abs().min()) >= 1e-3
    assert (state["disturbance"][:, 0, :] != 0).all()
    assert MIN_SHARE * N <= len(ids) <= (1 - MIN_SHARE) * N


def _obs_columns(what, width):
    names = {v: k for k, v in [(k, i) for k, s in TP.GROUPS.items() for i in range(*s.indices(width))]}
    return [f"{what}[{i}] ({names[i]})" for i in range(width)]


@pytest.mark.parametrize("task", TP.OBS_TASKS)
@pytest.mark.parametrize("variant", TP.OBS_VARIANTS)
def test_fp32_oracle_obs_within_the_bound(task, variant):
    """The fp32 oracle against the float64 reference: obs_buf[:, :45], privileged_obs_buf, the terminal rows and the
    terminal AMP rows, every column; the history shift of obs_buf bit for bit; the reset ids equal."""
    cfg = TP.obs_cfg(task, variant, N, CPU)
    state, hf, noise = TP.make_obs_probe(cfg, N)
    e64, ids64, term64, amp64 = TP.reference64_obs(cfg, state, hf, noise)
    e32, ids32, term32, amp32 = TP.reference32_obs(cfg, state, hf, noise)
    assert torch.equal(ids32, ids64)
    TP.check_bound(e32.obs_buf[:, :45].T, e64.obs_buf[:, :45].T, _obs_columns("obs", 45), "obs_buf")
    pw = e64.privileged_obs_buf.shape[1]
    TP.check_bound(e32.privileged_obs_buf.T, e64.privileged_obs_buf.T, _obs_columns("priv", pw), "privileged_obs_buf")
    TP.check_bound(term32.T, term64.T, _obs_columns("term", pw), "terminal rows")
    TP.check_bound(amp32.T, amp64.T, [f"amp[{i}]" for i in range(30)], "terminal AMP rows")
    assert torch.equal(e32.obs_buf[:, 45:], state["obs_buf"][:, :225].clamp(-cfg.clip_observations, cfg.clip_observations))


# ----------------------------------------------------------------------------- references of the rollout statistics
def test_float64_references_match_naive_numpy():
    """The references of tests/test_gpu_advantage_moments.py against naive float64 loops on small cases: the
    oracle's GAE returns (fp32, so within 1e-6), the unbiased normalisation (NaN for one element), two-pass column
    moments and the running mean/std merge."""
    import stats_reference as SR
    from oracle import torch_oracle as O
    rng = np.random.default_rng(5)
    for t, n in ((1, 1), (3, 2), (9, 5)):
        r = rng.normal(size=(t, n, 1)).astype(np.float32)
        v = rng.normal(size=(t, n, 1)).astype(np.float32)
        d = (rng.random((t, n, 1)) < 0.3).astype(np.uint8)
        lv = rng.normal(size=(n, 1)).astype(np.float32)
        ret = np.zeros((t, n, 1))
        for e in range(n):
            a, nxt = 0.0, float(lv[e, 0])
            for k in reversed(range(t)):
                live = 1.0 - d[k, e, 0]
                delta = float(r[k, e, 0]) + live * 0.99 * nxt - float(v[k, e, 0])
                a = delta + live * 0.99 * 0.95 * a
                ret[k, e, 0] = a + float(v[k, e, 0])
                nxt = float(v[k, e, 0])
        got, _ = O.compute_returns(*(torch.from_numpy(x) for x in (r, v, d, lv)), 0.99, 0.95)
        np.testing.assert_allclose(got.numpy(), ret, rtol=1e-6, atol=1e-6)
    for m in (2, 5, 48):
        a = rng.normal(3.0, 2.0, size=m).astype(np.float32)
        mean = sum(float(x) for x in a) / m
        for ddof in (0, 1):
            std = (sum((float(x) - mean) ** 2 for x in a) / (m - ddof)) ** 0.5
            want = [(float(x) - mean) / (std + 1e-8) for x in a]
            np.testing.assert_allclose(SR.normalize64(a, ddof), want, rtol=1e-12, atol=1e-12)
    assert np.isnan(SR.normalize64(np.ones(1, np.float32))).all()
    for rows, dim in ((1, 3), (7, 2), (33, 5)):
        x = rng.normal(size=(rows, dim)).astype(np.float32)
        mean, var = SR.moments64(x)
        for c in range(dim):
            col = [float(x[i, c]) for i in range(rows)]
            mu = sum(col) / rows
            assert abs(mean[c] - mu) <= 1e-14 * max(1.0, abs(mu))
            assert abs(var[c] - sum((y - mu) ** 2 for y in col) / rows) <= 1e-13
    rms = SR.RunningMeanStd64(3)
    batches = [rng.normal(1.0, 2.0, size=(k, 3)).astype(np.float32) for k in (4, 1, 9)]
    for b in batches:
        rms.update(b)
    allx = np.concatenate(batches).astype(np.float64)
    # RunningMeanStd starts from mean 0, var 1, count 1e-4: the merge equals the pooled moments up to that prior
    np.testing.assert_allclose(rms.mean, allx.mean(0), rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(rms.var, allx.var(0), rtol=1e-4, atol=1e-4)
    assert rms.count == pytest.approx(14 + 1e-4)
