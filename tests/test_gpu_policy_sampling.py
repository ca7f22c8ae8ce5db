"""-m gpu: the keyed policy sampling (hl_policy_sample, policy_sampling.keyed_act) -- HIMPPO.act's sample, log-probability,
mean and sigma in one launch, with the standard normals drawn from Philox stream 7.

* Arithmetic: fed the same standard normals, actions, mu and sigma equal torch's Normal(mean, mean*0. + std,
  validate_args=False).rsample() composition bit for bit (NaN, +-inf, +-0 and means beyond the action clip included);
  the log-probability is within a summation-order bound of the float64 sum of torch's per-action terms.
* Philox: the draws are Box-Muller of the stream-7 blocks of (seed, step, global env id), recomputed on the host; they
  are standard normal, bounded by sqrt(48 ln 2), and independent across columns, steps and streams 0 / 4.
* A captured launch draws what an eager one does, and two shards draw what one big env draws.
* With a storage the outputs are its slots and the transition record copies none of them; nothing syncs.
* A replayed rollout with a stochastic torch policy equals the eager public-step() loop, storage field for storage field.
"""
import ctypes

import numpy as np
import pytest
import torch

from test_gpu_keyed_domain_rand import _bits, _bufs, _cfg, _philox_block, _rollout_env, _special, _u01

pytestmark = pytest.mark.gpu

ZMAX = float(np.sqrt(48.0 * np.log(2.0))) * (1.0 + 1e-6)   # |z| bound of the 24-bit Box-Muller draw (+ fp32 rounding)


def _launch(c, b, mean, std, z, out, logp, mu=None, sigma=None, n=None):
    from isaacgymloco_b200 import _lib as L
    n = mean.shape[0] if n is None else n
    a = mean.shape[1]
    L.check(L.lib.hl_policy_sample(ctypes.byref(c), ctypes.byref(b), L.ptr(mean), L.ptr(std), a if std.dim() == 2 else 0,
                                   L.ptr(z), a, L.ptr(out), L.ptr(logp), L.ptr(mu), L.ptr(sigma), n, L.stream()))


def _draw(c, b, n, a, dev="cuda:0"):
    """The kernel's standard normals: actions of mean 0, std 1."""
    out, logp = torch.empty(n, a, device=dev), torch.empty(n, device=dev)
    _launch(c, b, torch.zeros(n, a, device=dev), torch.ones(a, device=dev), None, out, logp)
    return out


def _host_normals(seed, step, gid, a):
    """Stream 7 on the host: Box-Muller in float64 of the fp32 uniforms, block b -> columns 4b .. 4b+3."""
    cols, radii = [], []
    for blk in range((a + 3) // 4):
        x, y, zw, w = _philox_block(seed, step, gid, 7, block=blk)
        for p, q in ((x, y), (zw, w)):
            u1 = (np.float32(1.0) - _u01(p)).astype(np.float64)
            r = np.sqrt(-2.0 * np.log(u1))
            t = 2.0 * np.pi * _u01(q).astype(np.float64)
            cols += [r * np.cos(t), r * np.sin(t)]
            radii += [r, r]
    return np.stack(cols[:a], 1), np.stack(radii[:a], 1)


# ---------------------------------------------------------------------------------------------------- 1. arithmetic
def _torch_sample(mean, std, z, monkeypatch):
    """HIMActorCritic.update_distribution / act / get_actions_log_prob / action_mean / action_std with
    Normal(validate_args=False).rsample(), whose standard normals are `z`."""
    from torch.distributions import Normal, normal
    monkeypatch.setattr(normal, "_standard_normal", lambda shape, dtype, device: z)
    dist = Normal(mean, mean * 0. + std, validate_args=False)
    actions = dist.rsample()
    terms = dist.log_prob(actions)
    return actions, terms, dist.mean, dist.stddev


@pytest.mark.parametrize("n", [1, 4099, 65536])
def test_arithmetic_bit_for_bit(n, monkeypatch):
    dev = "cuda:0"
    g = torch.Generator().manual_seed(n)
    c, b = _cfg(n), _bufs()
    checked_nan = False
    for a in (12, 5, 16):
        for per_row in (False, True):
            mean = _special(3.0 * torch.randn(n, a, generator=g), g).to(dev)
            std = (0.2 + 0.8 * torch.rand(*((n, a) if per_row else (a,)), generator=g)).to(dev)
            z = torch.randn(n, a, generator=g).to(dev)
            want_a, terms, want_mu, want_s = _torch_sample(mean, std, z, monkeypatch)
            assert torch.equal(_bits(want_a), _bits(mean + z * (mean * 0. + std)))   # torch.normal's mul_(std).add_(mean)
            out, logp = torch.full((n, a), 7.0, device=dev), torch.full((n,), 7.0, device=dev)
            mu, sig = torch.full((n, a), 7.0, device=dev), torch.full((n, a), 7.0, device=dev)
            _launch(c, b, mean, std, z, out, logp, mu, sig)
            what = (a, per_row)
            assert torch.equal(_bits(out), _bits(want_a)), what
            assert torch.equal(_bits(mu), _bits(want_mu)), what
            assert torch.equal(_bits(sig), _bits(want_s)), what
            # log-probability: the float64 sum of torch's fp32 terms, within a summation-order bound
            ref = terms.double().sum(-1)
            bound = a * 2.0 ** -24 * terms.double().abs().sum(-1)
            nan = torch.isnan(ref)
            assert torch.equal(torch.isnan(logp), nan), what
            fin = ~nan
            assert ((logp.double()[fin] - ref[fin]).abs() <= bound[fin]).all(), what
            # the first PPO ratio exp(torch log-prob - kernel log-prob), on the rows of ordinary means
            plain = torch.isfinite(mean).all(-1) & (mean.abs() < 50.0).all(-1)
            assert n == 1 or plain.any()
            if plain.any():
                ratio = torch.exp(terms.sum(-1)[plain] - logp[plain])
                assert (ratio - 1.0).abs().max() <= 1e-5, what
            checked_nan |= bool(nan.any())
            # mu_out aliasing mean: skipped, everything else unchanged
            m2 = mean.clone()
            out2, logp2, sig2 = torch.empty_like(out), torch.empty_like(logp), torch.empty_like(sig)
            _launch(c, b, m2, std, z, out2, logp2, m2, sig2)
            assert torch.equal(_bits(m2), _bits(mean)) and torch.equal(_bits(out2), _bits(out)), what
            assert torch.equal(_bits(logp2), _bits(logp)) and torch.equal(_bits(sig2), _bits(sig)), what
            # mu / sigma NULL: actions and log-prob alone
            out3, logp3 = torch.empty_like(out), torch.empty_like(logp)
            _launch(c, b, mean, std, z, out3, logp3)
            assert torch.equal(_bits(out3), _bits(out)) and torch.equal(_bits(logp3), _bits(logp)), what
    assert n == 1 or checked_nan


# ---------------------------------------------------------------------------------------------------- 2. Philox
@pytest.mark.parametrize("a", [12, 5, 16])
def test_philox_draws_match_the_host(a):
    n, seed, off = 4099, 0x1234_5678_9ABC, 70001
    c = _cfg(1 << 20, offset=off)                        # a shard whose global ids start at `off`
    gid = np.arange(n, dtype=np.uint64) + np.uint64(off)
    for step in (0, 9, (1 << 33) + 9):
        got = _draw(c, _bufs(seed=seed, offset=step), n, a).double().cpu().numpy()
        want, r = _host_normals(seed, step, gid, a)
        err = np.abs(got - want) / np.maximum(1.0, r)
        assert err.max() <= 1e-6, (a, step, err.max())


def test_statistics():
    from scipy import stats
    n, a, steps, seed = 65536, 12, 8, 77
    c = _cfg(n)
    gid = np.arange(n, dtype=np.uint64)
    zs = np.stack([_draw(c, _bufs(seed=seed, offset=s), n, a).double().cpu().numpy() for s in range(steps)])   # (8, n, a)
    flat = zs.reshape(-1, a)
    m = flat.shape[0]
    for j in range(a):
        col = flat[:, j]
        assert stats.kstest(col, "norm").pvalue > 1e-4, j
        assert abs(col.mean()) < 5.0 / np.sqrt(m), j
        assert abs(col.var() - 1.0) < 5.0 * np.sqrt(2.0 / m), j
        for t, p in ((2.0, 2.0 * stats.norm.sf(2.0)), (3.0, 2.0 * stats.norm.sf(3.0))):
            k = int((np.abs(col) > t).sum())
            assert abs(k - m * p) < 5.0 * np.sqrt(m * p * (1 - p)), (j, t, k, m * p)
    assert np.abs(flat).max() <= ZMAX
    lim = 5.0 / np.sqrt(n)
    r = np.corrcoef(zs[0].T)                                                # between columns
    assert np.abs(r - np.eye(a)).max() < lim, r
    for s in range(steps - 1):                                              # consecutive steps
        for j in range(a):
            assert abs(np.corrcoef(zs[s, :, j], zs[s + 1, :, j])[0, 1]) < lim, (s, j)
    for s in (0, 5):                                                        # streams 0 and 4 at the same key
        for stream in (0, 4):
            u = _u01(_philox_block(seed, s, gid, stream)[0]).astype(np.float64)
            for j in range(a):
                assert abs(np.corrcoef(zs[s, :, j], u)[0, 1]) < lim, (s, stream, j)
    assert not np.array_equal(zs[0], zs[1])


# ---------------------------------------------------------------------------------------------------- 3. keys and sharding
def test_captured_launch_draws_the_eager_keys():
    n, a, seed = 4099, 12, 99
    dev = "cuda:0"
    c = _cfg(n)
    base = torch.zeros(1, dtype=torch.long, device=dev)
    mean, std = torch.randn(n, a, device=dev), 0.5 + torch.rand(a, device=dev)
    outs = [torch.empty(n, a, device=dev), torch.empty(n, device=dev), torch.empty(n, a, device=dev), torch.empty(n, a, device=dev)]
    bg = _bufs(seed=seed, offset=0, step_base=base)                  # step = *step_base
    _launch(c, bg, mean, std, None, *outs)                           # eager first: the kernel is loaded before capture
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.graph(gr, stream=s):
        _launch(c, bg, mean, std, None, *outs)
    torch.cuda.current_stream().wait_stream(s)
    prev = None
    for counter in (0, 40, 41, 1 << 34):
        base.fill_(counter)
        gr.replay()
        eager = [torch.empty_like(t) for t in outs]
        _launch(c, _bufs(seed=seed, offset=counter), mean, std, None, *eager)
        for x, y in zip(outs, eager):
            assert torch.equal(_bits(x), _bits(y)), counter
        if prev is not None:
            assert not torch.equal(prev, outs[0])
        prev = outs[0].clone()


def test_two_shards_equal_one_big_env():
    n, a, seed, step = 8192, 12, 5, 17
    dev = "cuda:0"
    mean, std = torch.randn(n, a, device=dev), 0.3 + torch.rand(n, a, device=dev)
    big = [torch.empty(n, a, device=dev), torch.empty(n, device=dev), torch.empty(n, a, device=dev), torch.empty(n, a, device=dev)]
    _launch(_cfg(n), _bufs(seed=seed, offset=step), mean, std, None, *big)
    h = n // 2
    for lo, hi in ((0, h), (h, n)):
        sh = [torch.empty(hi - lo, a, device=dev), torch.empty(hi - lo, device=dev), torch.empty(hi - lo, a, device=dev),
              torch.empty(hi - lo, a, device=dev)]
        _launch(_cfg(n, offset=lo), _bufs(seed=seed, offset=step), mean[lo:hi].contiguous(), std[lo:hi].contiguous(), None, *sh)
        for x, y in zip(big, sh):
            assert torch.equal(_bits(x[lo:hi]), _bits(y)), lo


# ---------------------------------------------------------------------------------------------------- 4. slots, no sync
def _small_env(n=2048):
    from isaacgymloco_b200 import config as C, synthetic as S
    from test_gpu_keyed_domain_rand import _keyed_env
    cfg = C.aliengo("flat", num_envs=n)
    hf = S.make_terrain(cfg, seed=1)
    return _keyed_env(cfg, S.make_state(cfg, n, hf, seed=9), hf)


def test_storage_slots_and_no_sync(monkeypatch):
    from isaacgymloco_b200 import _lib as L
    from isaacgymloco_b200.policy_sampling import keyed_act
    from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
    env = _small_env()
    n, a, dev = env.num_envs, 12, env.device
    mean = torch.randn(n, a, device=dev)
    std = torch.nn.Parameter(torch.full((a,), 0.7, device=dev))
    sa, sb = (HIMRolloutStorage(n, 3, [45], [None], [a], device=dev) for _ in range(2))
    seen = []
    record = L.lib.hl_record_transition

    def spy(t, n_, stream):
        tr = t._obj
        seen.append((tr.actions, tr.actions_out, tr.log_prob, tr.log_prob_out, tr.mu, tr.mu_out, tr.sigma, tr.sigma_out))
        return record(t, n_, stream)

    monkeypatch.setattr(L.lib, "hl_record_transition", spy)
    for k in range(3):
        ta, tb = HIMRolloutStorage.Transition(), HIMRolloutStorage.Transition()
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            got_a = keyed_act(env, mean, std, ta)                 # new tensors, then the four record copies
            got_b = keyed_act(env, mean, std, tb, sb)             # the slots: same counter, so the same draw
            keyed_act(env, mean, std, z=torch.zeros(n, a, device=dev))
        finally:
            torch.cuda.set_sync_debug_mode(0)
        assert got_a.data_ptr() != sa.actions[k].data_ptr() and ta.actions_log_prob.shape == (n,)
        assert got_b.data_ptr() == sb.actions[k].data_ptr() and tb.actions is got_b
        assert tb.actions_log_prob.data_ptr() == sb.actions_log_prob[k].data_ptr() and tb.actions_log_prob.shape == (n,)
        assert tb.action_mean.data_ptr() == sb.mu[k].data_ptr() and tb.action_sigma.data_ptr() == sb.sigma[k].data_ptr()
        seen.clear()
        sa.add_transitions(ta)
        assert all(seen[0]), "the path without storage copies all four"
        seen.clear()
        sb.add_transitions(tb)
        assert not any(seen[0]), "the slot outputs are not copied"
        env.step(got_a)
    for f in ("actions", "actions_log_prob", "mu", "sigma"):
        assert torch.equal(_bits(getattr(sa, f)), _bits(getattr(sb, f))), f
    assert torch.equal(sa.mu[0], mean) and (sa.sigma == 0.7).all() and not torch.equal(sa.actions[0], sa.actions[1])


# ---------------------------------------------------------------------------------------------------- 5. replay == eager
class _Policy(torch.nn.Module):
    """A small actor MLP with a std parameter (HIMActorCritic's shape of things) and a linear critic."""

    def __init__(self, obs_dim, priv_dim, dev):
        super().__init__()
        g = torch.Generator().manual_seed(3)
        self.actor = torch.nn.Sequential(torch.nn.Linear(obs_dim, 64), torch.nn.ELU(), torch.nn.Linear(64, 12)).to(dev)
        self.critic = torch.nn.Linear(priv_dim, 1).to(dev)
        with torch.no_grad():
            for p in self.parameters():
                p.copy_(0.1 * torch.randn(p.shape, generator=g))
        self.std = torch.nn.Parameter(torch.full((12,), 0.8, device=dev))


def _make_runner(task, n, eager, t_len):
    from test_gpu_rollout_schedule import GAMMA, _Runner
    from isaacgymloco_b200.policy_sampling import keyed_act

    class Runner(_Runner):
        def body(self, k):
            env, tr = self.env, self.tr
            env.episode_sums["tracking_lin_vel"].mul_(self.keep).add_(self.boost)
            pol = self.pol
            with torch.no_grad():
                keyed_act(env, pol.actor(env.obs_buf), pol.std, tr, self.st)
                tr.values = pol.critic(env.privileged_obs_buf)
            tr.observations, tr.critic_observations = env.obs_buf, env.privileged_obs_buf
            act = tr.actions
            if self.eager:
                obs, priv, rew, done, extras, ids, term = env.step(act)
                self.st.record_env_step(tr, rew, done, extras, priv, ids, term, GAMMA)
                m = ids.numel()
                self.ids[k, :m].copy_(ids)
                self.cnt[k] = m
                self.term[k, :m].copy_(term)
                if m:
                    self.ep.append({key: (v.clone() if isinstance(v, torch.Tensor) else v) for key, v in extras["episode"].items()})
            else:
                obs, priv, rew, done, extras, ids, n_dev, term, _ = env.step_device(act)
                self.st.record_env_step(tr, rew, done, extras, priv, ids, term, GAMMA, termination_count=n_dev)
                self.ids[k].copy_(ids)
                self.cnt[k:k + 1].copy_(n_dev)
                self.term[k].copy_(term)

        def finish(self):
            with torch.no_grad():
                self.last_values.copy_(self.pol.critic(self.env.privileged_obs_buf))
            super().finish()

    return Runner(_rollout_env(task, n), eager=eager, t_len=t_len)


@pytest.mark.parametrize("task,n", [("flat", 4096), ("stairs", 16385)])
def test_replay_equals_eager_with_a_stochastic_policy(task, n):
    """keyed_domain_rand on, capture_schedule=True, T = 20, pushes every 30 and the curriculum every 50 (host interval),
    and an Adam step on the actor and the std between rollouts: every rollout of RolloutGraph.run() equals the eager
    public-step() loop in every storage field."""
    from test_gpu_rollout_schedule import _compare
    from isaacgymloco_b200.rollout_graph import env_schedule, rollout_window
    tt = 20
    a, b = _make_runner(task, n, True, tt), _make_runner(task, n, False, tt)
    pol = a.pol = b.pol = _Policy(a.env.obs_buf.shape[1], a.env.num_privileged_obs, a.env.device)
    for e in (a.env, b.env):
        e.push_interval = 30
        e.max_episode_length = 50
    opt = torch.optim.Adam(list(pol.actor.parameters()) + [pol.std], lr=1e-2)
    rg = b.env.capture_rollout(b.body, tt, storage=b.st, finish=b.finish, capture_schedule=True)
    boost = {2: 1e3, 4: -1e3}
    keys = set()
    for r in range(7):
        for run in (a, b):
            run.keep.fill_(0.0 if r in boost else 1.0)
            run.boost.fill_(boost.get(r, 0.0))
        keys.add(rollout_window(b.env.common_step_counter, tt, **env_schedule(b.env), in_graph=True)[0])
        ra = a.rollout_eager()
        rb = rg.run()
        _compare(a, b, ra, rb, f"rollout {r}")
        for f in ("values", "actions_log_prob", "mu", "sigma"):
            assert torch.equal(_bits(getattr(a.st, f)), _bits(getattr(b.st, f))), (r, f)
        assert torch.equal(b.st.sigma, (b.st.mu * 0. + pol.std.detach()))
        assert not torch.equal(b.st.actions, b.st.mu)
        assert rg.last_mode == "eager" if r == 0 else rg.last_mode in ("replay", "capture+replay"), (r, rg.last_mode)
        # an in-place optimizer step on the actor and the std: the captured graph reads the new values
        opt.zero_grad()
        obs, act = a.st.observations.flatten(0, 1), a.st.actions.flatten(0, 1)
        loss = ((pol.actor(obs) - act) ** 2).mean() + 0.1 * (pol.std ** 2).sum()
        loss.backward()
        opt.step()
        a.st.clear()
        b.st.clear()
    assert rg.stats["eager"] == 1 and rg.stats["replays"] == 6
    assert any(k[1] for k in keys) and any(k[2] for k in keys)
    assert not torch.equal(pol.std.detach(), torch.full_like(pol.std, 0.8))


def test_two_replays_draw_different_actions():
    """One captured graph replayed twice from the same state (counters 0 and 8): the actions differ."""
    from isaacgymloco_b200.policy_sampling import keyed_act
    n, tt = 4096, 8
    env = _rollout_env("flat", n)
    pol = _Policy(env.obs_buf.shape[1], env.num_privileged_obs, env.device)
    rec = torch.zeros(tt, n, 12, device=env.device)

    def body(k):
        with torch.no_grad():
            act = keyed_act(env, pol.actor(env.obs_buf), pol.std)
        env.step_device(act)
        rec[k].copy_(act)

    state = {k: v.clone() for k, v in vars(env).items() if isinstance(v, torch.Tensor) and not k.endswith("_ws")
             and k != "_step_base"}
    with torch.no_grad():
        mean = pol.actor(state["obs_buf"])        # also sets cuBLAS up before the capture
    rg = env.capture_rollout(body, tt, warmup=0, capture_schedule=True)
    outs = []
    for r in range(2):
        for k, v in state.items():
            getattr(env, k).copy_(v)
        rg.run()
        outs.append(rec.clone())
    assert rg.stats == {"replays": 2, "captures": 1, "eager": 0}
    assert not torch.equal(outs[0][0], outs[1][0])
    z0, z1 = (outs[0][0] - mean) / 0.8, (outs[1][0] - mean) / 0.8
    assert z0.abs().max() <= ZMAX * 1.001 and z1.abs().max() <= ZMAX * 1.001 and 0.9 < z0.std().item() < 1.1
