"""-m gpu: the AMP env-step of the hybrid runner as one launch (hl_amp_transition) and inside a replayed rollout
(AMPRolloutStep + capture_rollout(..., amp=...)).

* One launch equals the public pieces it replaces -- get_amp_observations, clone + index_put of the terminal rows with
  the host ids, AMPDiscriminator.assemble_input, ReplayBuffer.insert, clone -- bit for bit: x, every ring row, the
  device cursor against the host step / num_samples, the carried amp_obs and the reward; x also equals the oracle's
  amp_disc_input.  Steps of the real chain, steps without resets and with every env reset, wrapping inserts into a
  ring whose size is not a multiple of N, normalizer=None, var = 0 and values landing exactly on +-clip.
* A replayed AMP rollout equals the runner's eager block over several rollouts (the ring wraps), with a normaliser
  update (it rebinds its tensors) and an in-place weight change between rollouts.
* Replays after the warm-up, a recapture when a discriminator layer is rebound, and N > ring rows rejected.

The torch-RNG hooks are replaced with deterministic ones (tests/test_gpu_rollout_graph.py), so in-kernel Philox and the
seeded discriminator are the only sources of randomness.
"""
import copy

import numpy as np
import pytest
import torch

from test_gpu_rollout_graph import _make_env, _policy

pytestmark = pytest.mark.gpu

GAMMA, LAM = 0.99, 0.95


def _disc(dev, hidden=(256, 128), seed=3):
    from isaacgymloco_b200.amp_discriminator import AMPDiscriminator
    torch.manual_seed(seed)
    return AMPDiscriminator(60, 2.0, list(hidden), dev, task_reward_lerp=0.3)


def _normalizer(dev, seed=4):
    from isaacgymloco_b200.amp_discriminator import Normalizer
    norm = Normalizer(30, device=dev)
    g = torch.Generator().manual_seed(seed)
    for _ in range(2):
        norm.update((torch.randn(512, 30, generator=g) * 0.7 + 0.2).to(dev))
    return norm


def _amp_policy(obs, amp_obs):
    return _policy(obs) + 0.1 * torch.tanh(amp_obs[:, :12])


@pytest.mark.parametrize("n", [4096, 16385, 65536])
def test_transition_equals_public_composition(n):
    from isaacgymloco_b200 import _lib as L
    from isaacgymloco_b200.amp_rollout import AMPRolloutStep
    from isaacgymloco_b200.replay_buffer import ReplayBuffer
    from oracle import torch_oracle as O
    env = _make_env("amp", n)
    dev = env.device
    disc, norm = _disc(dev), _normalizer(dev)
    size = 2 * n + n // 2 + 3                 # not a multiple of N: the third insert wraps
    rb_a, rb_b = ReplayBuffer(30, size, dev), ReplayBuffer(30, size, dev)
    steps = {True: AMPRolloutStep(env, disc, norm, rb_b), False: AMPRolloutStep(env, disc, None, rb_b)}
    steps[True].begin()
    steps[False].amp_obs = steps[True].amp_obs          # one carried observation, whichever launch runs the step
    amp_obs_a = env.get_amp_observations()
    g = torch.Generator().manual_seed(n)
    cases = ["chain", "none", "all", "chain", "no-normalizer", "clip-edge", "chain", "all"]
    for j, case in enumerate(cases):
        if case == "all":
            env.episode_length_buf.fill_(int(env.max_episode_length))      # every env times out in this step
        _, _, rew, _, _, ids, n_dev, _, term_amp = env.step_device(_amp_policy(env.obs_buf, amp_obs_a))
        if case == "none":
            env.reset_buf.zero_()
            n_dev.zero_()
        if case == "clip-edge":
            # integer joint positions, std exactly 1 on those columns and means 7 / -7: (v - mean) / std hits -10 / +10
            # exactly; var = 0 on the rest (std = sqrt(fp32(1e-4))) drives them far past the clip
            env.dof_state.view(n, 12, 2)[..., 0].copy_(torch.randint(-3, 4, (n, 12), generator=g).float().to(dev))
            norm.mean = torch.cat([torch.full((6,), 7.0), torch.full((6,), -7.0), torch.zeros(18)]).double().to(dev)
            norm.var = torch.cat([torch.full((12,), 1.0 - 1e-4, dtype=torch.float64), torch.zeros(18, dtype=torch.float64)]).to(dev)
        use_norm = case != "no-normalizer"
        normalizer = norm if use_norm else None
        amp = steps[use_norm]
        amp.refresh()
        r_b = amp.step(rew, ids, n_dev, term_amp).clone()
        # the runner's block on the public pieces
        m = int(n_dev.item())
        if case == "all":
            assert m == n
        next_amp_obs = env.get_amp_observations()
        nwt = next_amp_obs.clone()
        nwt[ids[:m]] = term_amp[:m]
        x_a = disc.assemble_input(amp_obs_a, nwt, normalizer)
        r_a = disc.predict_amp_reward(amp_obs_a, nwt, rew, normalizer)[0]
        rb_a.insert(amp_obs_a, nwt)
        x_o = (O.amp_disc_input(amp_obs_a, nwt, norm.mean.cpu().numpy(), norm.var.cpu().numpy()) if use_norm
               else torch.cat([amp_obs_a, nwt], dim=-1))
        amp_obs_a = next_amp_obs.clone()
        what = f"n={n} step {j} ({case})"
        assert torch.equal(amp.x, x_a), what
        assert torch.equal(x_a, x_o), what
        assert torch.equal(r_b, r_a), what
        assert torch.equal(amp.amp_obs, amp_obs_a), what
        assert torch.equal(rb_b.states, rb_a.states) and torch.equal(rb_b.next_states, rb_a.next_states), what
        assert (rb_b.step, rb_b.num_samples) == (rb_a.step, rb_a.num_samples), what
        assert amp._cursor.tolist() == [rb_a.step, rb_a.num_samples, 0], what
        if case == "clip-edge":
            assert (amp.x[:, 30:42] == 10.0).any() and (amp.x[:, 30:42] == -10.0).any(), "no value landed on the clip"
            assert (amp.x[:, 42:].abs() == 10.0).float().mean() > 0.5
    assert rb_a.num_samples == size and rb_a.step == (len(cases) * n) % size
    # the C entry point refuses more envs than ring rows
    small = ReplayBuffer(30, n - 1, dev)
    a = steps[True]
    rc = L.lib.hl_amp_transition(L.ptr(env.dof_state), L.ptr(env.base_lin_vel), L.ptr(env.base_ang_vel), L.ptr(env.reset_buf),
                                 L.ptr(env._reset_ids), L.ptr(env._n_reset), L.ptr(env._term_amp), None, 0.0, 0.0,
                                 L.ptr(a.amp_obs), L.ptr(a.x), L.ptr(small.states), L.ptr(small.next_states), n - 1,
                                 L.ptr(a._cursor), n, L.stream())
    assert rc != 0 and b"ring" in L.lib.hl_last_error()
    with pytest.raises(ValueError):
        AMPRolloutStep(env, disc, norm, small)


class _AmpRunner:
    """HybridPolicyRunner's rollout loop over one env.  eager=True: the public step() and the runner's AMP block
    verbatim (host ids, clone, index_put, predict_amp_reward, ReplayBuffer.insert, clone); otherwise step_device() and
    AMPRolloutStep.step()."""

    def __init__(self, env, eager, t_len, ring_rows, disc, norm):
        from isaacgymloco_b200.amp_rollout import AMPRolloutStep
        from isaacgymloco_b200.replay_buffer import ReplayBuffer
        from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
        n, dev = env.num_envs, env.device
        self.env, self.eager, self.t_len, self.disc, self.norm = env, eager, t_len, disc, norm
        env.extras["time_outs"] = env.time_out_buf
        self.st = HIMRolloutStorage(n, t_len, [270], [env.num_privileged_obs], [12], device=dev, env_writes_slots=True)
        env.bind_rollout(self.st)
        self.tr = HIMRolloutStorage.Transition()
        self.values, self.logp, self.sigma = torch.full((n, 1), 0.1, device=dev), torch.zeros(n, device=dev), torch.ones(n, 12, device=dev)
        self.last_values = torch.zeros(n, 1, device=dev)
        self.rb = ReplayBuffer(30, ring_rows, dev)
        if eager:
            self.amp_obs = env.get_amp_observations()
        else:
            self.amp = AMPRolloutStep(env, disc, norm, self.rb)
            self.amp.begin()

    def carried(self):
        return self.amp_obs if self.eager else self.amp.amp_obs

    def body(self, k):
        env, tr = self.env, self.tr
        act = _amp_policy(env.obs_buf, self.carried())
        tr.observations, tr.critic_observations, tr.actions = env.obs_buf, env.privileged_obs_buf, act
        tr.values, tr.actions_log_prob, tr.action_mean, tr.action_sigma = self.values, self.logp, act, self.sigma
        if self.eager:
            obs, priv, rew, done, extras, ids, term, term_amp = env.step(act)
            next_amp_obs = env.get_amp_observations()
            next_amp_obs_with_term = next_amp_obs.clone()
            next_amp_obs_with_term[ids] = term_amp
            rewards = self.disc.predict_amp_reward(self.amp_obs, next_amp_obs_with_term, rew, self.norm)[0]
            self.rb.insert(self.amp_obs, next_amp_obs_with_term)
            self.amp_obs = next_amp_obs.clone()
            self.st.record_env_step(tr, rewards, done, extras, priv, ids, term, GAMMA)
        else:
            obs, priv, rew, done, extras, ids, n_dev, term, term_amp = env.step_device(act)
            rewards = self.amp.step(rew, ids, n_dev, term_amp)
            self.st.record_env_step(tr, rewards, done, extras, priv, ids, term, GAMMA, termination_count=n_dev)

    def finish(self):
        self.st.compute_returns(self.last_values, GAMMA, LAM)

    def rollout_eager(self):
        for k in range(self.t_len):
            self.body(k)
        self.finish()

    def between_rollouts(self, seed):
        """The update's AMP side: one replay-buffer draw, Normalizer.update on it (rebinds mean / var), an in-place
        change of the discriminator's weights; returns the draw."""
        np.random.seed(seed)
        s, sn = next(self.rb.feed_forward_generator(1, 2048))
        self.norm.update(torch.cat([s, sn]))
        with torch.no_grad():
            for p in self.disc.parameters():
                p.mul_(0.98).add_(0.002)
        self.st.clear()
        return s, sn


@pytest.mark.parametrize("capture_schedule", [False, True])
def test_replayed_amp_rollout_equals_eager(capture_schedule):
    """T = 20 with a disturbance every 8 steps, the command curriculum every 70 steps and a push every 110 (host
    intervals), 4,096 envs, a 150,001-row ring (wraps on the 37th step and twice more); 7 rollouts."""
    n, tt, ring = 4096, 20, 150_001
    envs = [_make_env("amp", n, push=True, curriculum=True) for _ in range(2)]
    for e in envs:
        e.push_interval = 110
        e.max_episode_length = 70
    disc_a, norm_a = _disc(envs[0].device), _normalizer(envs[0].device)
    disc_b, norm_b = copy.deepcopy(disc_a), _normalizer(envs[1].device)
    a = _AmpRunner(envs[0], True, tt, ring, disc_a, norm_a)
    b = _AmpRunner(envs[1], False, tt, ring, disc_b, norm_b)
    rg = b.env.capture_rollout(b.body, tt, storage=b.st, finish=b.finish, capture_schedule=capture_schedule, amp=b.amp)
    wrapped = False
    for r in range(7):
        a.rollout_eager()
        rg.run()
        what = f"rollout {r} ({rg.last_mode})"
        sa, sb = a.env.snapshot(), b.env.snapshot()
        for k in sa:
            assert torch.equal(sa[k], sb[k]), f"{what}: {k}"
        # rewards included: the captured discriminator MLP runs the same cuBLAS kernels as the eager one on the B200
        for k in ("_obs_all", "_priv_all", "dones", "next_privileged_observations", "actions", "rewards", "returns",
                  "advantages"):
            assert torch.equal(getattr(a.st, k), getattr(b.st, k)), f"{what}: storage.{k}"
        assert torch.equal(b.amp._stats, torch.stack([norm_a.mean, norm_a.var])), what
        assert torch.equal(a.rb.states, b.rb.states) and torch.equal(a.rb.next_states, b.rb.next_states), what
        assert (a.rb.step, a.rb.num_samples) == (b.rb.step, b.rb.num_samples), what
        assert b.amp._cursor.tolist() == [a.rb.step, a.rb.num_samples, 0], what
        assert torch.equal(a.carried(), b.carried()), what
        assert a.env.common_step_counter == b.env.common_step_counter == (r + 1) * tt
        wrapped = wrapped or a.rb.num_samples == ring
        da, db = a.between_rollouts(100 + r), b.between_rollouts(100 + r)
        assert torch.equal(da[0], db[0]) and torch.equal(da[1], db[1]), f"{what}: feed_forward_generator draw"
        assert torch.equal(norm_a.mean, norm_b.mean) and torch.equal(norm_a.var, norm_b.var), what
    assert wrapped and a.rb.step == (7 * tt * n) % ring
    if capture_schedule:
        assert rg.stats["eager"] == 1 and rg.stats["replays"] == 6, rg.stats
    else:
        assert rg.stats["replays"] >= 3, rg.stats


def test_replays_and_recapture_on_rebound_layer():
    """After the warm-up every window replays; an in-place weight change or a normaliser update replays the same
    graph; rebinding a discriminator layer recaptures, and the rewards then come from the new layer."""
    from isaacgymloco_b200 import _lib as L
    n, tt = 4096, 12
    env = _make_env("amp", n, disturbance=False)
    disc, norm = _disc(env.device), _normalizer(env.device)
    b = _AmpRunner(env, False, tt, 10 * n + 1, disc, norm)
    rg = env.capture_rollout(b.body, tt, storage=b.st, finish=b.finish, amp=b.amp)
    modes = []
    for r in range(6):
        if r == 4:
            new = torch.nn.Linear(128, 1).to(env.device)
            with torch.no_grad():
                new.weight.copy_(-disc.amp_linear.weight)
                new.bias.copy_(disc.amp_linear.bias)
            disc.amp_linear = new
        rg.run()
        modes.append(rg.last_mode)
        # the last step's reward from its x, with the discriminator as it is now
        with torch.no_grad():
            d = disc(b.amp.x)
        want = torch.empty(n, device=env.device)
        L.check(L.lib.hl_amp_reward(L.ptr(d), L.ptr(env.rew_buf), 2.0, 0.3, L.ptr(want), n, L.stream()))
        torch.testing.assert_close(b.amp.reward, want, rtol=1e-5, atol=1e-6)
        assert (b.rb.step, b.rb.num_samples) == tuple(b.amp._cursor.tolist()[:2])
        b.between_rollouts(r)
    assert modes == ["eager", "capture+replay", "replay", "replay", "capture+replay", "replay"], modes
    assert rg.stats == {"replays": 5, "captures": 2, "eager": 1}
    assert b.amp.calls == 6 * tt and b.rb.step == (6 * tt * n) % (10 * n + 1)
