"""-m gpu: the runners' episode statistics on the device (EpisodeStats, hl_episode_stats) against the runners' own block.

* One launch per step equals the block below, run as torch on the same device, at 4,096, 16,385 and 65,536 envs:
  cur_reward_sum / cur_episode_length bit for bit after every step, and rewbuffer / lenbuffer as lists of Python floats
  for maxlen 1, 100 and 5,000 (the ring wraps within a step and across steps), for both id forms and with collect()
  after every step, every 7 steps and once at the end.  Rewards are signed, up to 1e30 in magnitude and subnormal;
  steps have no resets, every env resetting, 2 % resetting and more resets than maxlen.
* A replayed rollout (capture_rollout(..., episode_stats=stats)) fills the deques as the public step() loop with the
  block does, over push and curriculum windows, with and without capture_schedule; a replayed run() syncs once.  The
  eager loop with record() and one collect() per rollout matches too.
* The hybrid (AMP) loop, summing the AMP reward.
* record() captured alone in a CUDA graph and replayed K times equals K eager calls, the ring cursor included; it
  allocates nothing and does not sync.
"""
import warnings
from collections import deque

import pytest
import torch

from test_gpu_amp_rollout import _AmpRunner, _amp_policy, _disc, _normalizer
from test_gpu_rollout_graph import GAMMA, _make_env, _policy, _Runner

pytestmark = pytest.mark.gpu


class _Reference:
    """The runners' bookkeeping (him_on_policy_runner.py, hybrid_runner.py), verbatim."""

    def __init__(self, num_envs, dev, maxlen=100):
        self.rewbuffer = deque(maxlen=maxlen)
        self.lenbuffer = deque(maxlen=maxlen)
        self.cur_reward_sum = torch.zeros(num_envs, dtype=torch.float, device=dev)
        self.cur_episode_length = torch.zeros(num_envs, dtype=torch.float, device=dev)

    def step(self, rewards, dones):
        rewbuffer, lenbuffer = self.rewbuffer, self.lenbuffer
        cur_reward_sum, cur_episode_length = self.cur_reward_sum, self.cur_episode_length
        cur_reward_sum += rewards
        cur_episode_length += 1
        new_ids = (dones > 0).nonzero(as_tuple=False)
        rewbuffer.extend(cur_reward_sum[new_ids][:, 0].cpu().numpy().tolist())
        lenbuffer.extend(cur_episode_length[new_ids][:, 0].cpu().numpy().tolist())
        cur_reward_sum[new_ids] = 0
        cur_episode_length[new_ids] = 0


def _bits(t):
    return t.view(torch.int32)


def _assert_same(ref, stats, what, deques=True):
    assert torch.equal(_bits(ref.cur_reward_sum), _bits(stats.cur_reward_sum)), f"{what}: cur_reward_sum"
    assert torch.equal(_bits(ref.cur_episode_length), _bits(stats.cur_episode_length)), f"{what}: cur_episode_length"
    if deques:
        assert list(stats.rewbuffer) == list(ref.rewbuffer), f"{what}: rewbuffer"
        assert list(stats.lenbuffer) == list(ref.lenbuffer), f"{what}: lenbuffer"


def _rewards(n, g):
    r = torch.randn(n, generator=g) * 10.0
    pick = torch.randint(0, 4, (n,), generator=g)
    r = torch.where(pick == 1, torch.randn(n, generator=g) * 1e30, r)
    r = torch.where(pick == 2, torch.randn(n, generator=g) * 1e-39, r)      # fp32 subnormals (normal >= 1.18e-38)
    return r.float()


@pytest.mark.parametrize("n", [4096, 16385, 65536])
def test_launch_equals_the_runner_block(n):
    from isaacgymloco_b200.episode_stats import EpisodeStats
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(n)
    maxlens = (1, 100, 5000)
    refs = {m: _Reference(n, dev, m) for m in maxlens}
    cadences = {"every step": 1, "every 7 steps": 7, "at the end": 0}
    objs = {(m, form, cad): EpisodeStats(n, dev, maxlen=m) for m in maxlens for form in ("exact", "capacity")
            for cad in cadences}
    ids_cap = torch.empty(n, dtype=torch.long, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    kinds = ["2%", "none", "2%", "all", "2%", "more than maxlen", "2%"]
    steps = 40
    subnormal = False
    for k in range(steps):
        kind = kinds[k % len(kinds)]
        rewards = _rewards(n, g)
        subnormal = subnormal or bool(((rewards != 0) & (rewards.abs() < 1.1754944e-38)).any())
        rewards = rewards.to(dev)
        u = torch.rand(n, generator=g)
        p = {"none": 0.0, "all": 1.0, "2%": 0.02, "more than maxlen": 0.4}[kind]
        dones = (u < p).to(dev)
        ids = dones.nonzero().flatten()
        m = ids.numel()
        if kind == "more than maxlen":
            assert m > 100
        ids_cap.copy_(torch.randint(0, n, (n,), generator=g))          # the tail past the count is never read
        ids_cap[:m] = ids
        cnt.fill_(m)
        for (ml, form, cad), st in objs.items():
            if form == "exact":
                st.record(rewards, dones, ids)
            else:
                st.record(rewards, dones.view(torch.uint8), ids_cap, cnt)
        for ref in refs.values():
            ref.step(rewards, dones)
        for (ml, form, cad), st in objs.items():
            what = f"n={n} step {k} ({kind}) maxlen={ml} {form} ids, collect {cad}"
            every = cadences[cad]
            collect = every > 0 and (k + 1) % every == 0
            if collect:
                st.collect()
            _assert_same(refs[ml], st, what, deques=collect)
    assert subnormal
    for (ml, form, cad), st in objs.items():
        st.collect()
        _assert_same(refs[ml], st, f"n={n} end maxlen={ml} {form} ids, collect {cad}")
        assert len(st.rewbuffer) == ml and st._cursor[1].item() == 0


class _StatsRunner(_Runner):
    """_Runner plus the runner's episode statistics.  mode "reference": the public step() and the verbatim block
    (its syncs included); "eager": the public step() and EpisodeStats.record() with the exact ids; "graph":
    step_device() and record() with the capacity-N ids and the device count, inside a RolloutGraph."""

    def __init__(self, env, mode, t_len, maxlen=100):
        from isaacgymloco_b200.episode_stats import EpisodeStats
        super().__init__(env, eager=mode != "graph", t_len=t_len)
        self.mode = mode
        self.ref = _Reference(env.num_envs, env.device, maxlen) if mode == "reference" else None
        self.stats = None if mode == "reference" else EpisodeStats(env.num_envs, env.device, maxlen)

    def body(self, k):
        env, tr = self.env, self.tr
        if self.mode == "graph":
            super().body(k)
            self.stats.record(env.rew_buf, env.reset_buf, self.ids[k], self.cnt[k:k + 1])
            return
        act = _policy(env.obs_buf)
        tr.observations, tr.critic_observations, tr.actions = env.obs_buf, env.privileged_obs_buf, act
        tr.values, tr.actions_log_prob, tr.action_mean, tr.action_sigma = self.values, self.logp, act, self.sigma
        obs, priv, rewards, dones, extras, ids, term = env.step(act)
        self.st.record_env_step(tr, rewards, dones, extras, priv, ids, term, GAMMA)
        if self.ref is not None:
            self.ref.step(rewards, dones)
        else:
            self.stats.record(rewards, dones, ids)


def _run_counting_syncs(rg, monkeypatch):
    """rg.run(), and the host syncs it made: explicit stream syncs plus the implicit ones torch reports."""
    explicit = [0]
    sync = torch.cuda.Stream.synchronize

    def counted(stream):
        explicit[0] += 1
        torch.cuda.set_sync_debug_mode(0)
        try:
            sync(stream)
        finally:
            torch.cuda.set_sync_debug_mode("warn")

    monkeypatch.setattr(torch.cuda.Stream, "synchronize", counted)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            rg.run()
        finally:
            torch.cuda.set_sync_debug_mode(0)
            monkeypatch.undo()
    implicit = sum("synchroniz" in str(w.message) for w in caught)
    return explicit[0] + implicit


@pytest.mark.parametrize("capture_schedule", [False, True])
def test_replayed_rollout_equals_the_runner_block(capture_schedule, monkeypatch):
    """T = 20 with a disturbance every 8 steps, the command curriculum every 70 and a push every 110 (host intervals),
    4,096 envs, 8 rollouts: warm-up, replays, curriculum and push windows (eager, or replayed with capture_schedule)."""
    from isaacgymloco_b200.episode_stats import EpisodeStats
    n, tt = 4096, 20
    envs = [_make_env("flat", n, push=True, curriculum=True) for _ in range(3)]
    for e in envs:
        e.push_interval = 110
        e.max_episode_length = 70
    ref, eager, graph = (_StatsRunner(e, mode, tt) for e, mode in zip(envs, ("reference", "eager", "graph")))
    with pytest.raises(ValueError):
        graph.env.capture_rollout(graph.body, tt, episode_stats=EpisodeStats(n - 1, graph.env.device))
    rg = graph.env.capture_rollout(graph.body, tt, storage=graph.st, finish=graph.finish,
                                   capture_schedule=capture_schedule, episode_stats=graph.stats)
    replay_syncs = []
    for r in range(8):
        ref.rollout_eager()
        eager.rollout_eager()
        eager.stats.collect()
        syncs = _run_counting_syncs(rg, monkeypatch)
        if rg.last_mode == "replay":
            replay_syncs.append(syncs)
        what = f"rollout {r} ({rg.last_mode})"
        assert torch.equal(ref.st.rewards, graph.st.rewards) and torch.equal(ref.st.dones, graph.st.dones), what
        _assert_same(ref.ref, eager.stats, f"{what}, eager record()")
        _assert_same(ref.ref, graph.stats, f"{what}, run()")
        if r == 0:
            assert len(ref.ref.rewbuffer) > 0
        for x in (ref, eager, graph):
            x.st.clear()
    assert rg.stats["replays"] == (7 if capture_schedule else 4), rg.stats
    # (without capture_schedule a host curriculum move changes the ranges, and every later window may recapture)
    assert all(s == 1 for s in replay_syncs) and (replay_syncs or not capture_schedule), replay_syncs


class _AmpStatsRunner(_AmpRunner):
    """_AmpRunner plus the hybrid runner's episode statistics, summing the AMP reward."""

    def __init__(self, env, eager, t_len, ring_rows, disc, norm):
        from isaacgymloco_b200.episode_stats import EpisodeStats
        super().__init__(env, eager, t_len, ring_rows, disc, norm)
        self.ref = _Reference(env.num_envs, env.device) if eager else None
        self.stats = None if eager else EpisodeStats(env.num_envs, env.device)

    def body(self, k):
        env, tr = self.env, self.tr
        act = _amp_policy(env.obs_buf, self.carried())
        tr.observations, tr.critic_observations, tr.actions = env.obs_buf, env.privileged_obs_buf, act
        tr.values, tr.actions_log_prob, tr.action_mean, tr.action_sigma = self.values, self.logp, act, self.sigma
        if self.eager:
            obs, priv, rew, dones, extras, ids, term, term_amp = env.step(act)
            next_amp_obs = env.get_amp_observations()
            next_amp_obs_with_term = next_amp_obs.clone()
            next_amp_obs_with_term[ids] = term_amp
            rewards = self.disc.predict_amp_reward(self.amp_obs, next_amp_obs_with_term, rew, self.norm)[0]
            self.rb.insert(self.amp_obs, next_amp_obs_with_term)
            self.amp_obs = next_amp_obs.clone()
            self.st.record_env_step(tr, rewards, dones, extras, priv, ids, term, GAMMA)
            self.ref.step(rewards, dones)
        else:
            obs, priv, rew, dones, extras, ids, n_dev, term, term_amp = env.step_device(act)
            rewards = self.amp.step(rew, ids, n_dev, term_amp)
            self.st.record_env_step(tr, rewards, dones, extras, priv, ids, term, GAMMA, termination_count=n_dev)
            self.stats.record(rewards, dones, ids, n_dev)


def test_amp_rollout_equals_the_runner_block():
    """The hybrid loop of tests/test_gpu_amp_rollout.py with capture_schedule=True: 4,096 envs, T = 20, 6 rollouts with
    normaliser updates and weight changes between them."""
    import copy
    n, tt, ring = 4096, 20, 150_001
    envs = [_make_env("amp", n, push=True, curriculum=True) for _ in range(2)]
    for e in envs:
        e.push_interval = 110
        e.max_episode_length = 70
    disc_a, norm_a = _disc(envs[0].device), _normalizer(envs[0].device)
    disc_b, norm_b = copy.deepcopy(disc_a), _normalizer(envs[1].device)
    a = _AmpStatsRunner(envs[0], True, tt, ring, disc_a, norm_a)
    b = _AmpStatsRunner(envs[1], False, tt, ring, disc_b, norm_b)
    rg = b.env.capture_rollout(b.body, tt, storage=b.st, finish=b.finish, capture_schedule=True, amp=b.amp,
                               episode_stats=b.stats)
    for r in range(6):
        a.rollout_eager()
        rg.run()
        what = f"rollout {r} ({rg.last_mode})"
        assert torch.equal(a.st.rewards, b.st.rewards), what
        _assert_same(a.ref, b.stats, what)
        a.between_rollouts(100 + r)
        b.between_rollouts(100 + r)
    assert len(a.ref.rewbuffer) > 0
    assert rg.stats["eager"] == 1 and rg.stats["replays"] == 5, rg.stats


def test_record_captures_and_replays():
    """record() alone in a CUDA graph, replayed K times, equals K eager calls (running sums, ring, cursor, deques); a
    capture executes nothing; eager calls allocate nothing on the device and do not sync."""
    from isaacgymloco_b200.episode_stats import EpisodeStats
    n, K, dev = 16385, 9, torch.device("cuda", 0)
    g = torch.Generator().manual_seed(7)
    rewards = _rewards(n, g).to(dev)
    dones = (torch.rand(n, generator=g) < 0.01).to(dev)              # ~164 per call: more than maxlen = 100
    ids = dones.nonzero().flatten()
    m = ids.numel()
    assert m > 100
    ids_cap = torch.randint(0, n, (n,), generator=g).to(dev)
    ids_cap[:m] = ids
    cnt = torch.tensor([m], dtype=torch.int32, device=dev)
    for args in ((rewards, dones, ids), (rewards, dones, ids_cap, cnt)):
        eager, graphed = EpisodeStats(n, dev), EpisodeStats(n, dev)
        torch.cuda.synchronize()
        allocs = torch.cuda.memory_stats()["allocation.all.allocated"]
        torch.cuda.set_sync_debug_mode("error")
        try:
            for _ in range(K):
                eager.record(*args)
        finally:
            torch.cuda.set_sync_debug_mode(0)
        assert torch.cuda.memory_stats()["allocation.all.allocated"] == allocs
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=s):
            graphed.record(*args)
        torch.cuda.current_stream().wait_stream(s)
        assert graphed.cur_episode_length.count_nonzero().item() == 0 and graphed._cursor.tolist() == [0, 0]
        for _ in range(K):
            gr.replay()
        what = f"{len(args)} arguments"
        assert torch.equal(_bits(eager.cur_reward_sum), _bits(graphed.cur_reward_sum)), what
        assert torch.equal(_bits(eager.cur_episode_length), _bits(graphed.cur_episode_length)), what
        assert torch.equal(eager._ring.view(torch.int32), graphed._ring.view(torch.int32)), what
        assert eager._cursor.tolist() == graphed._cursor.tolist() == [K * m, 0], what
        eager.collect()
        graphed.collect()
        assert list(eager.rewbuffer) == list(graphed.rewbuffer) and list(eager.lenbuffer) == list(graphed.lenbuffer)
        assert len(graphed.rewbuffer) == 100 and set(graphed.lenbuffer) == {1.0}
        del gr
    with pytest.raises(RuntimeError, match="CPU fallback"):
        eager.record(rewards.cpu(), dones, ids)
