"""-m gpu: a captured rollout replayed every iteration (FusedLeggedRobot.capture_rollout / RolloutGraph.run()).

* Replay equals eager, bit for bit: env A runs R rollouts through the public step(); env B, built from the same seed
  and state, captures once and runs the same rollouts through RolloutGraph.run().  After every rollout the snapshot,
  the PhysX-side state, the curriculum / gain-factor state and the storage slots agree; every step's reset ids and
  terminal rows agree; the per-step episode logging matches extras["episode"] of the eager steps.
* Fresh draws: two consecutive replays from the same state draw different observation noise, resampled commands and
  reset states, and replay r equals the eager steps rT .. rT+T-1 (the keys come from the device counter).
* Schedule: windows with a push step or a command-curriculum step run eagerly, disturbance steps out of alignment
  with the rollout use a second cached graph, a change of the command ranges recaptures -- and each still equals the
  eager env and leaves the counters right.
* A sampled torch policy inside `body` captures (no host sync), fills the storage and acts differently per replay.

The torch-RNG hooks (action delay, disturbances, pushes) are replaced with deterministic ones here, so the library's
in-kernel Philox is the only source of randomness in the comparisons.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

T = 24
GAMMA, LAM = 0.99, 0.95


def _physics(e, k):
    """Standalone 'physics': the PD torques move the joints (deterministic, device-only)."""
    e.dof_state.view(e.num_envs, 12, 2)[..., 0].add_(0.001 * e.torques)
    e.dof_state.view(e.num_envs, 12, 2)[..., 1].add_(0.01 * e.torques)


def _make_env(task, n, seed=11, disturbance=True, push=False, curriculum=False):
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    from oracle.make_goldens import reset_inputs
    cfg, hf, state, _, ter, _ = reset_inputs(dict(task=task, n=n, seed=seed))
    cfg.reset.delay = False                       # _delay_actions without torch.randint
    cfg.reset.disturbance = disturbance
    cfg.reset.push_robots = push
    cfg.reset.commands_curriculum = curriculum
    state["episode_length_buf"][: n // 16] = 490  # these cross the 500-step resampling mark inside the first rollout
    env = FusedLeggedRobot(cfg, state, hf, device="cuda:0", physics_step_fn=_physics, seed=seed)
    env.custom_origins = True
    env.env_origins = ter["env_origins"].to(env.device).contiguous()
    env.terrain_origins = ter["origins"].to(env.device).contiguous()
    env.terrain_types = ter["types"].to(env.device).contiguous()
    env.max_terrain_level = cfg.num_rows
    env.refresh_buffers()
    # deterministic stand-ins for the torch-RNG hooks (they read device state only, so a replay stays exact)
    env._disturbance_robots = lambda: env.disturbance[:, 0, :].copy_(50.0 * env.base_lin_vel)
    env._push_robots = lambda: env.root_states[:, 7:9].copy_(0.5 * env.commands[:, :2])
    return env


def _policy(obs):
    return 0.5 * torch.tanh(obs[:, :12] + obs[:, 45:57])


class _Runner:
    """A runner's rollout loop over one env + HIMRolloutStorage(env_writes_slots=True).  eager=True drives the public
    step() (ids sliced on the host, extras["episode"] per step); otherwise step_device() (device counts)."""

    def __init__(self, env, eager, t_len=T):
        from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
        n, dev = env.num_envs, env.device
        self.env, self.eager, self.t_len = env, eager, t_len
        env.extras["time_outs"] = env.time_out_buf    # (the reference's extras carry it once the first reset happened)
        self.st = HIMRolloutStorage(n, t_len, [270], [env.num_privileged_obs], [12], device=dev, env_writes_slots=True)
        env.bind_rollout(self.st)
        self.tr = HIMRolloutStorage.Transition()
        self.values, self.logp, self.sigma = torch.full((n, 1), 0.1, device=dev), torch.zeros(n, device=dev), torch.ones(n, 12, device=dev)
        self.last_values = torch.zeros(n, 1, device=dev)
        self.ids = torch.zeros(t_len, n, dtype=torch.long, device=dev)
        self.cnt = torch.zeros(t_len, dtype=torch.int32, device=dev)
        self.term = torch.zeros(t_len, n, env.num_privileged_obs, device=dev)
        self.ep = []                              # eager: extras["episode"] of the steps with resets

    def body(self, k):
        env, tr = self.env, self.tr
        act = _policy(env.obs_buf)
        tr.observations, tr.critic_observations, tr.actions = env.obs_buf, env.privileged_obs_buf, act
        tr.values, tr.actions_log_prob, tr.action_mean, tr.action_sigma = self.values, self.logp, act, self.sigma
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
        self.st.compute_returns(self.last_values, GAMMA, LAM)

    def rollout_eager(self):
        self.ep = []
        for k in range(self.t_len):
            self.body(k)
        self.finish()
        return self.ep


def _compare(a, b, ra, rb, what):
    ea, eb = a.env, b.env
    sa, sb = ea.snapshot(), eb.snapshot()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), f"{what}: {k}"
    for k in ("root_states", "dof_state", "commands", "terrain_levels", "env_origins", "Kp_factors", "Kd_factors",
              "motor_strength_factors", "disturbance"):
        assert torch.equal(getattr(ea, k), getattr(eb, k)), f"{what}: {k}"
    for k in ("_obs_all", "_priv_all", "rewards", "dones", "next_privileged_observations", "actions", "returns", "advantages"):
        assert torch.equal(getattr(a.st, k), getattr(b.st, k)), f"{what}: storage.{k}"
    assert a.st.step == b.st.step == a.t_len and ea.common_step_counter == eb.common_step_counter
    ca, cb = a.cnt.cpu().tolist(), b.cnt.cpu().tolist()
    assert ca == cb, f"{what}: reset counts"
    for k, m in enumerate(ca):
        assert torch.equal(a.ids[k, :m], b.ids[k, :m]), f"{what}: ids of step {k}"
        assert torch.equal(a.term[k, :m], b.term[k, :m]), f"{what}: terminal rows of step {k}"
    assert len(ra) == len(rb) == sum(1 for m in ca if m), f"{what}: episode infos per step"
    for x, y in zip(ra, rb):
        assert set(x) == set(y), what
        for key in x:
            u, v = float(x[key]), float(y[key])
            assert abs(u - v) <= 1e-6 * max(abs(u), abs(v)) + 1e-9, (what, key, u, v)   # float64 atomics: summation order


@pytest.mark.parametrize("task,n,env_var", [("flat", 4096, None), ("stairs", 16385, None), ("flat", 65536, None),
                                            ("stairs", 16385, "HL_MERGED_RESET=1"), ("flat", 65536, "HL_FUSED_IMPL=persist")])
def test_replay_equals_eager_bit_for_bit(task, n, env_var, monkeypatch):
    from isaacgymloco_b200 import _lib as L
    if env_var:
        monkeypatch.setenv(*env_var.split("="))
    a, b = _Runner(_make_env(task, n), eager=True), _Runner(_make_env(task, n), eager=False)
    rg = b.env.capture_rollout(b.body, T, storage=b.st, finish=b.finish)
    for r in range(4):
        ra = a.rollout_eager()
        rb = rg.run()
        _compare(a, b, ra, rb, f"rollout {r}")
        assert rg.last_mode == ("eager" if r == 0 else "capture+replay" if r == 1 else "replay"), (r, rg.last_mode)
        a.st.clear()
        b.st.clear()
    assert rg.stats == {"replays": 3, "captures": 1, "eager": 1}
    assert b.env.common_step_counter == 4 * T and int(b.env._step_base.item()) == 4 * T
    if env_var == "HL_FUSED_IMPL=persist":
        assert L.lib.hl_fused_last_impl() == 1


def _state_tensors(env):
    """Every tensor the step mutates (the look-back workspaces and the device counter excepted)."""
    return {k: v for k, v in vars(env).items() if isinstance(v, torch.Tensor) and not k.endswith("_ws") and k != "_step_base"}


def test_consecutive_replays_draw_fresh_keys():
    """Two replays of one graph from the same state, at counters 0 and T: different observation noise, resampled
    commands and reset states (at the parent commit the keys repeat and they are equal); each equals the eager steps
    with the same keys."""
    n = 4096

    def recorder(env):
        rec = dict(obs=torch.zeros(T, n, 270, device=env.device), cmd=torch.zeros(T, n, 4, device=env.device),
                   root=torch.zeros(T, n, 13, device=env.device), ids=torch.zeros(T, n, dtype=torch.long, device=env.device),
                   cnt=torch.zeros(T, dtype=torch.int32, device=env.device))

        def body(k):
            _, _, _, _, _, ids, n_dev, _, _ = env.step_device(_policy(env.obs_buf))
            rec["obs"][k].copy_(env.obs_buf)
            rec["cmd"][k].copy_(env.commands)
            rec["root"][k].copy_(env.root_states)
            rec["ids"][k].copy_(ids)
            rec["cnt"][k:k + 1].copy_(n_dev)
        return rec, body

    env = _make_env("flat", n)
    start = {k: v.clone() for k, v in _state_tensors(env).items()}
    rec, body = recorder(env)
    rg = env.capture_rollout(body, T, warmup=0)
    outs = []
    for r in range(2):
        for k, v in _state_tensors(env).items():
            v.copy_(start[k])
        rg.run()
        outs.append({k: v.clone() for k, v in rec.items()})
    assert rg.stats == {"replays": 2, "captures": 1, "eager": 0} and env.common_step_counter == 2 * T
    o1, o2 = outs
    assert torch.equal(o1["cnt"][0], o2["cnt"][0])                        # same state, same terminations at step 0
    assert not torch.equal(o1["obs"][0, :, :45], o2["obs"][0, :, :45])    # obs noise (stream 0)
    assert torch.equal(o1["obs"][0, :, 45:], o2["obs"][0, :, 45:])        # the history slots carry no new noise
    m = int(o1["cnt"][0])
    ids = o1["ids"][0, :m]
    assert m > 0 and not torch.equal(o1["root"][0][ids], o2["root"][0][ids])   # reset re-draws (stream 3)
    marked = torch.arange(n // 16, device=env.device)                     # cross the resampling mark at step 9
    reset = torch.cat([o["ids"][k, :int(o["cnt"][k])] for o in outs for k in range(10)])
    keep = marked[~torch.isin(marked, reset)]                            # (an env that reset restarts its episode)
    assert keep.numel() > 0
    assert torch.equal(o1["cmd"][8][keep, :2], o2["cmd"][8][keep, :2])
    assert not torch.equal(o1["cmd"][9][keep, :2], o2["cmd"][9][keep, :2])  # pre-step resampling (stream 2)
    # replay r == the eager steps rT .. rT+T-1 from the same state
    for r in range(2):
        e = _make_env("flat", n)
        e.common_step_counter = r * T
        rec_e, body_e = recorder(e)
        for k in range(T):
            body_e(k)
        for key in rec_e:
            assert torch.equal(rec_e[key], outs[r][key]), (r, key)


def test_schedule_runs_push_and_curriculum_windows_eagerly():
    """T = 20 with a disturbance every 8 steps, the command curriculum every 70 steps (host interval) and a push every
    110: push / curriculum windows run eagerly, the two disturbance alignments use two graphs, a range change
    recaptures; every rollout equals the eager env and leaves the counters right."""
    n, tt = 4096, 20
    a = _Runner(_make_env("flat", n, push=True, curriculum=True), eager=True, t_len=tt)
    b = _Runner(_make_env("flat", n, push=True, curriculum=True), eager=False, t_len=tt)
    for e in (a.env, b.env):
        e.push_interval = 110
        e.max_episode_length = 70             # host-side curriculum interval only (the kernels keep cfg's)
    rg = b.env.capture_rollout(b.body, tt, storage=b.st, finish=b.finish)
    # windows: counters 1-20, 21-40 (disturbances at steps 3, 11, 19), 41-60 (7, 15), 61-80 (curriculum at 70),
    # 81-100 (7, 15; the curriculum may have moved the ranges), 101-120 (push at 110), 121-140 (curriculum at 140),
    # 141-160 (3, 11, 19, after a range change)
    want = [("eager", "warm-up"), ("capture+replay", None), ("capture+replay", None),
            ("eager", "command-curriculum step at counter 70"), (None, None), ("eager", "push step at counter 110"),
            ("eager", "command-curriculum step at counter 140"), ("capture+replay", None)]
    for r, (mode, reason) in enumerate(want):
        if r == 7:
            for e in (a.env, b.env):
                e.command_ranges["lin_vel_y"][1] += 0.25
        ra = a.rollout_eager()
        rb = rg.run()
        _compare(a, b, ra, rb, f"rollout {r}")
        if mode is not None:
            assert (rg.last_mode, rg.last_reason) == (mode, reason), (r, rg.last_mode, rg.last_reason)
        else:
            assert rg.last_mode in ("replay", "capture+replay"), (r, rg.last_mode)
        assert a.env.common_step_counter == b.env.common_step_counter == (r + 1) * tt
        assert int(b.env._step_base.item()) == (r + 1) * tt
        a.st.clear()
        b.st.clear()
    assert rg.stats["eager"] == 4 and rg.stats["replays"] == 4 and rg.stats["captures"] >= 3
    assert len(rg._graphs) == 2


def test_sampled_policy_in_the_loop():
    """A torch MLP policy with Normal sampling inside body: captures without a host sync, fills the storage, and the
    replays sample different actions (PyTorch's graph-safe Philox)."""
    from torch.distributions import Normal
    n = 4096
    env = _make_env("flat", n)
    r = _Runner(env, eager=False)
    torch.manual_seed(3)
    net = torch.nn.Sequential(torch.nn.Linear(270, 64), torch.nn.ELU(), torch.nn.Linear(64, 12)).to(env.device)
    std = torch.full((12,), 0.3, device=env.device)

    def body(k):
        with torch.no_grad():
            mu = net(env.obs_buf)
            dist = Normal(mu, std.expand_as(mu), validate_args=False)    # argument validation would sync
            act = dist.rsample()          # loc + scale * N(0,1); sample()'s torch.normal(loc, scale) checks scale on the host
            r.tr.observations, r.tr.critic_observations, r.tr.actions = env.obs_buf, env.privileged_obs_buf, act
            r.tr.values, r.tr.actions_log_prob = r.values, dist.log_prob(act).sum(dim=-1)
            r.tr.action_mean, r.tr.action_sigma = mu, dist.stddev
            obs, priv, rew, done, extras, ids, n_dev, term, _ = env.step_device(act)
            r.st.record_env_step(r.tr, rew, done, extras, priv, ids, term, GAMMA, termination_count=n_dev)

    rg = env.capture_rollout(body, T, storage=r.st, finish=r.finish)
    acts = []
    for _ in range(3):
        rg.run()
        assert r.st.step == T
        acts.append(r.st.actions.clone())
        assert r.st._obs_all[1:].abs().sum(dim=(1, 2)).min() > 0 and r.st.actions.abs().sum(dim=(1, 2)).min() > 0
        assert torch.isfinite(r.st.returns).all() and torch.isfinite(r.st.actions_log_prob).all()
        r.st.clear()
    assert rg.stats == {"replays": 2, "captures": 1, "eager": 1}
    assert not torch.equal(acts[1], acts[2])
