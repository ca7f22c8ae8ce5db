"""-m gpu: RolloutGraph(capture_schedule=True) -- push and command-curriculum windows replayed too.

* hl_command_curriculum equals the host update_command_curriculum bit for bit on the float64 ranges (empty, small and
  full id lists, decisions far from the threshold, 20 moves into saturation) and, near the threshold, decides as the
  exact float64 mean does.
* Device ranges (HlReset.cmd_ranges) and by-value ranges give bit-identical commands, re-draws and observations on
  every launch path that draws commands; with the ranges changed on the device only, every path follows them.
* Replay equals eager across a schedule with disturbance, push and curriculum steps: after the warm-up every window
  replays, every rollout (command_ranges and the per-step episode logging included) equals the eager public-step()
  env, neither a curriculum move nor a host edit of command_ranges recaptures.
* The default torch _push_robots inside a replay draws fresh pushes on every replay.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GAMMA, LAM = 0.99, 0.95


def _physics(e, k):
    """Standalone 'physics': the PD torques move the joints (deterministic, device-only)."""
    e.dof_state.view(e.num_envs, 12, 2)[..., 0].add_(0.001 * e.torques)
    e.dof_state.view(e.num_envs, 12, 2)[..., 1].add_(0.01 * e.torques)


def _make_env(task, n, seed=11, disturbance=True, push=False, curriculum=False, torch_push=False):
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
    if not torch_push:
        env._push_robots = lambda: env.root_states[:, 7:9].copy_(0.5 * env.commands[:, :2])
    return env


def _policy(obs):
    return 0.5 * torch.tanh(obs[:, :12] + obs[:, 45:57])


# ---------------------------------------------------------------------------------------------------- 1. the curriculum launch
def _host_ranges_after(env, ids):
    """update_command_curriculum on a copy of the host ranges."""
    saved = {k: list(v) for k, v in env.command_ranges.items()}
    env.update_command_curriculum(ids)
    out = env.command_ranges_flat()
    for k, v in saved.items():
        env.command_ranges[k][:] = v
    return out


def _device_move(env, ids, log):
    m = ids.numel()
    env._reset_ids[:m].copy_(ids)
    env._n_reset.fill_(m)
    env._command_curriculum_device(log)
    got = tuple(env._cmd_ranges_dev.cpu().tolist())
    env._cmd_ranges_mirror = got          # what run() records after it copies the device ranges back
    return got


def test_command_curriculum_launch_matches_host():
    n = 4096
    env = _make_env("flat", n, curriculum=True)
    sums = env.episode_sums["tracking_lin_vel"]
    thr = 0.8 * env.reward_scales["tracking_lin_vel"]
    L = env.max_episode_length
    g = torch.Generator(device="cpu").manual_seed(5)
    env._upload_command_ranges()
    log = torch.full((8,), float("nan"), dtype=torch.float64, device=env.device)
    checked = 0
    for size in (0, 1, 33, n):
        for above in (True, False):
            ids = torch.randperm(n, generator=g)[:size].sort().values.to(env.device)
            scale = 4.0 if above else 0.25                       # mean / L = scale * thr: far from the threshold
            sums.copy_((scale * thr * L * (0.5 + torch.rand(n, generator=g))).to(env.device))
            want = _host_ranges_after(env, ids)
            got = _device_move(env, ids, log)
            assert got == want, (size, above, got, want)
            assert tuple(log.cpu().tolist()) == got
            env.set_command_ranges_flat(got)
            checked += 1
    # 20 moves from the reference ranges into saturation at max_forward / max_backward / max_lat
    R = env.cfg_hot.reset
    env.set_command_ranges_flat([-1.0, 1.0, -0.6, 0.6, -1.0, 1.0, -3.14, 3.14])
    env._upload_command_ranges()
    ids = torch.arange(0, n, 3, device=env.device)
    sums.fill_(3.0 * thr * L)
    for i in range(20):
        want = _host_ranges_after(env, ids)
        got = _device_move(env, ids, log)
        assert got == want, (i, got, want)
        env.set_command_ranges_flat(got)
    assert got[:4] == (-R.max_backward_curriculum, R.max_forward_curriculum, -R.max_lat_curriculum, R.max_lat_curriculum)
    # near the threshold: the device decision equals the exact float64 mean's, a few fp32 ulp either side
    ids = torch.arange(0, n, 2, device=env.device)
    x = (torch.rand(n, generator=g, dtype=torch.float64) * 2.0 * thr * L).to(torch.float32)
    sums.copy_(x.to(env.device))
    exact = float(np.sum(x.numpy()[::2].astype(np.float64))) / ids.numel() / L
    for rel, widens in ((-4e-7, True), (4e-7, False)):
        env.set_command_ranges_flat([-0.5, 0.5, -0.3, 0.3, -1.0, 1.0, -3.14, 3.14])
        env._upload_command_ranges()
        env.reward_scales["tracking_lin_vel"] = exact * (1.0 + rel) / 0.8
        assert (exact > 0.8 * env.reward_scales["tracking_lin_vel"]) == widens
        got = _device_move(env, ids, log)
        assert (got[1] > 0.5) == widens, (rel, got)
    assert checked == 8


# ---------------------------------------------------------------------------------------------------- 2. device == by-value ranges
NEW_RANGES = [0.4, 0.9, 0.25, 0.45, -0.2, 0.35, 0.5, 1.25]


@pytest.mark.parametrize("uniforms", [True, False], ids=["parity-uniforms", "philox"])
@pytest.mark.parametrize("task,n,env_var,push", [
    ("flat", 4096, None, False), ("stairs", 16385, None, False), ("flat", 65536, None, False),
    ("flat", 65536, "HL_FUSED_EPB=64", False), ("flat", 65536, "HL_FUSED_IMPL=persist", False),
    ("stairs", 16385, "HL_MERGED_RESET=1", False), ("flat", 4096, None, True)])
def test_device_ranges_match_by_value(task, n, env_var, push, uniforms, monkeypatch):
    """Env A reads the host ranges by value, env B (device-schedule mode) the device copy: 12 public steps (resets every
    step, the pre-step resampling of the fused kernel at step 10, a staged push step at step 5 when `push`), the
    standalone resampling in both forms, all bit-identical.  Then B's ranges change on the device only and A's host dict
    takes the same values: every consumer still agrees, so every one reads the pointer."""
    from isaacgymloco_b200 import _lib as L
    if env_var:
        monkeypatch.setenv(*env_var.split("="))
    a, b = (_make_env(task, n, disturbance=False, push=push) for _ in range(2))
    for e in (a, b):
        e.push_interval = 5
        if uniforms:
            e.set_reset_uniforms(torch.rand(n, 44, generator=torch.Generator().manual_seed(3)))
    b._upload_command_ranges()
    b._device_schedule = True
    ids = torch.arange(0, n, 7, device=a.device)

    def check(what):
        sa, sb = a.snapshot(), b.snapshot()
        for k in sa:
            assert torch.equal(sa[k], sb[k]), (what, k)
        for k in ("root_states", "dof_state", "commands", "Kp_factors", "Kd_factors", "motor_strength_factors"):
            assert torch.equal(getattr(a, k), getattr(b, k)), (what, k)

    def steps(tag):
        resets = 0
        for s in range(12):
            act = _policy(a.obs_buf)
            _, _, _, _, _, ia, _ = a.step(act)
            _, _, _, _, _, ib, _ = b.step(act)
            assert torch.equal(ia, ib)
            resets += ia.numel()
            check(f"{tag} step {s}")
        assert resets > 0
        for e in (a, b):
            e._resample_commands(ids)                                   # hl_resample_commands on an id list
            e.episode_length_buf[: n // 4] = 2 * e.resample_interval - 1
            e._pre_step_callbacks()                                      # ... and in its pre-step form
        check(f"{tag} standalone resampling")

    steps("same ranges")
    if env_var == "HL_FUSED_IMPL=persist":
        assert L.lib.hl_fused_last_impl() == 1
    b._cmd_ranges_dev.copy_(torch.tensor(NEW_RANGES, dtype=torch.float64))    # B's host dict keeps the old values
    a.set_command_ranges_flat(NEW_RANGES)
    for e in (a, b):
        e.episode_length_buf[: n // 8] = 3 * e.resample_interval - 1        # the fused kernel resamples these at step 0
    steps("device-only change")
    assert b.command_ranges_flat() != tuple(NEW_RANGES)
    # the ids resampled last drew from the new ranges: the heading (or yaw-rate) column has no keep filter
    col, (lo, hi) = (3, NEW_RANGES[6:8]) if b.cfg_hot.heading_command else (2, NEW_RANGES[4:6])
    c = b.commands[ids, col]
    assert (c >= lo - 1e-6).all() and (c <= hi + 1e-6).all(), (c.min(), c.max())
    fast = ids[ids < b._high_vel_envs]
    vx = b.commands[fast, 0]
    assert ((vx == 0) | ((vx >= NEW_RANGES[0] - 1e-6) & (vx <= NEW_RANGES[1] + 1e-6))).all() and (vx != 0).any()


# ---------------------------------------------------------------------------------------------------- 3. replay == eager
class _Runner:
    """A runner's rollout loop over one env + HIMRolloutStorage(env_writes_slots=True).  eager=True drives the public
    step() (ids sliced on the host, extras["episode"] per step); otherwise step_device() (device counts).  Before each
    step the body sets the tracking_lin_vel sums to `boost` when `keep` is 0 (far above / below the curriculum
    threshold); keep = 1, boost = 0 leaves them alone.  Both are device tensors, so a replay reads their current values."""

    def __init__(self, env, eager, t_len):
        from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
        n, dev = env.num_envs, env.device
        self.env, self.eager, self.t_len = env, eager, t_len
        env.extras["time_outs"] = env.time_out_buf
        self.st = HIMRolloutStorage(n, t_len, [270], [env.num_privileged_obs], [12], device=dev, env_writes_slots=True)
        env.bind_rollout(self.st)
        self.tr = HIMRolloutStorage.Transition()
        self.values, self.logp, self.sigma = torch.full((n, 1), 0.1, device=dev), torch.zeros(n, device=dev), torch.ones(n, 12, device=dev)
        self.last_values = torch.zeros(n, 1, device=dev)
        self.ids = torch.zeros(t_len, n, dtype=torch.long, device=dev)
        self.cnt = torch.zeros(t_len, dtype=torch.int32, device=dev)
        self.term = torch.zeros(t_len, n, env.num_privileged_obs, device=dev)
        self.keep, self.boost = torch.ones(1, device=dev), torch.zeros(1, device=dev)
        self.ep = []

    def body(self, k):
        env, tr = self.env, self.tr
        env.episode_sums["tracking_lin_vel"].mul_(self.keep).add_(self.boost)
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
    assert ea.command_ranges == eb.command_ranges, f"{what}: command_ranges"
    ca, cb = a.cnt.cpu().tolist(), b.cnt.cpu().tolist()
    assert ca == cb, f"{what}: reset counts"
    for k, m in enumerate(ca):
        assert torch.equal(a.ids[k, :m], b.ids[k, :m]), f"{what}: ids of step {k}"
        assert torch.equal(a.term[k, :m], b.term[k, :m]), f"{what}: terminal rows of step {k}"
    assert len(ra) == len(rb) == sum(1 for m in ca if m), f"{what}: episode infos per step"
    for x, y in zip(ra, rb):
        assert set(x) == set(y), what
        assert x["max_command_x"] == y["max_command_x"], (what, x["max_command_x"], y["max_command_x"])
        for key in x:
            u, v = float(x[key]), float(y[key])
            assert abs(u - v) <= 1e-6 * max(abs(u), abs(v)) + 1e-9, (what, key, u, v)   # float64 atomics: summation order


@pytest.mark.parametrize("task,n,env_var", [("flat", 4096, None), ("stairs", 16385, None),
                                            ("stairs", 16385, "HL_MERGED_RESET=1"), ("flat", 65536, "HL_FUSED_IMPL=persist")])
def test_schedule_replays_push_and_curriculum_windows(task, n, env_var, monkeypatch):
    """T = 20, a disturbance every 8 steps, a push every 110, the curriculum every 70 (host interval): after the warm-up
    every window replays (6 graphs for 11 windows) and equals the eager env.  Counter 70 widens the ranges, 140 does not,
    210 widens again; a host edit of command_ranges after rollout 7 is uploaded without a recapture."""
    from isaacgymloco_b200.rollout_graph import rollout_window, env_schedule
    if env_var:
        monkeypatch.setenv(*env_var.split("="))
    tt = 20
    a = _Runner(_make_env(task, n, push=True, curriculum=True), eager=True, t_len=tt)
    b = _Runner(_make_env(task, n, push=True, curriculum=True), eager=False, t_len=tt)
    for e in (a.env, b.env):
        e.push_interval = 110
        e.max_episode_length = 70             # host-side curriculum interval only (the kernels keep cfg's)
    rg = b.env.capture_rollout(b.body, tt, storage=b.st, finish=b.finish, capture_schedule=True)
    boost = {3: 1e3, 6: -1e3, 10: 1e3}        # rollouts with the curriculum steps at counters 70, 140, 210
    keys = set()
    x_hi = []
    for r in range(12):
        if r == 8:
            for e in (a.env, b.env):
                e.command_ranges["lin_vel_y"][1] += 0.25
        for run in (a, b):
            run.keep.fill_(0.0 if r in boost else 1.0)
            run.boost.fill_(boost.get(r, 0.0))
        key = rollout_window(b.env.common_step_counter, tt, **env_schedule(b.env), in_graph=True)[0]
        ra = a.rollout_eager()
        rb = rg.run()
        _compare(a, b, ra, rb, f"rollout {r}")
        if r == 0:
            assert (rg.last_mode, rg.last_reason) == ("eager", "warm-up")
        else:
            new = key not in keys
            keys.add(key)
            assert rg.last_mode == ("capture+replay" if new else "replay"), (r, rg.last_mode, rg.last_reason)
            assert rg.stats["captures"] == len(keys), (r, rg.stats, keys)       # one capture per key, never a recapture
        assert int(b.env._step_base.item()) == (r + 1) * tt
        x_hi.append(b.env.command_ranges["lin_vel_x"][1])
        a.st.clear()
        b.st.clear()
    assert rg.stats["eager"] == 1 and rg.stats["replays"] == 11 and len(rg._graphs) <= rg.max_graphs
    assert len(keys) == 6 and any(k[1] for k in keys) and any(k[2] for k in keys)
    assert x_hi[3] > x_hi[2] and x_hi[6] == x_hi[5] and x_hi[10] > x_hi[9], x_hi


# ---------------------------------------------------------------------------------------------------- 4. torch pushes in a replay
def test_default_push_in_replay_draws_fresh_velocities():
    """The default _push_robots (torch.rand) captured in a graph: two replays from the same state push differently,
    within +-max_push_vel_xy; the step after the push leaves the pushed velocities of the envs that did not reset alone."""
    n, tt = 4096, 10
    env = _make_env("flat", n, disturbance=False, push=True, torch_push=True)
    env.push_interval = 5
    rec = dict(vel=torch.zeros(tt, n, 2, device=env.device), ids=torch.zeros(tt, n, dtype=torch.long, device=env.device),
               cnt=torch.zeros(tt, dtype=torch.int32, device=env.device))

    def body(k):
        _, _, _, _, _, ids, n_dev, _, _ = env.step_device(_policy(env.obs_buf))
        rec["vel"][k].copy_(env.root_states[:, 7:9])
        rec["ids"][k].copy_(ids)
        rec["cnt"][k:k + 1].copy_(n_dev)

    state = {k: v.clone() for k, v in vars(env).items() if isinstance(v, torch.Tensor) and not k.endswith("_ws")
             and k != "_step_base"}
    rg = env.capture_rollout(body, tt, warmup=0, capture_schedule=True)
    outs = []
    for r in range(2):
        for k, v in state.items():
            getattr(env, k).copy_(v)
        rg.run()
        assert rg.last_mode in ("replay", "capture+replay")
        outs.append({k: v.clone() for k, v in rec.items()})
    assert rg.stats == {"replays": 2, "captures": 1, "eager": 0}
    mv = env.cfg_hot.reset.max_push_vel_xy
    vels = []
    for o in outs:
        kept = torch.ones(n, dtype=torch.bool, device=env.device)
        kept[o["ids"][4, :int(o["cnt"][4])]] = False                 # step 4 = counter 5 (push); resets re-draw the velocity
        v4 = o["vel"][4][kept]
        assert v4.abs().max() <= mv and v4.abs().max() > 0.5 * mv
        kept5 = kept.clone()
        kept5[o["ids"][5, :int(o["cnt"][5])]] = False                # step 5: no push
        assert torch.equal(o["vel"][5][kept5], o["vel"][4][kept5])
        vels.append(o["vel"][4])
    assert not torch.equal(vels[0], vels[1])
