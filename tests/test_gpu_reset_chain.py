"""-m gpu: every launch path of post_physics_step() with the in-kernel reset (no reset hook overridden) against the
oracle run as eager torch on the same GPU, fed the same noise and reset uniforms.

The paths (legged_robot.py post_physics_step_device): the fused kernel emitting ids itself (<= 16,384 envs); the fused
kernel -> hl_select_and_terminal -> hl_reset_and_fixup (larger shards: the benchmarked chain); HL_MERGED_RESET=1
(ids, terminal rows, reset and fix-up in one launch); the persistent fused kernel; the push step (staged frame ->
_push_robots -> staged rest -> hl_reset_idx -> targeted re-scan); the command-curriculum step.  Every step checks the
ids, terrain levels, terminal rows, the whole snapshot, the re-drawn state and extras["episode"] (means against a
float64 restatement of LR:346-350), including steps where no env and where every env resets, ragged sizes
(n % 4 != 0) and the boundary of the high-speed command slice (num_envs a multiple of 5).
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _attach_terrain(env, ter):
    env.custom_origins = True
    env.env_origins = ter["env_origins"].to(DEV).contiguous()
    env.terrain_origins = ter["origins"].to(DEV).contiguous()
    env.terrain_types = ter["types"].to(DEV).contiguous()
    env.max_terrain_level = env.cfg_hot.num_rows
    env.refresh_buffers()


class Chain:
    """A FusedLeggedRobot and an OracleEnv on the same seeded state, stepped together."""

    def __init__(self, task, n, seed=71, marks=True, push=False):
        from isaacgymloco_b200 import synthetic as S
        from isaacgymloco_b200.legged_robot import FusedLeggedRobot
        from oracle import torch_oracle as O
        from oracle.make_goldens import reset_inputs
        cfg, hf, state, _, ter, _ = reset_inputs(dict(task=task, n=n, seed=seed))
        cfg.reset.push_robots = push
        cfg.reset.disturbance = push
        if marks:                                           # these hit the 500-step resampling mark on steps 1, 2
            state["episode_length_buf"][: n // 16] = 498
            state["episode_length_buf"][n // 16: n // 8] = 499
        self.cfg, self.hf, self.n, self.seed = cfg, hf, n, seed
        self.env = FusedLeggedRobot(cfg, state, hf, device=DEV)
        _attach_terrain(self.env, ter)
        assert self.env._kernel_reset_ok() and self.env.resample_interval == 500
        self.oenv = O.OracleEnv(cfg, S.to_device(state, DEV), hf.to(DEV))
        self.oenv.env_origins = ter["env_origins"].to(DEV).clone()
        self.oter = dict(origins=ter["origins"].to(DEV), types=ter["types"].to(DEV), max_level=cfg.num_rows,
                         env_length=cfg.terrain_length, max_episode_length_s=cfg.episode_length_s)
        self.total = 0
        self.reset_steps = 0
        self.history = []          # per step: (extras["episode"] object, float64 reference means or None)

    def both(self, fn):
        fn(self.env)
        fn(self.oenv)

    def step(self, step, mutate=None, push_vel=None, curriculum=False):
        from gpu_helpers import assert_close, assert_equal, compare_snapshots
        from isaacgymloco_b200 import config as C, synthetic as S
        env, oenv, n, cfg = self.env, self.oenv, self.n, self.cfg
        g = torch.Generator().manual_seed(500 + step)
        u = torch.rand(n, C.RESET_NU, generator=g).to(DEV)
        noise = S.make_noise(n, seed=600 + step)
        fresh = S.make_state(cfg, n, self.hf, seed=self.seed, step=step + 1)
        for k in ("contact_forces", "rigid_body_states", "actions"):        # (root / dof rows carry the reset draws forward)
            getattr(env, k).view(-1).copy_(fresh[k].view(-1).to(DEV))
            getattr(oenv, k).view(-1).copy_(fresh[k].view(-1).to(DEV))
        if mutate is not None:
            self.both(mutate)
        env.set_noise_tensors(**noise)
        env.set_reset_uniforms(u)
        prev_episode = env.extras.get("episode")
        # ---- oracle: LR:612-613 resampling on the mark (old ranges), the step, reset_idx with the same uniforms
        mark = ((oenv.episode_length_buf + 1) % 500 == 0).nonzero(as_tuple=False).flatten()
        oenv.resample_commands(mark, u, cfg.reset)
        nz = S.to_device(noise, DEV)
        oids, oterm, oamp = oenv.pre_reset(nz, push_vel=push_vel)
        if curriculum:
            _command_curriculum(oenv, oids, cfg)
        want = _episode_means_f64(oenv, oids) if len(oids) else None
        oenv.reset_idx_draw(oids, u, custom_origins=True, terrain=self.oter)
        oenv.apply_reset(oids, {})
        oenv.post_reset(nz)
        # ---- the public call
        ids, term_obs, term_amp = env.post_physics_step()
        self.total += len(ids)
        assert_equal(ids, oids, f"env_ids step {step}")
        assert_equal(env.terrain_levels, oenv.terrain_levels, f"terrain_levels step {step}")
        assert_close(term_obs, oterm, f"termination_privileged_obs step {step}")
        assert_close(term_amp, oamp, f"terminal_amp_states step {step}")
        compare_snapshots(env.snapshot(), oenv.snapshot())
        for k in ("root_states", "dof_state", "env_origins", "Kp_factors", "Kd_factors", "motor_strength_factors"):
            assert_close(getattr(env, k).reshape(getattr(oenv, k).shape), getattr(oenv, k), f"{k} step {step}", rtol=1e-6, atol=1e-6)
        ep = env.extras.get("episode")
        if want is None:
            assert ep is prev_episode, f"step {step} without resets replaced extras['episode']"
            self.history.append((ep, self.history[-1][1] if self.history else None))
            return oids
        self.reset_steps += 1
        assert ep is not prev_episode, f"step {step}: extras['episode'] is the previous step's dict"
        _check_means(ep, want, f"step {step}")
        level = oenv.terrain_levels.double().mean().item()          # LR:352-353, after this step's curriculum moves
        assert abs(float(ep["terrain_level"]) - level) <= 1e-6 * level + 1e-9, (float(ep["terrain_level"]), level)
        assert ep["max_command_x"] == oenv.command_ranges["lin_vel_x"][1]
        self.history.append((ep, want))
        return oids


def _episode_means_f64(oenv, ids):
    """LR:346-350 in float64 from the oracle's sums before apply_reset zeroes them:
    mean_e(sums[k, e] / max(len_e, 1) / dt) -> {name: (mean, mean_e |x_e|)}."""
    length = oenv.episode_length_buf[ids].double().clamp(min=1)
    out = {}
    for name in oenv.sum_names:
        x = oenv.episode_sums[name][ids].double() / length / oenv.dt
        out[name] = (x.mean().item(), x.abs().mean().item())
    return out


def _check_means(ep, want, what):
    """The kernel rounds each per-env quotient in fp32 (<= 2 ulp) and the mean once."""
    for name, (m, mabs) in want.items():
        got = float(ep["rew_" + name])
        assert abs(got - m) <= 1e-6 * mabs + 1e-9, f"{what} rew_{name}: {got} vs {m} (mean |x| {mabs})"


def _command_curriculum(oenv, ids, cfg):
    """LR:868-880 on the oracle's command ranges (the reset draws of this step see the widened ranges)."""
    R = cfg.reset
    mean = torch.mean(oenv.episode_sums["tracking_lin_vel"][ids]) / cfg.max_episode_length
    if float(mean) > 0.8 * oenv.term_scales["tracking_lin_vel"]:
        cr = oenv.command_ranges
        clip = lambda v, lo, hi: float(min(max(v, lo), hi))
        cr["lin_vel_x"][0] = clip(cr["lin_vel_x"][0] - 0.1, -R.max_backward_curriculum, 0.)      # np.clip of LR:877-880
        cr["lin_vel_x"][1] = clip(cr["lin_vel_x"][1] + 0.1, 0., R.max_forward_curriculum)
        cr["lin_vel_y"][0] = clip(cr["lin_vel_y"][0] - 0.1, -R.max_lat_curriculum, 0.)
        cr["lin_vel_y"][1] = clip(cr["lin_vel_y"][1] + 0.1, 0., R.max_lat_curriculum)


def _quiet(e):
    """No termination cause on this step: no base contact, no time-out, inside the border, not falling."""
    e.contact_forces[:, e.termination_contact_indices, :] = 0.0
    e.episode_length_buf.clamp_(max=e.cfg.max_episode_length - 10)
    e.root_states[:, 9].clamp_(min=-1.0)


def _everyone_times_out(e):
    e.episode_length_buf.fill_(e.cfg.max_episode_length)


# ------------------------------------------------------------------------------------------------ 1. the benchmarked chain
def test_bench_chain_65536_vs_oracle():
    """flat, 65,536 envs: fused (non-compact, resampling folded in) -> hl_select_and_terminal -> hl_reset_and_fixup."""
    ch = Chain("flat", 65536)
    assert not ch.env.single_launch
    for step in range(6):
        ch.step(step)
    assert ch.total > 6 and ch.reset_steps == 6 and ch.env.common_step_counter == 6


# ------------------------------------------------------------------------------------------------ 2. slice boundary, ragged size
@pytest.mark.parametrize("task,n", [("stairs", 16385), ("flat", 4100)])
def test_high_speed_slice_boundary_vs_oracle(task, n):
    """num_envs a multiple of 5: env n // 5 is the first env outside the high-speed slice (LR:649).  It and its
    neighbours are resampled on the mark (step 1, in the fused kernel) and re-drawn by a time-out reset (step 3).
    16,385 is also n % 4 != 0 (no aligned sums, no TMA) and the first size with the separate compaction launch;
    4,100 is a single-launch size."""
    ch = Chain(task, n)
    assert ch.env.single_launch == (n <= 16384) and n % 5 == 0
    b = slice(n // 5 - 1, n // 5 + 2)

    def on_mark(e):
        e.episode_length_buf[b] = 498

    def time_out(e):
        e.episode_length_buf[b] = e.cfg.max_episode_length

    ch.both(on_mark)
    for step in range(6):
        oids = ch.step(step, mutate=time_out if step == 3 else None)
        if step == 3:
            assert set(range(n // 5 - 1, n // 5 + 2)) <= set(oids.tolist())
    assert ch.reset_steps == 6


# ------------------------------------------------------------------------------------------------ 3. merged reset launch
@pytest.mark.parametrize("n", [65536, 16385])
def test_merged_reset_vs_oracle(n, monkeypatch):
    """HL_MERGED_RESET=1: ids, terminal rows, reset_idx and the fix-up in one launch after the fused kernel."""
    monkeypatch.setenv("HL_MERGED_RESET", "1")
    ch = Chain("flat", n)
    assert not ch.env.single_launch
    for step in range(6):
        ch.step(step)
    assert ch.total > 6 and ch.reset_steps == 6


# ------------------------------------------------------------------------------------------------ 4. persistent fused kernel
@pytest.mark.parametrize("n", [65536, 4096])
def test_persistent_kernel_with_kernel_reset_vs_oracle(n, monkeypatch):
    """HL_FUSED_IMPL=persist under the in-kernel reset: non-compact at 65,536, compact (ids from the kernel) at 4,096."""
    from isaacgymloco_b200 import _lib as L
    monkeypatch.setenv("HL_FUSED_IMPL", "persist")
    ch = Chain("flat", n)
    assert ch.env.single_launch == (n <= 16384)
    for step in range(6):
        ch.step(step)
        assert int(L.lib.hl_fused_last_impl()) == 1
    assert ch.total > 6 and ch.reset_steps == 6


# ------------------------------------------------------------------------------------------------ 5. push and disturbance steps
@pytest.mark.parametrize("n", [4096, 65536])
def test_push_and_disturbance_steps_vs_oracle(n):
    """push_interval 4 from step counter 2: pushes on counters 4 and 8, the disturbance on 8 (LR:624-632).  The hooks
    write fixed seeded tensors, so the oracle can be handed the same ones; the reset stays in the kernel."""
    ch = Chain("flat", n, push=True)
    env, oenv = ch.env, ch.oenv
    env.push_interval = 4
    env.common_step_counter = oenv.common_step_counter = 2
    g = torch.Generator().manual_seed(77)
    mv = ch.cfg.reset.max_push_vel_xy
    lo, hi = ch.cfg.reset.disturbance_range
    push_v = {c: ((2 * mv) * torch.rand(n, 2, generator=g) - mv).to(DEV) for c in (4, 8)}
    dist_v = {8: ((hi - lo) * torch.rand(n, 3, generator=g) + lo).to(DEV)}
    pushes, dists = [], []

    def push():
        pushes.append(env.common_step_counter)
        env.root_states[:, 7:9] = push_v[env.common_step_counter]

    def disturb():
        dists.append(env.common_step_counter)
        env.disturbance[:, 0, :] = dist_v[env.common_step_counter]

    env._push_robots, env._disturbance_robots = push, disturb
    assert env._kernel_reset_ok()
    for step in range(6):
        c = env.common_step_counter + 1

        def disturbed(e):
            if c in dist_v:
                e.disturbance[:, 0, :] = dist_v[c]

        ch.step(step, mutate=disturbed, push_vel=push_v.get(c))
    assert pushes == [4, 8] and dists == [8] and env.common_step_counter == 8
    assert ch.reset_steps == 6


# ------------------------------------------------------------------------------------------------ 6. command curriculum step
@pytest.mark.parametrize("n", [4096, 65536])
def test_command_curriculum_step_vs_oracle(n):
    """Step counter 1000 (= max_episode_length): update_command_curriculum widens the ranges before the reset launch
    (LR:306-307,868-880).  The reset draws of that step use the widened ranges; the pre-step resampling on the mark of
    the same step still uses the old ones."""
    ch = Chain("flat", n)
    env, oenv, cfg = ch.env, ch.oenv, ch.cfg
    env.common_step_counter = oenv.common_step_counter = cfg.max_episode_length - 2
    old_x = list(env.command_ranges["lin_vel_x"])

    def rich(e):                                            # every env tracked its command well: widen
        e.episode_sums["tracking_lin_vel"].fill_(100.0)

    for step in range(6):
        curriculum = env.common_step_counter + 1 == cfg.max_episode_length
        oids = ch.step(step, mutate=rich if curriculum else None, curriculum=curriculum)
        if curriculum:
            assert (oids < n // 5).any()
            assert oenv.command_ranges["lin_vel_x"][1] > old_x[1]
        assert env.command_ranges == oenv.command_ranges
    assert env.command_ranges["lin_vel_x"][1] == old_x[1] + 0.1
    assert ch.reset_steps == 6


# ------------------------------------------------------------------------------------------------ 7. edge steps
@pytest.mark.parametrize("n,merged", [(65536, False), (65536, True), (1, False), (33, False)])
def test_no_reset_and_all_reset_steps_vs_oracle(n, merged, monkeypatch):
    """Step 2: no env resets (extras['episode'] stays the previous step's dict).  Step 4: every env times out (at
    65,536: 65,536 terminal rows, the full grid-stride of the reset launch, means over every env)."""
    if merged:
        monkeypatch.setenv("HL_MERGED_RESET", "1")
    ch = Chain("flat", n)
    assert ch.env.single_launch == (n <= 16384)
    for step in range(6):
        if step == 0 and n < 64:
            oids = ch.step(step, mutate=_everyone_times_out)        # so the quiet step has a dict to keep
        elif step == 2:
            oids = ch.step(step, mutate=_quiet)
            assert len(oids) == 0
        elif step == 4:
            oids = ch.step(step, mutate=_everyone_times_out)
            assert len(oids) == n
        else:
            ch.step(step)
    assert ch.reset_steps >= 2 and (n < 64 or ch.reset_steps == 5)


# ------------------------------------------------------------------------------------------------ 9. runner-style collection
def test_runner_collects_each_steps_episode_means():
    """The reference runners keep infos['episode'] of every step (on_policy_runner: ep_infos.append(infos['episode'])):
    each kept entry must still hold its own step's means after later steps ran."""
    ch = Chain("flat", 65536)
    kept = []
    for step in range(8):
        ch.step(step, mutate=_quiet if step == 5 else None)
        if "episode" in ch.env.extras:
            kept.append(ch.env.extras["episode"])
    assert len(kept) == 8 and kept[5] is kept[4]
    for step, (ep, want) in enumerate(ch.history):
        assert kept[step] is ep
        _check_means(ep, want, f"kept entry of step {step}")
    distinct = {float(ep["rew_tracking_lin_vel"]) for ep in kept}
    assert len(distinct) >= 6
