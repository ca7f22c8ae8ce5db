"""-m gpu: reset_idx's re-draws, the pre-step command resampling and the post-reset fix-up of every launch path against
the float64 reference of tests/reset_probe.py, on probe states that switch every branch of the reset side.

Within the bound |got - ref64| <= 1e-5 |ref64| + 1e-6 max_e |ref64[:, col]| (reward_probe's): root_states, dof_state,
commands and the three gain factors of the reset envs, and after the fix-up obs_buf[:, :45] and privileged_obs_buf.
Exact: terrain levels and origins, zeroed commands, u = 0 draws, the fallback fields, the clipped history, every
buffer of the envs a launch on an id list does not reset.  The three copies of the command arithmetic
(hl_resample_env, hl_resample_kernel, hl_fused_resample) agree bit for bit, and a launch with HlReset.parts set to
one part writes only that part's fields.
"""
import ctypes

import pytest
import torch

import reset_probe as RP

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
PUSH_VEL_SEED = 91


def _env(cfg, pr, cls=None, device_ranges=False):
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    env = (cls or FusedLeggedRobot)(cfg, pr["state"], pr["hf"], device=DEV)
    ter = pr["ter"]
    env.env_origins = ter["env_origins"].to(DEV).contiguous()
    if not cfg.is_plane:
        env.terrain_origins = ter["origins"].to(DEV).contiguous()
        env.terrain_types = ter["types"].to(DEV).contiguous()
        env.max_terrain_level = cfg.num_rows
    env.refresh_buffers()
    env.set_reset_uniforms(pr["u"])
    env.set_noise_tensors(**pr["noise"])
    if device_ranges:
        env._device_schedule = True
        env._upload_command_ranges()
    return env


WATCHED = ("root_states", "dof_state", "commands", "Kp_factors", "Kd_factors", "motor_strength_factors", "terrain_levels",
           "env_origins", "obs_buf", "privileged_obs_buf", "last_actions", "last_last_actions", "last_dof_pos",
           "last_dof_vel", "last_torques", "last_root_vel", "feet_air_time", "episode_length_buf", "reset_buf",
           "measured_heights", "disturbance")


def _rows(env):
    n = env.num_envs
    out = {k: getattr(env, k).detach().reshape(n, -1).clone() for k in WATCHED}
    out["episode_sums"] = env._episode_sums_buf.detach().T.clone()
    return out


def _assert_others_unchanged(before, env, ids, what):
    after = _rows(env)
    keep = torch.ones(env.num_envs, dtype=torch.bool, device=DEV)
    keep[ids.to(DEV)] = False
    for k, v in before.items():
        assert torch.equal(after[k][keep], v[keep]), f"{what}: {k} of an env off the reset list changed"


def _check(cfg, pr, env, what, pre_step, obs=True, push_vel=None):
    ref = RP.reference64_reset(cfg, pr, pre_step=pre_step, push_vel=push_vel, root32_after=env.root_states.detach().cpu())
    if pre_step:
        ids, n = env._reset_ids, int(env._n_reset.item())
        assert torch.equal(ids[:n].cpu(), ref.ids), f"{what}: reset ids"
        # the envs the step resampled on the mark and did not reset: the pre-step copy of the command arithmetic
        stay = pr["mark"].clone()
        stay[ref.ids] = False
        cols = [0, 1, 3 if cfg.heading_command else 2]
        if stay.any():
            RP.check_bound(env.commands.cpu()[stay][:, cols].T, ref.commands[stay][:, cols].T,
                           [f"commands[{c}]" for c in cols], f"{what}: commands resampled on the mark")
    RP.check_reset_rows(env, ref, ref.ids, what, obs=obs)
    bad = RP.exact_failures(cfg, pr, env, ref, obs=obs, shifted=pre_step)
    assert not bad, f"{what}:\n" + "\n".join(bad)
    return ref


# ------------------------------------------------------------------------------------------------ torch stand-ins of the hooks
def _hook_env(which):
    """A FusedLeggedRobot with one reset hook overridden by torch code that reads the same uniform table (LR:634-820 as
    the oracle restates them): the step then takes the hook fallback (fused -> sync -> reset_idx -> fix-up)."""
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot

    def dofs(self, ids):
        R, n, U = self.cfg_hot.reset, self.num_envs, self._reset_uniforms[ids]
        dp = self.dof_state.view(n, 12, 2)
        pr = R.dof_init_pos_ratio_range
        dp[ids, :, 0] = (self.default_dof_pos * ((pr[1] - pr[0]) * U[:, 0:12] + pr[0]) if pr is not None
                         else self.default_dof_pos.expand(len(ids), 12))
        r = R.dof_init_vel_range
        dp[ids, :, 1] = U[:, 12:24] * abs(r[1] - r[0]) + min(r) if R.randomize_dof_vel else 0.0

    def root(self, ids):
        R, U = self.cfg_hot.reset, self._reset_uniforms[ids]
        rng = lambda k, lohi: (lohi[1] - lohi[0]) * U[:, k] + lohi[0]
        rs = self.root_states
        rs[ids] = self.base_init_state
        rs[ids, :3] += self.env_origins[ids]
        if self.custom_origins:
            p = R.base_init_pos_range or dict(x=(-1.0, 1.0), y=(-1.0, 1.0), z=None)
            rs[ids, 0] += rng(24, p["x"])
            rs[ids, 1] += rng(25, p["y"])
            if p["z"] is not None:
                rs[ids, 2] += rng(26, p["z"])
        rr = R.base_init_rot_range
        if rr is not None:
            roll, pitch, yaw = rng(27, rr["roll"]), rng(28, rr["pitch"]), rng(29, rr.get("yaw", [-3.141592653589793, 3.141592653589793]))
            cy, sy, cr, sr = torch.cos(yaw * 0.5), torch.sin(yaw * 0.5), torch.cos(roll * 0.5), torch.sin(roll * 0.5)
            cp, sp = torch.cos(pitch * 0.5), torch.sin(pitch * 0.5)
            rs[ids, 3:7] = torch.stack([cy * sr * cp - sy * cr * sp, cy * cr * sp + sy * sr * cp,
                                        sy * cr * cp - cy * sr * sp, cy * cr * cp + sy * sr * sp], dim=-1)
        vr = R.base_init_vel_range
        for k, ax in enumerate(("x", "y", "z", "roll", "pitch", "yaw")):
            rs[ids, 7 + k] = rng(30 + k, vr[ax] if isinstance(vr, dict) else vr)

    def commands(self, ids):
        if len(ids) == 0:
            return
        U, cr, c = self._reset_uniforms[ids], self.command_ranges, self.commands
        rng = lambda k, lohi: (lohi[1] - lohi[0]) * U[:, k] + lohi[0]
        c[ids, 0] = rng(36, (-1.0, 1.0))
        c[ids, 1] = rng(37, cr["lin_vel_y"])
        if self.cfg_hot.heading_command:
            c[ids, 3] = rng(38, cr["heading"])
        else:
            c[ids, 2] = rng(38, cr["ang_vel_yaw"])
        hi = (ids + self.cfg_hot.env_id_offset) < self._high_vel_envs
        hid = ids[hi]
        c[hid, 0] = rng(39, cr["lin_vel_x"])[hi]
        c[hid, 1:2] *= (torch.norm(c[hid, 0:1], dim=1) < 1.0).unsqueeze(1)
        c[ids, :2] *= (torch.norm(c[ids, :2], dim=1) > 0.2).unsqueeze(1)

    name = {"dofs": "_reset_dofs", "root": "_reset_root_states", "commands": "_resample_commands"}[which]
    fn = {"dofs": dofs, "root": root, "commands": commands}[which]
    return type(f"Hook_{which}", (FusedLeggedRobot,), {name: fn})


# ------------------------------------------------------------------------------------------------ 1. every config through hl_reset_and_fixup
@pytest.mark.parametrize("task", RP.TASKS)
@pytest.mark.parametrize("variant", RP.VARIANTS)
def test_reset_idx_device_every_config_vs_float64(task, variant):
    """reset_idx_device(ids, fixup=True) at 4,099 envs: every task's ranges, the None / off fallbacks and the wide
    ranges; the envs off the list keep every buffer bit for bit."""
    cfg = RP.reset_cfg(task, variant, 4099)
    pr = RP.make_reset_probe(cfg, 4099)
    env = _env(cfg, pr)
    before = _rows(env)
    ids = pr["ids"].to(DEV)
    env.reset_idx_device(ids, fixup=True)
    _check(cfg, pr, env, f"{task} {variant}", pre_step=False)
    _assert_others_unchanged(before, env, ids, f"{task} {variant}")


# ------------------------------------------------------------------------------------------------ 2. the launch paths
PATHS = [
    # path, task, variant, n, reset share
    ("reset_idx", "flat", "wide", 7, 0.4),
    ("reset_idx", "stairs", "default", 65536, 0.4),
    ("reset_idx_fixup", "recover", "fallbacks", 16385, 1.0),
    ("reset_idx_fixup", "plane", "wide", 65536, 0.4),
    ("chain", "flat", "wide", 4099, 0.4),
    ("chain", "amp", "default", 4099, 0.0),
    ("chain", "recover", "wide", 7, 1.0),
    ("chain", "stairs", "default", 65536, 0.4),
    ("chain", "plane", "fallbacks", 16385, 1.0),
    ("chain_select", "recover", "wide", 4099, 0.4),
    ("chain_devranges", "flat", "wide", 4099, 0.4),
    ("chain_devranges", "stairs", "wide", 65536, 0.4),
    ("merged", "flat", "wide", 65536, 0.4),
    ("merged", "stairs", "default", 16385, 1.0),
    ("persist", "stairs", "wide", 4099, 0.4),
    ("persist", "flat", "default", 65536, 1.0),
    ("persist_devranges", "flat", "wide", 65536, 0.4),
    ("push", "flat", "wide", 4099, 0.4),
    ("push", "stairs", "default", 16385, 0.4),
    ("hook_dofs", "flat", "default", 4099, 0.4),
    ("hook_root", "recover", "default", 16385, 0.4),
    ("hook_root", "stairs", "fallbacks", 4099, 0.4),
    ("hook_commands", "flat", "wide", 4099, 0.4),
    ("hook_commands", "plane", "default", 4099, 1.0),
    ("post_reset_zero", "stairs", "default", 4099, 0.4),
    ("post_reset_zero", "flat", "wide", 65536, 0.4),
]


@pytest.mark.parametrize("path,task,variant,n,share", PATHS, ids=[f"{p}-{t}-{v}-{n}-{s}" for p, t, v, n, s in PATHS])
def test_launch_path_vs_float64(path, task, variant, n, share, monkeypatch):
    from isaacgymloco_b200 import _lib as L
    cfg = RP.reset_cfg(task, variant, n)
    pr = RP.make_reset_probe(cfg, n, reset_share=share)
    what = f"{path} {task} {variant} n={n}"
    if path.startswith("merged"):
        monkeypatch.setenv("HL_MERGED_RESET", "1")
    if path.startswith("persist"):
        monkeypatch.setenv("HL_FUSED_IMPL", "persist")
    cls = _hook_env(path[5:]) if path.startswith("hook_") else None
    env = _env(cfg, pr, cls, device_ranges=path.endswith("devranges"))
    if path in ("reset_idx", "reset_idx_fixup", "post_reset_zero"):
        before = _rows(env)
        ids = pr["ids"].to(DEV)
        if path == "post_reset_zero":            # draws (every part, no zeroing), then the fix-up with the zeroing
            env._reset_part(ids, 0)
            env._reset_ids[:len(ids)] = ids
            env._n_reset.fill_(len(ids))
            env.fused_post_reset(with_reset_zero=True)
        else:
            env.reset_idx_device(ids, fixup=path == "reset_idx_fixup")
        _check(cfg, pr, env, what, pre_step=False, obs=path != "reset_idx")
        _assert_others_unchanged(before, env, ids, what)
        return
    push_vel = None
    if path == "chain_select" or path.startswith("merged"):
        env.single_launch = False
        env.refresh_buffers()
    if path == "push":
        cfg.reset.push_robots = True
        env.push_interval = 1
        g = torch.Generator().manual_seed(PUSH_VEL_SEED)
        push_vel = (2 * torch.rand(n, 2, generator=g) - 1).to(DEV)
        env._push_robots = lambda: env.root_states[:, 7:9].copy_(push_vel)
    if path.startswith("hook_"):
        assert not env._kernel_reset_ok()
    else:
        assert env._kernel_reset_ok()
    env.post_physics_step()
    if path.startswith("persist"):
        assert int(L.lib.hl_fused_last_impl()) == 1
    _check(cfg, pr, env, what, pre_step=True, push_vel=push_vel)
    if share == 0:
        assert int(env._n_reset.item()) == 0


def test_shard_with_offset_vs_float64():
    """A shard with env_id_offset = 3,000 of 20,000 envs: its first 1,000 envs lie in the high-speed slice."""
    cfg = RP.reset_cfg("flat", "wide", 4099, num_envs=20000, env_id_offset=3000)
    pr = RP.make_reset_probe(cfg, 4099, reset_share=1.0)
    env = _env(cfg, pr)
    env.post_physics_step()
    _check(cfg, pr, env, "shard", pre_step=True)


# ------------------------------------------------------------------------------------------------ 3. the three resampling copies
@pytest.mark.parametrize("variant", ["default", "wide"])
@pytest.mark.parametrize("device_ranges", [False, True])
@pytest.mark.parametrize("task", ["flat", "recover"])
def test_resampling_copies_bit_equal(variant, device_ranges, task, monkeypatch):
    """Every env on the mark: hl_resample_commands (interval form and id form), hl_reset_draw with
    HL_RESET_COMMANDS (hl_resample_env) and the tiled and persistent fused kernels (hl_fused_resample) write the same
    bits into the resampled command columns, by value and from the device copy of the ranges; all within the bound of
    the float64 resample_commands."""
    from isaacgymloco_b200 import _lib as L
    n = 4100
    cfg = RP.reset_cfg(task, variant, n)
    pr = RP.make_reset_probe(cfg, n, reset_share=0.0)
    pr["state"]["episode_length_buf"].fill_(499)
    cols = [0, 1, 3 if cfg.heading_command else 2]
    got = {}
    # (the persistent kernel takes the flat task only; it falls back to the tiled one for recover)
    for form in ("interval", "ids", "draw", "tiled") + (("persist",) if task == "flat" else ()):
        env = _env(cfg, pr, device_ranges=device_ranges)
        ids = torch.arange(n, device=DEV)
        cnt = torch.tensor([n], dtype=torch.int32, device=DEV)
        r = env._reset_struct(L.RESET_COMMANDS)
        c, b = ctypes.byref(env._c), ctypes.byref(env._buffers())
        if form == "interval":
            L.check(L.lib.hl_resample_commands(c, b, ctypes.byref(r), None, None, 500, n, L.stream()))
        elif form == "ids":
            L.check(L.lib.hl_resample_commands(c, b, ctypes.byref(r), L.ptr(ids), L.ptr(cnt), 0, n, L.stream()))
        elif form == "draw":
            L.check(L.lib.hl_reset_draw(c, b, ctypes.byref(r), L.ptr(ids), L.ptr(cnt), n, L.stream()))
        else:
            if form == "persist":
                monkeypatch.setenv("HL_FUSED_IMPL", "persist")
            else:
                monkeypatch.delenv("HL_FUSED_IMPL", raising=False)
            env.post_physics_step()
            assert int(L.lib.hl_fused_last_impl()) == (1 if form == "persist" else 0)
            assert int(env._n_reset.item()) == 0
        got[form] = env.commands[:, cols].cpu()
    for form, v in got.items():
        assert torch.equal(v, got["interval"]), f"{form} != interval form"
    with RP.default_dtype(torch.float64):
        from oracle import torch_oracle as O
        st = {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in pr["state"].items()}
        o = O.OracleEnv(cfg, st, pr["hf"])
        o.resample_commands(torch.arange(n), pr["u"].double(), cfg.reset)
    RP.check_bound(got["interval"].T, o.commands[:, cols].T, [f"commands[{k}]" for k in cols], "resampled commands")


# ------------------------------------------------------------------------------------------------ 4. one part at a time
PART_FIELDS = {"DOFS": ("dof_state",), "ROOT": ("root_states",), "COMMANDS": ("commands",),
               "FACTORS": ("Kp_factors", "Kd_factors", "motor_strength_factors"),
               "CURRICULUM": ("terrain_levels", "env_origins")}


@pytest.mark.parametrize("part", list(PART_FIELDS))
def test_one_part_writes_only_its_fields(part):
    """hl_reset_draw with HlReset.parts = one bit: that part's fields change on the reset envs (and match a launch of
    every part), nothing else changes anywhere."""
    from isaacgymloco_b200 import _lib as L
    cfg = RP.reset_cfg("stairs", "default", 4099)
    pr = RP.make_reset_probe(cfg, 4099)
    ids = pr["ids"].to(DEV)
    full = _env(cfg, pr)
    full._reset_part(ids, 0)
    env = _env(cfg, pr)
    before = _rows(env)
    env._reset_part(ids, getattr(L, "RESET_" + part))
    after = _rows(env)
    for k, v in before.items():
        if k in PART_FIELDS[part]:
            assert not torch.equal(after[k][ids], v[ids]), f"{part}: {k} did not change"
            if part != "ROOT":      # (the root draw adds env_origins, which the curriculum of the full launch moved)
                assert torch.equal(getattr(env, k), getattr(full, k)), f"{part}: {k} differs from the all-parts launch"
        else:
            assert torch.equal(after[k], v), f"{part}: {k} changed"


# ------------------------------------------------------------------------------------------------ 5. capacity buffers
@pytest.mark.parametrize("fixup", [False, True])
def test_ids_past_the_device_count_are_ignored(fixup):
    """A capacity-N id buffer whose tail (past the device count) holds valid ids of envs that do not reset: those envs
    keep every buffer bit for bit."""
    cfg = RP.reset_cfg("flat", "default", 4099)
    pr = RP.make_reset_probe(cfg, 4099)
    env = _env(cfg, pr)
    ids = pr["ids"]
    others = torch.ones(4099, dtype=torch.bool)
    others[ids] = False
    buf = torch.cat([ids, others.nonzero(as_tuple=False).flatten()]).to(DEV)
    assert len(buf) == 4099
    cnt = torch.tensor([len(ids)], dtype=torch.int32, device=DEV)
    before = _rows(env)
    env.reset_idx_device(buf, cnt, fixup=fixup)
    _check(cfg, pr, env, "capacity buffer", pre_step=False, obs=fixup)
    _assert_others_unchanged(before, env, ids, "capacity buffer")


# ------------------------------------------------------------------------------------------------ 6. gain factors under a torch hook
def test_reset_idx_draws_gain_factors_with_a_torch_dof_hook():
    """LR:336-341: reset_idx draws the Kp, Kd and motor-strength factors after the hooks, also when _reset_dofs is a
    torch override (LeggedRobotB200._reset_dofs = LeggedRobot._reset_dofs, INTEGRATION.md): columns 40-42."""
    cfg = RP.reset_cfg("flat", "default", 4099)
    pr = RP.make_reset_probe(cfg, 4099)
    env = _env(cfg, pr, _hook_env("dofs"))
    ids = pr["ids"].to(DEV)
    before = {k: getattr(env, k).clone() for k in ("Kp_factors", "Kd_factors", "motor_strength_factors")}
    env.reset_idx(ids)
    R, u = cfg.reset, pr["u"][pr["ids"]].double()
    for name, col, (lo, hi) in (("Kp_factors", 40, R.kp_range), ("Kd_factors", 41, R.kd_range),
                                ("motor_strength_factors", 42, R.motor_strength_range)):
        got = getattr(env, name)[ids, 0].cpu()
        assert not torch.equal(got, before[name][ids, 0].cpu()), f"{name} kept its pre-reset values"
        RP.check_bound(got, (hi - lo) * u[:, col] + lo, [name], f"{name} from uniform column {col}")
