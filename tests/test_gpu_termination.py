"""-m gpu: check_termination, the contact filter, the heading command and the base frame of every path that decides
termination, against the float64 reference of tests/termination_probe.py on probes that switch every termination
clause (and make each the only reason to reset for some envs).

Exact: the ascending reset ids equal nonzero(reset64); reset_buf, time_out_buf, extras["time_outs"], contact_filt and
last_contacts; the stairs task's termination row of episode_sums equals scale * (reset & ~time_out); the terminal AMP
rows come in the reference's id order (their dof columns are the probe's rows of those envs); commands[:, 2] is
untouched where heading_command is off (off the resampling mark).  Within the bound |got - ref64| <= 1e-5 |ref64| +
1e-6 max_e |ref64[:, col]| (reward_probe's): base_lin_vel, base_ang_vel, projected_gravity, commands[:, 2] and the
terminal AMP rows' velocity columns.
"""
import functools

import numpy as np
import pytest
import torch

import termination_probe as TP

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
PUSH_VEL_SEED = 57


@functools.lru_cache(maxsize=4)
def _case(task, variant, n, num_envs=None, offset=0):
    cfg = TP.termination_cfg(task, variant, n, num_envs=num_envs, env_id_offset=offset)
    pr = TP.make_termination_probe(cfg, n)
    return cfg, pr, TP.reference64_termination(cfg, pr)


def _push_vel(n):
    g = torch.Generator().manual_seed(PUSH_VEL_SEED)
    return 2 * torch.rand(n, 2, generator=g) - 1


def _env_class():
    from isaacgymloco_b200 import _lib as L
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot

    class Env(FusedLeggedRobot):
        """Keeps the episode sums as the step's reward pass left them, before reset_idx zeroes the reset envs' rows
        (the reset itself stays the in-kernel one)."""
        sums_after_reward = None

        def fused_pre_reset(self, select=True):
            super().fused_pre_reset(select)
            self.sums_after_reward = self._episode_sums_buf.clone()

        def _stages(self, stages, env_ids=None, n_ids=None):
            super()._stages(stages, env_ids, n_ids)
            if stages & L.ST_REWARD:
                self.sums_after_reward = self._episode_sums_buf.clone()

    return Env


def _env(cfg, pr):
    env = _env_class()(cfg, pr["state"], pr["hf"], device=DEV)
    ter = pr["ter"]
    env.env_origins = ter["env_origins"].to(DEV).contiguous()
    if not cfg.is_plane:
        env.terrain_origins = ter["origins"].to(DEV).contiguous()
        env.terrain_types = ter["types"].to(DEV).contiguous()
        env.max_terrain_level = cfg.num_rows
    env.refresh_buffers()
    env.set_reset_uniforms(pr["u"])
    env.set_noise_tensors(**pr["noise"])
    return env


def _run(monkeypatch, path, cfg, pr):
    """One step of `path` on the probe -> (env, reset ids, terminal AMP rows)."""
    from isaacgymloco_b200 import _lib as L
    monkeypatch.delenv("HL_FUSED_EPB", raising=False)
    monkeypatch.delenv("HL_MERGED_RESET", raising=False)
    monkeypatch.setenv("HL_FUSED_IMPL", "persist" if path == "persist" else "tiled")
    if path == "tiled-epb64":
        monkeypatch.setenv("HL_FUSED_EPB", "64")
    if path == "merged":
        monkeypatch.setenv("HL_MERGED_RESET", "1")
    n = pr["u"].shape[0]
    env = _env(cfg, pr)
    if path == "stages":
        env.episode_length_buf += 1
        env.update_base_frame()
        env._resample_commands((env.episode_length_buf % env.resample_interval == 0).nonzero(as_tuple=False).flatten())
        env.update_heading_command()
        env.check_termination()
        env.compute_reward()
        env.sums_after_reward = env._episode_sums_buf.clone()
        ids = env.reset_buf.nonzero(as_tuple=False).flatten()
        amp = env.get_amp_observations()[ids]
        torch.cuda.synchronize()
        return env, ids.cpu(), amp.cpu()
    if path in ("tiled-single", "tiled-separate", "merged"):
        env.single_launch = path == "tiled-single"
        env.refresh_buffers()
    if path == "push":
        cfg.reset.push_robots = True
        env.push_interval = 1
        pv = _push_vel(n).to(DEV)
        env._push_robots = lambda: env.root_states[:, 7:9].copy_(pv)
    assert env._kernel_reset_ok()
    ids, amp = env.post_physics_step()[::2]
    if path == "persist":
        assert int(L.lib.hl_fused_last_impl()) == 1, "the persistent kernel did not run"
    elif path != "push":
        assert int(L.lib.hl_fused_last_impl()) == 0, "the tiled kernel did not run"
    torch.cuda.synchronize()
    return env, ids.cpu(), amp.cpu()


def _check(cfg, pr, ref, env, ids, amp, what, extras=True):
    cpu = lambda t: t.detach().cpu()
    n = ref.num_envs
    st = pr["state"]
    assert torch.equal(ids, ref.reset_buf.nonzero(as_tuple=False).flatten()), f"{what}: reset ids"
    assert torch.equal(ids, ref.ids)
    for k in ("reset_buf", "time_out_buf", "contact_filt", "last_contacts"):
        got, want = cpu(getattr(env, k)), getattr(ref, k)
        assert torch.equal(got, want), f"{what}: {k} differs on {int((got != want).reshape(n, -1).any(dim=1).sum())} envs"
    if extras and len(ids):
        assert torch.equal(cpu(env.extras["time_outs"]), ref.time_out_buf), f"{what}: extras['time_outs']"
    if cfg.termination_scale is not None:
        row = cpu(env.sums_after_reward)[len(env.episode_sums) - 1]
        init = st["episode_sums"][-1]
        want = init + float(np.float32(cfg.termination_scale)) * (ref.reset_buf & ~ref.time_out_buf).float()
        assert torch.equal(row, want), f"{what}: episode_sums['termination'] != scale * (reset & ~time_out)"
    # terminal AMP rows: (dof_pos, base_lin_vel, base_ang_vel, dof_vel) of the reset envs in the reference's id order
    assert amp.shape[0] == len(ref.ids), f"{what}: {amp.shape[0]} terminal rows, the reference has {len(ref.ids)}"
    dof = st["dof_state"].view(n, 12, 2)[ref.ids]
    assert torch.equal(amp[:, :12], dof[..., 0]) and torch.equal(amp[:, 18:], dof[..., 1]), \
        f"{what}: terminal AMP rows are not the reset envs' rows in id order"
    if len(ref.ids):
        TP.check_bound(amp[:, 12:18].T, ref.term_amp[:, 12:18].T, [f"amp[{c}]" for c in range(12, 18)],
                       f"{what}: terminal AMP velocity columns")
    # the frame of every env; commands[:, 2]: the heading command of every env (reset_idx re-draws column 3 then), else
    # the envs the step did not reset (reset_idx re-draws their column 2)
    TP.check_frame(env, ref, torch.ones(n, dtype=torch.bool), what, cmd2=False)
    got2 = cpu(env.commands)[:, 2]
    if cfg.heading_command:
        TP.check_bound(got2, ref.commands[:, 2], ["commands[2]"], f"{what}: heading command")
    else:
        keep = ~ref.reset_buf
        mk = pr["mark"]
        assert torch.equal(got2[keep & ~mk], st["commands"][keep & ~mk, 2]), f"{what}: commands[:, 2] changed"
        TP.check_bound(got2[keep & mk], ref.commands[keep & mk, 2], ["commands[2]"], f"{what}: resampled commands[2]")


# ------------------------------------------------------------------------------------------------ every path
PATHS = [
    # path, task, variant, n
    ("tiled-single", "stairs", "default", 7),
    ("tiled-single", "flat", "all-on", 4099),
    ("tiled-single", "recover", "default", 16384),
    ("tiled-separate", "stairs", "default", 16385),
    ("tiled-separate", "plane", "default", 4099),
    ("tiled-separate", "amp", "default", 65536),
    ("tiled-default", "stairs", "default", 65536),
    ("tiled-default", "flat", "all-off", 16385),
    ("tiled-default", "flat", "default", 4099),
    ("tiled-epb64", "flat", "all-on", 16384),
    ("tiled-epb64", "recover", "default", 4099),
    ("persist", "stairs", "default", 65536),
    ("persist", "flat", "all-on", 4099),
    ("persist", "flat", "default", 16385),
    ("merged", "stairs", "default", 16385),
    ("merged", "flat", "all-on", 65536),
    ("stages", "stairs", "default", 4099),
    ("stages", "flat", "all-on", 7),
    ("stages", "recover", "default", 16385),
    ("stages", "plane", "default", 4099),
    ("push", "stairs", "default", 16384),
    ("push", "flat", "all-on", 65536),
    ("push", "amp", "default", 4099),
]


@pytest.mark.parametrize("path,task,variant,n", PATHS, ids=[f"{p}-{t}-{v}-{n}" for p, t, v, n in PATHS])
def test_termination_path_vs_float64(path, task, variant, n, monkeypatch):
    """The reset ids, the termination buffers, the contact filter, the termination reward, the terminal rows' order,
    the frame and the heading command of one step of `path` against the float64 reference."""
    cfg, pr, ref = _case(task, variant, n)
    if path == "push":
        cfg = TP.termination_cfg(task, variant, n)
        ref = TP.reference64_termination(cfg, pr, push_vel=_push_vel(n))
        if cfg.base_vel_violate_commands:
            # the push must matter: a frame taken after it would flip base_vel_violate_commands for some envs
            pushed = {**pr, "state": {**pr["state"], "root_states": pr["state"]["root_states"].clone()}}
            pushed["state"]["root_states"][:, 7:9] = _push_vel(n)
            after = TP.reference64_termination(cfg, pushed)
            assert (after.vel_violate != ref.vel_violate).double().mean() > 0.05
    env, ids, amp = _run(monkeypatch, path, cfg, pr)
    _check(cfg, pr, ref, env, ids, amp, f"{path} {task} {variant} n={n}", extras=path != "stages")


def test_shard_with_offset_vs_float64(monkeypatch):
    """A shard with env_id_offset = 3,000 of 20,000 envs (its first 1,000 envs in the high-speed slice)."""
    cfg, pr, ref = _case("stairs", "default", 4099, num_envs=20000, offset=3000)
    env, ids, amp = _run(monkeypatch, "tiled-default", cfg, pr)
    _check(cfg, pr, ref, env, ids, amp, "shard")
