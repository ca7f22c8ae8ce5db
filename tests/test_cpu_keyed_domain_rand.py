"""CPU (-m "not gpu"): keyed domain randomisation is opt-in and its host side checks its inputs.

* aliengo(task) and from_reference_cfg() leave ResetCfg.keyed_domain_rand off, whatever the domain_rand settings;
* set_domain_rand_draws rejects bad shapes, dtypes and ranges with ValueError before anything is launched;
* there is no CPU fallback: the launches refuse CPU tensors.
"""
import ctypes
import dataclasses
from types import SimpleNamespace as NS

import pytest
import torch

from isaacgymloco_b200 import config as C


def _reference_like(task):
    """A duck-typed stand-in for the reference's nested config classes, built from the preset, with every domain_rand
    switch on (the reference sources are not needed)."""
    hc = C.aliengo(task, num_envs=64)
    R = hc.reset
    scales = NS(**hc.reward_scales)
    return NS(
        env=NS(num_envs=64, episode_length_s=hc.episode_length_s),
        terrain=NS(mesh_type=hc.mesh_type, measure_heights=hc.measure_heights, horizontal_scale=hc.horizontal_scale,
                   vertical_scale=hc.vertical_scale, border_size=hc.border_size, terrain_length=hc.terrain_length,
                   terrain_width=hc.terrain_width, num_rows=hc.num_rows, num_cols=hc.num_cols,
                   terrain_proportions=hc.terrain_proportions, measured_points_x=hc.measured_points_x,
                   measured_points_y=hc.measured_points_y, curriculum=True),
        control=NS(control_type=hc.control_type, stiffness={"joint": hc.stiffness}, damping={"joint": hc.damping},
                   action_scale=hc.action_scale, decimation=hc.decimation, hip_reduction=hc.hip_reduction),
        rewards=NS(scales=scales, only_positive_rewards=hc.only_positive_rewards, tracking_sigma=hc.tracking_sigma,
                   soft_dof_pos_limit=hc.soft_dof_pos_limit, soft_dof_vel_limit=hc.soft_dof_vel_limit,
                   soft_torque_limit=hc.soft_torque_limit, base_height_target=hc.base_height_target,
                   max_contact_force=hc.max_contact_force),
        noise=NS(add_noise=hc.add_noise, noise_level=hc.noise_level,
                 noise_scales=NS(dof_pos=hc.noise_dof_pos, dof_vel=hc.noise_dof_vel, ang_vel=hc.noise_ang_vel,
                                 gravity=hc.noise_gravity, height_measurements=hc.noise_height)),
        normalization=NS(obs_scales=NS(lin_vel=hc.obs_lin_vel, ang_vel=hc.obs_ang_vel, dof_pos=hc.obs_dof_pos,
                                       dof_vel=hc.obs_dof_vel, height_measurements=hc.obs_height),
                         clip_observations=hc.clip_observations, clip_actions=hc.clip_actions),
        commands=NS(heading_command=hc.heading_command, resampling_time=hc.resampling_time, curriculum=True,
                    ranges=NS(lin_vel_x=R.lin_vel_x, lin_vel_y=R.lin_vel_y, ang_vel_yaw=R.ang_vel_yaw, heading=R.heading)),
        domain_rand=NS(push_robots=True, max_push_vel_xy=1.0, disturbance=True, disturbance_range=[-30.0, 30.0], delay=True,
                       disturbance_interval=8, push_interval_s=16),
        init_state=NS(pos=R.base_init_state[:3], rot=R.base_init_state[3:7], lin_vel=R.base_init_state[7:10],
                      ang_vel=R.base_init_state[10:13]),
    )


@pytest.mark.parametrize("task", ["flat", "stairs", "amp", "recover"])
def test_presets_and_reference_configs_leave_the_flag_off(task):
    from oracle import ref_harness as H
    cfgs = [C.aliengo(task, num_envs=64), C.from_reference_cfg(_reference_like(task), num_envs=64)]
    if H.reference_available():
        cfgs.append(C.from_reference_cfg(H.reference_cfg(task), num_envs=64))
    for cfg in cfgs:
        assert cfg.reset.keyed_domain_rand is False
    assert cfgs[1].reset.delay and cfgs[1].reset.disturbance and cfgs[1].reset.push_robots
    # an opt-in on one config does not leak into another, and the reference-config record does not carry the flag
    cfgs[0].reset.keyed_domain_rand = True
    assert C.aliengo(task).reset.keyed_domain_rand is False and C.ResetCfg().keyed_domain_rand is False
    assert "keyed_domain_rand" not in dataclasses.asdict(cfgs[0].reset)


class _Host:
    """The host-side state set_domain_rand_draws reads, without a device (the checks run before any launch)."""

    def __init__(self, n=6, dec=4):
        self.num_envs, self.device = n, torch.device("cpu")
        self.cfg_hot = C.aliengo("flat", num_envs=n, decimation=dec)
        self._noise = {}


def _set(h, **kw):
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    FusedLeggedRobot.set_domain_rand_draws(h, **kw)


def test_set_domain_rand_draws_checks_its_inputs():
    n, dec = 6, 4
    h = _Host(n, dec)
    good = dict(delay=torch.tensor([0, 1, 2, 3, 0, 3]), disturbance=torch.rand(n, 3), push=torch.rand(n, 2, dtype=torch.float64))
    _set(h, **good)
    assert h._noise["delay"].dtype == torch.int64 and h._noise["push"].dtype == torch.float32
    assert torch.equal(h._noise["delay"], good["delay"])
    bad = [
        dict(delay=torch.tensor([0, 1, 2, 3, 0, 4])),                    # == decimation
        dict(delay=torch.tensor([0, 1, 2, 3, 0, -1])),
        dict(delay=torch.tensor([0, 1, 2, 3, 0, 1], dtype=torch.int32)),  # dtype
        dict(delay=torch.tensor([0.0, 1, 2, 3, 0, 1])),
        dict(delay=torch.zeros(n, 1, dtype=torch.long)),                 # shape
        dict(delay=[0, 1, 2, 3, 0, 1]),                                  # not a tensor
        dict(disturbance=torch.rand(n, 2)),
        dict(disturbance=torch.rand(n + 1, 3)),
        dict(disturbance=torch.ones(n, 3)),                              # 1.0 is outside [0, 1)
        dict(disturbance=torch.full((n, 3), -1e-7)),
        dict(disturbance=torch.full((n, 3), float("nan"))),
        dict(disturbance=torch.zeros(n, 3, dtype=torch.int64)),
        dict(push=torch.rand(n, 3)),
        dict(push=torch.rand(n)),
        dict(push=torch.ones(n, 2, dtype=torch.float64) - 1e-12),        # rounds to 1.0 in float32
        dict(push=torch.zeros(n, 2, dtype=torch.bool)),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            _set(h, **kw)
    _set(h, delay=None, push=good["push"])
    assert h._noise["delay"] is None and h._noise["disturbance"] is None and h._noise["push"] is not None


def test_the_launches_refuse_cpu_tensors():
    from isaacgymloco_b200 import _lib as L
    n = 4
    a = torch.zeros(n, 12)
    with pytest.raises(RuntimeError, match="CUDA"):
        L.ptr(a)
    cfg = C.aliengo("flat", num_envs=n).to_c()
    b = L.HlEnvBuffers()
    b.struct_bytes = ctypes.sizeof(L.HlEnvBuffers)
    # bad arguments are refused on the host, before a launch: these run without a device
    assert L.lib.hl_delay_actions(ctypes.byref(cfg), ctypes.byref(b), None, None, None, 4, 1, 100.0, None, n, None) != 0
    assert L.lib.hl_uniform_rows(ctypes.byref(cfg), ctypes.byref(b), None, 13, 2, -1.0, 1.0, None, 6, n, None) != 0
    assert L.lib.hl_uniform_rows(ctypes.byref(cfg), ctypes.byref(b), 16, 13, 2, -1.0, 1.0, None, 3, n, None) != 0
    assert b"stream_id" in L.lib.hl_last_error()
