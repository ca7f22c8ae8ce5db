"""TEST INFRASTRUCTURE ONLY (the checker) -- never imported by the product path.

Tier-1 oracle: an independent eager-torch restatement of the reference hot path.  It travels to
the GPU box (where /root/reference does not exist) and runs on CPU or on CUDA beside the
kernels.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import it.

Pinning: the reference has no golden vectors of its own (SURVEY.md §4/§8c), so this oracle is
pinned against outputs of the reference itself: tests/golden/*.npz are minted in the build
container by oracle/make_goldens.py, which executes the real reference classes
(oracle/ref_harness.py) on the same seeded inputs; tests/test_oracle_golden.py asserts this
restatement reproduces them (bit-exact for flags/ids/indices; fp32 rounding-level for floats).
The `isaacgym.torch_utils` helpers are third-party and absent (Isaac Gym Preview 4, proprietary,
un-vendored): restated from their public definitions => parity unpinned at that boundary.

Each function cites the reference lines it follows (paths relative to /root/reference, `LR` =
legged_gym/legged_gym/envs/base/legged_robot.py).
"""
import math
from typing import Dict, List, Optional

import numpy as np
import torch

# --------------------------------------------------------------------------- isaacgym helpers
def quat_rotate_inverse(q, v):
    """isaacgym.torch_utils.quat_rotate_inverse (public definition; SURVEY Appendix B.2)."""
    w = q[:, 3]
    qv = q[:, :3]
    a = v * (2.0 * w ** 2 - 1.0).unsqueeze(-1)
    b = torch.cross(qv, v, dim=-1) * w.unsqueeze(-1) * 2.0
    c = qv * torch.bmm(qv.reshape(-1, 1, 3), v.reshape(-1, 3, 1)).squeeze(-1) * 2.0
    return a - b + c


def quat_apply(a, b):
    """isaacgym.torch_utils.quat_apply."""
    shp = b.shape
    a = a.reshape(-1, 4)
    b = b.reshape(-1, 3)
    xyz = a[:, :3]
    t = xyz.cross(b, dim=-1) * 2
    return (b + a[:, 3:] * t + xyz.cross(t, dim=-1)).view(shp)


def quat_apply_yaw(quat, vec):
    """legged_gym/legged_gym/utils/math.py:38-42 with torch_utils.normalize inlined."""
    qy = quat.clone().view(-1, 4)
    qy[:, :2] = 0.0
    qy = qy / qy.norm(p=2, dim=-1).clamp(min=1e-9).unsqueeze(-1)
    return quat_apply(qy, vec)


def wrap_to_pi(angles):
    """math.py:45-48 (Python-sign modulo, in place on a fresh tensor)."""
    angles = angles.clone()
    angles %= 2 * np.pi
    angles -= 2 * np.pi * (angles > np.pi)
    return angles


# --------------------------------------------------------------------------- environment
class OracleEnv:
    """State container + the hot-path methods, named as on the reference's LeggedRobot."""

    def __init__(self, cfg, state: Dict[str, torch.Tensor], height_samples: torch.Tensor):
        self.cfg = cfg
        dev = state["root_states"].device
        self.device = dev
        n = state["root_states"].shape[0]
        self.num_envs = n
        for k, v in state.items():
            setattr(self, k, v.clone())
        self.contact_forces = self.contact_forces.view(n, -1, 3)
        self.dof_pos = self.dof_state.view(n, 12, 2)[..., 0]
        self.dof_vel = self.dof_state.view(n, 12, 2)[..., 1]
        self.base_quat = self.root_states[:, 3:7]
        self.default_dof_pos = self.default_dof_pos.view(1, 12)
        self.height_samples = height_samples.to(dev)
        t = cfg.dof_tables()
        self.p_gains = torch.tensor(t["p_gains"], device=dev)
        self.d_gains = torch.tensor(t["d_gains"], device=dev)
        li = lambda v: torch.tensor(v, dtype=torch.long, device=dev)
        self.feet_indices = li(cfg.feet_indices)
        self.penalised_contact_indices = li(cfg.penalised_contact_indices)
        self.termination_contact_indices = li(cfg.termination_contact_indices)
        self.gravity_vec = torch.tensor([0.0, 0.0, -1.0], device=dev).repeat(n, 1)
        self.forward_vec = torch.tensor([1.0, 0.0, 0.0], device=dev).repeat(n, 1)
        self.commands_scale = torch.tensor([cfg.obs_lin_vel, cfg.obs_lin_vel, cfg.obs_ang_vel],
                                           device=dev)
        self.noise_scale_vec = torch.tensor(cfg.noise_scale_vec(), device=dev)
        self.dt = cfg.dt
        self.rew_buf = torch.zeros(n, device=dev)
        self.reset_buf = torch.ones(n, dtype=torch.long, device=dev)
        self.time_out_buf = torch.zeros(n, dtype=torch.bool, device=dev)
        self.term_names, scales = cfg.active_terms()
        self.term_scales = dict(zip(self.term_names, scales))
        self.sum_names = cfg.episode_sum_names()
        self.episode_sums = {nm: self.episode_sums[k].clone() if k < self.episode_sums.shape[0]
                             else torch.zeros(n, device=dev)
                             for k, nm in enumerate(self.sum_names)} if self.sum_names else {}
        self.height_points = self._grid(cfg.measured_points_x, cfg.measured_points_y)
        self.base_height_points = self._grid(
            [-0.15, -0.1, -0.05, 0., 0.05, 0.1, 0.15],
            [-0.2, -0.15, -0.1, -0.05, 0., 0.05, 0.1, 0.15, 0.2])
        sr = cfg.stumble_ranges()
        off = cfg.env_id_offset
        clampi = lambda v: int(min(max(v - off, 0), n))
        self._stumble_slices = [(clampi(sr["stairsup_start"]), clampi(sr["stairsup_end"])),
                                (clampi(sr["pit_start"]), clampi(sr["gap_end"]))]
        self.measured_heights = self._get_heights()
        self.common_step_counter = 0
        self.last_height_indices = None
        rs = getattr(cfg, "reset", None)
        if rs is not None:
            self.command_ranges = dict(lin_vel_x=list(rs.lin_vel_x), lin_vel_y=list(rs.lin_vel_y),
                                       ang_vel_yaw=list(rs.ang_vel_yaw), heading=list(rs.heading))
        if not hasattr(self, "env_origins"):
            self.env_origins = torch.zeros(n, 3, device=dev)
        if not hasattr(self, "motor_strength_factors"):
            self.motor_strength_factors = torch.ones(n, 1, device=dev)

    def _grid(self, xs, ys):
        """LR:1286-1316: x-major meshgrid of body-frame sample points, z = 0."""
        x = torch.tensor(xs, device=self.device)
        y = torch.tensor(ys, device=self.device)
        gx, gy = torch.meshgrid(x, y, indexing="ij")
        pts = torch.zeros(self.num_envs, gx.numel(), 3, device=self.device)
        pts[:, :, 0] = gx.flatten()
        pts[:, :, 1] = gy.flatten()
        return pts

    # ------------------------------------------------------------------ a1: PD torques
    def _compute_torques(self, actions):
        """LR:658-688."""
        c = self.cfg
        a = self.motor_strength * actions
        scaled = a * c.action_scale
        scaled[:, [0, 3, 6, 9]] *= c.hip_reduction
        self.joint_pos_target = self.default_dof_pos + scaled
        if c.control_type == "P":
            tq = self.p_gains * self.Kp_factors * (self.joint_pos_target - self.dof_pos) \
                - self.d_gains * self.Kd_factors * self.dof_vel
        elif c.control_type == "V":
            tq = self.p_gains * (scaled - self.dof_vel) \
                - self.d_gains * (self.dof_vel - self.last_dof_vel) / c.sim_dt
        elif c.control_type == "T":
            tq = scaled
        else:
            raise NameError(f"Unknown controller type: {c.control_type}")
        return torch.clip(tq, -self.torque_limits, self.torque_limits)

    # ------------------------------------------------------------------ a5/a6: height scans
    def _scan(self, pts_body, root_states=None, quat=None):
        """LR:1339-1355 (and :1378-1392): yaw-rotate, translate, +border, /hscale, trunc to int64,
        clip, min of three int16 neighbours.  Returns (heights_raw int16 (N,P), px, py)."""
        root_states = self.root_states if root_states is None else root_states
        quat = root_states[:, 3:7]
        p = pts_body.shape[1]
        pts = quat_apply_yaw(quat.repeat(1, p), pts_body) + root_states[:, :3].unsqueeze(1)
        pts += self.cfg.border_size
        pts = (pts / self.cfg.horizontal_scale).long()
        px = torch.clip(pts[:, :, 0].reshape(-1), 0, self.height_samples.shape[0] - 2)
        py = torch.clip(pts[:, :, 1].reshape(-1), 0, self.height_samples.shape[1] - 2)
        h = torch.min(torch.min(self.height_samples[px, py], self.height_samples[px + 1, py]),
                      self.height_samples[px, py + 1])
        return h.view(self.num_envs, -1), px.view(self.num_envs, -1), py.view(self.num_envs, -1)

    def _get_heights(self, env_ids=None):
        """LR:1318-1355."""
        if self.cfg.is_plane:
            return torch.zeros(self.num_envs, self.height_points.shape[1], device=self.device)
        h, px, py = self._scan(self.height_points)
        self.last_height_indices = (px, py)
        return h * self.cfg.vertical_scale

    def _get_base_heights(self):
        """LR:1357-1398."""
        if self.cfg.is_plane:
            return self.root_states[:, 2].clone()
        h, _, _ = self._scan(self.base_height_points)
        bh = h * self.cfg.vertical_scale
        return torch.mean(self.root_states[:, 2].unsqueeze(1) - bh, dim=1)

    # ------------------------------------------------------------------ a7: termination
    def check_termination(self):
        """LR:249-286 (the dead termination_counts/.item() bookkeeping is not restated)."""
        c = self.cfg
        f = self.contact_forces[:, self.termination_contact_indices, :]
        self.reset_buf = torch.any(torch.norm(f, dim=-1) > 1.0, dim=1)
        self.time_out_buf = self.episode_length_buf > c.max_episode_length
        self.reset_buf |= self.time_out_buf
        if c.base_vel_violate_commands:
            err = self.base_lin_vel[:, 0] - self.commands[:, 0]
            viol = ((err > 2) & (self.commands[:, 0] < 0.0)) | ((err < -2) & (self.commands[:, 0] > 0.0))
            viol = viol & (self.terrain_levels > 3)
            self.vel_violate = viol
            self.reset_buf |= viol
        if c.out_of_border and not c.is_plane:
            lim = torch.tensor([c.x_size + c.border_size / 2, c.y_size + c.border_size / 2],
                               device=self.device)
            xy = self.root_states[:, :2]
            inside = torch.logical_and(xy >= 0, xy < lim).all(dim=-1)      # terrain.py:220-227
            self.reset_buf |= inside.logical_not()
        if c.fall_down:
            self.reset_buf |= self.root_states[:, 9] < -5.0

    # ------------------------------------------------------------------ a8/a9: rewards
    def compute_reward(self):
        """LR:363-380: alphabetical accumulation, optional clip, then the termination term."""
        self.rew_buf[:] = 0.0
        for name in self.term_names:
            r = getattr(self, "_r_" + name)() * self.term_scales[name]
            self.rew_buf += r
            self.episode_sums[name] += r
        if self.cfg.only_positive_rewards:
            self.rew_buf[:] = torch.clip(self.rew_buf[:], min=0.0)
        ts = self.cfg.termination_scale
        if ts is not None:
            r = self._r_termination() * ts
            self.rew_buf += r
            self.episode_sums["termination"] += r

    # helpers shared by several terms
    def _up(self):
        return torch.clamp(-self.projected_gravity[:, 2], 0, 1)

    def _cmd_norm(self):
        return torch.norm(self.commands[:, :2], dim=1)

    def _feet_force(self):
        return self.contact_forces[:, self.feet_indices, :]

    def _foot_body_frame(self, what):
        """LR:1612-1618 / 1685-1697: foot pos or vel relative to base, rotated into the body frame."""
        src, ref = (self.feet_pos, self.root_states[:, 0:3]) if what == "pos" \
            else (self.feet_vel, self.root_states[:, 7:10])
        rel = src - ref.unsqueeze(1)
        out = torch.zeros(self.num_envs, 4, 3, device=self.device)
        for i in range(4):
            out[:, i, :] = quat_rotate_inverse(self.base_quat, rel[:, i, :])
        return out

    def _r_tracking_lin_vel(self):      # LR:1444-1452
        small = self._cmd_norm() < 0.1
        track = self.commands[:, :2] * (~small.unsqueeze(-1))
        err = torch.sum(torch.square(track - self.base_lin_vel[:, :2]), dim=1)
        return torch.exp(-err / self.cfg.tracking_sigma)

    def _r_tracking_ang_vel(self):      # LR:1454-1457
        err = torch.square(self.commands[:, 2] - self.base_ang_vel[:, 2])
        return torch.exp(-err / self.cfg.tracking_sigma)

    def _r_feet_air_time(self):         # LR:1459-1470 (stateful)
        contact = self.contact_forces[:, self.feet_indices, 2] > 1.0
        filt = torch.logical_or(contact, self.last_contacts)
        self.last_contacts = contact
        first = (self.feet_air_time > 0.0) * filt
        self.feet_air_time += self.dt
        r = torch.sum((self.feet_air_time - 0.5) * first, dim=1)
        r *= self._cmd_norm() > 0.1
        self.feet_air_time *= ~filt
        return r

    def _r_upward(self):                # LR:1472-1474
        return 1 - self.projected_gravity[:, 2]

    def _r_has_contact(self):           # LR:1476-1479
        return (self._cmd_norm() < 0.1) * torch.sum(1.0 * self.contact_filt, dim=-1) / 4

    def _r_lin_vel_z(self):             # LR:1482-1484
        return torch.square(self.base_lin_vel[:, 2])

    def _r_lin_vel_z_up(self):
        return self._r_lin_vel_z() * self._up()

    def _r_ang_vel_xy(self):            # LR:1488-1490
        return torch.sum(torch.square(self.base_ang_vel[:, :2]), dim=1)

    def _r_ang_vel_xy_up(self):
        return self._r_ang_vel_xy() * self._up()

    def _r_orientation(self):           # LR:1494-1496
        return torch.sum(torch.square(self.projected_gravity[:, :2]), dim=1)

    def _r_orientation_up(self):
        return self._r_orientation() * self._up()

    def _r_base_height(self):           # LR:1500-1503
        return torch.square(self._get_base_heights() - self.cfg.base_height_target)

    def _r_base_height_up(self):
        return self._r_base_height() * self._up()

    def _r_dof_vel(self):               # LR:1509-1511
        return torch.sum(torch.square(self.dof_vel), dim=1)

    def _r_dof_acc(self):               # LR:1513-1515
        return torch.sum(torch.square((self.last_dof_vel - self.dof_vel) / self.dt), dim=1)

    def _r_dof_vel_limits(self):        # LR:1517-1520
        lim = self.dof_vel_limits * self.cfg.soft_dof_vel_limit
        return torch.sum((torch.abs(self.dof_vel) - lim).clip(min=0.0, max=1.0), dim=1)

    def _r_dof_pos_dif(self):           # LR:1523-1525
        return torch.sum(torch.square(self.last_dof_pos - self.dof_pos), dim=1)

    def _r_dof_pos_limits(self):        # LR:1527-1531
        out = -(self.dof_pos - self.dof_pos_limits[:, 0]).clip(max=0.0)
        out += (self.dof_pos - self.dof_pos_limits[:, 1]).clip(min=0.0)
        return torch.sum(out, dim=1)

    def _r_action_rate(self):           # LR:1534-1536
        return torch.sum(torch.square(self.last_actions - self.actions), dim=1)

    def _r_smoothness(self):            # LR:1538-1540
        return torch.sum(torch.square(
            self.actions - self.last_actions - self.last_actions + self.last_last_actions), dim=1)

    def _r_torques(self):               # LR:1543-1545
        return torch.sum(torch.square(self.torques), dim=1)

    def _r_torques_distribution(self):  # LR:1547-1549
        return torch.var(torch.abs(self.torques), dim=1)

    def _r_torques_dif(self):           # LR:1551-1553
        return torch.sum(torch.square(self.torques - self.last_torques), dim=1)

    def _r_torque_limits(self):         # LR:1555-1557
        lim = self.torque_limits * self.cfg.soft_torque_limit
        return torch.sum((torch.abs(self.torques) - lim).clip(min=0.0), dim=1)

    def _r_joint_power(self):           # LR:1560-1562
        return torch.sum(torch.abs(self.dof_vel) * torch.abs(self.torques), dim=1)

    def _r_power(self):                 # LR:1564-1566
        return torch.sum(torch.abs(self.torques * self.dof_vel), dim=1)

    def _r_power_distribution(self):    # LR:1568-1570
        return torch.var(torch.abs(self.torques * self.dof_vel), dim=1)

    def _r_collision(self):             # LR:1573-1576
        f = self.contact_forces[:, self.penalised_contact_indices, :]
        return torch.sum(1.0 * (torch.norm(f, dim=-1) > 0.1), dim=1)

    def _r_collision_up(self):
        return self._r_collision() * self._up()

    def _r_termination(self):           # LR:1580-1582
        return self.reset_buf * ~self.time_out_buf

    def _r_feet_contact_forces(self):   # LR:1628-1630 (second definition wins; identical)
        return torch.sum((torch.norm(self._feet_force(), dim=-1)
                          - self.cfg.max_contact_force).clip(min=0.0), dim=1)

    def _stumble(self, factor):         # LR:1589-1608
        ff = self._feet_force()
        r = torch.any(torch.norm(ff[:, :, :2], dim=2) > factor * torch.abs(ff[:, :, 2]), dim=1)
        r = (r * (self.terrain_levels > 3)).float()
        out = torch.zeros_like(r)
        for lo, hi in self._stumble_slices:
            out[lo:hi] = r[lo:hi]
        return out

    def _r_feet_stumble(self):
        return self._stumble(5)

    def _r_feet_stumble_up(self):
        return self._stumble(4) * self._up()

    def _r_feet_slide(self):            # LR:1610-1619
        v = self._foot_body_frame("vel")
        lat = torch.sqrt(torch.sum(torch.square(v[:, :, :2]), dim=2)).view(self.num_envs, -1)
        return torch.sum(self.contact_filt * lat, dim=1)

    def _r_feet_slide_up(self):
        return self._r_feet_slide() * self._up()

    def _r_feet_mirror(self):           # LR:1632-1636
        q = self.dof_pos
        d1 = torch.sum(torch.square(q[:, [1, 2]] - q[:, [10, 11]]), dim=-1)
        d2 = torch.sum(torch.square(q[:, [4, 5]] - q[:, [7, 8]]), dim=-1)
        return 0.5 * (d1 + d2)

    def _r_feet_mirror_up(self):
        return self._r_feet_mirror() * self._up()

    def _r_stand_still(self):           # LR:1643-1645
        return torch.sum(torch.abs(self.dof_pos - self.default_dof_pos), dim=1) * (self._cmd_norm() < 0.1)

    def _r_stand_nice(self):            # LR:1647-1649
        return self._r_stand_still() * (1 - self.projected_gravity[:, 2])

    def _r_stuck(self):                 # LR:1651-1654
        return (torch.abs(self.base_lin_vel[:, 0]) < 0.1) * (torch.abs(self.commands[:, 0]) > 0.1)

    def _r_hip_action_magnitude(self):  # LR:1657-1660
        a = self.actions[:, [0, 3, 6, 9]]
        return torch.sum(torch.square(torch.maximum(torch.abs(a) - 1.0, torch.zeros_like(a))), dim=1)

    def _pose(self, idx):               # LR:1662-1679
        return torch.sum(torch.abs(self.dof_pos[:, idx] - self.default_dof_pos[:, idx]), dim=1)

    def _r_hip_pos(self):
        return self._pose([0, 3, 6, 9])

    def _r_hip_pos_up(self):
        return self._pose([0, 3, 6, 9]) * self._up()

    def _r_thigh_pose(self):
        return self._pose([1, 4, 7, 10])

    def _r_thigh_pose_up(self):
        return self._pose([1, 4, 7, 10]) * self._up()

    def _r_calf_pose(self):
        return self._pose([2, 5, 8, 11])

    def _r_calf_pose_up(self):
        return self._pose([2, 5, 8, 11]) * self._up()

    def _r_foot_clearance_base(self):   # LR:1682-1698
        p = self._foot_body_frame("pos")
        v = self._foot_body_frame("vel")
        herr = torch.square(p[:, :, 2] - self.cfg.foot_height_target_base).view(self.num_envs, -1)
        lat = torch.sqrt(torch.sum(torch.square(v[:, :, :2]), dim=2)).view(self.num_envs, -1)
        return torch.sum(herr * lat, dim=1)

    def _r_foot_clearance_base_up(self):
        return self._r_foot_clearance_base() * self._up()

    def _r_foot_clearance_terrain(self):  # LR:1717-1743 incl. the in-place `points += border` quirk
        c = self.cfg
        if c.is_plane:
            fh = self.feet_pos[:, :, 2]
        else:
            pts = self.feet_pos
            pts += c.border_size                       # mutates self.feet_pos (all 3 coords)
            ip = (pts / c.horizontal_scale).long()
            px = torch.clip(ip[:, :, 0].reshape(-1), 0, self.height_samples.shape[0] - 2)
            py = torch.clip(ip[:, :, 1].reshape(-1), 0, self.height_samples.shape[1] - 2)
            h = torch.min(torch.min(self.height_samples[px, py], self.height_samples[px + 1, py]),
                          self.height_samples[px, py + 1])
            ground = h.reshape(self.num_envs, -1) * c.vertical_scale
            fh = self.feet_pos[:, :, 2] - ground
        lat = torch.norm(self.feet_vel[:, :, :2], dim=-1)
        return torch.sum(lat * torch.square(fh - c.foot_height_target_terrain), dim=-1)

    def _r_foot_clearance_terrain_up(self):
        return self._r_foot_clearance_terrain() * self._up()

    # ------------------------------------------------------------------ a11/a12/a13: observations
    def _current_obs(self, u45, u187):
        """LR:385-401 (shared body of compute_observations / compute_termination_observations).
        `u45`, `u187` are the U[0,1) draws that `torch.rand_like` would return there."""
        c = self.cfg
        cur = torch.cat((self.commands[:, :3] * self.commands_scale,
                         self.base_ang_vel * c.obs_ang_vel,
                         self.projected_gravity,
                         (self.dof_pos - self.default_dof_pos) * c.obs_dof_pos,
                         self.dof_vel * c.obs_dof_vel,
                         self.actions), dim=-1)
        if c.add_noise:
            cur += (2 * u45 - 1) * self.noise_scale_vec[0:45]
        cur = torch.cat((cur, self.base_lin_vel * c.obs_lin_vel, self.disturbance[:, 0, :]), dim=-1)
        if c.measure_heights:
            h = torch.clip(self.root_states[:, 2].unsqueeze(1) - 0.5 - self.measured_heights, -1, 1.0) \
                * c.obs_height
            h += (2 * u187 - 1) * self.noise_scale_vec[45:45 + h.shape[1]]
            cur = torch.cat((cur, h), dim=-1)
        return cur

    def compute_observations(self, u45, u187):
        """LR:382-404."""
        cur = self._current_obs(u45, u187)
        self.obs_buf = torch.cat((cur[:, :45], self.obs_buf[:, :-45]), dim=-1)
        self.privileged_obs_buf = cur.clone()

    def compute_termination_observations(self, env_ids, u45, u187):
        """LR:439-460."""
        return self._current_obs(u45, u187)[env_ids]

    def get_amp_observations(self):
        """LR:406-416."""
        return torch.cat((self.dof_pos, self.base_lin_vel, self.base_ang_vel, self.dof_vel), dim=-1)

    # ------------------------------------------------------------------ the step
    def pre_reset(self, noise, push_vel=None):
        """LR:193-228 minus the RNG-driven calls (_resample_commands, pushes, disturbances).  `push_vel` (N,2): the
        root xy velocities a push step's _push_robots writes (LR:627-628, 822-828), applied where
        _post_physics_step_callback applies them (LR:607-632): after the heading command and the height scan,
        before termination and rewards."""
        c = self.cfg
        n = self.num_envs
        self.episode_length_buf += 1
        self.common_step_counter += 1
        self.base_lin_vel = quat_rotate_inverse(self.base_quat, self.root_states[:, 7:10])
        self.base_ang_vel = quat_rotate_inverse(self.base_quat, self.root_states[:, 10:13])
        self.projected_gravity = quat_rotate_inverse(self.base_quat, self.gravity_vec)
        rb = self.rigid_body_states.view(n, c.num_bodies, 13)
        self.feet_pos = rb[:, self.feet_indices, 0:3]
        self.feet_vel = rb[:, self.feet_indices, 7:10]
        contact = self.contact_forces[:, self.feet_indices, 2] > 1.0
        self.contact_filt = torch.logical_or(contact, self.last_contacts)
        self.last_contacts = contact
        if c.heading_command:                                       # LR:616-620
            fwd = quat_apply(self.base_quat, self.forward_vec)
            heading = torch.atan2(fwd[:, 1], fwd[:, 0])
            self.commands[:, 2] = torch.clip(0.5 * wrap_to_pi(self.commands[:, 3] - heading), -2.0, 2.0)
        if c.measure_heights:
            self.measured_heights = self._get_heights()
        if push_vel is not None:                                    # LR:627-628
            self.root_states[:, 7:9] = push_vel
        self.check_termination()
        self.compute_reward()
        env_ids = self.reset_buf.nonzero(as_tuple=False).flatten()
        term_obs = self.compute_termination_observations(env_ids, noise["term45"], noise["term187"])
        term_amp = self.get_amp_observations()[env_ids]
        return env_ids, term_obs, term_amp

    def apply_reset(self, env_ids, targets):
        """The deterministic part of reset_idx (LR:288-361) with the RNG-driven state draws
        replaced by rows of `targets` (see synthetic.make_reset_targets)."""
        if len(env_ids) == 0:
            return
        n = self.num_envs
        if "dof_state" in targets:
            self.dof_state.view(n, 12, 2)[env_ids] = targets["dof_state"].view(n, 12, 2)[env_ids]
        if "root_states" in targets:
            self.root_states[env_ids] = targets["root_states"][env_ids]
        if "commands" in targets:
            self.commands[env_ids] = targets["commands"][env_ids]
        for name in ("last_actions", "last_last_actions", "last_dof_pos", "last_dof_vel",
                     "last_torques", "feet_air_time"):
            getattr(self, name)[env_ids] = 0.0
        self.reset_buf[env_ids] = 1
        if self.cfg.measure_heights:
            self.measured_heights = self._get_heights()
        for k in self.episode_sums:
            self.episode_sums[k][env_ids] = 0.0
        self.episode_length_buf[env_ids] = 0

    def post_reset(self, noise):
        """LR:232-241 and the obs clip of step() (LR:167-171)."""
        self.compute_observations(noise["obs45"], noise["obs187"])
        self.disturbance[:, :, :] = 0.0
        self.last_last_actions[:] = self.last_actions[:]
        self.last_actions[:] = self.actions[:]
        self.last_dof_pos[:] = self.dof_pos[:]
        self.last_dof_vel[:] = self.dof_vel[:]
        self.last_torques[:] = self.torques[:]
        self.last_root_vel[:] = self.root_states[:, 7:13]
        clip = self.cfg.clip_observations
        self.obs_buf = torch.clip(self.obs_buf, -clip, clip)
        self.privileged_obs_buf = torch.clip(self.privileged_obs_buf, -clip, clip)

    def post_physics_step(self, noise, reset_targets=None):
        env_ids, term_obs, term_amp = self.pre_reset(noise)
        if reset_targets is not None:
            self.apply_reset(env_ids, reset_targets)
        self.post_reset(noise)
        return env_ids, term_obs, term_amp

    # ------------------------------------------------------------------ f2: reset_idx with its draws
    # Every `torch_rand_float(lo, hi, ...)` of the reference becomes lo + (hi - lo) * u[:, k] with the column map of
    # include/himloco_b200.h (HL_RESET_NU): the same uniforms the kernel consumes in parity mode.
    def resample_commands(self, env_ids, u, rs):
        """LR:634-656.  `rs` = cfg.reset (+ the live command ranges in rs_ranges)."""
        if len(env_ids) == 0:
            return
        cr = self.command_ranges
        U = u[env_ids]
        rng = lambda k, lohi: (lohi[1] - lohi[0]) * U[:, k] + lohi[0]
        self.commands[env_ids, 0] = rng(36, (-1.0, 1.0))
        self.commands[env_ids, 1] = rng(37, cr["lin_vel_y"])
        if self.cfg.heading_command:
            self.commands[env_ids, 3] = rng(38, cr["heading"])
        else:
            self.commands[env_ids, 2] = rng(38, cr["ang_vel_yaw"])
        gid = env_ids + self.cfg.env_id_offset
        high = gid < (self.cfg.num_envs * 0.2)
        hi_ids = env_ids[high.nonzero(as_tuple=True)]
        self.commands[hi_ids, 0] = ((cr["lin_vel_x"][1] - cr["lin_vel_x"][0]) * u[hi_ids, 39] + cr["lin_vel_x"][0])
        self.commands[hi_ids, 1:2] *= (torch.norm(self.commands[hi_ids, 0:1], dim=1) < 1.0).unsqueeze(1)
        self.commands[env_ids, :2] *= (torch.norm(self.commands[env_ids, :2], dim=1) > 0.2).unsqueeze(1)

    def reset_idx_draw(self, env_ids, u, custom_origins=True, terrain=None):
        """LR:288-341: terrain curriculum, _reset_dofs, _reset_root_states, _resample_commands, gain factors.
        `terrain` = dict(origins (L,T,3), types (N,), max_level, env_length, max_episode_length_s) or None."""
        if len(env_ids) == 0:
            return
        rs = self.cfg.reset
        n = self.num_envs
        U = u[env_ids]
        rng = lambda k, lohi: (lohi[1] - lohi[0]) * U[:, k] + lohi[0]
        if terrain is not None and rs.terrain_curriculum:                     # LR:845-866
            dist = torch.norm(self.root_states[env_ids, :2] - self.env_origins[env_ids, :2], dim=1)
            up = dist > terrain["env_length"] / 2
            down = (dist < torch.norm(self.commands[env_ids, :2], dim=1) * terrain["max_episode_length_s"] * 0.5) * ~up
            lv = self.terrain_levels[env_ids] + 1 * up - 1 * down
            rand_lv = (U[:, 43] * terrain["max_level"]).long().clamp(max=terrain["max_level"] - 1)
            lv = torch.where(lv >= terrain["max_level"], rand_lv, torch.clip(lv, 0))
            self.terrain_levels[env_ids] = lv
            self.env_origins[env_ids] = terrain["origins"][lv, terrain["types"][env_ids]]
        # _reset_dofs (LR:690-716)
        dp = self.dof_state.view(n, 12, 2)
        if rs.dof_init_pos_ratio_range is not None:
            dp[env_ids, :, 0] = self.default_dof_pos * ((rs.dof_init_pos_ratio_range[1] - rs.dof_init_pos_ratio_range[0]) * U[:, 0:12]
                                                        + rs.dof_init_pos_ratio_range[0])
        else:
            dp[env_ids, :, 0] = self.default_dof_pos.expand(len(env_ids), 12)
        if rs.randomize_dof_vel:
            r = rs.dof_init_vel_range
            dp[env_ids, :, 1] = U[:, 12:24] * abs(r[1] - r[0]) + min(r)
        else:
            dp[env_ids, :, 1] = 0.0
        # _reset_root_states (LR:718-820)
        base = torch.tensor(rs.base_init_state, device=self.device)
        self.root_states[env_ids] = base
        self.root_states[env_ids, :3] += self.env_origins[env_ids]
        if custom_origins:
            pr = rs.base_init_pos_range
            if pr is not None:
                self.root_states[env_ids, 0] += rng(24, pr["x"])
                self.root_states[env_ids, 1] += rng(25, pr["y"])
                self.root_states[env_ids, 2] += rng(26, pr["z"])
            else:
                self.root_states[env_ids, 0] += rng(24, (-1.0, 1.0))
                self.root_states[env_ids, 1] += rng(25, (-1.0, 1.0))
        rr = rs.base_init_rot_range
        if rr is not None:
            roll, pitch, yaw = rng(27, rr["roll"]), rng(28, rr["pitch"]), rng(29, rr.get("yaw", [-np.pi, np.pi]))
            cy, sy = torch.cos(yaw * 0.5), torch.sin(yaw * 0.5)
            cr_, sr = torch.cos(roll * 0.5), torch.sin(roll * 0.5)
            cp, sp = torch.cos(pitch * 0.5), torch.sin(pitch * 0.5)
            self.root_states[env_ids, 3:7] = torch.stack([cy * sr * cp - sy * cr_ * sp, cy * cr_ * sp + sy * sr * cp,
                                                          sy * cr_ * cp - cy * sr * sp, cy * cr_ * cp + sy * sr * sp], dim=-1)
        vr = rs.base_init_vel_range if rs.base_init_vel_range is not None else (-0.5, 0.5)
        for k, ax in enumerate(("x", "y", "z", "roll", "pitch", "yaw")):
            self.root_states[env_ids, 7 + k] = rng(30 + k, vr[ax] if isinstance(vr, dict) else vr)
        self.resample_commands(env_ids, u, rs)
        if rs.randomize_kp:
            self.Kp_factors[env_ids, 0] = rng(40, rs.kp_range)
        if rs.randomize_kd:
            self.Kd_factors[env_ids, 0] = rng(41, rs.kd_range)
        if rs.randomize_motor_strength:
            self.motor_strength_factors[env_ids, 0] = rng(42, rs.motor_strength_range)

    def snapshot(self) -> Dict[str, torch.Tensor]:
        """Everything a parity test compares, as detached CPU tensors."""
        out = {}
        for k in ("base_lin_vel", "base_ang_vel", "projected_gravity", "measured_heights", "reset_buf",
                  "time_out_buf", "rew_buf", "contact_filt", "last_contacts", "feet_air_time",
                  "commands", "episode_length_buf", "obs_buf", "privileged_obs_buf", "last_actions",
                  "last_last_actions", "last_dof_pos", "last_dof_vel", "last_torques", "last_root_vel"):
            if hasattr(self, k):
                out[k] = getattr(self, k).detach().cpu().clone()
        if self.sum_names:
            out["episode_sums"] = torch.stack([self.episode_sums[k] for k in self.sum_names]).cpu()
        return out


# --------------------------------------------------------------------------- a15: GAE
def compute_returns(rewards, values, dones, last_values, gamma, lam):
    """rsl_rl/rsl_rl/storage/him_rollout_storage.py:113-127 (== amp_rollout_storage.py:141-155).
    Returns (returns, normalised advantages), both (T,N,1)."""
    t_len = rewards.shape[0]
    returns = torch.zeros_like(rewards)
    adv = 0
    for t in reversed(range(t_len)):
        nxt = last_values if t == t_len - 1 else values[t + 1]
        live = 1.0 - dones[t].float()
        delta = rewards[t] + live * gamma * nxt - values[t]
        adv = delta + live * gamma * lam * adv
        returns[t] = adv + values[t]
    a = returns - values
    a = (a - a.mean()) / (a.std() + 1e-8)
    return returns, a


# --------------------------------------------------------------------------- f1: record one rollout step
def record_env_step(storage, step, tr, gamma):
    """Runner patch + process_env_step + add_transitions for slot `step`:
    rsl_rl/rsl_rl/runners/him_on_policy_runner.py:122-123,
    rsl_rl/rsl_rl/algorithms/him_ppo.py:104-115,
    rsl_rl/rsl_rl/storage/him_rollout_storage.py:92-108.
    `storage`: dict of (T,N,.) tensors; `tr`: dict with obs, critic_obs, privileged_obs (after the
    env step), termination_ids, termination_privileged_obs, actions, rewards, dones, values,
    time_outs (or None), log_prob, mu, sigma."""
    nxt = tr["privileged_obs"].clone()
    nxt[tr["termination_ids"]] = tr["termination_privileged_obs"].clone()
    rewards = tr["rewards"].clone()
    if tr.get("time_outs") is not None:
        rewards += gamma * torch.squeeze(tr["values"] * tr["time_outs"].unsqueeze(1), 1)
    storage["observations"][step].copy_(tr["obs"])
    storage["privileged_observations"][step].copy_(tr["critic_obs"])
    storage["next_privileged_observations"][step].copy_(nxt)
    storage["actions"][step].copy_(tr["actions"])
    storage["rewards"][step].copy_(rewards.view(-1, 1))
    storage["dones"][step].copy_(tr["dones"].view(-1, 1))
    storage["values"][step].copy_(tr["values"])
    storage["actions_log_prob"][step].copy_(tr["log_prob"].view(-1, 1))
    storage["mu"][step].copy_(tr["mu"])
    storage["sigma"][step].copy_(tr["sigma"])


# --------------------------------------------------------------------------- f3: minibatch gather
MINIBATCH_ORDER = ("observations", "privileged_observations", "actions", "next_privileged_observations", "values",
                   "advantages", "returns", "actions_log_prob", "mu", "sigma")


def mini_batches(storage, num_mini_batches, num_epochs, indices):
    """rsl_rl/rsl_rl/storage/him_rollout_storage.py:137-177 with the permutation given: yields the
    ten `x.flatten(0,1)[batch_idx]` tensors in the reference's order."""
    t, n = storage["observations"].shape[:2]
    mb = (t * n) // num_mini_batches
    flat = {k: storage[k].flatten(0, 1) for k in MINIBATCH_ORDER}
    for _ in range(num_epochs):
        for i in range(num_mini_batches):
            idx = indices[i * mb:(i + 1) * mb]
            yield tuple(flat[k][idx] for k in MINIBATCH_ORDER)


# --------------------------------------------------------------------------- f3: AMP replay ring
class OracleReplayBuffer:
    """rsl_rl/rsl_rl/storage/replay_buffer.py:35-74 restated (ring insert with the two-slice wrap,
    host-RNG sampling)."""

    def __init__(self, obs_dim, buffer_size, device="cpu"):
        self.states = torch.zeros(buffer_size, obs_dim, device=device)
        self.next_states = torch.zeros(buffer_size, obs_dim, device=device)
        self.buffer_size, self.device, self.step, self.num_samples = buffer_size, device, 0, 0

    def insert(self, states, next_states):
        num, size = states.shape[0], self.buffer_size
        end = self.step + num
        if end > size:
            head = size - self.step
            self.states[self.step:size] = states[:head]
            self.next_states[self.step:size] = next_states[:head]
            self.states[:end - size] = states[head:]
            self.next_states[:end - size] = next_states[head:]
        else:
            self.states[self.step:end] = states
            self.next_states[self.step:end] = next_states
        self.num_samples = min(size, max(end, self.num_samples))
        self.step = (self.step + num) % size

    def feed_forward_generator(self, num_mini_batch, mini_batch_size):
        for _ in range(num_mini_batch):
            idx = np.random.choice(self.num_samples, size=mini_batch_size)
            yield self.states[idx], self.next_states[idx]


# --------------------------------------------------------------------------- a16-a19: AMP
_EPS = np.finfo(float).eps * 4.0        # rsl_rl/rsl_rl/utils/utils.py:35


def quaternion_slerp(q0, q1, fraction):
    """rsl_rl/rsl_rl/utils/utils.py:153-186 (spin=0, shortestpath=True).  Divides by the angle,
    not its sine, and does not renormalise -- reproduced as is."""
    q0, q1 = q0.clone(), q1.clone()
    out = torch.zeros_like(q0)
    m_zero = torch.isclose(fraction, torch.zeros_like(fraction)).squeeze(-1)
    m_one = torch.isclose(fraction, torch.ones_like(fraction)).squeeze(-1)
    out[m_zero] = q0[m_zero]
    out[m_one] = q1[m_one]
    d = torch.sum(q0 * q1, dim=-1, keepdim=True)
    m_dist = (torch.abs(torch.abs(d) - 1.0) < _EPS).squeeze(-1)
    out[m_dist] = q0[m_dist]
    neg = d < 0
    d = torch.where(neg, -d, d)
    q1 = torch.where(neg, -q1, q1)
    angle = torch.acos(d)
    m_ang = (torch.abs(angle) < _EPS).squeeze(-1)
    out[m_ang] = q0[m_ang]
    general = torch.logical_not(m_zero | m_one | m_dist | m_ang)
    inv = 1.0 / angle
    mix = q0 * (torch.sin((1.0 - fraction) * angle) * inv) + q1 * (torch.sin(fraction * angle) * inv)
    out[general] = mix[general]
    return out


class OracleMotionTable:
    """The numeric half of AMPLoader (rsl_rl/rsl_rl/datasets/motion_loader.py): per-clip (n_i,49)
    fp32 tables, lens/num_frames/frame_durations/weights as float64 numpy arrays."""

    def __init__(self, frames: List[torch.Tensor], frame_durations, weights, dt):
        self.trajectories_full = frames
        self.trajectory_frame_durations = np.asarray(frame_durations, dtype=np.float64)
        self.trajectory_num_frames = np.asarray([float(f.shape[0]) for f in frames])
        self.trajectory_lens = (self.trajectory_num_frames - 1) * self.trajectory_frame_durations
        w = np.asarray(weights, dtype=np.float64)
        self.trajectory_weights = w / np.sum(w)
        self.time_between_frames = dt

    def get_full_frame_at_time_batch(self, traj_idxs, times):
        """motion_loader.py:231-255; index math in float64 numpy exactly as there."""
        p = times / self.trajectory_lens[traj_idxs]
        n = self.trajectory_num_frames[traj_idxs]
        lo = np.floor(p * n).astype(int)
        hi = np.ceil(p * n).astype(int)
        dev = self.trajectories_full[0].device
        start = torch.zeros(len(traj_idxs), 49, device=dev)
        end = torch.zeros(len(traj_idxs), 49, device=dev)
        for i in set(traj_idxs.tolist()):
            m = traj_idxs == i
            start[m] = self.trajectories_full[i][lo[m]]
            end[m] = self.trajectories_full[i][hi[m]]
        blend = torch.tensor(p * n - lo, device=dev, dtype=torch.float32).unsqueeze(-1)
        lerp = lambda a, b: (1.0 - blend) * a + blend * b       # AMPLoader.slerp (:189-190)
        return torch.cat([lerp(start[:, 0:3], end[:, 0:3]),
                          quaternion_slerp(start[:, 3:7], end[:, 3:7], blend),
                          lerp(start[:, 7:49], end[:, 7:49])], dim=-1), lo, hi


def amp_pairs(pre_s, pre_s_next, idxs):
    """motion_loader.py:321-330 (preload branch): columns [7:19] + [31:49] of the two tables."""
    pick = lambda t: torch.cat([t[idxs, 7:19], t[idxs, 31:49]], dim=-1)
    return pick(pre_s), pick(pre_s_next)


def normalize_torch(x, mean64, var64, eps=1e-4, clip=10.0):
    """rsl_rl/rsl_rl/utils/utils.py:124-130."""
    mean = torch.tensor(mean64, device=x.device, dtype=torch.float32)
    std = torch.sqrt(torch.tensor(var64 + eps, device=x.device, dtype=torch.float32))
    return torch.clamp((x - mean) / std, -clip, clip)


def amp_disc_input(state, next_state, mean64, var64):
    """amp_discriminator.py:59-63."""
    return torch.cat([normalize_torch(state, mean64, var64),
                      normalize_torch(next_state, mean64, var64)], dim=-1)


def amp_reward_from_logit(d, task_reward, coef, lerp):
    """amp_discriminator.py:64-68,70-72."""
    r = coef * torch.clamp(1 - (1 / 4) * torch.square(d - 1), min=0)
    if lerp > 0:
        r = (1.0 - lerp) * r + lerp * task_reward.unsqueeze(-1)
    return r.squeeze()


def running_moments_update(mean, var, count, arr):
    """rsl_rl/rsl_rl/utils/utils.py:90-110 in numpy, on `arr` as the reference passes it (fp32)."""
    bm, bv, bc = np.mean(arr, axis=0), np.var(arr, axis=0), arr.shape[0]
    delta = bm - mean
    tot = count + bc
    new_mean = mean + delta * bc / tot
    m2 = var * count + bv * bc + np.square(delta) * count * bc / (count + bc)
    return new_mean, m2 / (count + bc), bc + count
