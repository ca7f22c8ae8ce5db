"""Hot-path constants: one POD config (`HlCfg`, see include/himloco_b200.h) built from the
same nested config object the reference uses.

Reference: the values come from legged_gym/legged_gym/envs/aliengo/aliengo_config.py:33-292
(flat), aliengo_stairs_config.py:40-221 (stairs), aliengo_amp_config.py:41-293 (AMP),
aliengo_recover_config.py:34-174 (recover); the derived quantities follow
LeggedRobot._parse_cfg (legged_robot.py:1252-1263), _prepare_reward_function (:1035-1059),
_get_noise_scale_vec (:883-910), _process_dof_props (:560-580) and __init__ (:70-90).
"""
import ctypes
import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np

HL_MAX_TERMS = 64
HL_MAX_PTS = 32
HL_MAX_BODIES_IDX = 16

# All 51 unique `_reward_*` names of legged_robot.py:1444-1770 in sorted() order; the id of a
# term is its position here (mirrored by the enum in csrc/himloco_kernels.cuh).
REWARD_TERMS = [
    "action_rate", "ang_vel_xy", "ang_vel_xy_up", "base_height", "base_height_up", "calf_pose",
    "calf_pose_up", "collision", "collision_up", "dof_acc", "dof_pos_dif", "dof_pos_limits",
    "dof_vel", "dof_vel_limits", "feet_air_time", "feet_contact_forces", "feet_mirror",
    "feet_mirror_up", "feet_slide", "feet_slide_up", "feet_stumble", "feet_stumble_up",
    "foot_clearance_base", "foot_clearance_base_up", "foot_clearance_terrain",
    "foot_clearance_terrain_up", "has_contact", "hip_action_magnitude", "hip_pos", "hip_pos_up",
    "joint_power", "lin_vel_z", "lin_vel_z_up", "orientation", "orientation_up", "power",
    "power_distribution", "smoothness", "stand_nice", "stand_still", "stuck", "termination",
    "thigh_pose", "thigh_pose_up", "torque_limits", "torques", "torques_dif",
    "torques_distribution", "tracking_ang_vel", "tracking_lin_vel", "upward",
]
TERM_ID = {n: i for i, n in enumerate(REWARD_TERMS)}

# index-path arithmetic flavours (SURVEY.md §7 hard part 1): what eager torch does on each device
INDEX_MATH_TORCH_CUDA = 0   # x * float(1/hscale); norm(0,0,z,w) as torch's CUDA reduce rounds it
INDEX_MATH_TORCH_CPU = 1    # x / hscale (true divide); norm as torch's CPU reduce rounds it

MESH_PLANE = 0
MESH_HEIGHTFIELD = 1  # 'heightfield' and 'trimesh' both sample height_samples


class HlCfg(ctypes.Structure):
    """ctypes mirror of `struct HlCfg` in include/himloco_b200.h (keep field order identical)."""
    _fields_ = [
        ("struct_bytes", ctypes.c_int32),
        ("num_bodies", ctypes.c_int32),
        ("control_type", ctypes.c_int32),
        ("only_positive_rewards", ctypes.c_int32),
        ("n_terms", ctypes.c_int32),
        ("has_termination_term", ctypes.c_int32),
        ("add_noise", ctypes.c_int32),
        ("mesh_type", ctypes.c_int32),
        ("measure_heights", ctypes.c_int32),
        ("terrain_rows", ctypes.c_int32),
        ("terrain_cols", ctypes.c_int32),
        ("term_base_vel_violate", ctypes.c_int32),
        ("term_out_of_border", ctypes.c_int32),
        ("term_fall_down", ctypes.c_int32),
        ("heading_command", ctypes.c_int32),
        ("index_math", ctypes.c_int32),
        ("n_px", ctypes.c_int32),
        ("n_py", ctypes.c_int32),
        ("n_bx", ctypes.c_int32),
        ("n_by", ctypes.c_int32),
        ("n_penalised", ctypes.c_int32),
        ("n_term_contact", ctypes.c_int32),
        ("feet_idx", ctypes.c_int32 * 4),
        ("penalised_idx", ctypes.c_int32 * HL_MAX_BODIES_IDX),
        ("term_contact_idx", ctypes.c_int32 * HL_MAX_BODIES_IDX),
        ("term_id", ctypes.c_int32 * HL_MAX_TERMS),
        ("max_episode_length", ctypes.c_int64),
        ("env_id_offset", ctypes.c_int64),
        ("stairsup_start", ctypes.c_int64),
        ("stairsup_end", ctypes.c_int64),
        ("pit_start", ctypes.c_int64),
        ("gap_end", ctypes.c_int64),
        ("dt", ctypes.c_float),
        ("action_scale", ctypes.c_float),
        ("hip_reduction", ctypes.c_float),
        ("sim_dt", ctypes.c_float),
        ("soft_dof_vel_limit", ctypes.c_float),
        ("soft_torque_limit", ctypes.c_float),
        ("tracking_sigma", ctypes.c_float),
        ("base_height_target", ctypes.c_float),
        ("foot_height_target_base", ctypes.c_float),
        ("foot_height_target_terrain", ctypes.c_float),
        ("max_contact_force", ctypes.c_float),
        ("termination_scale", ctypes.c_float),
        ("obs_lin_vel", ctypes.c_float),
        ("obs_ang_vel", ctypes.c_float),
        ("obs_dof_pos", ctypes.c_float),
        ("obs_dof_vel", ctypes.c_float),
        ("obs_height", ctypes.c_float),
        ("clip_obs", ctypes.c_float),
        ("noise_height", ctypes.c_float),
        ("horizontal_scale", ctypes.c_float),
        ("inv_horizontal_scale", ctypes.c_float),
        ("vertical_scale", ctypes.c_float),
        ("border_size", ctypes.c_float),
        ("x_limit", ctypes.c_float),
        ("y_limit", ctypes.c_float),
        ("commands_scale", ctypes.c_float * 3),
        ("p_gains", ctypes.c_float * 12),
        ("d_gains", ctypes.c_float * 12),
        ("torque_limits", ctypes.c_float * 12),
        ("default_dof_pos", ctypes.c_float * 12),
        ("dof_pos_lo", ctypes.c_float * 12),
        ("dof_pos_hi", ctypes.c_float * 12),
        ("dof_vel_limits", ctypes.c_float * 12),
        ("noise45", ctypes.c_float * 45),
        ("term_scale", ctypes.c_float * HL_MAX_TERMS),
        ("px", ctypes.c_float * HL_MAX_PTS),
        ("py", ctypes.c_float * HL_MAX_PTS),
        ("bx", ctypes.c_float * HL_MAX_PTS),
        ("by", ctypes.c_float * HL_MAX_PTS),
    ]


# aliengo URDF limits (legged_gym/resources/robots/aliengo/urdf/aliengo.urdf:363,416,470),
# per-leg order hip, thigh, calf; DOF order FL,FR,RL,RR (legged_robot.py:1145).
_ALIENGO_POS_LIMITS = [(-0.873, 1.047), (-0.524, 3.927), (-2.775, -0.611)]
_ALIENGO_EFFORT = [44.0, 44.0, 55.0]
_ALIENGO_VELOCITY = [20.0, 20.0, 15.89]
_ALIENGO_DEFAULT = [0.0, 0.8, -1.5]

_BASE_POINTS_Y = [-0.2, -0.15, -0.1, -0.05, 0., 0.05, 0.1, 0.15, 0.2]   # legged_robot.py:1308
_BASE_POINTS_X = [-0.15, -0.1, -0.05, 0., 0.05, 0.1, 0.15]              # legged_robot.py:1309


RESET_NU = 44   # include/himloco_b200.h: HL_RESET_NU


class HlReset(ctypes.Structure):
    """Mirror of `struct HlReset` (keep field order identical to the header)."""
    _fields_ = [(n, ctypes.c_int32) for n in (
        "struct_bytes", "custom_origins", "has_pos_range", "has_rot_range", "vel_range_is_dict", "randomize_dof_pos",
        "randomize_dof_vel", "randomize_kp", "randomize_kd", "randomize_motor_strength", "heading_command",
        "terrain_curriculum", "max_terrain_level", "n_terrain_types", "parts", "pad_")] + [
        ("num_envs_global", ctypes.c_int64), ("high_vel_envs", ctypes.c_int64),
        ("base_init_state", ctypes.c_float * 13), ("pos_range", ctypes.c_float * 6), ("rot_range", ctypes.c_float * 6),
        ("vel_range", ctypes.c_float * 12), ("dof_pos_ratio", ctypes.c_float * 2), ("dof_vel_range", ctypes.c_float * 2),
        ("kp_range", ctypes.c_float * 2), ("kd_range", ctypes.c_float * 2), ("motor_strength_range", ctypes.c_float * 2),
        ("cmd_lin_vel_x", ctypes.c_float * 2), ("cmd_lin_vel_y", ctypes.c_float * 2), ("cmd_ang_vel_yaw", ctypes.c_float * 2),
        ("cmd_heading", ctypes.c_float * 2), ("env_length", ctypes.c_float),
        ("max_episode_length_s", ctypes.c_float)] + [(n, ctypes.c_void_p) for n in (
        "root_states", "dof_state", "commands", "env_origins", "terrain_origins", "terrain_levels", "terrain_types",
        "kp_factors", "kd_factors", "motor_strength_factors", "uniforms", "means_out", "means_ws", "cmd_ranges")]


def high_vel_env_count(num_envs: int) -> int:
    """Size of the high-speed command slice of _resample_commands: the global env ids with `env_ids < num_envs * 0.2`
    (LR:649), computed once per env object.  torch compares the int64 ids with the Python float in fp32, so the count
    is the number of ids below the fp32-rounded product (ids are exact in fp32 below 2**24).  The kernels compare the
    id with this integer; a product with the fp32 0.2f takes one env too many whenever num_envs is a multiple of 5."""
    n = int(num_envs)
    return min(n, math.ceil(float(np.float32(n * 0.2))))


def _f32(x) -> float:
    return float(np.float32(x))


@dataclass
class ResetCfg:
    """reset_idx / command-resampling / domain-rand settings (aliengo_config.py:102-215; the reference keeps
    them in cfg.init_state, cfg.commands and cfg.domain_rand).  `None` ranges = the reference's
    `hasattr(...)` / `getattr(..., None)` fallbacks (legged_robot.py:698,707,728,753,774)."""
    base_init_state: List[float] = field(default_factory=lambda: [0., 0., 0.50, 0., 0., 0., 1., 0., 0., 0., 0., 0., 0.])
    base_init_pos_range: Optional[Dict[str, List[float]]] = field(
        default_factory=lambda: dict(x=[-1.0, 1.0], y=[-1.0, 1.0], z=[0.0, 0.05]))
    base_init_rot_range: Optional[Dict[str, List[float]]] = field(
        default_factory=lambda: dict(roll=[-0.2, 0.2], pitch=[-0.2, 0.2], yaw=[-0.0, 0.0]))
    base_init_vel_range: object = field(
        default_factory=lambda: dict(x=[-0.5, 0.5], y=[-0.5, 0.5], z=[-0.5, 0.5], roll=[-0.5, 0.5], pitch=[-0.5, 0.5], yaw=[-0.5, 0.5]))
    dof_init_pos_ratio_range: Optional[List[float]] = field(default_factory=lambda: [0.5, 1.5])
    randomize_dof_vel: bool = True
    # the cfg file says `dof_init_vel_range = [-0.1, 0.1]` (aliengo_config.py:201) but legged_robot.py:708 reads
    # `init_dof_vel_range`, which does not exist => the reference really draws from its fallback [-1, 1]
    dof_init_vel_range: List[float] = field(default_factory=lambda: [-1.0, 1.0])
    max_forward_curriculum: float = 1.5   # aliengo_config.py:104-106
    max_backward_curriculum: float = 1.0
    max_lat_curriculum: float = 1.0
    randomize_kp: bool = True
    kp_range: List[float] = field(default_factory=lambda: [0.9, 1.1])
    randomize_kd: bool = True
    kd_range: List[float] = field(default_factory=lambda: [0.9, 1.1])
    randomize_motor_strength: bool = True
    motor_strength_range: List[float] = field(default_factory=lambda: [0.9, 1.1])
    # commands (aliengo_config.py:102-115); the curriculum moves these at run time (legged_robot.py:868-880)
    lin_vel_x: List[float] = field(default_factory=lambda: [-1.0, 1.0])
    lin_vel_y: List[float] = field(default_factory=lambda: [-0.5, 0.5])
    ang_vel_yaw: List[float] = field(default_factory=lambda: [-1.0, 1.0])
    heading: List[float] = field(default_factory=lambda: [-math.pi, math.pi])
    commands_curriculum: bool = True
    terrain_curriculum: bool = True
    # interval domain randomisation (legged_robot.py:627-632)
    push_robots: bool = True
    max_push_vel_xy: float = 1.0
    disturbance: bool = True
    disturbance_range: List[float] = field(default_factory=lambda: [-30.0, 30.0])
    delay: bool = True                   # legged_robot.py:134-138


@dataclass
class HotPathCfg:
    """Everything the kernels need, in plain Python.  Build with `aliengo(task, num_envs)` or
    `from_reference_cfg(cfg_obj, num_envs, ...)`."""
    num_envs: int = 4096                 # GLOBAL env count (all shards)
    env_id_offset: int = 0               # first global env id owned by this shard
    num_bodies: int = 17
    feet_indices: List[int] = field(default_factory=lambda: [4, 8, 12, 16])
    penalised_contact_indices: List[int] = field(
        default_factory=lambda: [2, 6, 10, 14, 3, 7, 11, 15, 0])
    termination_contact_indices: List[int] = field(default_factory=lambda: [0])
    # control (aliengo_config.py:94-100)
    control_type: str = "P"
    stiffness: float = 40.0
    damping: float = 2.0
    action_scale: float = 0.5
    hip_reduction: float = 1.0
    decimation: int = 4
    sim_dt: float = 0.005
    # env
    episode_length_s: float = 20.0
    # terrain
    mesh_type: str = "trimesh"
    measure_heights: bool = True
    horizontal_scale: float = 0.1
    vertical_scale: float = 0.005
    border_size: float = 15
    terrain_length: float = 8.0
    terrain_width: float = 8.0
    num_rows: int = 10
    num_cols: int = 20
    terrain_proportions: List[float] = field(default_factory=lambda: [0.3, 0.3, 0.2, 0.2])
    measured_points_x: List[float] = field(
        default_factory=lambda: [-0.8, -0.7, -0.6, -0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.2,
                                 0.3, 0.4, 0.5, 0.6, 0.7, 0.8])
    measured_points_y: List[float] = field(
        default_factory=lambda: [-0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.2, 0.3, 0.4, 0.5])
    # commands
    heading_command: bool = True
    resampling_time: float = 10.0
    # termination
    base_vel_violate_commands: bool = False
    out_of_border: bool = True
    fall_down: bool = True
    # rewards: raw (un-multiplied-by-dt) scales exactly as in the cfg class
    reward_scales: Dict[str, float] = field(default_factory=dict)
    only_positive_rewards: bool = False
    tracking_sigma: float = 0.25
    soft_dof_pos_limit: float = 0.95
    soft_dof_vel_limit: float = 0.95
    soft_torque_limit: float = 0.95
    base_height_target: float = 0.43
    foot_height_target_base: float = -0.27
    foot_height_target_terrain: float = 0.15
    max_contact_force: float = 100.0
    # normalisation / noise
    obs_lin_vel: float = 2.0
    obs_ang_vel: float = 0.25
    obs_dof_pos: float = 1.0
    obs_dof_vel: float = 0.05
    obs_height: float = 5.0
    clip_observations: float = 100.0
    clip_actions: float = 100.0
    add_noise: bool = True
    noise_level: float = 1.0
    noise_dof_pos: float = 0.01
    noise_dof_vel: float = 1.5
    noise_ang_vel: float = 0.2
    noise_gravity: float = 0.05
    noise_height: float = 0.1
    # domain-rand intervals (only used by the host-side step bookkeeping)
    disturbance_interval: int = 8
    push_interval_s: float = 16
    # PPO
    gamma: float = 0.99
    lam: float = 0.95
    # AMP (aliengo_amp_config.py:325,342-346)
    amp_reward_coef: float = 0.01
    amp_task_reward_lerp: float = 0.3
    # numerics
    index_math: int = INDEX_MATH_TORCH_CUDA
    # reset_idx / resampling / interval domain-rand (hooks and the in-kernel re-draws)
    reset: ResetCfg = field(default_factory=ResetCfg)
    using_amp: bool = False              # step() returns the 8-tuple of legged_robot.py:173-174

    # ----------------------------------------------------------------- derived (reference rules)
    @property
    def dt(self) -> float:                       # legged_robot.py:1253
        return self.decimation * self.sim_dt

    @property
    def max_episode_length(self) -> int:         # legged_robot.py:1261 (np.ceil)
        return int(np.ceil(self.episode_length_s / self.dt))

    @property
    def resample_interval(self) -> int:          # legged_robot.py:612
        return int(self.resampling_time / self.dt)

    @property
    def push_interval(self) -> int:              # legged_robot.py:1263
        return int(np.ceil(self.push_interval_s / self.dt))

    @property
    def is_plane(self) -> bool:
        return self.mesh_type == "plane"

    @property
    def terrain_shape(self):                     # terrain.py:55-62
        wpp = int(self.terrain_width / self.horizontal_scale)
        lpp = int(self.terrain_length / self.horizontal_scale)
        border = int(self.border_size / self.horizontal_scale)
        return (int(self.num_rows * lpp) + 2 * border, int(self.num_cols * wpp) + 2 * border)

    @property
    def x_size(self) -> float:                   # terrain.py:49
        return self.terrain_length * self.num_rows

    @property
    def y_size(self) -> float:
        return self.terrain_width * self.num_cols

    def active_terms(self):
        """(names, scales*dt) in accumulation order: sorted(name) with zero scales dropped and
        `termination` taken out of the loop (legged_robot.py:1041-1055; helpers.py:45-60 walks
        dir(), hence alphabetical)."""
        names, scales = [], []
        for name in sorted(self.reward_scales.keys()):
            s = self.reward_scales[name]
            if s == 0 or name == "termination":
                continue
            if name not in TERM_ID:
                raise AttributeError(f"'LeggedRobot' object has no attribute '_reward_{name}'")
            names.append(name)
            scales.append(s * self.dt)
        return names, scales

    @property
    def termination_scale(self) -> Optional[float]:
        s = self.reward_scales.get("termination", 0)
        return None if s == 0 else s * self.dt

    def episode_sum_names(self):
        """Row order of the (R, N) episode_sums buffer: loop terms then `termination`."""
        names, _ = self.active_terms()
        if self.termination_scale is not None:
            names = names + ["termination"]
        return names

    def noise_scale_vec(self) -> np.ndarray:     # legged_robot.py:883-910
        n = 45 + (len(self.measured_points_x) * len(self.measured_points_y) if self.measure_heights else 0)
        v = np.zeros(n, dtype=np.float32)
        lvl = self.noise_level
        v[3:6] = self.noise_ang_vel * lvl * self.obs_ang_vel
        v[6:9] = self.noise_gravity * lvl
        v[9:21] = self.noise_dof_pos * lvl * self.obs_dof_pos
        v[21:33] = self.noise_dof_vel * lvl * self.obs_dof_vel
        if self.measure_heights:
            v[45:] = self.noise_height * lvl * self.obs_height
        return v

    def dof_tables(self):
        """p_gains, d_gains, torque_limits, default_dof_pos, soft pos limits, vel limits (12,)."""
        lo, hi, eff, vel, dflt = [], [], [], [], []
        for _leg in range(4):
            for j in range(3):
                l, h = np.float32(_ALIENGO_POS_LIMITS[j][0]), np.float32(_ALIENGO_POS_LIMITS[j][1])
                # legged_robot.py:574-578, evaluated in fp32 tensors there
                m = (l + h) / np.float32(2)
                r = h - l
                soft = self.soft_dof_pos_limit
                lo.append(np.float32(m - np.float32(0.5) * r * np.float32(soft)))
                hi.append(np.float32(m + np.float32(0.5) * r * np.float32(soft)))
                eff.append(_ALIENGO_EFFORT[j])
                vel.append(_ALIENGO_VELOCITY[j])
                dflt.append(_ALIENGO_DEFAULT[j])
        f = lambda x: np.asarray(x, dtype=np.float32)
        return dict(p_gains=f([self.stiffness] * 12), d_gains=f([self.damping] * 12),
                    torque_limits=f(eff), default_dof_pos=f(dflt), dof_pos_lo=f(lo),
                    dof_pos_hi=f(hi), dof_vel_limits=f(vel))

    def stumble_ranges(self):
        """Global env-index slices of legged_robot.py:71-90,1597-1598."""
        tp = list(self.terrain_proportions) + [0.0] * 10
        n = self.num_envs
        return dict(stairsup_start=math.ceil(n * sum(tp[:4])), stairsup_end=math.ceil(n * sum(tp[:5])),
                    pit_start=math.ceil(n * sum(tp[:8])), gap_end=n)

    # ----------------------------------------------------------------- C struct
    def to_c(self) -> HlCfg:
        c = HlCfg()
        c.struct_bytes = ctypes.sizeof(HlCfg)
        c.num_bodies = self.num_bodies
        c.control_type = {"P": 0, "V": 1, "T": 2}.get(self.control_type, -1)
        if c.control_type < 0:
            raise NameError(f"Unknown controller type: {self.control_type}")  # legged_robot.py:687
        c.only_positive_rewards = int(self.only_positive_rewards)
        names, scales = self.active_terms()
        if len(names) > HL_MAX_TERMS:
            raise ValueError("too many reward terms")
        c.n_terms = len(names)
        for k, (nm, sc) in enumerate(zip(names, scales)):
            c.term_id[k] = TERM_ID[nm]
            c.term_scale[k] = sc
        ts = self.termination_scale
        c.has_termination_term = int(ts is not None)
        c.termination_scale = 0.0 if ts is None else ts
        c.add_noise = int(self.add_noise)
        if self.mesh_type == "none":
            raise NameError("Can't measure height with terrain mesh type 'none'")  # legged_robot.py:1334
        c.mesh_type = MESH_PLANE if self.is_plane else MESH_HEIGHTFIELD
        c.measure_heights = int(self.measure_heights)
        rows, cols = self.terrain_shape if not self.is_plane else (2, 2)
        c.terrain_rows, c.terrain_cols = rows, cols
        c.term_base_vel_violate = int(self.base_vel_violate_commands)
        c.term_out_of_border = int(self.out_of_border and not self.is_plane)
        c.term_fall_down = int(self.fall_down)
        c.heading_command = int(self.heading_command)
        c.index_math = self.index_math
        c.n_px, c.n_py = len(self.measured_points_x), len(self.measured_points_y)
        c.n_bx, c.n_by = len(_BASE_POINTS_X), len(_BASE_POINTS_Y)
        for i, v in enumerate(self.measured_points_x):
            c.px[i] = v
        for i, v in enumerate(self.measured_points_y):
            c.py[i] = v
        for i, v in enumerate(_BASE_POINTS_X):
            c.bx[i] = v
        for i, v in enumerate(_BASE_POINTS_Y):
            c.by[i] = v
        c.n_penalised = len(self.penalised_contact_indices)
        c.n_term_contact = len(self.termination_contact_indices)
        for i, v in enumerate(self.feet_indices):
            c.feet_idx[i] = v
        for i, v in enumerate(self.penalised_contact_indices):
            c.penalised_idx[i] = v
        for i, v in enumerate(self.termination_contact_indices):
            c.term_contact_idx[i] = v
        c.max_episode_length = self.max_episode_length
        c.env_id_offset = self.env_id_offset
        sr = self.stumble_ranges()
        c.stairsup_start, c.stairsup_end = sr["stairsup_start"], sr["stairsup_end"]
        c.pit_start, c.gap_end = sr["pit_start"], sr["gap_end"]
        c.dt = self.dt
        c.action_scale = self.action_scale
        c.hip_reduction = self.hip_reduction
        c.sim_dt = self.sim_dt
        c.soft_dof_vel_limit = self.soft_dof_vel_limit
        c.soft_torque_limit = self.soft_torque_limit
        c.tracking_sigma = self.tracking_sigma
        c.base_height_target = self.base_height_target
        c.foot_height_target_base = self.foot_height_target_base
        c.foot_height_target_terrain = self.foot_height_target_terrain
        c.max_contact_force = self.max_contact_force
        c.obs_lin_vel, c.obs_ang_vel = self.obs_lin_vel, self.obs_ang_vel
        c.obs_dof_pos, c.obs_dof_vel = self.obs_dof_pos, self.obs_dof_vel
        c.obs_height = self.obs_height
        c.clip_obs = self.clip_observations
        nv = self.noise_scale_vec()
        for i in range(45):
            c.noise45[i] = float(nv[i])
        c.noise_height = float(nv[45]) if self.measure_heights else 0.0
        c.horizontal_scale = self.horizontal_scale
        # torch CUDA `tensor / python_scalar` multiplies by the fp32 reciprocal (div_true_kernel_cuda)
        c.inv_horizontal_scale = float(np.float32(1.0) / np.float32(self.horizontal_scale))
        c.vertical_scale = self.vertical_scale
        c.border_size = self.border_size
        c.x_limit = self.x_size + self.border_size / 2      # terrain.py:226
        c.y_limit = self.y_size + self.border_size / 2
        c.commands_scale[0] = c.commands_scale[1] = self.obs_lin_vel   # legged_robot.py:968
        c.commands_scale[2] = self.obs_ang_vel
        t = self.dof_tables()
        for name in ("p_gains", "d_gains", "torque_limits", "default_dof_pos", "dof_pos_lo",
                     "dof_pos_hi", "dof_vel_limits"):
            arr = getattr(c, name)
            for i in range(12):
                arr[i] = float(t[name][i])
        return c


_FLAT_SCALES = dict(                       # aliengo_config.py:217-256
    termination=-0.0, tracking_lin_vel=1.5, tracking_ang_vel=1.5, lin_vel_z=-2.0, ang_vel_xy=-0.05,
    orientation=-2.0, base_height=-8.0, torques=-0.0002, torque_limits=-0.0, dof_vel=-0.0,
    dof_acc=-2.5e-7, stand_still=-0.1, hip_pos=-0.2, thigh_pose=-0.05, calf_pose=-0.05,
    dof_pos_limits=-0.0, dof_vel_limits=-0.0, joint_power=-2e-5, feet_mirror=-0.05,
    action_rate=-0.02, smoothness=-0.01, hip_action_magnitude=-0.0, collision=-0.0,
    feet_contact_forces=-0.00015, feet_air_time=0.25, has_contact=0.0, feet_stumble=-0.0,
    feet_slide=-0.01, foot_clearance_base=-0.1, foot_clearance_base_terrain=-0.0, stuck=-0.01,
    upward=0.0)
_STAIRS_SCALES = dict(                     # aliengo_stairs_config.py:171-210
    termination=-50., tracking_lin_vel=1.5, tracking_ang_vel=0.75, lin_vel_z=-2.0, ang_vel_xy=-0.05,
    orientation=-0.2, base_height=-5.0, torques=-0.0002, torque_limits=-0.0, dof_vel=-0.0,
    dof_acc=-2.5e-7, stand_still=-0.01, hip_pos=-0.2, thigh_pose=-0.1, calf_pose=-0.1,
    dof_pos_limits=-0.0, dof_vel_limits=-0.0, joint_power=-6e-5, feet_mirror=-0.0,
    action_rate=-0.01, smoothness=-0.0, hip_action_magnitude=-0.0, collision=-3.0,
    feet_contact_forces=-0.00015, feet_air_time=0.1, has_contact=0.0, feet_stumble=-1.0,
    feet_slide=-0.01, foot_clearance_base=-0.0, foot_clearance_base_terrain=-0.0, stuck=-1.,
    upward=0.0)
_RECOVER_SCALES = dict(                    # aliengo_recover_config.py:113-146
    termination=-0.0, tracking_lin_vel=2.0, tracking_ang_vel=1.0, lin_vel_z_up=-2.0,
    ang_vel_xy_up=-0.05, orientation_up=-2.0, base_height_up=-5.0, torques=-0.0002,
    torque_limits=-0.0, dof_vel=-0.0, dof_acc=-2.5e-7, stand_nice=-0.1, hip_pos_up=-0.3,
    thigh_pose_up=-0.05, calf_pose_up=-0.05, dof_pos_limits=-0.0, dof_vel_limits=-0.0,
    joint_power=-2e-5, feet_mirror_up=-0.05, action_rate=-0.02, smoothness=-0.01,
    hip_action_magnitude=-0.01, collision_up=-0.0, feet_contact_forces=-0.00015,
    feet_air_time=0.25, has_contact=0.3, feet_stumble_up=-0.0, feet_slide_up=-0.01,
    foot_clearance_base_up=-0.1, foot_clearance_base_terrain=-0.0, stuck=-0.05, upward=1.0)


def aliengo(task: str = "flat", num_envs: int = 4096, **overrides) -> HotPathCfg:
    """The four aliengo task configs of the reference, as constants."""
    if task == "flat":
        cfg = HotPathCfg(num_envs=num_envs, reward_scales=dict(_FLAT_SCALES))
    elif task == "amp":
        sc = dict(_FLAT_SCALES)
        sc["base_height"] = -10.0                      # aliengo_amp_config.py:226
        # aliengo_amp_config.py has no `termination` class: check_termination (LR:266-283) then keeps
        # only the contact and time-out clauses
        cfg = HotPathCfg(num_envs=num_envs, reward_scales=sc, out_of_border=False, fall_down=False, using_amp=True)
        cfg.reset.max_forward_curriculum = 2.0          # aliengo_amp_config.py (commands.max_forward_curriculum)
    elif task == "stairs":
        cfg = HotPathCfg(
            num_envs=num_envs, reward_scales=dict(_STAIRS_SCALES), terrain_length=10.0,
            terrain_width=10.0,
            terrain_proportions=[0.0, 0.0, 0.1, 0.1, 0.3, 0.3, 0.2, 0.0, 0.0, 0.0],
            base_vel_violate_commands=True)
    elif task == "recover":
        # aliengo_recover_config.py:70,79,89,95-96,153: two terrain types, no heading command,
        # base contact does not terminate, clipped-at-zero rewards
        cfg = HotPathCfg(num_envs=num_envs, reward_scales=dict(_RECOVER_SCALES),
                         only_positive_rewards=True, heading_command=False,
                         terrain_proportions=[0.5, 0.5], termination_contact_indices=[])
        cfg.reset.max_forward_curriculum = 2.0
        cfg.reset.base_init_rot_range = dict(roll=[-3.14, 3.14], pitch=[-3.14, 3.14], yaw=[-3.14, 3.14])   # aliengo_recover_config.py
    else:
        raise ValueError(f"unknown task {task!r}")
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


def _scales_to_dict(obj) -> Dict[str, float]:
    return {k: getattr(obj, k) for k in dir(obj) if not k.startswith("_")
            and isinstance(getattr(obj, k), (int, float))}


def from_reference_cfg(rc, num_envs: Optional[int] = None, sim_dt: float = 0.005, env=None) -> HotPathCfg:
    """Build from an instance of the reference's nested config classes (duck-typed; this module
    never imports the reference).  `env` (optional) = the reference LeggedRobot being patched: its
    own body index tensors (`feet_indices`, `penalised_contact_indices`,
    `termination_contact_indices`, resolved from the asset at LR:1207-1218) then replace the
    aliengo defaults."""
    t, ctl, rw, nz, norm = rc.terrain, rc.control, rc.rewards, rc.noise, rc.normalization
    term = getattr(rc, "termination", None)
    idx = {}
    for name in ("feet_indices", "penalised_contact_indices", "termination_contact_indices"):
        v = getattr(env, name, None) if env is not None else None
        if v is not None:
            idx[name] = [int(x) for x in (v.tolist() if hasattr(v, "tolist") else v)]
    asset = getattr(rc, "asset", None)
    if "termination_contact_indices" not in idx and asset is not None and \
            list(getattr(asset, "terminate_after_contacts_on", ["base"])) == []:
        idx["termination_contact_indices"] = []          # e.g. aliengo_recover_config.py:97
    cfg = HotPathCfg(
        num_envs=num_envs or rc.env.num_envs,
        control_type=ctl.control_type, stiffness=list(ctl.stiffness.values())[0],
        damping=list(ctl.damping.values())[0], action_scale=ctl.action_scale,
        hip_reduction=getattr(ctl, "hip_reduction", 1.0), decimation=ctl.decimation, sim_dt=sim_dt,
        episode_length_s=rc.env.episode_length_s, mesh_type=t.mesh_type,
        measure_heights=t.measure_heights, horizontal_scale=t.horizontal_scale,
        vertical_scale=t.vertical_scale, border_size=t.border_size,
        terrain_length=t.terrain_length, terrain_width=t.terrain_width, num_rows=t.num_rows,
        num_cols=t.num_cols, terrain_proportions=list(t.terrain_proportions),
        measured_points_x=list(t.measured_points_x), measured_points_y=list(t.measured_points_y),
        heading_command=rc.commands.heading_command, resampling_time=rc.commands.resampling_time,
        base_vel_violate_commands=bool(getattr(term, "base_vel_violate_commands", False)),
        out_of_border=bool(getattr(term, "out_of_border", False)),
        fall_down=bool(getattr(term, "fall_down", False)),
        reward_scales=_scales_to_dict(rw.scales), only_positive_rewards=rw.only_positive_rewards,
        tracking_sigma=rw.tracking_sigma, soft_dof_pos_limit=rw.soft_dof_pos_limit,
        soft_dof_vel_limit=rw.soft_dof_vel_limit, soft_torque_limit=rw.soft_torque_limit,
        base_height_target=rw.base_height_target,
        foot_height_target_base=getattr(rw, "foot_height_target_base", -0.27),
        foot_height_target_terrain=getattr(rw, "foot_height_target_terrain", 0.15),
        max_contact_force=rw.max_contact_force,
        obs_lin_vel=norm.obs_scales.lin_vel, obs_ang_vel=norm.obs_scales.ang_vel,
        obs_dof_pos=norm.obs_scales.dof_pos, obs_dof_vel=norm.obs_scales.dof_vel,
        obs_height=norm.obs_scales.height_measurements, clip_observations=norm.clip_observations,
        clip_actions=norm.clip_actions, add_noise=nz.add_noise, noise_level=nz.noise_level,
        noise_dof_pos=nz.noise_scales.dof_pos, noise_dof_vel=nz.noise_scales.dof_vel,
        noise_ang_vel=nz.noise_scales.ang_vel, noise_gravity=nz.noise_scales.gravity,
        noise_height=nz.noise_scales.height_measurements,
        disturbance_interval=getattr(rc.domain_rand, "disturbance_interval", 8),
        push_interval_s=getattr(rc.domain_rand, "push_interval_s", 16),
        **idx,
    )
    dr, init, cmd = rc.domain_rand, rc.init_state, rc.commands
    g = lambda o, k, d=None: getattr(o, k, d)
    cfg.reset = ResetCfg(
        base_init_state=list(init.pos) + list(init.rot) + list(init.lin_vel) + list(init.ang_vel),
        base_init_pos_range=g(dr, "base_init_pos_range"), base_init_rot_range=g(dr, "base_init_rot_range"),
        base_init_vel_range=g(dr, "base_init_vel_range") if g(dr, "base_init_vel_range") is not None else (-0.5, 0.5),
        dof_init_pos_ratio_range=g(dr, "dof_init_pos_ratio_range"), randomize_dof_vel=bool(g(dr, "randomize_dof_vel", False)),
        dof_init_vel_range=list(g(dr, "init_dof_vel_range", [-1.0, 1.0])),        # sic: legged_robot.py:708 reads `init_dof_vel_range`
        randomize_kp=bool(g(dr, "randomize_kp", False)), kp_range=list(g(dr, "kp_range", [1.0, 1.0])),
        randomize_kd=bool(g(dr, "randomize_kd", False)), kd_range=list(g(dr, "kd_range", [1.0, 1.0])),
        randomize_motor_strength=bool(g(dr, "randomize_motor_strength", False)),
        motor_strength_range=list(g(dr, "motor_strength_range", [1.0, 1.0])),
        lin_vel_x=list(cmd.ranges.lin_vel_x), lin_vel_y=list(cmd.ranges.lin_vel_y), ang_vel_yaw=list(cmd.ranges.ang_vel_yaw),
        heading=list(cmd.ranges.heading), commands_curriculum=bool(g(cmd, "curriculum", False)),
        terrain_curriculum=bool(g(t, "curriculum", False)), push_robots=bool(g(dr, "push_robots", False)),
        max_push_vel_xy=float(g(dr, "max_push_vel_xy", 1.0)), disturbance=bool(g(dr, "disturbance", False)),
        disturbance_range=list(g(dr, "disturbance_range", [-30.0, 30.0])), delay=bool(g(dr, "delay", False)),
        max_forward_curriculum=float(g(cmd, "max_forward_curriculum", 1.5)),
        max_backward_curriculum=float(g(cmd, "max_backward_curriculum", 1.0)), max_lat_curriculum=float(g(cmd, "max_lat_curriculum", 1.0)))
    return cfg
