"""FusedLeggedRobot: the post-physics half of `LeggedRobot`
(reference: legged_gym/legged_gym/envs/base/legged_robot.py, cited as LR) behind the same method
names, attribute names, dtypes and in-place side effects, executed by libhimloco_b200's CUDA
kernels.

What stays torch / host (out of scope, SURVEY.md §2): PhysX itself and every `gym.*` call (issued here in the
reference's order when `self.gym` exists), pushes and disturbances (torch RNG written into PhysX-owned tensors),
the host-side command curriculum, friction re-randomisation.  The reset hooks (`_reset_dofs`, `_reset_root_states`,
`_resample_commands`, `_update_terrain_curriculum`) run in the kernels by default (Philox, or pre-drawn uniforms in
parity mode); overriding any of them with torch code (subclass / mix in the reference class, INTEGRATION.md) makes
the step fall back to fused -> host sync -> torch reset_idx -> fix-up.  `physics_step_fn` feeds replayed or synthetic
PhysX state.

One env-step (post_physics_step_device, no host sync, CUDA-graph capturable):
    gym.refresh_* x4, common_step_counter += 1                                      LR:187-194
    [torch] disturbance / push on their interval steps (the push step takes the staged path)   LR:624-632
    hl_post_physics_fused      command resampling on the interval mark, counters, frame, contacts, heading,
                               187+63-point scans, termination, rewards, speculative obs + last_* roll
                               [+ ordered reset ids and terminal rows for shards <= 16,384 envs]   LR:193-241,612-613
    hl_select_and_terminal     env_ids = reset_buf.nonzero().flatten(); termination_privileged_obs,
                               terminal_amp_states of those envs                     LR:225-228
    hl_reset_and_fixup         reset_idx (curriculum, dof / root / command re-draws, gain factors, buffer zeroing,
                               extras["episode"] means) + re-scan, obs slot 0 and roll of the reset envs
                                                                                    LR:229-241,288-361
post_physics_step() adds the one `.item()` its return signature needs, after everything is queued, hands the
re-drawn rows to PhysX (`set_*_state_tensor_indexed`) and, on a step with resets, builds extras["episode"].
"""
import ctypes
import math
import os
from typing import Callable, Dict, Optional

import torch

from . import _lib as L
from .config import HlReset, HotPathCfg, high_vel_env_count


class FusedLeggedRobot:
    """Standalone env shard over replayed/synthetic PhysX tensors.  All tensors live on `device`
    (a CUDA device) and carry the reference's attribute names."""

    def __init__(self, cfg: HotPathCfg, state: Dict[str, torch.Tensor], height_samples: torch.Tensor,
                 device="cuda:0", physics_step_fn: Optional[Callable] = None, seed: int = 0):
        self.cfg = cfg
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("FusedLeggedRobot runs on CUDA only (no CPU fallback)")
        n = state["root_states"].shape[0]
        self.num_envs = n
        self.num_actions = self.num_dof = self.num_dofs = 12
        self.num_bodies = cfg.num_bodies
        self.num_one_step_obs = 45
        self.num_height_points = len(cfg.measured_points_x) * len(cfg.measured_points_y)
        self.num_one_step_privileged_obs = 51 + (self.num_height_points if cfg.measure_heights else 0)
        self.num_obs, self.num_privileged_obs = 270, self.num_one_step_privileged_obs
        self.dt = cfg.dt
        self.max_episode_length = cfg.max_episode_length
        self.common_step_counter = 0
        self.extras = {}
        self.physics_step_fn = physics_step_fn
        dev = self.device
        f32 = lambda k: state[k].to(dev, torch.float32).contiguous()
        # --- PhysX-owned tensors, Isaac Gym layouts (LR:929-944)
        self.root_states = f32("root_states")
        self.dof_state = f32("dof_state")
        self.dof_pos = self.dof_state.view(n, 12, 2)[..., 0]
        self.dof_vel = self.dof_state.view(n, 12, 2)[..., 1]
        self.base_quat = self.root_states[:, 3:7]
        self.rigid_body_states = f32("rigid_body_states")
        self.contact_forces = f32("contact_forces").view(n, -1, 3)
        # --- policy-side buffers (LR:954-1032)
        for k in ("actions", "last_actions", "last_last_actions", "last_dof_pos", "last_dof_vel", "torques",
                  "last_torques", "last_root_vel", "commands", "feet_air_time", "motor_strength",
                  "Kp_factors", "Kd_factors", "disturbance", "obs_buf", "privileged_obs_buf"):
            setattr(self, k, f32(k))
        self.episode_length_buf = state["episode_length_buf"].to(dev, torch.long).contiguous()
        self.terrain_levels = state["terrain_levels"].to(dev, torch.long).contiguous()
        self.last_contacts = state["last_contacts"].to(dev, torch.bool).contiguous()
        self.base_lin_vel = f32("base_lin_vel")
        self.base_ang_vel = f32("base_ang_vel")
        self.projected_gravity = f32("projected_gravity")
        self.rew_buf = torch.zeros(n, device=dev)
        self.reset_buf = torch.ones(n, dtype=torch.bool, device=dev)
        self.time_out_buf = torch.zeros(n, dtype=torch.bool, device=dev)
        self.height_samples = height_samples.to(dev, torch.int16).contiguous()
        self._initial_episode_sums = state.get("episode_sums")
        self._hl_attach(cfg, seed=seed)

    def _hl_attach(self, cfg: HotPathCfg, seed: int = 0):
        """Everything the kernels need on top of the reference's own buffers (LR:913-1032).  Also the
        hook for mixing this class into the reference's LeggedRobot (INTEGRATION.md §2): call it at
        the end of `_init_buffers` once the PhysX tensors are wrapped."""
        self.cfg_hot = cfg
        if not hasattr(self, "cfg") or self.cfg is None:
            self.cfg = cfg
        dev = self.device = torch.device(self.device)
        n = self.num_envs
        self.num_height_points = len(cfg.measured_points_x) * len(cfg.measured_points_y)
        self.num_one_step_privileged_obs = 51 + (self.num_height_points if cfg.measure_heights else 0)
        for name, shape, dt in (("contact_filt", (n, 4), torch.bool), ("feet_pos", (n, 4, 3), torch.float32),
                                ("feet_vel", (n, 4, 3), torch.float32),
                                ("measured_heights", (n, self.num_height_points), torch.float32),
                                ("joint_pos_target", (n, 12), torch.float32),
                                ("delayed_actions", (n, cfg.decimation, 12), torch.float32)):
            cur = getattr(self, name, None)
            if not (isinstance(cur, torch.Tensor) and tuple(cur.shape) == shape and cur.dtype == dt
                    and cur.is_contiguous() and cur.device == dev):
                setattr(self, name, torch.zeros(*shape, dtype=dt, device=dev))
        if self.reset_buf.dtype != torch.bool:                 # base_task.py:72 starts it as int64 ones
            self.reset_buf = self.reset_buf.to(torch.bool)
        self._base_heights = torch.zeros(n, device=dev)
        # episode sums: one (R,N) buffer; the dict holds row views so reference code keeps working
        names = cfg.episode_sum_names()
        self._episode_sums_buf = torch.zeros(max(len(names), 1), n, device=dev)
        init = getattr(self, "_initial_episode_sums", None)
        if init is not None and len(names):
            self._episode_sums_buf[:len(names)].copy_(init[:len(names)].to(dev))
        self.episode_sums = {nm: self._episode_sums_buf[k] for k, nm in enumerate(names)}
        self.reward_names, scales = cfg.active_terms()
        self.reward_scales = dict(zip(self.reward_names, scales))
        if cfg.termination_scale is not None:
            self.reward_scales["termination"] = cfg.termination_scale
        # constants the reference keeps as tensors
        t = cfg.dof_tables()
        tt = lambda a: torch.tensor(a, device=dev)
        self.default_dof_pos = tt(t["default_dof_pos"]).view(1, 12)
        self.p_gains, self.d_gains = tt(t["p_gains"]), tt(t["d_gains"])
        self.torque_limits, self.dof_vel_limits = tt(t["torque_limits"]), tt(t["dof_vel_limits"])
        self.dof_pos_limits = torch.stack([tt(t["dof_pos_lo"]), tt(t["dof_pos_hi"])], dim=-1)
        self.noise_scale_vec = tt(cfg.noise_scale_vec())
        self.add_noise = cfg.add_noise
        self.feet_indices = torch.tensor(cfg.feet_indices, dtype=torch.long, device=dev)
        self.penalised_contact_indices = torch.tensor(cfg.penalised_contact_indices, dtype=torch.long, device=dev)
        self.termination_contact_indices = torch.tensor(cfg.termination_contact_indices, dtype=torch.long, device=dev)
        # terrain: the one-off min-of-3 table
        self._height_min3 = None
        self._height_min3f = None
        # reset-id compaction + terminal rows (capacity N; counts live on the device)
        self._reset_ids = torch.zeros(n, dtype=torch.long, device=dev)
        self._n_reset = torch.zeros(1, dtype=torch.int32, device=dev)
        self._term_priv = torch.zeros(n, self.num_one_step_privileged_obs, device=dev)
        self._term_amp = torch.zeros(n, 30, device=dev)
        self._select_ws = torch.zeros(int(L.lib.hl_select_workspace_bytes(n)), dtype=torch.uint8, device=dev)
        self._fused_ws = torch.zeros(int(L.lib.hl_fused_workspace_bytes(n)), dtype=torch.uint8, device=dev)
        self._selterm_ws = torch.zeros(int(L.lib.hl_select_terminal_workspace_bytes(n)), dtype=torch.uint8, device=dev)
        # ids + terminal rows straight from the fused kernel: wins in the launch-bound small-N regime,
        # costs more than the separate compaction launch at large N (measured, DESIGN.md §4)
        self.single_launch = n <= 16384
        if os.environ.get("HL_SINGLE_LAUNCH") in ("0", "1"):      # A/B knob
            self.single_launch = os.environ["HL_SINGLE_LAUNCH"] == "1"
        # noise: Philox by default; parity tests install pre-drawn tensors
        self._noise = {}
        self._philox_seed = int(seed)
        self._c = cfg.to_c()
        self._bufs = None
        self._fused_event_hook = None      # bench.py: CUDA-event pair around the fused kernel
        self._rollout = None               # bind_rollout(): storage whose slots the env writes in place
        self._philox_bias = 0
        # device step counter for replayed rollouts (capture_rollout): while a graph is captured the kernels key step k
        # as *_step_base + k (_capture_base = the host counter the capture started at); None = keys by value
        self._step_base = torch.zeros(1, dtype=torch.long, device=dev)
        self._capture_base = None
        self._ep_log = None                # RolloutGraph: (tables, row) the step's episode logging goes to
        self._reset_sets_physx = False
        self._prepare_terrain()
        self._init_reset_state()

    # ------------------------------------------------------------------ plumbing
    def _prepare_terrain(self):
        if self.cfg_hot.is_plane:
            return
        rows, cols = self.height_samples.shape
        if (rows, cols) != tuple(self.cfg_hot.terrain_shape):
            raise ValueError(f"height_samples is {rows}x{cols}, cfg expects {self.cfg_hot.terrain_shape}")
        self._height_min3 = torch.empty(rows - 1, cols - 1, dtype=torch.int16, device=self.device)
        L.check(L.lib.hl_terrain_prepare(L.ptr(self.height_samples), rows, cols, L.ptr(self._height_min3), L.stream()))
        # the same table in metres (fp32): one gather per scan point in the persistent fused kernel
        self._height_min3f = torch.empty(rows - 1, cols - 1, dtype=torch.float32, device=self.device)
        L.check(L.lib.hl_terrain_prepare_f32(L.ptr(self.height_samples), rows, cols, float(self.cfg_hot.vertical_scale),
                                             L.ptr(self._height_min3f), L.stream()))

    def set_noise_tensors(self, obs45=None, obs187=None, term45=None, term187=None):
        """Parity mode: the U[0,1) draws `torch.rand_like` would return at LR:394,400 (obs) and
        LR:451,457 (terminal obs).  None => in-kernel Philox."""
        cv = lambda t: None if t is None else t.to(self.device, torch.float32).contiguous()
        self._noise = dict(obs45=cv(obs45), obs187=cv(obs187), term45=cv(term45), term187=cv(term187))
        self._bufs = None

    def refresh_buffers(self):
        """Call after rebinding any tensor attribute (pointers are cached in a C struct)."""
        self._bufs = None

    # ------------------------------------------------------------------ zero-copy rollout slots
    def bind_rollout(self, storage):
        """Make the env read its observation history from rollout slot `storage.step` and write the
        new observations / privileged observations into slot step+1 of a
        HIMRolloutStorage(env_writes_slots=True): add_transitions' two largest copies
        (him_rollout_storage.py:97-98) disappear because transition.observations and
        .critic_observations already ARE the slots.  bind_rollout(None) detaches."""
        if storage is None:
            if getattr(self, "_rollout", None) is not None:
                self.obs_buf, self.privileged_obs_buf = self.obs_buf.clone(), self.privileged_obs_buf.clone()
            self._rollout = None
            self._bufs = None
            return
        if not getattr(storage, "env_writes_slots", False):
            raise ValueError("bind_rollout needs HIMRolloutStorage(env_writes_slots=True)")
        s = storage.step
        storage.obs_slot(s).copy_(self.obs_buf)
        storage.priv_slot(s).copy_(self.privileged_obs_buf)
        self.obs_buf, self.privileged_obs_buf = storage.obs_slot(s), storage.priv_slot(s)
        self._rollout = storage
        self._bufs = None

    def _bind_rollout_slot(self, bufs):
        st = self._rollout
        s = st.step
        if s >= st.num_transitions_per_env:
            raise AssertionError("Rollout buffer overflow")     # as add_transitions would (him_rollout_storage.py:94)
        self.obs_buf, self.privileged_obs_buf = st.obs_slot(s + 1), st.priv_slot(s + 1)
        bufs.obs_buf_in = L.ptr(st.obs_slot(s))
        bufs.obs_buf_out = L.ptr(self.obs_buf)
        bufs.privileged_obs_buf = L.ptr(self.privileged_obs_buf)

    def _step_key(self):
        """(philox_offset, step_base): the step index by value, or relative to the device counter while a rollout
        graph is captured (a replay then keys its steps by the counter it finds on the device)."""
        k = self.common_step_counter + self._philox_bias
        if self._capture_base is None:
            return k, None
        return k - self._capture_base, L.ptr(self._step_base)

    def _buffers(self) -> L.HlEnvBuffers:
        if self._bufs is not None:
            self._bufs.philox_offset, self._bufs.step_base = self._step_key()
            return self._bufs
        b = L.HlEnvBuffers()
        b.struct_bytes = ctypes.sizeof(L.HlEnvBuffers)
        p = L.ptr
        b.root_states, b.dof_state = p(self.root_states), p(self.dof_state)
        b.contact_forces, b.rigid_body_states = p(self.contact_forces), p(self.rigid_body_states)
        b.foot_records = p(getattr(self, "foot_records", None))     # optional packed (N,4,13): replaces rigid_body_states[:, feet]
        b.height_samples = p(self.height_samples)
        b.height_min3 = p(self._height_min3)
        b.height_min3f = p(self._height_min3f)
        b.fused_ws = p(self._fused_ws)        # tile ticket of the persistent kernel (+ look-back states)
        b.actions, b.last_actions, b.last_last_actions = p(self.actions), p(self.last_actions), p(self.last_last_actions)
        b.last_dof_pos, b.last_dof_vel = p(self.last_dof_pos), p(self.last_dof_vel)
        b.torques, b.last_torques, b.last_root_vel = p(self.torques), p(self.last_torques), p(self.last_root_vel)
        b.commands, b.episode_length_buf = p(self.commands), p(self.episode_length_buf)
        b.last_contacts, b.contact_filt = p(self.last_contacts), p(self.contact_filt)
        b.feet_air_time, b.disturbance = p(self.feet_air_time), p(self.disturbance)
        b.terrain_levels, b.episode_sums = p(self.terrain_levels), p(self._episode_sums_buf)
        b.base_lin_vel, b.base_ang_vel = p(self.base_lin_vel), p(self.base_ang_vel)
        b.projected_gravity, b.measured_heights = p(self.projected_gravity), p(self.measured_heights)
        b.feet_pos, b.feet_vel = p(self.feet_pos), p(self.feet_vel)
        b.reset_buf, b.time_out_buf, b.rew_buf = p(self.reset_buf), p(self.time_out_buf), p(self.rew_buf)
        b.obs_buf_in = b.obs_buf_out = p(self.obs_buf)
        b.privileged_obs_buf = p(self.privileged_obs_buf)
        b.noise_u45, b.noise_u187 = p(self._noise.get("obs45")), p(self._noise.get("obs187"))
        b.philox_seed = self._philox_seed
        b.philox_offset, b.step_base = self._step_key()
        b.height_idx_out = None
        b.base_height_out = p(self._base_heights)
        if self.single_launch:
            b.reset_ids_out, b.n_reset_out = p(self._reset_ids), p(self._n_reset)
            b.term_priv_out, b.term_amp_out = p(self._term_priv), p(self._term_amp)
            b.term_noise_u45, b.term_noise_u187 = p(self._noise.get("term45")), p(self._noise.get("term187"))
        self._bufs = b
        return b

    def _stages(self, stages: int, env_ids: Optional[torch.Tensor] = None, n_ids: Optional[torch.Tensor] = None):
        if env_ids is not None and n_ids is None:
            if env_ids.numel() == 0:
                return
            env_ids = env_ids.to(self.device, torch.long).contiguous()
            n_ids = torch.tensor([env_ids.numel()], dtype=torch.int32, device=self.device)
        L.check(L.lib.hl_post_physics_stages(ctypes.byref(self._c), ctypes.byref(self._buffers()), stages,
                                             L.ptr(env_ids), L.ptr(n_ids), self.num_envs, L.stream()))

    # ------------------------------------------------------------------ the reference's methods
    def _compute_torques(self, actions):
        """LR:658-688.  `actions` may be a column slice of delayed_actions (row-strided)."""
        if actions.stride(-1) != 1:
            actions = actions.contiguous()
        out = torch.empty(self.num_envs, 12, device=self.device)
        L.check(L.lib.hl_pd_torque(ctypes.byref(self._c), L.ptr(actions), actions.stride(0), L.ptr(self.dof_state),
                                   L.ptr(self.motor_strength), L.ptr(self.Kp_factors), L.ptr(self.Kd_factors),
                                   L.ptr(self.last_dof_vel), L.ptr(out), L.ptr(self.joint_pos_target), self.num_envs,
                                   L.stream()))
        return out

    def _compute_torques_into(self, actions, out):
        """Same, writing into a preallocated (N,12) tensor (no allocation; graph-capturable)."""
        L.check(L.lib.hl_pd_torque(ctypes.byref(self._c), L.ptr(actions), actions.stride(0), L.ptr(self.dof_state),
                                   L.ptr(self.motor_strength), L.ptr(self.Kp_factors), L.ptr(self.Kd_factors),
                                   L.ptr(self.last_dof_vel), L.ptr(out), L.ptr(self.joint_pos_target), self.num_envs,
                                   L.stream()))
        return out

    def _get_heights(self, env_ids=None):
        """LR:1318-1355 -> (N,187); the scan itself always covers every env like the reference's
        `env_ids=None` path (the only one it ever takes)."""
        self._stages(L.ST_HEIGHTS)
        return self.measured_heights

    def _get_base_heights(self, env_ids=None):
        """LR:1357-1398 -> (N,)."""
        self._stages(L.ST_BASE_HEIGHT)
        return self._base_heights

    def get_height_indices(self):
        """Debug/parity: the clipped (px,py) cell of every scan point, (N,187,2) int32."""
        idx = torch.empty(self.num_envs, self.num_height_points, 2, dtype=torch.int32, device=self.device)
        b = self._buffers()
        b.height_idx_out = L.ptr(idx)
        try:
            self._stages(L.ST_HEIGHTS)
        finally:
            b.height_idx_out = None
        return idx

    def update_base_frame(self):
        """LR:197-209: base_lin_vel, base_ang_vel, projected_gravity, feet_pos/vel, contacts."""
        self._stages(L.ST_FRAME | L.ST_CONTACTS)

    def update_heading_command(self):
        """LR:616-620."""
        self._stages(L.ST_HEADING)

    def check_termination(self):
        """LR:249-286 (sets reset_buf, time_out_buf; the dead .item() bookkeeping is dropped)."""
        self._stages(L.ST_TERMINATION)

    def compute_reward(self):
        """LR:363-380."""
        self._stages(L.ST_REWARD)

    def compute_observations(self):
        """LR:382-404."""
        self._stages(L.ST_OBS)

    def compute_termination_observations(self, env_ids):
        """LR:439-460 -> (len(env_ids), 238)."""
        env_ids = env_ids.to(self.device, torch.long).contiguous()
        if env_ids.numel() == 0:
            return self._term_priv[:0]
        n_ids = torch.tensor([env_ids.numel()], dtype=torch.int32, device=self.device)
        self._terminal_rows(env_ids, n_ids)
        return self._term_priv[:env_ids.numel()]

    def get_amp_observations(self):
        """LR:406-416 -> (N,30)."""
        out = torch.empty(self.num_envs, 30, device=self.device)
        L.check(L.lib.hl_amp_observations(L.ptr(self.dof_state), L.ptr(self.base_lin_vel), L.ptr(self.base_ang_vel),
                                          L.ptr(out), self.num_envs, L.stream()))
        return out

    def _terminal_rows(self, env_ids, n_ids):
        L.check(L.lib.hl_terminal_rows(ctypes.byref(self._c), ctypes.byref(self._buffers()), L.ptr(env_ids), L.ptr(n_ids),
                                       L.ptr(self._noise.get("term45")), L.ptr(self._noise.get("term187")),
                                       L.ptr(self._term_priv), L.ptr(self._term_amp), self.num_envs, L.stream()))

    # ------------------------------------------------------------------ fused step pieces
    def fused_pre_reset(self, select=True):
        """Launch the fused kernel, the id compaction and the terminal rows; no host sync.  select=False: the caller
        runs the compaction itself (hl_select_terminal_reset: ids + terminal rows + reset + fix-up in one launch)."""
        bufs = self._buffers()
        if getattr(self, "_rollout", None) is not None:
            self._bind_rollout_slot(bufs)
        c, b = ctypes.byref(self._c), ctypes.byref(bufs)
        ev = self._fused_event_hook() if self._fused_event_hook is not None else None
        L.check(L.lib.hl_post_physics_fused(c, b, self.num_envs, L.stream()))
        if ev is not None:
            ev()
        bufs.flags |= 1          # HL_BUF_HISTORY_CLIPPED: the step just clipped the whole obs_buf (LR:168)
        bufs.resample_host, bufs.resample_interval = None, 0      # (set per step by post_physics_step_device)
        if self.single_launch or not select:
            return               # ids, count and terminal rows came out of the same launch (or the caller's next one)
        L.check(L.lib.hl_select_and_terminal(c, b, L.ptr(self._noise.get("term45")), L.ptr(self._noise.get("term187")),
                                             L.ptr(self._reset_ids), L.ptr(self._n_reset), L.ptr(self._term_priv),
                                             L.ptr(self._term_amp), L.ptr(self._selterm_ws), self.num_envs, L.stream()))

    def fused_post_reset(self, with_reset_zero: bool = False):
        """Patch the reset envs after reset_idx.  with_reset_zero=True also applies reset_idx's own
        RNG-free buffer resets in the kernel (for replay loops that skip the torch reset_idx)."""
        L.check(L.lib.hl_post_reset_fixup(ctypes.byref(self._c), ctypes.byref(self._buffers()), L.ptr(self._reset_ids),
                                          L.ptr(self._n_reset), int(with_reset_zero), self.num_envs, L.stream()))

    # ------------------------------------------------------------------ reset state (LR:288-361) in the kernel chain
    def _init_reset_state(self):
        """Buffers reset_idx needs on top of the hot-path ones (LR:1221-1250,1013-1023); idempotent."""
        dev, n, R = self.device, self.num_envs, self.cfg_hot.reset
        z = lambda *shape, **kw: torch.zeros(*shape, device=dev, **kw)
        if not isinstance(getattr(self, "env_origins", None), torch.Tensor):
            self.env_origins = z(n, 3)
        if not hasattr(self, "custom_origins"):
            self.custom_origins = not self.cfg_hot.is_plane            # LR:1226
        if not hasattr(self, "terrain_origins"):
            self.terrain_origins, self.terrain_types = None, None
        if not hasattr(self, "max_terrain_level"):
            self.max_terrain_level = self.cfg_hot.num_rows               # LR:1235
        if not isinstance(getattr(self, "motor_strength_factors", None), torch.Tensor):
            self.motor_strength_factors = torch.ones(n, 1, device=dev)  # LR:1013
        if not isinstance(getattr(self, "base_init_state", None), torch.Tensor):
            self.base_init_state = torch.tensor(R.base_init_state, device=dev)
        self._base_init_host = [float(x) for x in self.base_init_state.tolist()]   # host copy: no sync per step
        if not hasattr(self, "command_ranges"):
            self.command_ranges = dict(lin_vel_x=list(R.lin_vel_x), lin_vel_y=list(R.lin_vel_y),
                                       ang_vel_yaw=list(R.ang_vel_yaw), heading=list(R.heading))
        if not hasattr(self, "init_done"):
            self.init_done = True
        # device copy of command_ranges (HlReset.cmd_ranges order), read by the kernels only in the device-schedule mode of
        # RolloutGraph.run(); _cmd_ranges_mirror = the host values it holds (None = not uploaded yet)
        self._cmd_ranges_dev = z(8, dtype=torch.float64)
        self._cmd_ranges_mirror = None
        self._device_schedule = False
        self._high_vel_envs = high_vel_env_count(self.cfg_hot.num_envs)         # LR:649, keyed by the global env id
        self._reset_uniforms = None           # parity mode: (N, RESET_NU) pre-drawn U[0,1)
        self._episode_means = z(max(self._episode_sums_buf.shape[0], 1))
        self._means_ws = z(self._episode_sums_buf.shape[0] + 1, dtype=torch.float64)      # zeroed once; the kernel re-arms it
        self.push_interval = int(math.ceil(self.cfg_hot.push_interval_s / self.dt))     # LR:1263
        self.resample_interval = int(self.cfg_hot.resampling_time / self.dt)            # LR:612
        self.max_episode_length_s = self.cfg_hot.episode_length_s

    def set_reset_uniforms(self, u):
        """Parity mode for the in-kernel reset_idx / _resample_commands: row e of `u` (N, 44) holds the
        U[0,1) draws env e consumes (column map: include/himloco_b200.h).  None => in-kernel Philox."""
        self._reset_uniforms = None if u is None else u.to(self.device, torch.float32).contiguous()

    def _reset_struct(self, parts: int = 0) -> HlReset:
        R, r = self.cfg_hot.reset, HlReset()
        r.struct_bytes = ctypes.sizeof(HlReset)
        r.custom_origins = int(bool(self.custom_origins))
        pr, rr, vr = R.base_init_pos_range, R.base_init_rot_range, R.base_init_vel_range
        r.has_pos_range = int(pr is not None)
        if pr is not None:
            r.pos_range[:] = [*pr["x"], *pr["y"], *pr["z"]]
        r.has_rot_range = int(rr is not None)
        if rr is not None:
            r.rot_range[:] = [*rr["roll"], *rr["pitch"], *rr.get("yaw", [-math.pi, math.pi])]
        if isinstance(vr, dict):
            r.vel_range_is_dict = 1
            r.vel_range[:] = [*vr["x"], *vr["y"], *vr["z"], *vr["roll"], *vr["pitch"], *vr["yaw"]]
        elif isinstance(vr, (tuple, list)):
            r.vel_range[0], r.vel_range[1] = vr[0], vr[1]
        else:
            raise NameError(f"Unknown base_vel_range type: {type(vr)}")           # LR:818
        r.randomize_dof_pos = int(R.dof_init_pos_ratio_range is not None)
        if R.dof_init_pos_ratio_range is not None:
            r.dof_pos_ratio[:] = R.dof_init_pos_ratio_range
        r.randomize_dof_vel = int(R.randomize_dof_vel)
        r.dof_vel_range[:] = R.dof_init_vel_range
        r.randomize_kp, r.randomize_kd, r.randomize_motor_strength = int(R.randomize_kp), int(R.randomize_kd), int(R.randomize_motor_strength)
        r.kp_range[:], r.kd_range[:], r.motor_strength_range[:] = R.kp_range, R.kd_range, R.motor_strength_range
        r.heading_command = int(self.cfg_hot.heading_command)
        if self._device_schedule:
            # the kernels read the device copy; the by-value fields stay zero, so a captured graph's signature does not
            # change when the curriculum or the user moves the ranges
            r.cmd_ranges = L.ptr(self._cmd_ranges_dev)
        else:
            cr = self.command_ranges
            r.cmd_lin_vel_x[:], r.cmd_lin_vel_y[:] = cr["lin_vel_x"], cr["lin_vel_y"]
            r.cmd_ang_vel_yaw[:], r.cmd_heading[:] = cr["ang_vel_yaw"], cr["heading"]
        r.num_envs_global = self.cfg_hot.num_envs
        r.high_vel_envs = self._high_vel_envs
        has_cur = R.terrain_curriculum and self.init_done and self.terrain_origins is not None and self.terrain_types is not None
        r.terrain_curriculum = int(bool(has_cur))
        r.max_terrain_level = int(self.max_terrain_level)
        r.n_terrain_types = int(self.terrain_origins.shape[1]) if self.terrain_origins is not None else 0
        r.env_length = float(self.cfg_hot.terrain_length)
        r.max_episode_length_s = float(self.max_episode_length_s)
        r.base_init_state[:] = self._base_init_host
        r.parts = parts
        p = L.ptr
        r.root_states, r.dof_state, r.commands = p(self.root_states), p(self.dof_state), p(self.commands)
        r.env_origins, r.terrain_origins = p(self.env_origins), p(self.terrain_origins)
        r.terrain_levels, r.terrain_types = p(self.terrain_levels), p(self.terrain_types)
        r.kp_factors, r.kd_factors = p(self.Kp_factors), p(self.Kd_factors)
        r.motor_strength_factors = p(self.motor_strength_factors)
        r.uniforms = p(self._reset_uniforms)
        return r

    def _uw(self, t):
        """gymtorch.unwrap_tensor when mixed into the reference env (set `self._unwrap = gymtorch.unwrap_tensor`,
        INTEGRATION.md §2); identity for replayed / synthetic PhysX state."""
        f = getattr(self, "_unwrap", None)
        return f(t) if f is not None else t

    def _ids_arg(self, env_ids):
        env_ids = env_ids.to(self.device, torch.long).contiguous()
        return env_ids, torch.tensor([env_ids.numel()], dtype=torch.int32, device=self.device)

    def _reset_part(self, env_ids, parts):
        if len(env_ids) == 0:
            return
        ids, cnt = self._ids_arg(env_ids)
        r = self._reset_struct(parts)
        if parts == L.RESET_COMMANDS:
            L.check(L.lib.hl_resample_commands(ctypes.byref(self._c), ctypes.byref(self._buffers()), ctypes.byref(r), L.ptr(ids),
                                               L.ptr(cnt), 0, self.num_envs, L.stream()))
            return
        # the individual hooks: only that part, no buffer zeroing
        L.check(L.lib.hl_reset_draw(ctypes.byref(self._c), ctypes.byref(self._buffers()), ctypes.byref(r), L.ptr(ids), L.ptr(cnt),
                                   self.num_envs, L.stream()))

    # the reference's hooks: in-kernel by default (Philox); subclass / mix in torch versions to override
    def _reset_dofs(self, env_ids):
        """LR:690-716 (the PhysX setter the reference calls at the end stays with the caller)."""
        self._reset_part(env_ids, L.RESET_DOFS)
        gym = getattr(self, "gym", None)
        if gym is not None and len(env_ids):
            gym.set_dof_state_tensor_indexed(self.sim, self._uw(self.dof_state), self._uw(env_ids.to(torch.int32)), len(env_ids))

    def _reset_root_states(self, env_ids):
        """LR:718-820."""
        self._reset_part(env_ids, L.RESET_ROOT)
        gym = getattr(self, "gym", None)
        if gym is not None and len(env_ids):
            gym.set_actor_root_state_tensor_indexed(self.sim, self._uw(self.root_states), self._uw(env_ids.to(torch.int32)), len(env_ids))

    def _resample_commands(self, env_ids):
        """LR:634-656."""
        self._reset_part(env_ids, L.RESET_COMMANDS)

    def _update_terrain_curriculum(self, env_ids):
        """LR:845-866."""
        if self.init_done and self.terrain_origins is not None:
            self._reset_part(env_ids, L.RESET_CURRICULUM)

    def reset_idx_device(self, env_ids, n_ids_dev=None, fixup=False):
        """reset_idx's kernel form on a device id list (count on the device): curriculum, state re-draws, buffer
        zeroing [+ the post-reset fix-up].  No host sync."""
        if n_ids_dev is None:
            env_ids, n_ids_dev = self._ids_arg(env_ids)
        r = self._reset_struct()
        fn = L.lib.hl_reset_and_fixup if fixup else L.lib.hl_reset_idx
        L.check(fn(ctypes.byref(self._c), ctypes.byref(self._buffers()), ctypes.byref(r), L.ptr(env_ids), L.ptr(n_ids_dev),
                   self.num_envs, L.stream()))

    def _kernel_reset_ok(self) -> bool:
        """True when none of the three state hooks is overridden: reset_idx then runs in the kernel chain."""
        base = FusedLeggedRobot
        t = type(self)
        return (t._reset_dofs is base._reset_dofs and t._reset_root_states is base._reset_root_states
                and t._resample_commands is base._resample_commands and t.reset_idx is base.reset_idx)

    def _push_robots(self):
        """LR:822-828 (torch RNG; PhysX-facing)."""
        mv = self.cfg_hot.reset.max_push_vel_xy
        self.root_states[:, 7:9] = (2 * mv) * torch.rand(self.num_envs, 2, device=self.device) - mv
        gym = getattr(self, "gym", None)
        if gym is not None:
            gym.set_actor_root_state_tensor(self.sim, self._uw(self.root_states))

    def _disturbance_robots(self):
        """LR:838-844 (torch RNG; PhysX-facing)."""
        lo, hi = self.cfg_hot.reset.disturbance_range
        self.disturbance[:, 0, :] = (hi - lo) * torch.rand(self.num_envs, 3, device=self.device) + lo
        gym = getattr(self, "gym", None)
        if gym is not None:
            gym.apply_rigid_body_force_tensors(self.sim, forceTensor=self._uw(self.disturbance), space=getattr(self, "_local_space", "LOCAL_SPACE"))

    def update_command_curriculum(self, env_ids):
        """LR:868-880 (host state: the shared command ranges)."""
        import numpy as np
        R = self.cfg_hot.reset
        if "tracking_lin_vel" not in self.episode_sums or len(env_ids) == 0:
            return
        mean = torch.mean(self.episode_sums["tracking_lin_vel"][env_ids]) / self.max_episode_length
        if float(mean) > 0.8 * self.reward_scales["tracking_lin_vel"]:
            cr = self.command_ranges
            cr["lin_vel_x"][0] = float(np.clip(cr["lin_vel_x"][0] - 0.1, -getattr(R, "max_backward_curriculum", 1.0), 0.))
            cr["lin_vel_x"][1] = float(np.clip(cr["lin_vel_x"][1] + 0.1, 0., getattr(R, "max_forward_curriculum", 1.5)))
            cr["lin_vel_y"][0] = float(np.clip(cr["lin_vel_y"][0] - 0.1, -getattr(R, "max_lat_curriculum", 1.0), 0.))
            cr["lin_vel_y"][1] = float(np.clip(cr["lin_vel_y"][1] + 0.1, 0., getattr(R, "max_lat_curriculum", 1.0)))

    # ------------------------------------------------------------------ device-resident command ranges
    COMMAND_RANGE_KEYS = ("lin_vel_x", "lin_vel_y", "ang_vel_yaw", "heading")

    def command_ranges_flat(self):
        """command_ranges as the 8 floats of HlReset.cmd_ranges (lo, hi of lin_vel_x, lin_vel_y, ang_vel_yaw, heading)."""
        return tuple(float(self.command_ranges[k][j]) for k in self.COMMAND_RANGE_KEYS for j in (0, 1))

    def set_command_ranges_flat(self, vals):
        """Write 8 floats into command_ranges, in place (the lists keep their identity)."""
        for i, k in enumerate(self.COMMAND_RANGE_KEYS):
            self.command_ranges[k][0], self.command_ranges[k][1] = float(vals[2 * i]), float(vals[2 * i + 1])

    def _upload_command_ranges(self):
        """Copy command_ranges to the device copy when they differ from what it holds (a host edit, or the first use)."""
        host = self.command_ranges_flat()
        if host != self._cmd_ranges_mirror:
            self._cmd_ranges_dev.copy_(torch.tensor(host, dtype=torch.float64))
            self._cmd_ranges_mirror = host

    def _device_curriculum_ok(self) -> bool:
        """The command curriculum can run on the device: update_command_curriculum is not overridden."""
        return type(self).update_command_curriculum is FusedLeggedRobot.update_command_curriculum

    def _command_curriculum_device(self, ranges_log=None):
        """update_command_curriculum(reset ids) on the device copy of the ranges: one launch, no host sync
        (hl_command_curriculum; its float64 sum can decide differently from torch's fp32 mean only within a few ulp of
        the threshold).  ranges_log: an (8,) float64 row that receives the ranges after the decision, or None."""
        if "tracking_lin_vel" not in self.episode_sums:
            return
        R = self.cfg_hot.reset
        L.check(L.lib.hl_command_curriculum(
            L.ptr(self.episode_sums["tracking_lin_vel"]), L.ptr(self._reset_ids), L.ptr(self._n_reset),
            0.8 * self.reward_scales["tracking_lin_vel"], int(self.max_episode_length),
            float(getattr(R, "max_backward_curriculum", 1.0)), float(getattr(R, "max_forward_curriculum", 1.5)),
            float(getattr(R, "max_lat_curriculum", 1.0)), L.ptr(self._cmd_ranges_dev), L.ptr(ranges_log), self.num_envs,
            L.stream()))

    def _pre_step_callbacks(self, resample_in_fused=False):
        """The RNG-driven part of _post_physics_step_callback that precedes the fused step (LR:612-613,631-632):
        commands of the envs whose incremented episode length hits the resampling interval (in-kernel, Philox
        stream 2 or the parity uniforms; `resample_in_fused`: the fused kernel does it itself), then the interval
        disturbance."""
        R = self.cfg_hot.reset
        if resample_in_fused:
            pass
        elif self.resample_interval > 0 and type(self)._resample_commands is FusedLeggedRobot._resample_commands:
            r = self._reset_struct(L.RESET_COMMANDS)
            L.check(L.lib.hl_resample_commands(ctypes.byref(self._c), ctypes.byref(self._buffers()), ctypes.byref(r), None, None,
                                               self.resample_interval, self.num_envs, L.stream()))
        elif self.resample_interval > 0:
            ids = ((self.episode_length_buf + 1) % self.resample_interval == 0).nonzero(as_tuple=False).flatten()
            self._resample_commands(ids)
        if R.disturbance and self.common_step_counter % self.cfg_hot.disturbance_interval == 0:
            self._disturbance_robots()

    def _log_episode(self):
        """extras of reset_idx (LR:344-359) after a kernel-chain step with resets.  Like the reference, every such step
        gets a fresh dict of fresh tensors (a runner that keeps infos["episode"] of every step sees each step's own
        means) and a step without resets leaves the previous dict in place.  The masked means come from the reset launch
        itself; terrain_level is taken from the post-reset levels, after this step's curriculum moves (LR:352-353)."""
        means = self._episode_means.clone()
        ep = {"rew_" + key: means[k] for k, key in enumerate(self.episode_sums.keys())}
        if self.cfg_hot.reset.terrain_curriculum and self.terrain_origins is not None:
            ep["terrain_level"] = torch.mean(self.terrain_levels.float())
        if self.cfg_hot.reset.commands_curriculum:
            ep["max_command_x"] = self.command_ranges["lin_vel_x"][1]
        self.extras["episode"] = ep
        self.extras["time_outs"] = self.time_out_buf

    def post_physics_step_device(self):
        """LR:178-247 as ONE chain of launches without a host sync (CUDA-graph capturable when no torch hook is
        overridden): returns the capacity-N id / terminal-row buffers and the device count.  post_physics_step()
        is this plus the one `.item()` the reference's return signature needs, issued after everything is queued.
        With the in-kernel reset this chain only writes the episode means to a device buffer: building
        extras["episode"] (allocations, and only on steps with resets) is left to the caller, post_physics_step()."""
        R = self.cfg_hot.reset
        gym = getattr(self, "gym", None)
        if gym is not None:                                   # LR:187-190
            gym.refresh_actor_root_state_tensor(self.sim)
            gym.refresh_net_contact_force_tensor(self.sim)
            gym.refresh_force_sensor_tensor(self.sim)
            gym.refresh_rigid_body_state_tensor(self.sim)
        self.common_step_counter += 1                         # LR:194 (episode_length_buf += 1 happens in the kernel)
        self._philox_bias = -1                                # noise streams stay keyed by the step index 0, 1, 2, ...
        try:
            push_now = R.push_robots and self.push_interval > 0 and self.common_step_counter % self.push_interval == 0
            merged = False
            # the default callbacks: the fused kernel resamples the commands on the mark itself (one launch less)
            own_cb = type(self)._pre_step_callbacks is FusedLeggedRobot._pre_step_callbacks
            in_fused = (own_cb and not push_now and self.resample_interval > 0
                        and type(self)._resample_commands is FusedLeggedRobot._resample_commands)
            self._resample_struct = self._reset_struct(L.RESET_COMMANDS) if in_fused else None
            bufs = self._buffers()
            bufs.resample_host = ctypes.cast(ctypes.pointer(self._resample_struct), ctypes.c_void_p) if in_fused else None
            bufs.resample_interval = self.resample_interval if in_fused else 0
            if own_cb:
                self._pre_step_callbacks(resample_in_fused=in_fused)
            else:
                self._pre_step_callbacks()
            if push_now:
                # LR:627-628: the push changes root_states[:, 7:9] AFTER base_lin_vel was taken and BEFORE rewards /
                # observations: the staged path splits the step around it (1 step in push_interval)
                if getattr(self, "_rollout", None) is not None:
                    self._bind_rollout_slot(self._buffers())   # read slot step, write slot step+1, as the fused path does
                self._stages(L.ST_COUNTERS | L.ST_FRAME | L.ST_CONTACTS)
                self._push_robots()
                self._stages(L.ST_HEADING | L.ST_HEIGHTS | L.ST_TERMINATION | L.ST_REWARD)
                bufs = self._buffers()
                L.check(L.lib.hl_select_and_terminal(ctypes.byref(self._c), ctypes.byref(bufs), L.ptr(self._noise.get("term45")),
                                                     L.ptr(self._noise.get("term187")), L.ptr(self._reset_ids), L.ptr(self._n_reset),
                                                     L.ptr(self._term_priv), L.ptr(self._term_amp), L.ptr(self._selterm_ws),
                                                     self.num_envs, L.stream()))
            else:
                # HL_MERGED_RESET=1: ids + terminal rows + reset + fix-up as ONE launch after the fused kernel.  Measured at
                # 65,536 envs: 34.3 us vs 16.2 + 17.3 us for the two launches (256 CTAs do serially what the separate
                # fix-up spreads over the whole GPU), so the two-launch form stays the default.
                merged = (os.environ.get("HL_MERGED_RESET") == "1" and self._kernel_reset_ok() and not self.single_launch
                          and not (R.commands_curriculum and self.common_step_counter % self.max_episode_length == 0))
                self.fused_pre_reset(select=not merged)
            if self._kernel_reset_ok():
                if R.commands_curriculum and self.common_step_counter % self.max_episode_length == 0:   # LR:306-307 (1 step in 1000)
                    if self._device_schedule and self._device_curriculum_ok():
                        log = None if self._ep_log is None else self._ep_log[0].ranges_log[self._ep_log[1]]
                        self._command_curriculum_device(log)
                    else:
                        self.update_command_curriculum(self._reset_ids[:int(self._n_reset.item())])
                r = self._reset_struct()
                means = self._episode_means if self._ep_log is None else self._ep_log[0].means[self._ep_log[1]]
                r.means_out, r.means_ws = L.ptr(means), L.ptr(self._means_ws)
                c, b = ctypes.byref(self._c), ctypes.byref(self._buffers())
                if push_now:
                    L.check(L.lib.hl_reset_idx(c, b, ctypes.byref(r), L.ptr(self._reset_ids), L.ptr(self._n_reset), self.num_envs, L.stream()))
                    self._stages(L.ST_HEIGHTS, self._reset_ids, self._n_reset)
                    self._stages(L.ST_OBS | L.ST_OBS_CLIP | L.ST_ROLL)
                elif merged:
                    L.check(L.lib.hl_select_terminal_reset(c, b, ctypes.byref(r), L.ptr(self._noise.get("term45")),
                                                           L.ptr(self._noise.get("term187")), L.ptr(self._reset_ids), L.ptr(self._n_reset),
                                                           L.ptr(self._term_priv), L.ptr(self._term_amp), L.ptr(self._selterm_ws),
                                                           self.num_envs, L.stream()))
                else:
                    L.check(L.lib.hl_reset_and_fixup(c, b, ctypes.byref(r), L.ptr(self._reset_ids), L.ptr(self._n_reset), self.num_envs,
                                                     L.stream()))
                self._reset_sets_physx = True
                if self._ep_log is not None:
                    self._ep_log[0].record(self, self._ep_log[1])
            else:
                n_reset = int(self._n_reset.item())          # torch hooks need the ids on the host side (LR:225,298)
                self.reset_idx(self._reset_ids[:n_reset])
                if push_now:
                    self._stages(L.ST_HEIGHTS, self._reset_ids, self._n_reset)
                    self._stages(L.ST_OBS | L.ST_OBS_CLIP | L.ST_ROLL)
                else:
                    self.fused_post_reset()
        finally:
            self._philox_bias = 0
        return self._reset_ids, self._n_reset, self._term_priv, self._term_amp

    def post_physics_step(self):
        """LR:178-247 -> (env_ids, termination_privileged_obs, terminal_amp_states)."""
        ids, n_dev, term_priv, term_amp = self.post_physics_step_device()
        n_reset = int(n_dev.item())                          # after the whole chain is queued: the GPU never waits for it
        env_ids = ids[:n_reset]
        gym = getattr(self, "gym", None)
        if gym is not None and n_reset and getattr(self, "_reset_sets_physx", False):
            ids32 = env_ids.to(torch.int32)                   # LR:713-716,817-820: hand the re-drawn rows to PhysX
            gym.set_dof_state_tensor_indexed(self.sim, self._uw(self.dof_state), self._uw(ids32), n_reset)
            gym.set_actor_root_state_tensor_indexed(self.sim, self._uw(self.root_states), self._uw(ids32), n_reset)
        if n_reset and self._kernel_reset_ok():
            self._log_episode()                               # LR:344-359 (the torch-hook reset_idx logs itself)
        if n_reset and getattr(self, "_reset_sets_physx", False) and hasattr(self, "refresh_actor_rigid_shape_props"):
            self.refresh_actor_rigid_shape_props(env_ids)     # LR:343: friction / restitution re-draw (PhysX actor props)
        return env_ids, term_priv[:n_reset], term_amp[:n_reset]

    def step(self, actions):
        """LR:122-176.  7-tuple, or the 8-tuple with terminal_amp_states when cfg.using_amp (LR:173-176)."""
        clip = self.cfg_hot.clip_actions
        torch.clamp(actions.to(self.device), -clip, clip, out=self.actions)
        self._delay_actions()
        gym = getattr(self, "gym", None)
        if gym is not None and hasattr(self, "render"):
            self.render()                                     # LR:131
        for k in range(self.cfg_hot.decimation):
            self._compute_torques_into(self.delayed_actions[:, k], self.torques)
            if gym is not None:                               # LR:148-152
                gym.set_dof_actuation_force_tensor(self.sim, self._uw(self.torques))
                gym.simulate(self.sim)
                gym.fetch_results(self.sim, True)
                gym.refresh_dof_state_tensor(self.sim)
            if self.physics_step_fn is not None:
                self.physics_step_fn(self, k)
        env_ids, term_priv, term_amp = self.post_physics_step()
        self.extras["terminal_amp_states"] = term_amp
        out = (self.obs_buf, self.privileged_obs_buf, self.rew_buf, self.reset_buf, self.extras, env_ids, term_priv)
        return out + (term_amp,) if self.cfg_hot.using_amp else out

    def step_device(self, actions):
        """step() without the host sync, for CUDA-graph capture: clip, delay, `decimation` x (PD torques,
        physics_step_fn), post_physics_step_device().  Returns (obs_buf, privileged_obs_buf, rew_buf, reset_buf, extras,
        reset_ids, n_reset, termination_privileged_obs, terminal_amp_states): the id and terminal-row buffers have
        capacity N and the count n_reset is a (1,) int32 device tensor (HIMRolloutStorage.record_env_step takes it as
        termination_count).  extras["episode"] is not built here (RolloutGraph.run() returns the episode logging).
        A live Isaac Gym sim cannot be stepped this way: gym.simulate is a host call that a graph cannot capture."""
        if getattr(self, "gym", None) is not None:
            raise RuntimeError("step_device() needs standalone physics (physics_step_fn): gym.simulate cannot be captured")
        clip = self.cfg_hot.clip_actions
        torch.clamp(actions.to(self.device), -clip, clip, out=self.actions)
        self._delay_actions()
        for k in range(self.cfg_hot.decimation):
            self._compute_torques_into(self.delayed_actions[:, k], self.torques)
            if self.physics_step_fn is not None:
                self.physics_step_fn(self, k)
        ids, n_dev, term_priv, term_amp = self.post_physics_step_device()
        self.extras["time_outs"] = self.time_out_buf
        self.extras["terminal_amp_states"] = term_amp
        return (self.obs_buf, self.privileged_obs_buf, self.rew_buf, self.reset_buf, self.extras, ids, n_dev, term_priv,
                term_amp)

    def capture_rollout(self, body: Callable[[int], None], num_steps: int, storage=None, finish: Optional[Callable[[], None]] = None,
                        max_graphs: int = 8, warmup: int = 1, capture_schedule: bool = False, amp=None, episode_stats=None):
        """A RolloutGraph that runs `body(0) .. body(num_steps - 1)` then `finish()` as one captured CUDA graph whenever
        the rollout window allows it, and eagerly otherwise (rollout_graph.py).  `body(k)` is the runner's per-step
        code (act -> step_device -> storage.record_env_step(..., termination_count=n_reset)); `finish` e.g.
        compute_returns; `storage`: the HIMRolloutStorage the body records into.  `max_graphs` bounds the cache of
        captured graphs; the first `warmup` rollouts run eagerly.  `capture_schedule=True` also replays windows with
        push and command-curriculum steps: inside run() the command ranges live on the device and the curriculum
        decides there (its float64 sum can differ from the host's fp32 mean within a few ulp of the threshold).
        `amp`: the AMPRolloutStep (amp_rollout.py) whose step() `body` calls, for the hybrid (AMP) runner.
        `episode_stats`: the EpisodeStats (episode_stats.py) whose record() `body` calls; run() fills its rewbuffer /
        lenbuffer."""
        from .rollout_graph import RolloutGraph
        return RolloutGraph(self, body, num_steps, storage=storage, finish=finish, max_graphs=max_graphs, warmup=warmup,
                            capture_schedule=capture_schedule, amp=amp, episode_stats=episode_stats)

    # ------------------------------------------------------------------ torch-side hooks (RNG / PhysX)
    def _delay_actions(self):
        """LR:133-138: per-env random action delay, only when cfg.domain_rand.delay."""
        dec = self.cfg_hot.decimation
        if not self.cfg_hot.reset.delay:
            self.delayed_actions.copy_(self.actions.unsqueeze(1).expand(-1, dec, -1))
            return
        delay = torch.randint(0, dec, (self.num_envs, 1), device=self.device)
        steps = torch.arange(dec, device=self.device).view(1, dec, 1)
        mask = (steps >= delay.view(-1, 1, 1)).to(self.actions.dtype)
        torch.add(self.last_actions.unsqueeze(1), (self.actions - self.last_actions).unsqueeze(1) * mask,
                  out=self.delayed_actions)

    def reset_idx(self, env_ids):
        """LR:288-361 through the hooks (used when a hook is overridden with torch code, or when called directly);
        post_physics_step runs the same work as one launch when no hook is overridden.  The full-N height re-scan
        of LR:332-333 is replaced by the targeted re-scan of the fix-up (non-reset envs did not move)."""
        if len(env_ids) == 0:
            return
        R = self.cfg_hot.reset
        if R.terrain_curriculum:
            self._update_terrain_curriculum(env_ids)
        if R.commands_curriculum and (self.common_step_counter % self.max_episode_length == 0):
            self.update_command_curriculum(env_ids)
        self._reset_dofs(env_ids)
        self._reset_root_states(env_ids)
        self._resample_commands(env_ids)
        self.last_actions[env_ids] = 0.0
        self.last_last_actions[env_ids] = 0.0
        self.last_dof_pos[env_ids] = 0.0
        self.last_dof_vel[env_ids] = 0.0
        self.last_torques[env_ids] = 0.0
        self.feet_air_time[env_ids] = 0.0
        self.reset_buf[env_ids] = True
        if type(self)._reset_dofs is FusedLeggedRobot._reset_dofs:   # LR:336-341 (kernel form: same uniform columns)
            self._reset_part(env_ids, L.RESET_FACTORS)
        self.extras["episode"] = {}
        if self.episode_sums:   # LR:346-350 as one launch (means of every row over the reset ids, rows zeroed)
            ids, cnt = self._ids_arg(env_ids)
            rows = self._episode_sums_buf.shape[0]
            means = torch.empty(rows, device=self.device)
            L.check(L.lib.hl_episode_means(L.ptr(self._episode_sums_buf), L.ptr(self.episode_length_buf), L.ptr(ids),
                                           L.ptr(cnt), rows, self.num_envs, float(self.dt), 1, L.ptr(means), L.stream()))
            for k, key in enumerate(self.episode_sums.keys()):
                self.extras["episode"]["rew_" + key] = means[k]
        self.extras["time_outs"] = self.time_out_buf
        self.episode_length_buf[env_ids] = 0

    def snapshot(self) -> Dict[str, torch.Tensor]:
        out = {}
        for k in ("base_lin_vel", "base_ang_vel", "projected_gravity", "measured_heights", "reset_buf",
                  "time_out_buf", "rew_buf", "contact_filt", "last_contacts", "feet_air_time", "commands",
                  "episode_length_buf", "obs_buf", "privileged_obs_buf", "last_actions", "last_last_actions",
                  "last_dof_pos", "last_dof_vel", "last_torques", "last_root_vel"):
            out[k] = getattr(self, k).detach().cpu().clone()
        if self.episode_sums:
            out["episode_sums"] = self._episode_sums_buf[:len(self.episode_sums)].detach().cpu().clone()
        return out
