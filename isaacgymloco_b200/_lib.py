"""ctypes binding of libhimloco_b200.so (the C ABI of include/himloco_b200.h).

There is no CPU fallback: if the shared library is missing and cannot be built, importing this
module raises.  Tensors are passed as raw device pointers; work is enqueued on torch's current
CUDA stream.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int32, c_int64, c_uint32, c_uint64, c_void_p

import torch

from . import build as _build
from .config import HlCfg, HlReset

_vp = c_void_p


class HlEnvBuffers(ctypes.Structure):
    """Mirror of `struct HlEnvBuffers` (keep field order identical to the header)."""
    _fields_ = [("struct_bytes", c_int32), ("flags", c_uint32)] + [(n, _vp) for n in (
        "root_states", "dof_state", "contact_forces", "rigid_body_states", "height_samples",
        "height_min3", "actions", "last_actions", "last_last_actions", "last_dof_pos", "last_dof_vel",
        "torques", "last_torques", "last_root_vel", "commands", "episode_length_buf", "last_contacts",
        "contact_filt", "feet_air_time", "disturbance", "terrain_levels", "episode_sums",
        "base_lin_vel", "base_ang_vel", "projected_gravity", "measured_heights", "feet_pos",
        "feet_vel", "reset_buf", "time_out_buf", "rew_buf", "obs_buf_in", "obs_buf_out",
        "privileged_obs_buf", "noise_u45", "noise_u187")] + [
        ("philox_seed", c_uint64), ("philox_offset", c_uint64), ("height_idx_out", _vp),
        ("base_height_out", _vp), ("reset_ids_out", _vp), ("n_reset_out", _vp), ("term_priv_out", _vp),
        ("term_amp_out", _vp), ("term_noise_u45", _vp), ("term_noise_u187", _vp), ("fused_ws", _vp),
        ("foot_records", _vp), ("resample_host", _vp), ("resample_interval", c_int64), ("height_min3f", _vp),
        ("step_base", _vp)]


class HlTransition(ctypes.Structure):
    """Mirror of `struct HlTransition` (keep field order identical to the header)."""
    _fields_ = [("struct_bytes", c_int32), ("obs_dim", c_int32), ("priv_dim", c_int32), ("act_dim", c_int32),
                ("gamma", c_float), ("pad_", c_int32)] + [(n, _vp) for n in (
        "obs", "critic_obs", "next_critic_obs", "term_ids", "n_term_dev", "term_rows", "actions", "rewards", "dones",
        "values", "time_outs", "log_prob", "mu", "sigma", "obs_out", "critic_out", "next_critic_out", "actions_out",
        "rewards_out", "dones_out", "values_out", "log_prob_out", "mu_out", "sigma_out")]


MAX_GATHER_FIELDS = 12


class HlGatherFields(ctypes.Structure):
    """Mirror of `struct HlGatherFields`."""
    _fields_ = [("struct_bytes", c_int32), ("n_fields", c_int32), ("src", _vp * MAX_GATHER_FIELDS),
                ("dst", _vp * MAX_GATHER_FIELDS), ("width", c_int32 * MAX_GATHER_FIELDS)]


class HlAmpUpdateBatch(ctypes.Structure):
    """Mirror of `struct HlAmpUpdateBatch` (keep field order identical to the header)."""
    _fields_ = [("struct_bytes", c_int32), ("clip", c_float), ("ring_states", _vp), ("ring_next", _vp), ("ring_rows", c_int64),
                ("ring_cursor", _vp), ("num_samples", c_int64), ("preloaded_s", _vp), ("preloaded_s_next", _vp),
                ("n_preloaded", c_int64), ("norm_mean", _vp), ("norm_var", _vp), ("eps", c_double), ("seed", c_uint64),
                ("draw_counter", _vp), ("row_offset", c_int64), ("idx_in", _vp), ("idx_out", _vp)] + [(n, _vp) for n in (
        "policy_s", "policy_sn", "expert_s", "expert_sn", "x_policy", "x_expert")] + [("mb", c_int64)]


MAX_FINITE_FIELDS = 16
FINITE_WORKSPACE_WORDS = 2 * MAX_FINITE_FIELDS + 1
FINITE, FINITE_POSITIVE = 0, 1          # HlFiniteField.kind


class HlFiniteField(ctypes.Structure):
    """Mirror of `struct HlFiniteField`."""
    _fields_ = [("src", _vp), ("row_stride", c_int64), ("width", c_int32), ("kind", c_int32)]


class HlFiniteFields(ctypes.Structure):
    """Mirror of `struct HlFiniteFields`."""
    _fields_ = [("struct_bytes", c_int32), ("n_fields", c_int32), ("field", HlFiniteField * MAX_FINITE_FIELDS)]


# stage bits (include/himloco_b200.h)
ST_COUNTERS, ST_FRAME, ST_CONTACTS, ST_HEADING, ST_HEIGHTS = 0x001, 0x002, 0x004, 0x008, 0x010
ST_TERMINATION, ST_REWARD, ST_OBS, ST_OBS_NOSHIFT, ST_OBS_CLIP = 0x020, 0x040, 0x080, 0x100, 0x200
ST_ROLL, ST_BASE_HEIGHT, ST_RESET_ZERO, ST_RESET_DRAW = 0x400, 0x800, 0x1000, 0x2000

# bits of HlReset.parts (include/himloco_b200.h)
RESET_DOFS, RESET_ROOT, RESET_COMMANDS, RESET_FACTORS, RESET_CURRICULUM = 1, 2, 4, 8, 16

EXPORTS = {
    "hl_version": (c_int32, []),
    "hl_last_error": (c_char_p, []),
    "hl_sizeof_cfg": (c_int32, []),
    "hl_sizeof_env_buffers": (c_int32, []),
    "hl_pd_torque": (c_int32, [POINTER(HlCfg), _vp, c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, c_int64, _vp]),
    "hl_terrain_prepare": (c_int32, [_vp, c_int32, c_int32, _vp, _vp]),
    "hl_terrain_prepare_f32": (c_int32, [_vp, c_int32, c_int32, c_float, _vp, _vp]),
    "hl_post_physics_fused": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), c_int64, _vp]),
    "hl_fused_workspace_bytes": (c_int64, [c_int64]),
    "hl_fused_last_impl": (c_int32, []),
    "hl_post_physics_stages": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), c_uint32, _vp, _vp, c_int64, _vp]),
    "hl_select_workspace_bytes": (c_int64, [c_int64]),
    "hl_select_reset_ids": (c_int32, [_vp, c_int64, _vp, _vp, _vp, _vp]),
    "hl_terminal_rows": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), _vp, _vp, _vp, _vp, _vp, _vp, c_int64, _vp]),
    "hl_select_terminal_workspace_bytes": (c_int64, [c_int64]),
    "hl_select_and_terminal": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), _vp, _vp, _vp, _vp, _vp, _vp, _vp, c_int64, _vp]),
    "hl_select_terminal_reset": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), POINTER(HlReset), _vp, _vp, _vp, _vp, _vp, _vp, _vp, c_int64, _vp]),
    "hl_post_reset_fixup": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), _vp, _vp, c_int32, c_int64, _vp]),
    "hl_sizeof_reset": (c_int32, []),
    "hl_reset_idx": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), POINTER(HlReset), _vp, _vp, c_int64, _vp]),
    "hl_reset_draw": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), POINTER(HlReset), _vp, _vp, c_int64, _vp]),
    "hl_reset_and_fixup": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), POINTER(HlReset), _vp, _vp, c_int64, _vp]),
    "hl_resample_commands": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), POINTER(HlReset), _vp, _vp, c_int64, c_int64, _vp]),
    "hl_command_curriculum": (c_int32, [_vp, _vp, _vp, c_double, c_int64, c_double, c_double, c_double, _vp, _vp, c_int64, _vp]),
    "hl_episode_means": (c_int32, [_vp, _vp, _vp, _vp, c_int32, c_int64, c_float, c_int32, _vp, _vp]),
    "hl_amp_observations": (c_int32, [_vp, _vp, _vp, _vp, c_int64, _vp]),
    "hl_gae_scan": (c_int32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, c_int32, c_int64, c_float, c_float, _vp]),
    "hl_adv_normalize": (c_int32, [_vp, _vp, c_int64, _vp]),
    "hl_sizeof_transition": (c_int32, []),
    "hl_record_transition": (c_int32, [POINTER(HlTransition), c_int64, _vp]),
    "hl_delay_actions": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), _vp, _vp, _vp, c_int32, c_int32, c_float, _vp, c_int64, _vp]),
    "hl_uniform_rows": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), _vp, c_int64, c_int32, c_double, c_double, _vp, c_int32,
                                  c_int64, _vp]),
    "hl_policy_sample": (c_int32, [POINTER(HlCfg), POINTER(HlEnvBuffers), _vp, _vp, c_int64, _vp, c_int32, _vp, _vp, _vp, _vp,
                                   c_int64, _vp]),
    "hl_ring_insert": (c_int32, [_vp, _vp, _vp, _vp, c_int64, c_int32, c_int64, c_int64, _vp]),
    "hl_episode_stats": (c_int32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, c_int64, _vp, c_int64, _vp]),
    "hl_sizeof_gather_fields": (c_int32, []),
    "hl_minibatch_gather": (c_int32, [POINTER(HlGatherFields), _vp, c_int64, c_int64, _vp]),
    "hl_amp_frame_blend": (c_int32, [_vp, _vp, _vp, _vp, c_int32, _vp, _vp, _vp, _vp, _vp, c_int64, _vp]),
    "hl_amp_gather_pairs": (c_int32, [_vp, _vp, c_int64, _vp, _vp, _vp, c_int64, _vp]),
    "hl_amp_disc_input": (c_int32, [_vp, _vp, _vp, _vp, c_float, _vp, _vp, _vp, _vp, _vp, c_int64, _vp]),
    "hl_amp_transition": (c_int32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, c_double, c_float, _vp, _vp, _vp, _vp, c_int64,
                                    _vp, c_int64, _vp]),
    "hl_amp_reward": (c_int32, [_vp, _vp, c_float, c_float, _vp, c_int64, _vp]),
    "hl_sizeof_amp_update_batch": (c_int32, []),
    "hl_amp_update_batch": (c_int32, [POINTER(HlAmpUpdateBatch), _vp]),
    "hl_sizeof_finite_fields": (c_int32, []),
    "hl_finite_scan": (c_int32, [POINTER(HlFiniteFields), c_int64, _vp, _vp, _vp]),
    "hl_moments_workspace_bytes": (c_int64, [c_int32]),
    "hl_column_moments": (c_int32, [_vp, c_int64, c_int32, _vp, _vp, _vp]),
}


def _load():
    path = _build.LIB
    if not os.path.exists(path):
        # built in-tree by __graft_entry__.build(); build on demand if a toolchain is present
        _build.build()
    lib = ctypes.CDLL(path)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)          # AttributeError here = the .so is stale
        fn.restype = res
        fn.argtypes = args
    if lib.hl_sizeof_cfg() != ctypes.sizeof(HlCfg):
        raise ImportError(f"HlCfg layout mismatch: python {ctypes.sizeof(HlCfg)} vs library {lib.hl_sizeof_cfg()}")
    if lib.hl_sizeof_env_buffers() != ctypes.sizeof(HlEnvBuffers):
        raise ImportError(f"HlEnvBuffers layout mismatch: python {ctypes.sizeof(HlEnvBuffers)} vs "
                          f"library {lib.hl_sizeof_env_buffers()}")
    if lib.hl_sizeof_reset() != ctypes.sizeof(HlReset):
        raise ImportError(f"HlReset layout mismatch: python {ctypes.sizeof(HlReset)} vs library {lib.hl_sizeof_reset()}")
    if lib.hl_sizeof_gather_fields() != ctypes.sizeof(HlGatherFields):
        raise ImportError("HlGatherFields layout mismatch")
    if lib.hl_sizeof_transition() != ctypes.sizeof(HlTransition):
        raise ImportError(f"HlTransition layout mismatch: python {ctypes.sizeof(HlTransition)} vs "
                          f"library {lib.hl_sizeof_transition()}")
    if lib.hl_sizeof_amp_update_batch() != ctypes.sizeof(HlAmpUpdateBatch):
        raise ImportError(f"HlAmpUpdateBatch layout mismatch: python {ctypes.sizeof(HlAmpUpdateBatch)} vs "
                          f"library {lib.hl_sizeof_amp_update_batch()}")
    if lib.hl_sizeof_finite_fields() != ctypes.sizeof(HlFiniteFields):
        raise ImportError(f"HlFiniteFields layout mismatch: python {ctypes.sizeof(HlFiniteFields)} vs "
                          f"library {lib.hl_sizeof_finite_fields()}")
    return lib


lib = _load()
LIB_PATH = _build.LIB


def check(rc: int):
    if rc != 0:
        raise RuntimeError(f"libhimloco_b200: {lib.hl_last_error().decode()} (code {rc})")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("libhimloco_b200 kernels need CUDA tensors (there is no CPU fallback)")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream
