"""Probe states for the PD torques and the observations, and their float64 references (plain helper module of
tests/test_cpu_torque_obs_probe.py and tests/test_gpu_torques_obs.py).

`make_torque_probe` edits synthetic.make_state env by env so that, for every DOF, the raw PD torque lies above
+torque_limit, below -torque_limit and inside the limits on a sizeable share of the envs each, every value at least
5 % of the limit away from it.  `make_obs_probe` does the same for the clips of the observations: the +-1 clip of the
height scan, the +-clip_observations clip of step(), noise draws at both ends of [0, 1), heading commands away from
the wrap_to_pi discontinuity, resets (time-outs) for the terminal rows.  `reference64_torques` and `reference64_obs`
run the oracle's own code on those states in float64 (terrain cells from the fp32 index arithmetic, as
reward_probe.Oracle64 does), and `torque_gates` / `obs_gates` return each branch as a boolean tensor.
"""
import math

import numpy as np
import torch

from isaacgymloco_b200 import config as C
from isaacgymloco_b200 import synthetic as S
from oracle import torch_oracle as O
from reward_probe import Oracle64, bound, check_bound, default_dtype, scan_cells  # noqa: F401  (re-exported)

CONTROL_TYPES = ("P", "V", "T")
OBS_TASKS = ("flat", "stairs", "plane")
OBS_VARIANTS = ("noise", "clip", "plain")
U_TOP = float(np.float32(1.0) - np.float32(2.0 ** -24))     # the largest fp32 below 1
CLIP_OBS = 3.0                                                # the clip_observations of the "clip" obs variant
HEIGHT_MARGIN = 0.05                                          # |z - 0.5 - h| stays this far from 1


# ----------------------------------------------------------------------------- configs
def torque_cfg(control_type, n, index_math=C.INDEX_MATH_TORCH_CUDA):
    """The flat task with a non-default hip_reduction and the given control type."""
    return C.aliengo("flat", num_envs=n, index_math=index_math, control_type=control_type, hip_reduction=0.8)


def obs_cfg(task, variant, n, index_math=C.INDEX_MATH_TORCH_CUDA):
    """`task` in OBS_TASKS ("plane" = the flat task on a plane mesh, as the `plane` golden case), `variant` in
    OBS_VARIANTS: "noise": add_noise on, default clip_observations (it cannot bind on the heights, so the fused kernels
    take their fast height path); "clip": add_noise on, clip_observations = CLIP_OBS (binds on several groups);
    "plain": add_noise off, the kernels' noise-free switch (the +-1 height clip alone decides the heights).  The
    reference's add_noise gates the 45 proprioceptive columns only (LR:393) and still noises the heights (LR:399-400);
    with noise_level 0 that noise is zero too, so the oracle and the kernels describe the same step (DESIGN
    "Tolerances")."""
    kw = {"noise": dict(add_noise=True), "clip": dict(add_noise=True, clip_observations=CLIP_OBS),
          "plain": dict(add_noise=False, noise_level=0.0)}[variant]
    cfg = C.aliengo("flat" if task == "plane" else task, num_envs=n, index_math=index_math, **kw)
    if task == "plane":
        cfg.mesh_type = "plane"
        cfg.out_of_border = False
    return cfg


def _rng(seed):
    g = torch.Generator().manual_seed(seed)
    rand = lambda *sh: torch.rand(*sh, generator=g)
    uni = lambda lo, hi, *sh: lo + (hi - lo) * rand(*sh)
    sgn = lambda *sh: torch.where(rand(*sh) < 0.5, -1.0, 1.0)
    return g, rand, uni, sgn


def _tables64(cfg):
    t = cfg.dof_tables()
    return {k: torch.from_numpy(np.asarray(v, dtype=np.float64)) for k, v in t.items()}


def _hip_factor(cfg):
    f = torch.ones(12, dtype=torch.float64)
    f[[0, 3, 6, 9]] = float(np.float32(cfg.hip_reduction))
    return f


# ----------------------------------------------------------------------------- torque probe
def make_torque_probe(cfg, n, seed=21):
    """(state, hf): for each (env, DOF) the raw torque of cfg.control_type is drawn from one of three bands --
    (1.05, 2) x limit, -(1.05, 2) x limit, (-0.95, 0.95) x limit -- and the state is solved for it: dof_pos for P,
    last_dof_vel for V, the action itself for T.  Kp/Kd factors and motor strengths are drawn away from 1."""
    hf = S.make_terrain(cfg, seed=seed)
    s = S.make_state(cfg, n, hf, seed=seed)
    g, rand, uni, sgn = _rng(seed + 500)
    t = _tables64(cfg)
    p, d, lim, dflt = t["p_gains"], t["d_gains"], t["torque_limits"], t["default_dof_pos"]
    s["motor_strength"] = torch.where(rand(n, 12) < 0.5, uni(0.8, 0.97, n, 12), uni(1.03, 1.2, n, 12))
    s["Kp_factors"] = torch.where(rand(n, 1) < 0.5, uni(0.8, 0.97, n, 1), uni(1.03, 1.2, n, 1))
    s["Kd_factors"] = torch.where(rand(n, 1) < 0.5, uni(0.8, 0.97, n, 1), uni(1.03, 1.2, n, 1))
    band = torch.randint(0, 3, (n, 12), generator=g)
    want = torch.where(band == 0, uni(1.05, 2.0, n, 12), torch.where(band == 1, -uni(1.05, 2.0, n, 12),
                                                                      uni(-0.95, 0.95, n, 12))).double() * lim
    ms = s["motor_strength"].double()
    hip = _hip_factor(cfg)
    scale = float(np.float32(cfg.action_scale))
    dp = s["dof_state"].view(n, 12, 2)
    vel = dp[..., 1].double()
    if cfg.control_type == "T":
        s["actions"] = (want / (ms * scale * hip)).float()
    else:
        scaled = ms * s["actions"].double() * scale * hip
        if cfg.control_type == "P":
            kp, kd = s["Kp_factors"].double(), s["Kd_factors"].double()
            dp[..., 0] = (dflt + scaled - (want + d * kd * vel) / (p * kp)).float()
        else:
            s["last_dof_vel"] = (vel + (want - p * (scaled - vel)) * cfg.sim_dt / d).float()
    return s, hf


def reference64_torques(cfg, state, hf, actions=None, index_math=None):
    """The oracle's _compute_torques in float64 -> (torques, joint_pos_target, raw torques before the clip)."""
    im = cfg.index_math if index_math is None else index_math
    with default_dtype(torch.float64):
        st = {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in state.items()}
        env = Oracle64(cfg, st, hf, im)
        a = (state["actions"] if actions is None else actions).double()
        tq = env._compute_torques(a)
        target = env.joint_pos_target.clone()
        env.torque_limits = torch.full_like(env.torque_limits, math.inf)
        raw = env._compute_torques(a)
    return tq, target, raw


def torque_gates(cfg, raw):
    """(N, 12) boolean tensors: the raw torque above +limit, below -limit, inside."""
    lim = _tables64(cfg)["torque_limits"]
    return {"raw torque > +limit": raw > lim, "raw torque < -limit": raw < -lim, "inside the limits": raw.abs() < lim}


def torque_margin(cfg, raw):
    """Smallest | |raw| - limit | / limit: how far every raw torque stays from the clip."""
    lim = _tables64(cfg)["torque_limits"]
    return float(((raw.abs() - lim).abs() / lim).min())


# ----------------------------------------------------------------------------- observation probe
def _scan_heights(cfg, hf, root):
    """(N, 187) float64 heights of the scan under both fp32 index flavours, stacked (2, N, 187)."""
    n = root.shape[0]
    if cfg.is_plane:
        return torch.zeros(2, n, len(cfg.measured_points_x) * len(cfg.measured_points_y), dtype=torch.float64)
    xs, ys = cfg.measured_points_x, cfg.measured_points_y
    pts = torch.tensor([[x, y, 0.0] for x in xs for y in ys], dtype=torch.float32).expand(n, -1, -1)
    out = [scan_cells(cfg, hf, root, pts, im)[0].double() * cfg.vertical_scale
           for im in (C.INDEX_MATH_TORCH_CPU, C.INDEX_MATH_TORCH_CUDA)]
    return torch.stack(out)


def make_obs_probe(cfg, n, seed=31):
    """(state, hf, noise): synthetic.make_state and make_noise edited so that every clip of the observation binds on
    both sides for a sizeable share of the entries, clear of its threshold."""
    hf = S.make_terrain(cfg, seed=seed)
    s = S.make_state(cfg, n, hf, seed=seed)
    noise = S.make_noise(n, seed=seed + 1)
    g, rand, uni, sgn = _rng(seed + 500)
    root = s["root_states"]
    q = root[:, 3:7].double()

    # body-frame angular velocity: per component |w| in (13, 20) (x obs_ang_vel 0.25 -> 3.25..5, beyond CLIP_OBS) on
    # half of the envs, |w| < 1 on the others
    big = rand(n, 3) < 0.5
    wb = torch.where(big, sgn(n, 3) * uni(13.0, 20.0, n, 3), uni(-1.0, 1.0, n, 3)).double()
    root[:, 10:13] = O.quat_apply(q, wb).float()
    # dof velocities: |v| in (65, 100) (x obs_dof_vel 0.05 -> 3.25..5) on half of the entries
    dp = s["dof_state"].view(n, 12, 2)
    dp[..., 1] = torch.where(rand(n, 12) < 0.5, sgn(n, 12) * uni(65.0, 100.0, n, 12), uni(-2.0, 2.0, n, 12))

    # heading command: wrap_to_pi(cmd_heading - heading) at least 1e-2 away from +-pi
    fwd = O.quat_apply(q, torch.tensor([[1.0, 0.0, 0.0]], dtype=torch.float64).expand(n, 3))
    heading = torch.atan2(fwd[:, 1], fwd[:, 0])
    delta = uni(-math.pi + 0.01, math.pi - 0.01, n).double()
    s["commands"][:, 3] = O.wrap_to_pi(heading + delta).float()
    s["disturbance"][:, 0, :] = sgn(n, 3) * uni(1.0, 30.0, n, 3)

    # base height: every scan entry of an env on one side of the +-1 clip, or all inside it
    h = _scan_heights(cfg, hf, root)
    hmin, hmax = h.amin(dim=(0, 2)), h.amax(dim=(0, 2))
    kind = rand(n)
    fits = (hmax - hmin) < 2 * (1 - HEIGHT_MARGIN) - 0.4
    inside = (kind < 0.4) & fits
    below = (kind >= 0.4) & (kind < 0.7)
    z = torch.where(inside, 0.5 + 0.5 * (hmin + hmax) + uni(-0.2, 0.2, n).double(),
                    torch.where(below, 0.5 + hmin - uni(1.1, 1.6, n).double(), 0.5 + hmax + uni(1.1, 1.6, n).double()))
    nb = cfg.num_bodies
    rb = s["rigid_body_states"].view(n, nb, 13)
    rb[:, :, 2] += (z.float() - root[:, 2])[:, None]
    root[:, 2] = z.float()

    # resets for the terminal rows: time-out on a quarter of the envs
    ep = s["episode_length_buf"]
    ep[:] = torch.where(rand(n) < 0.25, torch.full_like(ep, cfg.max_episode_length), ep.clamp(max=cfg.max_episode_length - 1))

    # noise draws at both ends of [0, 1) in every table
    for k, v in noise.items():
        r = rand(*v.shape)
        noise[k] = torch.where(r < 0.15, torch.zeros_like(v), torch.where(r > 0.85, torch.full_like(v, U_TOP), v))
    return s, hf, noise


def reference64_obs(cfg, state, hf, noise, index_math=None):
    """The oracle's pre_reset + post_reset (no reset applied) in float64.  Returns the env (obs_buf, privileged_obs_buf
    after the clip) and the (ids, terminal rows, terminal AMP rows), plus the pre-clip privileged rows of this step."""
    im = cfg.index_math if index_math is None else index_math
    with default_dtype(torch.float64):
        st = {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in state.items()}
        nz = {k: v.double() for k, v in noise.items()}
        env = Oracle64(cfg, st, hf, im)
        ids, term_obs, term_amp = env.pre_reset(nz)
        env.unclipped = env._current_obs(nz["obs45"], nz["obs187"])    # the step's rows before the obs clip
        env.post_reset(nz)
    return env, ids, term_obs, term_amp


def reference32_obs(cfg, state, hf, noise, device="cpu"):
    """The plain fp32 oracle's step (torch arithmetic on `device`) -> (env, ids, terminal rows, terminal AMP rows)."""
    env = O.OracleEnv(cfg, S.to_device(state, device), hf.to(device))
    nz = S.to_device(noise, device)
    ids, term_obs, term_amp = env.pre_reset(nz)
    env.post_reset(nz)
    return env, ids, term_obs, term_amp


def height_arg(env):
    """(N, P) float64 z - 0.5 - h of the reference env (the argument of the +-1 clip)."""
    return env.root_states[:, 2:3] - 0.5 - env.measured_heights


# column groups of the 51 + P privileged row
GROUPS = {"commands": slice(0, 3), "ang_vel": slice(3, 6), "gravity": slice(6, 9), "dof_pos": slice(9, 21),
          "dof_vel": slice(21, 33), "actions": slice(33, 45), "lin_vel": slice(45, 48), "disturbance": slice(48, 51),
          "heights": slice(51, None)}


def obs_gates(cfg, env, clip_margin=1e-3):
    """Boolean tensors over the entries each clip decides: the +-1 height clip on the scan entries, and (when the
    clip_observations clip can bind) that clip per group, judged on the float64 pre-clip value with a margin."""
    x = height_arg(env)
    out = {"height z-0.5-h > +1": x > 1 + HEIGHT_MARGIN, "height z-0.5-h < -1": x < -1 - HEIGHT_MARGIN,
           "height z-0.5-h inside": x.abs() < 1 - HEIGHT_MARGIN}
    if cfg.clip_observations < 10:
        cl = cfg.clip_observations
        for grp in ("ang_vel", "dof_vel", "heights"):
            v = env.unclipped[:, GROUPS[grp]]
            out[f"{grp} > +clip_observations"] = v > cl + clip_margin
            out[f"{grp} < -clip_observations"] = v < -cl - clip_margin
    return out
