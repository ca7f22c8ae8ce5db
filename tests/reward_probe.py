"""A reward probe state and a float64 reference of the reward pass (plain helper module of
tests/test_cpu_reward_terms.py and tests/test_gpu_reward_terms.py).

`make_probe` starts from `synthetic.make_state` and edits it env by env so that every gate of every
`_r_*` term of oracle/torch_oracle.py is on for a sizeable share of the envs and off for another, each
value kept well clear of its threshold (so fp32 and float64 agree on which side it lies).
`reference64` runs the oracle's step up to compute_reward in float64 on that state.  The terrain
cells are the one discrete choice the reward pass makes from coordinates: the reference picks them
in fp32, so `Oracle64` takes them from the fp32 index arithmetic (torch-CPU true division or the
torch-CUDA fp32 reciprocal) and does everything else in float64.
"""
import contextlib
import math

import numpy as np
import torch

from isaacgymloco_b200 import config as C
from isaacgymloco_b200 import synthetic as S
from oracle import torch_oracle as O

RTOL, FLOOR = 1e-5, 1e-6      # |got - ref64| <= RTOL |ref64| + FLOOR max_e |ref64[k]|
TASKS = ("flat", "stairs", "amp")


@contextlib.contextmanager
def default_dtype(dt):
    old = torch.get_default_dtype()
    torch.set_default_dtype(dt)
    try:
        yield
    finally:
        torch.set_default_dtype(old)


def probe_cfg(task, n, index_math=C.INDEX_MATH_TORCH_CUDA, **kw):
    """`task` in TASKS, or "allterms": the stairs task with all 51 terms at distinct scales."""
    from oracle.make_goldens import all_term_scales
    cfg = C.aliengo("stairs" if task == "allterms" else task, num_envs=n, index_math=index_math, **kw)
    if task == "allterms":
        cfg.reward_scales = all_term_scales()
    return cfg


# ----------------------------------------------------------------------------- terrain cells in fp32
def cell_heights(cfg, hs, pts32, index_math):
    """int16 min-of-3 height under world points (N,P,3) that already carry `+= border` (LR:1342-1353)."""
    n = pts32.shape[0]
    if index_math == C.INDEX_MATH_TORCH_CPU:
        g = pts32 / cfg.horizontal_scale
    else:
        g = pts32 * torch.tensor(np.float32(1.0) / np.float32(cfg.horizontal_scale))
    g = g.long()
    px = torch.clip(g[:, :, 0].reshape(-1), 0, hs.shape[0] - 2)
    py = torch.clip(g[:, :, 1].reshape(-1), 0, hs.shape[1] - 2)
    h = torch.min(torch.min(hs[px, py], hs[px + 1, py]), hs[px, py + 1])
    return h.view(n, -1), px.view(n, -1), py.view(n, -1)


def scan_cells(cfg, hs, root32, pts_body32, index_math):
    """The body-frame scan of LR:1339-1355 in fp32, with the given division flavour."""
    p = pts_body32.shape[1]
    pts = O.quat_apply_yaw(root32[:, 3:7].repeat(1, p), pts_body32) + root32[:, :3].unsqueeze(1)
    pts += cfg.border_size
    return cell_heights(cfg, hs, pts, index_math)


class Oracle64(O.OracleEnv):
    """The oracle in float64 (build it under default_dtype(torch.float64)), terrain cells picked in fp32."""

    def __init__(self, cfg, state, hf, index_math):
        self._index_math = index_math
        self._feet32 = None
        super().__init__(cfg, state, hf)

    def _scan(self, pts_body, root_states=None, quat=None):
        root = self.root_states if root_states is None else root_states
        return scan_cells(self.cfg, self.height_samples, root.float(), pts_body.float(), self._index_math)

    def pre_reset(self, noise, push_vel=None):
        self._feet32 = None
        return super().pre_reset(noise, push_vel)

    def _r_foot_clearance_terrain(self):    # LR:1717-1743; the in-place `feet_pos += border` runs in both precisions
        c = self.cfg
        if c.is_plane:
            return super()._r_foot_clearance_terrain()
        if self._feet32 is None:
            self._feet32 = self.feet_pos.float()
        self._feet32 += c.border_size
        self.feet_pos += c.border_size
        h, _, _ = cell_heights(c, self.height_samples, self._feet32, self._index_math)
        fh = self.feet_pos[:, :, 2] - h * c.vertical_scale
        lat = torch.norm(self.feet_vel[:, :, :2], dim=-1)
        return torch.sum(lat * torch.square(fh - c.foot_height_target_terrain), dim=-1)


def _noise(n):
    return S.make_noise(n, seed=7)


def reference64(cfg, state, hf, index_math=None):
    """The oracle's pre-reset step (frame, contacts, heading, heights, termination, compute_reward) in float64.
    Returns the env: rows via `rows64(env)`, plus rew_buf, reset_buf, time_out_buf, feet_air_time, last_contacts."""
    im = cfg.index_math if index_math is None else index_math
    with default_dtype(torch.float64):
        st = {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in state.items()}
        env = Oracle64(cfg, st, hf, im)
        env.pre_reset({k: v.double() for k, v in _noise(env.num_envs).items()})
    return env


def reference32(cfg, state, hf):
    """The plain fp32 oracle's pre-reset step on CPU (torch-CPU index arithmetic)."""
    env = O.OracleEnv(cfg, {k: v.clone() for k, v in state.items()}, hf)
    env.pre_reset(_noise(env.num_envs))
    return env


def rows64(env):
    """(R, N) episode_sums rows in cfg.episode_sum_names() order."""
    return torch.stack([env.episode_sums[k] for k in env.sum_names]) if env.sum_names else torch.zeros(0, env.num_envs)


def bound(ref):
    """Per-element tolerance of a (R, N) or (N,) float64 reference."""
    ref = ref.double()
    mx = ref.abs().amax(dim=-1, keepdim=True) if ref.shape[-1] else ref.abs()
    return RTOL * ref.abs() + FLOOR * mx


def check_bound(got, ref, names, what):
    """Assert |got - ref| <= bound(ref) everywhere; the message names the row, the worst env and the counts."""
    got, ref = got.detach().cpu().double(), ref.detach().cpu().double()
    if got.dim() == 1:
        got, ref = got[None], ref[None]
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    err, tol = (got - ref).abs(), bound(ref)
    bad = ~(err <= tol)
    msgs = []
    for k in range(ref.shape[0]):
        if bad[k].any():
            e = int(torch.argmax(torch.where(bad[k], err[k] / tol[k].clamp(min=1e-300), torch.zeros_like(err[k]))))
            msgs.append(f"{names[k]}: {int(bad[k].sum())} envs out of bound, worst env {e}: got {float(got[k, e])!r} "
                        f"ref64 {float(ref[k, e])!r} tol {float(tol[k, e]):.3g}")
    assert not msgs, f"{what}:\n  " + "\n  ".join(msgs)


# ----------------------------------------------------------------------------- the probe state
def make_probe(cfg, n, seed=14):
    """(state, hf): synthetic.make_state edited per env so that every reward gate is exercised on both sides."""
    hf = S.make_terrain(cfg, seed=seed)
    s = S.make_state(cfg, n, hf, seed=seed)
    g = torch.Generator().manual_seed(seed + 500)
    rand = lambda *sh: torch.rand(*sh, generator=g)
    uni = lambda lo, hi, *sh: lo + (hi - lo) * rand(*sh)
    sgn = lambda *sh: torch.where(rand(*sh) < 0.5, -1.0, 1.0)
    pick = lambda p, *sh: rand(*sh) < p
    nb = cfg.num_bodies
    tabs = cfg.dof_tables()
    f32 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float32))

    # commands: standing (|cmd_xy| < 0.06), lateral-only (|cmd_x| < 0.05, |cmd_xy| >= 0.2), forward (|cmd_x| >= 0.2)
    cmd = s["commands"]
    kind = rand(n)
    stand, lateral = kind < 0.3, (kind >= 0.3) & (kind < 0.45)
    cx = torch.where(stand | lateral, sgn(n) * uni(0.0, 0.04, n), sgn(n) * uni(0.2, 1.0, n))
    cy = torch.where(stand, sgn(n) * uni(0.0, 0.04, n), torch.where(lateral, sgn(n) * uni(0.2, 0.5, n), uni(-0.5, 0.5, n)))
    cmd[:, 0], cmd[:, 1] = cx, cy

    # base velocity given in the body frame.  Tracking envs follow the command (v_xy = cmd_xy, yaw rate = the heading
    # command of LR:616-620) so that their summed reward can be positive; the others have |v_x| < 0.05 (stuck when
    # |cmd_x| > 0.1) or 0.2 <= |v_x| <= 0.9
    root = s["root_states"]
    q = root[:, 3:7].double()
    track = pick(0.4, n)
    vb = torch.stack([torch.where(pick(0.4, n), sgn(n) * uni(0.0, 0.05, n), sgn(n) * uni(0.2, 0.9, n)),
                      (0.5 * torch.randn(n, generator=g)).clamp(-1.0, 1.0),
                      (0.3 * torch.randn(n, generator=g)).clamp(-1.0, 1.0)], dim=-1).double()
    vb[:, :2] = torch.where(track[:, None], cmd[:, :2].double() + uni(-0.02, 0.02, n, 2).double(), vb[:, :2])
    root[:, 7:10] = O.quat_apply(q, vb).float()
    fwd = O.quat_apply(q, torch.tensor([[1.0, 0.0, 0.0]], dtype=torch.float64).expand(n, 3))
    yaw_cmd = torch.clip(0.5 * O.wrap_to_pi(cmd[:, 3].double() - torch.atan2(fwd[:, 1], fwd[:, 0])), -2.0, 2.0)
    wb = (0.5 * torch.randn(n, 3, generator=g)).double()
    wb[:, 2] = torch.where(track, yaw_cmd + uni(-0.05, 0.05, n).double(), wb[:, 2])
    root[:, 10:13] = O.quat_apply(q, wb).float()

    # feet: Fz on both sides of 1 N, first contacts, stumbling feet (|Fxy| = 4.5 or 8 |Fz|), |F| on both sides of 100 N
    cf = s["contact_forces"].view(n, nb, 3)
    feet = cfg.feet_indices
    fz = torch.where(pick(0.5, n, 4), uni(2.0, 150.0, n, 4), uni(0.0, 0.8, n, 4))
    ratio = uni(0.0, 1.0, n, 4)
    stumbler = torch.randint(0, 4, (n,), generator=g)
    hit = torch.nn.functional.one_hot(stumbler, 4).bool() & pick(0.7, n)[:, None]
    ratio = torch.where(hit, torch.where(pick(0.7, n, 4), 8.0, 4.5), ratio)
    ang = uni(-math.pi, math.pi, n, 4)
    cf[:, feet, 0] = ratio * fz * torch.cos(ang)
    cf[:, feet, 1] = ratio * fz * torch.sin(ang)
    cf[:, feet, 2] = fz
    s["last_contacts"] = pick(0.5, n, 4)
    s["feet_air_time"] = torch.where(pick(0.4, n, 4), uni(0.05, 0.6, n, 4), torch.zeros(n, 4))
    s["terrain_levels"] = torch.where(pick(0.85, n), torch.randint(4, 10, (n,), generator=g),
                                      torch.randint(0, 4, (n,), generator=g))

    # penalised bodies (other than the termination ones): norms in (0.5, 20) or below 0.06
    pen = [b for b in cfg.penalised_contact_indices if b not in cfg.termination_contact_indices]
    dirs = torch.randn(n, len(pen), 3, generator=g)
    dirs = dirs / dirs.norm(dim=-1, keepdim=True)
    colliding = pick(0.3, n)[:, None] & (pick(0.3, n, len(pen)) |
                                          torch.nn.functional.one_hot(torch.randint(0, len(pen), (n,), generator=g),
                                                                      len(pen)).bool())
    mag = torch.where(colliding, uni(0.5, 20.0, n, len(pen)), uni(0.0, 0.06, n, len(pen)) * pick(0.5, n, len(pen)))
    cf[:, pen, :] = dirs * mag[..., None]

    # resets: base contact (|F| in 5..50 N) without time-out, time-out (episode_length 1000 -> 1001), neither
    ep = s["episode_length_buf"]
    timeout = pick(0.25, n)
    ep[:] = torch.where(timeout, torch.full_like(ep, cfg.max_episode_length), torch.randint(0, cfg.max_episode_length - 1, (n,), generator=g))
    base_hit = pick(0.25, n)
    for b in cfg.termination_contact_indices:
        d = torch.randn(n, 3, generator=g)
        cf[:, b, :] = d / d.norm(dim=-1, keepdim=True) * (uni(5.0, 50.0, n) * base_hit)[:, None]

    # DOF positions outside the soft limits on either side, |dof_vel| and |torque| above theirs
    dp = s["dof_state"].view(n, 12, 2)
    lo, hi = f32(tabs["dof_pos_lo"]), f32(tabs["dof_pos_hi"])
    side = rand(n, 12)
    dp[..., 0] = torch.where(side < 0.04, lo - uni(0.05, 0.3, n, 12),
                             torch.where(side > 0.96, hi + uni(0.05, 0.3, n, 12), dp[..., 0]))
    vlim = f32(tabs["dof_vel_limits"]) * np.float32(cfg.soft_dof_vel_limit)
    over = torch.where(pick(0.5, n, 12), uni(0.3, 0.9, n, 12), uni(1.5, 4.0, n, 12))
    dp[..., 1] = torch.where(pick(0.03, n, 12), sgn(n, 12) * (vlim + over), dp[..., 1])
    tlim = f32(tabs["torque_limits"]) * np.float32(cfg.soft_torque_limit)
    s["torques"] = torch.where(pick(0.03, n, 12), sgn(n, 12) * (tlim + uni(0.5, 10.0, n, 12)), s["torques"])

    # base height: 3..7 cm off the target, or within 5 mm of it (the feet move with the base)
    if not cfg.is_plane:
        bpts = torch.tensor([[x, y, 0.0] for x in C._BASE_POINTS_X for y in C._BASE_POINTS_Y], dtype=torch.float32).expand(n, -1, -1)
        h, _, _ = scan_cells(cfg, hf, root, bpts, C.INDEX_MATH_TORCH_CPU)
        ground = (h.double() * cfg.vertical_scale).mean(dim=1)
    else:
        ground = torch.zeros(n, dtype=torch.float64)
    off = torch.where(pick(0.5, n), sgn(n) * uni(0.03, 0.07, n), sgn(n) * uni(0.0, 0.005, n)).double()
    z = (ground + cfg.base_height_target + off).float()
    rb = s["rigid_body_states"].view(n, nb, 13)
    rb[:, :, 2] += (z - root[:, 2])[:, None]
    root[:, 2] = z

    s["episode_sums"] = torch.zeros_like(s["episode_sums"])
    return s, hf


def gates(cfg, state, env):
    """Every gate the reward terms branch on, as boolean tensors over envs (or env x foot), from the probe state and
    the float64 reference env after its step."""
    n, nb = env.num_envs, cfg.num_bodies
    cf = state["contact_forces"].view(n, nb, 3).double()
    ff = cf[:, cfg.feet_indices]
    fxy, fz = ff[..., :2].norm(dim=-1), ff[..., 2].abs()
    contact = ff[..., 2] > 1.0
    dp = state["dof_state"].view(n, 12, 2).double()
    lim = env.dof_pos_limits
    pen = cf[:, cfg.penalised_contact_indices].norm(dim=-1)
    bh = env._get_base_heights() - cfg.base_height_target
    cmd = state["commands"].double()
    cmd_small = cmd[:, :2].norm(dim=1) < 0.1
    blv = env.base_lin_vel
    return {
        "|cmd_xy| < 0.1": cmd_small,
        "|cmd_x| > 0.1": cmd[:, 0].abs() > 0.1,
        "|base_lin_vel_x| < 0.1": blv[:, 0].abs() < 0.1,
        "stuck (|v_x| < 0.1 and |cmd_x| > 0.1)": (blv[:, 0].abs() < 0.1) & (cmd[:, 0].abs() > 0.1),
        "foot Fz > 1 N (per foot)": contact,
        "first contact (air time > 0, contact_filt)": ((state["feet_air_time"] > 0) & (contact | state["last_contacts"])).any(dim=1),
        "|Fxy| > 5 |Fz| (any foot)": (fxy > 5 * fz).any(dim=1),
        "|Fxy| > 4 |Fz| (any foot)": (fxy > 4 * fz).any(dim=1),
        "terrain_level > 3": state["terrain_levels"] > 3,
        "feet_stumble active": env._stumble(5) > 0,
        "foot |F| > max_contact_force (per foot)": ff.norm(dim=-1) > cfg.max_contact_force,
        "penalised-body |F| > 0.1 (any)": (pen > 0.1).any(dim=1),
        "dof_pos below the soft lower limit (any)": (dp[..., 0] < lim[:, 0]).any(dim=1),
        "dof_pos above the soft upper limit (any)": (dp[..., 0] > lim[:, 1]).any(dim=1),
        "|dof_vel| above the soft limit (any)": (dp[..., 1].abs() > env.dof_vel_limits * cfg.soft_dof_vel_limit).any(dim=1),
        "|torque| above the soft limit (any)": (state["torques"].double().abs() > env.torque_limits * cfg.soft_torque_limit).any(dim=1),
        "base height off target by > 2 cm": bh.abs() > 0.02,
        "reset with time-out": env.reset_buf & env.time_out_buf,
        "reset without time-out": env.reset_buf & ~env.time_out_buf,
        "no reset": ~env.reset_buf,
    }


def loop_sum(env):
    """Sum of the loop terms before the clip of only_positive_rewards (LR:367-375), float64."""
    names, _ = env.cfg.active_terms()
    return sum(env.episode_sums[k] for k in names)
