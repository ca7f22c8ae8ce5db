"""A probe state and uniform table for reset_idx's re-draws, the pre-step command resampling and the post-reset
fix-up, and their float64 reference (plain helper module of tests/test_cpu_reset_probe.py and
tests/test_gpu_reset_draws.py).

`make_reset_probe` starts from `synthetic.make_state` and edits it env by env, together with the (N, 44) uniform
table the kernels read in parity mode (include/himloco_b200.h: HL_RESET_NU), so that every branch of the reset side
switches on a sizeable share of the reset envs: the terrain curriculum moves up, down or not at all, wraps from the
top level to a random one and clips at level 0; the command keep gate sees norms just above 0.2 and below 0.19; in
the high-speed slice |c0| lies below 1, above 1 (wide ranges) and exactly at 1; envs on the 500-step resampling mark
reset on the same step.  Every decided value stays at least 1e-3 (relative) from its threshold, unless fp32 computes
it exactly (then both precisions agree by construction).

`reference64_reset` runs the oracle's resample_commands (on the mark), pre_reset, reset_idx_draw, apply_reset and
post_reset in float64 from the same fp32 uniform table, through reward_probe.Oracle64.  The height cells after the
reset are a discrete choice made from the fp32 root state: the reference takes them from the root state of the
implementation under test (`root32_after`), which the same bound checks on its own.
"""
import math

import numpy as np
import torch

from isaacgymloco_b200 import config as C
from isaacgymloco_b200 import synthetic as S
from oracle import torch_oracle as O
from reward_probe import Oracle64, bound, check_bound, default_dtype, scan_cells  # noqa: F401  (re-exported)

TASKS = ("flat", "stairs", "amp", "recover", "plane")
VARIANTS = ("default", "fallbacks", "wide")
U_TOP = float(np.float32(1.0) - np.float32(2.0 ** -24))     # the largest fp32 below 1
WIDE_X, WIDE_Y = [-2.0, 2.0], [-1.0, 1.0]
WIDE_DOF_VEL = [0.5, -1.0]                                    # reversed: |hi - lo| u + min(lo, hi)
MARGIN = 1e-3


# ----------------------------------------------------------------------------- configs
def reset_cfg(task, variant, n, index_math=C.INDEX_MATH_TORCH_CUDA, num_envs=None, env_id_offset=0):
    """`task` in TASKS ("plane" = the flat task on a plane mesh: no custom origins, no terrain curriculum), `variant`
    in VARIANTS.  "fallbacks": every `None` / off branch of LR:690-820 and LR:336-341 (position and rotation ranges
    None, a scalar velocity range, no dof-position ratio, no dof-velocity draw, no gain randomisation); "wide": the
    command ranges a widened curriculum reaches (lin_vel_x = [-2, 2], lin_vel_y = [-1, 1]) and a reversed
    dof_init_vel_range.  Pushes and disturbances are off.  `num_envs`: the global env count (default n)."""
    cfg = C.aliengo("flat" if task == "plane" else task, num_envs=num_envs or n, index_math=index_math,
                    env_id_offset=env_id_offset)
    if task == "plane":
        cfg.mesh_type = "plane"
        cfg.out_of_border = False
    R = cfg.reset
    R.push_robots = False
    R.disturbance = False
    if variant == "fallbacks":
        R.base_init_pos_range = None
        R.base_init_rot_range = None
        R.base_init_vel_range = (-0.5, 0.5)
        R.dof_init_pos_ratio_range = None
        R.randomize_dof_vel = False
        R.randomize_kp = R.randomize_kd = R.randomize_motor_strength = False
    elif variant == "wide":
        R.lin_vel_x, R.lin_vel_y = list(WIDE_X), list(WIDE_Y)
        R.dof_init_vel_range = list(WIDE_DOF_VEL)
    else:
        assert variant == "default", variant
    return cfg


def terrain_tables(cfg, n, seed):
    """Terrain-curriculum tables as reset_inputs builds them: origins (rows, cols, 3) and the shard's types (N,)."""
    g = torch.Generator().manual_seed(seed + 7000)
    origins = torch.zeros(cfg.num_rows, cfg.num_cols, 3)
    origins[..., 0] = (torch.arange(cfg.num_rows).float()[:, None] + 0.5) * cfg.terrain_length
    origins[..., 1] = (torch.arange(cfg.num_cols).float()[None, :] + 0.5) * cfg.terrain_width
    origins[..., 2] = 0.1 * torch.rand(cfg.num_rows, cfg.num_cols, generator=g)
    gid = torch.arange(n) + cfg.env_id_offset
    types = torch.div(gid, (cfg.num_envs / cfg.num_cols), rounding_mode="floor").to(torch.long)      # LR:1234
    return origins, types


def command_ranges(cfg):
    R = cfg.reset
    return dict(lin_vel_x=list(R.lin_vel_x), lin_vel_y=list(R.lin_vel_y), ang_vel_yaw=list(R.ang_vel_yaw),
                heading=list(R.heading))


def draw_commands64(cfg, u, ids):
    """(c0, c1) of LR:641-653 in float64 before the keep gate of LR:656, for env ids `ids` of the shard."""
    cr = command_ranges(cfg)
    U = u[ids].double()
    c0 = 2.0 * U[:, 36] - 1.0
    c1 = (cr["lin_vel_y"][1] - cr["lin_vel_y"][0]) * U[:, 37] + cr["lin_vel_y"][0]
    hi = (ids + cfg.env_id_offset) < C.high_vel_env_count(cfg.num_envs)
    x0, x1 = cr["lin_vel_x"]
    c0 = torch.where(hi, (x1 - x0) * U[:, 39] + x0, c0)
    c1 = torch.where(hi & (c0.abs() >= 1.0), torch.zeros_like(c1), c1)
    return c0, c1, hi


# ----------------------------------------------------------------------------- the probe
def make_reset_probe(cfg, n, seed=41, reset_share=0.4, mark_share=0.25):
    """dict(state, hf, u, ids, ter, noise): the shard's state, its (N, 44) uniform table, the ids the step resets
    (time-outs; the other envs cannot terminate), the terrain tables and the step's noise.  reset_share 0 / 1: no env
    / every env resets.  A `mark_share` of the reset envs sits on the 500-step resampling mark too (episode length
    1,499: the step increments it to 1,500, a time-out on the mark), as does a share of the other envs (499)."""
    off = cfg.env_id_offset
    hf = S.make_terrain(cfg, seed=seed)
    s = S.make_state(cfg, n, hf, seed=seed, env_id_offset=off)
    g = torch.Generator().manual_seed(seed + 500 + off)
    rand = lambda *sh: torch.rand(*sh, generator=g)
    uni = lambda lo, hi, *sh: lo + (hi - lo) * rand(*sh)
    sgn = lambda *sh: torch.where(rand(*sh) < 0.5, -1.0, 1.0)
    f32 = lambda x: torch.as_tensor(x, dtype=torch.float64).float()
    R = cfg.reset
    gid = torch.arange(n) + off
    hi = gid < C.high_vel_env_count(cfg.num_envs)
    reset = rand(n) < reset_share if 0 < reset_share < 1 else torch.full((n,), bool(reset_share))
    mark = torch.where(reset, rand(n) < mark_share, rand(n) < 0.1)

    # ---- episode lengths: time-outs reset, nothing else terminates
    ep = s["episode_length_buf"].clamp(max=cfg.max_episode_length - 10)
    ep = torch.where((ep + 1) % 500 == 0, ep - 1, ep)
    ep = torch.where(reset, torch.full_like(ep, cfg.max_episode_length), ep)
    ep = torch.where(mark, torch.where(reset, torch.full_like(ep, 1499), torch.full_like(ep, 499)), ep)
    s["episode_length_buf"] = ep
    nb = cfg.num_bodies
    cf = s["contact_forces"].view(n, nb, 3)
    for b in cfg.termination_contact_indices:
        cf[:, b, :] = 0.0
    root = s["root_states"]
    root[:, 7:10].clamp_(-0.5, 0.5)                 # no fall-down, no base_vel_violate_commands
    if not cfg.is_plane:
        root[:, 0].clamp_(1.0, cfg.x_size - 1.0)     # inside the border
        root[:, 1].clamp_(1.0, cfg.y_size - 1.0)
    s["base_lin_vel"] = 0.5 * torch.randn(n, 3, generator=g)
    s["base_ang_vel"] = 0.5 * torch.randn(n, 3, generator=g)
    pg = torch.randn(n, 3, generator=g) + torch.tensor([0.0, 0.0, -4.0])
    s["projected_gravity"] = pg / pg.norm(dim=1, keepdim=True)

    # ---- the uniform table: commands by design (inverting LR:641-656), extremes on some rows
    u = rand(n, C.RESET_NU)
    cr = command_ranges(cfg)
    x0, x1 = cr["lin_vel_x"]
    y0, y1 = cr["lin_vel_y"]
    kind = rand(n)
    near, low = kind < 0.35, (kind >= 0.35) & (kind < 0.65)
    r = torch.where(near, uni(0.2 * (1 + 3 * MARGIN), 0.25, n), torch.where(low, uni(0.0, 0.19, n), uni(0.3, 0.9, n)))
    th = uni(-math.pi, math.pi, n)
    c1 = (r * torch.sin(th)).clamp(y0 * 0.99, y1 * 0.99)
    c0 = torch.sign(torch.cos(th)) * (r ** 2 - c1 ** 2).clamp(min=0).sqrt()
    c0 = torch.where(r >= 0.3, c0.clamp(-0.95, 0.95), c0)
    u[:, 36] = f32((c0.double() + 1.0) / 2.0)
    u[:, 37] = f32((c1.double() - y0) / (y1 - y0))
    # high-speed slice: c0 from column 39; |c0| > 1 (wide ranges only), exactly 1, or below 1
    hk = rand(n)
    c0h = torch.where(hk < 0.2, sgn(n) * uni(1.05, 1.95, n), c0) if x1 - x0 > 2 else c0
    u[:, 39] = f32((c0h.double() - x0) / (x1 - x0))
    exact = (hk >= 0.2) & (hk < 0.4)
    if x1 - x0 > 2:      # [-2, 2]: u = 0.25 / 0.75 give exactly -1 / +1 in both precisions
        u[:, 39] = torch.where(exact, torch.where(rand(n) < 0.5, 0.25, 0.75), u[:, 39])
    else:                # [-1, 1]: only u = 0 gives |c0| = 1 (c0 = -1)
        u[:, 39] = torch.where(exact, 0.0, u[:, 39])
    edge = rand(n)
    u[edge < 0.03] = 0.0
    u[edge > 0.97] = U_TOP

    # ---- terrain curriculum (LR:845-866) of the reset envs: up, down or neither, from the pre-reset command (the
    # fresh one on the mark)
    origins, types = terrain_tables(cfg, n, seed)
    L = cfg.num_rows
    levels = torch.randint(1, L - 1, (n,), generator=g)
    cmd = s["commands"]
    if not cfg.is_plane:
        ck = rand(n)
        up, down = ck < 0.35, (ck >= 0.35) & (ck < 0.7)
        levels = torch.where(up & (rand(n) < 0.45), torch.full_like(levels, L - 1), levels)
        levels = torch.where(down & (rand(n) < 0.45), torch.zeros_like(levels), levels)
        # top level + up: u[43] at 0, at 1 - 2^-24, or interior (at least 0.02 / L from every k / L)
        wk = rand(n)
        interior = (torch.randint(0, L, (n,), generator=g).double() + uni(0.02, 0.98, n).double()) / L
        u[:, 43] = torch.where(wk < 0.25, 0.0, torch.where(wk < 0.5, U_TOP, f32(interior)))
        # pre-reset commands of the envs off the mark: a norm in (0.3, 1) for up / down, zero or in (0.05, 0.3) else
        rc = torch.where(up | down, uni(0.3, 1.0, n), torch.where(rand(n) < 0.5, torch.zeros(n), uni(0.05, 0.3, n)))
        phi = uni(-math.pi, math.pi, n)
        cmd[:, 0] = torch.where(mark, 0.0, rc * torch.cos(phi))
        cmd[:, 1] = torch.where(mark, 0.0, rc * torch.sin(phi))
        # what the curriculum sees: the fresh draw on the mark (old command 0: down fires only with the fresh one)
        f0, f1, _ = draw_commands64(cfg, u, torch.arange(n))
        fn = torch.hypot(f0, f1)
        fn = torch.where(fn > 0.2, fn, torch.zeros_like(fn))
        seen = torch.where(mark, fn, torch.hypot(cmd[:, 0].double(), cmd[:, 1].double()))
        half = cfg.terrain_length / 2
        dthr = seen * cfg.episode_length_s * 0.5
        d_up = half * uni(1.05, 1.5, n).double()
        d_down = uni(0.05, 0.95, n).double() * torch.minimum(dthr, torch.full_like(dthr, half))
        lo_n = torch.maximum(dthr * 1.05, torch.full_like(dthr, 0.01))
        d_nei = torch.where(lo_n < half * 0.9, lo_n + (half * 0.95 - lo_n) * rand(n).double(), d_up)
        dist = torch.where(up, d_up, torch.where(down & (seen > 0), d_down, d_nei))
        env_origins = origins[levels, types].clone()
        psi = uni(-math.pi, math.pi, n).double()
        newxy = env_origins[:, :2].double() + dist[:, None] * torch.stack([torch.cos(psi), torch.sin(psi)], dim=1)
        root[:, 0:2] = torch.where(reset[:, None], newxy.float(), root[:, 0:2])
    else:
        env_origins = torch.zeros(n, 3)
    if cfg.base_vel_violate_commands:       # levels <= 3 off the reset list: the wide commands cannot terminate them
        levels = torch.where(reset, levels, levels.clamp(max=3))
    s["terrain_levels"] = levels
    s["obs_buf"][:, :8] = 1.5 * cfg.clip_observations * sgn(n, 8)             # history entries beyond the clip
    ids = reset.nonzero(as_tuple=False).flatten()
    noise = S.make_noise(n, seed=seed + 1, n_points=len(cfg.measured_points_x) * len(cfg.measured_points_y))
    return dict(state=s, hf=hf, u=u, ids=ids, mark=mark, noise=noise,
                ter=dict(origins=origins, types=types, env_origins=env_origins))


# ----------------------------------------------------------------------------- references
def _terrain_arg(cfg, ter, dtype):
    if cfg.is_plane:
        return None
    return dict(origins=ter["origins"].to(dtype), types=ter["types"], max_level=cfg.num_rows, env_length=cfg.terrain_length,
                max_episode_length_s=cfg.episode_length_s)


class ResetOracle64(Oracle64):
    """Oracle64 whose height re-scan after the reset takes its cells from a given fp32 root state."""
    root32_after = None

    def _scan(self, pts_body, root_states=None, quat=None):
        if self.root32_after is not None and root_states is None:
            return scan_cells(self.cfg, self.height_samples, self.root32_after, pts_body.float(), self._index_math)
        return super()._scan(pts_body, root_states, quat)


def _run_reset(env, cfg, u, ids, noise, ter, pre_step, push_vel, root32_after=None, dtype=torch.float32):
    """The oracle's side of one reset step on `env` (any precision)."""
    env.env_origins = ter["env_origins"].to(dtype).clone()
    if pre_step:
        mark = ((env.episode_length_buf + 1) % cfg.resample_interval == 0).nonzero(as_tuple=False).flatten()
        env.resample_commands(mark, u, cfg.reset)                               # LR:612-613
        ids, _, _ = env.pre_reset(noise, push_vel=push_vel)
    env.pre = dict(root_states=env.root_states.clone(), commands=env.commands.clone(),
                   terrain_levels=env.terrain_levels.clone(), obs_buf=env.obs_buf.clone(),
                   Kp_factors=env.Kp_factors.clone(), Kd_factors=env.Kd_factors.clone(),
                   motor_strength_factors=env.motor_strength_factors.clone())
    env.reset_idx_draw(ids, u, custom_origins=not cfg.is_plane, terrain=_terrain_arg(cfg, ter, dtype))
    if root32_after is not None:
        env.root32_after = root32_after(env) if callable(root32_after) else root32_after.float().cpu()
    env.apply_reset(ids, {})
    env.post_reset(noise)
    env.ids = ids
    return env


def reference64_reset(cfg, probe, pre_step=True, ids=None, push_vel=None, root32_after=None, index_math=None):
    """The float64 reference of one reset step on the probe: resample_commands on the mark + pre_reset (pre_step), or
    the given ids alone; then reset_idx_draw, apply_reset and post_reset.  `root32_after`: the fp32 root state whose
    cells the post-reset height scan takes (default: the float64 root rounded to fp32)."""
    im = cfg.index_math if index_math is None else index_math
    st = probe["state"]
    with default_dtype(torch.float64):
        s64 = {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in st.items()}
        env = ResetOracle64(cfg, s64, probe["hf"], im)
        nz = {k: v.double() for k, v in probe["noise"].items()}
        pv = None if push_vel is None else push_vel.double().cpu()
        return _run_reset(env, cfg, probe["u"].double(), probe["ids"] if ids is None else ids, nz, probe["ter"], pre_step,
                          pv, root32_after, torch.float64)


def reference32_reset(cfg, probe, pre_step=True, ids=None):
    """The plain fp32 oracle's reset step on CPU."""
    env = O.OracleEnv(cfg, {k: v.clone() for k, v in probe["state"].items()}, probe["hf"])
    return _run_reset(env, cfg, probe["u"].clone(), probe["ids"] if ids is None else ids, probe["noise"], probe["ter"],
                      pre_step, None)


# ----------------------------------------------------------------------------- gates and checks
def gates(cfg, probe, env):
    """Every decision of the reset side as {name: boolean tensor over the envs it applies to}, from the float64
    reference env after its step (`env.pre`: the state reset_idx started from)."""
    ids = env.ids
    u = probe["u"]
    out = {}
    if not cfg.is_plane and cfg.reset.terrain_curriculum:
        pre = env.pre
        dist = torch.norm(pre["root_states"][ids, :2] - probe["ter"]["env_origins"][ids, :2].double(), dim=1)
        up = dist > cfg.terrain_length / 2
        cn = torch.norm(pre["commands"][ids, :2], dim=1)
        down = (dist < cn * cfg.episode_length_s * 0.5) & ~up
        lv = pre["terrain_levels"][ids]
        L = cfg.num_rows
        out["curriculum: up"] = up
        out["curriculum: down"] = down
        out["curriculum: neither"] = ~up & ~down
        out["curriculum: top level + up (wraps)"] = up & (lv == L - 1)
        out["curriculum: level 0 + down (clips)"] = down & (lv == 0)
        out["curriculum: zero pre-reset command"] = cn == 0
        mk = probe["mark"][ids]
        out["reset on the resampling mark"] = mk
    c0, c1, hi = draw_commands64(cfg, u, ids)
    nrm = torch.hypot(c0, c1)
    out["keep: |c_xy| in (0.2, 0.25]"] = (nrm > 0.2) & (nrm <= 0.25)
    out["keep: |c_xy| < 0.19"] = nrm < 0.19
    out["keep: |c_xy| > 0.2"] = nrm > 0.2
    if hi.any():
        c0h = c0[hi]
        out["high slice: |c0| < 1"] = c0h.abs() < 1
        out["high slice: |c0| == 1"] = c0h.abs() == 1
        if cfg.reset.lin_vel_x[1] - cfg.reset.lin_vel_x[0] > 2:
            out["high slice: |c0| > 1"] = c0h.abs() > 1
    return out


def margins_ok(cfg, probe, env):
    """Envs whose decided values sit within MARGIN (relative) of a threshold without being exact in fp32: [] when
    the probe is clean."""
    ids = env.ids
    u = probe["u"]
    bad = []
    c0, c1, hi = draw_commands64(cfg, u, ids)
    nrm = torch.hypot(c0, c1)
    near = ((nrm - 0.2).abs() < MARGIN * 0.2) & (nrm != 0)
    bad += [f"env {int(e)}: |c_xy| = {float(v)!r}" for e, v in zip(ids[near], nrm[near])]
    h1 = hi & ((c0.abs() - 1).abs() < MARGIN) & (c0.abs() != 1)
    # exact in fp32 when the fp32 draw of column 39 equals the float64 one (e.g. u = 1 - 2^-24 on [-1, 1])
    x0, x1 = cfg.reset.lin_vel_x
    c0_32 = (np.float32(x1 - x0) * u[ids, 39].numpy().astype(np.float32) + np.float32(x0)).astype(np.float64)
    h1 &= torch.from_numpy(c0_32) != c0
    bad += [f"env {int(e)}: high-slice c0 = {float(v)!r}" for e, v in zip(ids[h1], c0[h1])]
    if not cfg.is_plane and cfg.reset.terrain_curriculum:
        pre = env.pre
        dist = torch.norm(pre["root_states"][ids, :2] - probe["ter"]["env_origins"][ids, :2].double(), dim=1)
        half = cfg.terrain_length / 2
        thr = torch.norm(pre["commands"][ids, :2], dim=1) * cfg.episode_length_s * 0.5
        up = dist > half
        for name, t, live in (("env_length / 2", torch.full_like(dist, half), torch.ones_like(up)), ("|cmd| T / 2", thr, ~up)):
            m = ((dist - t).abs() < MARGIN * t) & (t > 0) & live
            bad += [f"env {int(e)}: dist {float(d)!r} vs {name} {float(x)!r}" for e, d, x in zip(ids[m], dist[m], t[m])]
        L = cfg.num_rows
        g = u[ids, 43].double() * L
        m = ((g - g.round()).abs() < MARGIN) & (g != g.round()) & (u[ids, 43] != U_TOP)
        bad += [f"env {int(e)}: u[43] L = {float(v)!r}" for e, v in zip(ids[m], g[m])]
    return bad


# ----------------------------------------------------------------------------- compared fields
def drawn_fields(env):
    """{name: (N, C) tensor} of what reset_idx draws, any precision."""
    n = env.root_states.shape[0]
    return dict(root_states=env.root_states, dof_state=env.dof_state.reshape(n, 24), commands=env.commands,
                Kp_factors=env.Kp_factors.reshape(n, 1), Kd_factors=env.Kd_factors.reshape(n, 1),
                motor_strength_factors=env.motor_strength_factors.reshape(n, 1))


def check_reset_rows(got, ref, ids, what, obs=True):
    """The bound on every drawn field and (obs) on obs_buf[:, :45] and privileged_obs_buf of the reset envs; `got` and
    `ref` are env-like objects (FusedLeggedRobot, OracleEnv)."""
    ids_c = ids.cpu()
    g, r = drawn_fields(got), drawn_fields(ref)
    pairs = list(g.keys())
    if obs:
        g.update(obs45=got.obs_buf[:, :45], priv=got.privileged_obs_buf)
        r.update(obs45=ref.obs_buf[:, :45], priv=ref.privileged_obs_buf)
        pairs += ["obs45", "priv"]
    for k in pairs:
        a, b = g[k].detach().cpu()[ids_c], r[k].detach().cpu()[ids_c]
        if len(ids_c) == 0:
            continue
        check_bound(a.T, b.T, [f"{k}[{c}]" for c in range(b.shape[1])], f"{what}: {k}")


def exact_failures(cfg, probe, got, ref, obs=True, shifted=True):
    """The exactness claims on the reset envs of `got` (env-like, any device), judged against the float64 reference
    `ref` of the same step: [] when they all hold.  `shifted`: the history of obs_buf moved by one slot on this step
    (a whole step); False for the fix-up alone, which writes slot 0 and leaves the history as it was."""
    ids = ref.ids
    R = cfg.reset
    cpu = lambda t: t.detach().cpu()
    bad = []
    if not torch.equal(cpu(got.terrain_levels), ref.terrain_levels):
        bad.append("terrain_levels differ")
    lv = cpu(got.terrain_levels)[ids]
    if not cfg.is_plane and not torch.equal(cpu(got.env_origins)[ids], probe["ter"]["origins"][lv, probe["ter"]["types"][ids]]):
        bad.append("env_origins != terrain_origins[level, type]")
    f = {k: cpu(v)[ids] for k, v in drawn_fields(got).items()}
    zero = ref.commands[ids, :2] == 0
    if not (f["commands"][:, :2][zero] == 0).all():
        bad.append("a zeroed command is not exactly 0")
    u = probe["u"][ids]
    f32 = lambda x: float(np.float32(x))
    vr = R.base_init_vel_range
    for k, ax in enumerate(("x", "y", "z", "roll", "pitch", "yaw")):
        lo = (vr[ax] if isinstance(vr, dict) else vr)[0]
        m = u[:, 30 + k] == 0
        if not (f["root_states"][m, 7 + k] == f32(lo)).all():
            bad.append(f"u[{30 + k}] = 0 does not give exactly lo = {lo} of {ax}")
    for col, name, rng, on in ((40, "Kp_factors", R.kp_range, R.randomize_kp), (41, "Kd_factors", R.kd_range, R.randomize_kd),
                               (42, "motor_strength_factors", R.motor_strength_range, R.randomize_motor_strength)):
        pre = ref.pre[name].reshape(-1)[ids].float()
        if on and not (f[name][u[:, col] == 0, 0] == f32(rng[0])).all():
            bad.append(f"u[{col}] = 0 does not give exactly the lower {name}")
        if not on and not torch.equal(f[name][:, 0], pre):
            bad.append(f"{name} changed with its randomisation off")
    dof = f["dof_state"].view(-1, 12, 2)
    dflt = torch.tensor(cfg.dof_tables()["default_dof_pos"], dtype=torch.float32)
    if R.dof_init_pos_ratio_range is None and not torch.equal(dof[..., 0], dflt.expand_as(dof[..., 0])):
        bad.append("dof positions != defaults without a ratio range")
    if not R.randomize_dof_vel and not (dof[..., 1] == 0).all():
        bad.append("dof velocities != 0 without randomize_dof_vel")
    if R.randomize_dof_vel:
        m = u[:, 12:24] == 0
        if not (dof[..., 1][m] == f32(min(R.dof_init_vel_range))).all():
            bad.append("u = 0 does not give exactly min(dof_init_vel_range)")
    if R.base_init_rot_range is None:
        q0 = torch.tensor(R.base_init_state[3:7], dtype=torch.float32)
        if not torch.equal(f["root_states"][:, 3:7], q0.expand(len(ids), 4)):
            bad.append("quaternion != base_init_state[3:7] without a rotation range")
    if obs:
        clip = cfg.clip_observations
        old = ref.pre["obs_buf"][ids].float()
        want = old[:, :225].clamp(-clip, clip) if shifted else old[:, 45:]
        if not torch.equal(cpu(got.obs_buf)[ids, 45:], want):
            bad.append("history columns of the reset envs != " + ("old rows, clipped" if shifted else "old history"))
    return bad
