"""A probe state for check_termination and the stages it reads (the base frame, the contact filter and the heading
command), and its float64 reference (plain helper module of tests/test_cpu_termination_probe.py and
tests/test_gpu_termination.py).

`make_termination_probe` starts from `synthetic.make_state` and edits it env by env, together with the (N, 44) uniform
table the kernels read on the 500-step resampling mark, so that every termination clause the config applies is on for
a sizeable share of the envs, off for another, and the only reason to reset for a third: termination-body contact
(one body or several), time-out, base_vel_violate_commands (both signs, the wrong signs, a zero command, levels 3 and
4), out-of-border (each of the four sides, and the border strip [x_size, x_limit) that stays inside) and fall-down.
The clauses a config turns off see the same values and must not reset.  Envs on the resampling mark are decided on
their fresh command: some of them would violate with the old one and not with the fresh one, or the reverse.  Every
decided value stays at least MARGIN from its threshold, except the exact slices, which both precisions compute
exactly: a body force (0, 0, 1) and (0, 0, nextafter(1, inf)), foot forces Fz = 1 and nextafter(1, inf), positions
0, x_limit and nextafter(x_limit, -inf) (and the same in y), root v_z = -5 and nextafter(-5, -inf).

`reference64_termination` runs the oracle's resample_commands on the mark and pre_reset in float64 through
reward_probe.Oracle64.
"""
import math

import numpy as np
import torch

from isaacgymloco_b200 import config as C
from isaacgymloco_b200 import synthetic as S
from oracle import torch_oracle as O
from reset_probe import terrain_tables
from reward_probe import FLOOR, RTOL, Oracle64, bound, check_bound, default_dtype  # noqa: F401  (re-exported)

TASKS = ("flat", "stairs", "amp", "recover", "plane")
VARIANTS = ("default", "all-on", "all-off")
CONFIGS = [(t, "default") for t in TASKS] + [("flat", "all-on"), ("flat", "all-off")]
CLAUSES = ("contact", "time-out", "velocity", "border", "fall-down")
THIGH = 2                     # FL_thigh of the AlienGo body list (the base is body 0)
MARGIN = 0.05                 # forces, velocities, positions: distance from a threshold
HEADING_MARGIN = 1e-2         # radians: cmd[3] - heading from 0 and +-pi, heading from the atan2 cut
ONE_UP = float(np.nextafter(np.float32(1.0), np.float32(np.inf)))
FIVE_DOWN = float(np.nextafter(np.float32(-5.0), np.float32(-np.inf)))


# ----------------------------------------------------------------------------- configs
def termination_cfg(task, variant, n, index_math=C.INDEX_MATH_TORCH_CUDA, num_envs=None, env_id_offset=0):
    """`task` in TASKS ("plane": the flat task on a plane mesh with out_of_border left True, so that the is_plane gate
    is what turns the border clause off), `variant` in VARIANTS.  "all-on": the flat task with
    base_vel_violate_commands and two termination bodies (the base and a thigh); "all-off": no border, fall-down or
    velocity clause (contacts and time-out only).  Pushes and disturbances are off."""
    cfg = C.aliengo("flat" if task == "plane" else task, num_envs=num_envs or n, index_math=index_math,
                    env_id_offset=env_id_offset)
    if task == "plane":
        cfg.mesh_type = "plane"
    if variant == "all-on":
        assert task == "flat", task
        cfg.base_vel_violate_commands = True
        cfg.termination_contact_indices = [0, THIGH]
    elif variant == "all-off":
        cfg.out_of_border = cfg.fall_down = cfg.base_vel_violate_commands = False
    else:
        assert variant == "default", variant
    cfg.reset.push_robots = False
    cfg.reset.disturbance = False
    return cfg


def clauses(cfg):
    """The termination clauses the config applies (check_termination, LR:249-286)."""
    on = dict(contact=bool(cfg.termination_contact_indices), velocity=cfg.base_vel_violate_commands,
              border=cfg.out_of_border and not cfg.is_plane, **{"time-out": True, "fall-down": cfg.fall_down})
    return [c for c in CLAUSES if on[c]]


def limits(cfg):
    """(x_limit, y_limit) of terrain.py:226 (the flat task's values on a plane mesh, whose clause is off)."""
    return cfg.x_size + cfg.border_size / 2, cfg.y_size + cfg.border_size / 2


def wide_rotations(cfg):
    rr = cfg.reset.base_init_rot_range
    return rr is not None and rr["roll"][1] > 3.0


# ----------------------------------------------------------------------------- the probe
def make_termination_probe(cfg, n, seed=23):
    """dict(state, hf, u, mark, noise, ter): the shard's state, its (N, 44) uniform table, the envs on the
    resampling mark, the step's noise and the terrain tables the in-kernel reset reads."""
    off = cfg.env_id_offset
    hf = S.make_terrain(cfg, seed=seed)
    s = S.make_state(cfg, n, hf, seed=seed, env_id_offset=off)
    g = torch.Generator().manual_seed(seed + 900 + off)
    rand = lambda *sh: torch.rand(*sh, generator=g, dtype=torch.float64)
    uni = lambda lo, hi, *sh: lo + (hi - lo) * rand(*sh)
    sgn = lambda *sh: torch.where(rand(*sh) < 0.5, -1.0, 1.0).double()
    pick = lambda p, *sh: rand(*sh) < p
    choose = lambda p, a, b: torch.where(pick(p, n), torch.as_tensor(a, dtype=torch.float64),
                                         torch.as_tensor(b, dtype=torch.float64))
    f32 = lambda x: torch.as_tensor(x, dtype=torch.float64).float()
    nb, cl = cfg.num_bodies, clauses(cfg)
    interval, max_len = cfg.resample_interval, cfg.max_episode_length

    # ---- which clauses fire: none (20 %), exactly one (55 %, split evenly) or each with probability 1/2 (25 %)
    k = rand(n)
    none, multi = k < 0.2, k >= 0.75
    sole = ((k - 0.2) / 0.55 * len(cl)).floor().long().clamp(0, len(cl) - 1)
    on = {}
    for c in CLAUSES:
        if c in cl:
            on[c] = ~none & ((~multi & (sole == cl.index(c))) | (multi & pick(0.5, n)))
        else:
            on[c] = pick(0.3, n)            # a clause the config turns off sees the same values

    # ---- episode lengths: time-out at max -> max + 1 or beyond (1499: on the mark too); none at 0, max - 1 -> max
    # (on the mark), 499 (on the mark) or in between
    mark = pick(0.15, n)
    r = torch.randint(1, max_len - 1, (n,), generator=g)
    r = torch.where((r + 1) % interval == 0, r - 1, r)
    ep = torch.where(mark, torch.where(on["time-out"], 1499, torch.where(pick(0.5, n), 499, max_len - 1)),
                     torch.where(on["time-out"], torch.where(pick(0.5, n), max_len, 5000),
                                 torch.where(pick(0.3, n), 0, r)))
    s["episode_length_buf"] = ep.long()
    mark = (ep + 1) % interval == 0

    # ---- rotations: yaw over (-pi, pi], some envs upside down (recover: +-3.14 on every axis)
    if wide_rotations(cfg):
        roll, pitch, yaw = uni(-3.14, 3.14, n), uni(-3.14, 3.14, n), uni(-3.14, 3.14, n)
    else:
        roll = torch.where(pick(0.15, n), sgn(n) * (math.pi - uni(0.0, 0.4, n)), (0.15 * torch.randn(n, generator=g)).double())
        pitch = (0.15 * torch.randn(n, generator=g)).double().clamp(-0.4, 0.4)
        yaw = uni(-math.pi, math.pi, n)
    ex = torch.tensor([[1.0, 0.0, 0.0]], dtype=torch.float64).expand(n, 3)
    for _ in range(4):                      # keep the heading clear of the atan2 cut
        q32 = S._quat_from_euler_xyz(roll, pitch, yaw).float()
        fwd = O.quat_apply(q32.double(), ex)
        heading = torch.atan2(fwd[:, 1], fwd[:, 0])
        cut = (math.pi - heading.abs()) < 2 * HEADING_MARGIN
        if not cut.any():
            break
        yaw = torch.where(cut, yaw + 5 * HEADING_MARGIN, yaw)
    root = s["root_states"]
    root[:, 3:7] = q32

    # ---- termination bodies: |F| in (1.5, 50) when hit, below 0.5 else; (0, 0, 1) and (0, 0, nextafter(1, inf))
    cf = s["contact_forces"].view(n, nb, 3)
    K = list(cfg.termination_contact_indices)
    if K:
        which = torch.randint(0, len(K) + 1, (n,), generator=g)        # len(K) = every body, else that body alone
        for j, b in enumerate(K):
            hit = on["contact"] & ((which == j) | (which == len(K)))
            d = torch.randn(n, 3, generator=g)
            d = d / d.norm(dim=1, keepdim=True)
            mag = torch.where(hit, uni(1.5, 50.0, n), uni(0.0, 0.5, n) * pick(0.6, n)).float()
            cf[:, b, :] = d * mag[:, None]
            exact = pick(0.12, n)
            cf[:, b, :] = torch.where((exact & hit)[:, None], torch.tensor([0.0, 0.0, ONE_UP]), cf[:, b, :])
            cf[:, b, :] = torch.where((exact & ~hit)[:, None], torch.tensor([0.0, 0.0, 1.0]), cf[:, b, :])
    else:                                   # a base contact that must not terminate
        d = torch.randn(n, 3, generator=g)
        cf[:, 0, :] = d / d.norm(dim=1, keepdim=True) * torch.where(on["contact"], uni(1.5, 50.0, n), 0.0).float()[:, None]

    # ---- feet: Fz in (1.05, 150) or (0, 0.95), exactly 1 or nextafter(1, inf); last_contacts both ways
    feet = cfg.feet_indices
    fz = torch.where(pick(0.5, n, 4), uni(1.05, 150.0, n, 4), uni(0.0, 0.95, n, 4))
    ek = rand(n, 4)
    fz = torch.where(ek < 0.08, 1.0, torch.where(ek < 0.16, ONE_UP, fz))
    cf[:, feet, 2] = fz.float()
    s["last_contacts"] = pick(0.5, n, 4)

    # ---- fall-down: root v_z below -5.05 (or nextafter(-5, -inf)) or above -4.95 (or exactly -5)
    ek = rand(n)
    wz = torch.where(on["fall-down"], torch.where(ek < 0.15, FIVE_DOWN, uni(-8.0, -5.05, n)),
                     torch.where(ek < 0.15, -5.0, uni(-4.95, 1.5, n)))

    # ---- velocity: err = v_x - cmd_x (cmd_x the command check_termination sees: the fresh one on the mark)
    #   V+: err in (2.05, 3), cmd_x < 0   V-: err in (-3, -2.05), cmd_x > 0   (violate; reset at levels 4 and 9 only)
    #   W+: err in (2.05, 3), cmd_x > 0   W-: err in (-3, -2.05), cmd_x < 0   Z: |err| in (2.05, 3), cmd_x == 0
    #   S: |err| < 1.95
    L = cfg.num_rows
    vk = rand(n)
    viol = on["velocity"] | (vk < 0.3)                                  # V+/-: on, or off by the level gate
    kind_w, kind_z = ~viol & (vk >= 0.3) & (vk < 0.55), ~viol & (vk >= 0.55) & (vk < 0.7)
    kind_s = ~viol & ~kind_w & ~kind_z
    e_sign = sgn(n)
    err = torch.where(kind_s, uni(-1.95, 1.95, n), e_sign * uni(2.05, 3.0, n))
    mag = uni(0.3, 0.95, n)
    c_seen = torch.where(viol, -e_sign * mag, torch.where(kind_w, e_sign * mag, torch.where(kind_z, 0.0, sgn(n) * mag)))
    c_seen = torch.where(kind_s & pick(0.2, n), 0.0, c_seen)
    levels = torch.randint(0, L, (n,), generator=g)
    hi_lv = torch.where(pick(0.5, n), 4, L - 1)
    lo_lv = torch.where(pick(0.5, n), 3, 0)
    levels = torch.where(viol, torch.where(on["velocity"], hi_lv, lo_lv), levels)
    v_x = c_seen + err
    # the old command of the envs on the mark: violating where the fresh one does not (level > 3), and not where it does
    seen_viol = viol & on["velocity"]
    e_old = uni(2.1, 2.9, n)
    c_old = torch.where(v_x - e_old < -MARGIN, v_x - e_old, v_x + e_old)          # (err > 2, cmd < 0) or (err < -2, cmd > 0)
    c_old = torch.where(seen_viol, v_x - uni(-1.5, 1.5, n), c_old)
    levels = torch.where(mark & ~seen_viol & ~viol, torch.randint(4, L, (n,), generator=g), levels)
    s["terrain_levels"] = levels.long()
    cmd = s["commands"]
    cmd[:, 0] = torch.where(mark, c_old, c_seen).float()

    # world velocity with body-frame v_x = v_x and world v_z = wz (LR:197: base_lin_vel = quat_rotate_inverse(q, v))
    fxy = fwd[:, :2]
    nn = fxy.norm(dim=1)
    if wide_rotations(cfg):
        assert not cfg.base_vel_violate_commands
        wxy = (0.5 * torch.randn(n, 2, generator=g)).double()
    else:
        t = v_x - fwd[:, 2] * wz
        perp = torch.stack([-fxy[:, 1], fxy[:, 0]], dim=1) / nn[:, None]
        wxy = t[:, None] * fxy / (nn ** 2)[:, None] + uni(-0.5, 0.5, n)[:, None] * perp
    root[:, 7:9] = wxy.float()
    root[:, 9] = wz.float()

    # ---- the uniform table: fresh commands of the envs on the mark (LR:641-656) by design
    u = torch.rand(n, C.RESET_NU, generator=g)
    x0, x1 = cfg.reset.lin_vel_x
    assert (x0, x1) == (-1.0, 1.0)          # column 36 and column 39 (high-speed slice) then give the same c0
    u0 = f32((c_seen + 1.0) / 2.0)          # c_seen == 0: u = 0.5, c0 = 0 exactly
    u[:, 36] = torch.where(mark, u0, u[:, 36])
    u[:, 39] = torch.where(mark, u0, u[:, 39])
    y0, y1 = cfg.reset.lin_vel_y
    c1 = torch.where(pick(0.5, n), sgn(n) * uni(0.25, 0.45, n), uni(-0.15, 0.15, n))   # clear of the 0.2 keep gate
    u[:, 37] = torch.where(mark, f32((c1 - y0) / (y1 - y0)), u[:, 37])

    # ---- heading command: d = cmd[3] - heading in (-2 pi, 2 pi), both signs and both sides of +-pi
    band = torch.randint(0, 4, (n,), generator=g)
    lo = torch.tensor([-2 * math.pi, -math.pi, 0.0, math.pi], dtype=torch.float64)[band] + HEADING_MARGIN
    d = lo + (math.pi - 2 * HEADING_MARGIN) * rand(n)
    h0, h1 = cfg.reset.heading
    c3 = heading + d
    c3m = torch.where(c3 >= h1, c3 - 2 * math.pi, torch.where(c3 < h0, c3 + 2 * math.pi, c3))      # the fresh draw's range
    cmd[:, 3] = torch.where(mark & torch.tensor(cfg.heading_command), cmd[:, 3], c3.float())
    u[:, 38] = torch.where(mark, f32((c3m - h0) / (h1 - h0)).clamp(max=float(np.float32(1) - np.float32(2 ** -24))), u[:, 38])

    # ---- positions: each side of the border, the strip [size, limit), the exact slices
    xl, yl = limits(cfg)

    def coord(size, lim, side_lo, side_hi):
        inside = torch.where(pick(0.2, n), uni(size, lim - MARGIN, n), uni(MARGIN, size, n))
        ek = rand(n)
        inside = torch.where(ek < 0.05, 0.0, torch.where(ek < 0.1, float(np.nextafter(np.float32(lim), np.float32(-np.inf))), inside))
        out_hi = torch.where(pick(0.15, n), lim, lim + uni(MARGIN, 5.0, n))
        return torch.where(side_lo, -uni(MARGIN, 5.0, n), torch.where(side_hi, out_hi, inside))

    side = torch.randint(0, 4, (n,), generator=g)
    b = on["border"]
    root[:, 0] = coord(cfg.x_size, xl, b & (side == 0), b & (side == 2)).float()
    root[:, 1] = coord(cfg.y_size, yl, b & (side == 1), b & (side == 3)).float()

    s["episode_sums"] = torch.zeros_like(s["episode_sums"]) if cfg.termination_scale is not None else s["episode_sums"]
    noise = S.make_noise(n, seed=seed + 1, n_points=len(cfg.measured_points_x) * len(cfg.measured_points_y))
    origins, types = terrain_tables(cfg, n, seed)
    env_origins = torch.zeros(n, 3) if cfg.is_plane else origins[levels.clamp(0, L - 1), types].clone()
    return dict(state=s, hf=hf, u=u, mark=mark, noise=noise,
                ter=dict(origins=origins, types=types, env_origins=env_origins))


# ----------------------------------------------------------------------------- references
def _step(env, cfg, u, noise, push_vel):
    mark = ((env.episode_length_buf + 1) % cfg.resample_interval == 0).nonzero(as_tuple=False).flatten()
    env.resample_commands(mark, u, cfg.reset)                                   # LR:612-613 before LR:249
    env.ids, _, env.term_amp = env.pre_reset(noise, push_vel=push_vel)
    if not cfg.base_vel_violate_commands:
        env.vel_violate = torch.zeros(env.num_envs, dtype=torch.bool)
    return env


def reference64_termination(cfg, probe, push_vel=None, index_math=None):
    """The float64 reference of the step up to check_termination (and its reward pass): resample_commands on the mark
    from the probe's uniform table, then pre_reset.  The env carries reset_buf, time_out_buf, vel_violate,
    base_lin_vel, base_ang_vel, projected_gravity, commands, contact_filt, last_contacts, episode_sums, ids (the
    reset ids) and term_amp (the terminal AMP rows).  `push_vel` (N, 2): the push step's root xy velocities."""
    im = cfg.index_math if index_math is None else index_math
    with default_dtype(torch.float64):
        s64 = {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in probe["state"].items()}
        env = Oracle64(cfg, s64, probe["hf"], im)
        nz = {k: v.double() for k, v in probe["noise"].items()}
        pv = None if push_vel is None else push_vel.double().cpu()
        return _step(env, cfg, probe["u"].double(), nz, pv)


def reference32_termination(cfg, probe):
    """The plain fp32 oracle's step on CPU."""
    env = O.OracleEnv(cfg, {k: v.clone() for k, v in probe["state"].items()}, probe["hf"])
    return _step(env, cfg, probe["u"].clone(), probe["noise"], None)


# ----------------------------------------------------------------------------- gates and checks
def clause_decisions(cfg, probe, env):
    """{clause: bool (N,)} of every clause the config applies, from the float64 reference env after its step."""
    st = probe["state"]
    n = env.num_envs
    cf = st["contact_forces"].view(n, cfg.num_bodies, 3).double()
    root = st["root_states"].double()
    xl, yl = limits(cfg)
    out = {}
    K = list(cfg.termination_contact_indices)
    if K:
        out["contact"] = (cf[:, K].norm(dim=-1) > 1.0).any(dim=1)
    out["time-out"] = env.time_out_buf.clone()
    if cfg.base_vel_violate_commands:
        out["velocity"] = env.vel_violate.clone()
    if cfg.out_of_border and not cfg.is_plane:
        out["border"] = ~((root[:, 0] >= 0) & (root[:, 1] >= 0) & (root[:, 0] < xl) & (root[:, 1] < yl))
    if cfg.fall_down:
        out["fall-down"] = root[:, 9] < -5.0
    return out


def gates(cfg, probe, env):
    """Every decision of the probed stages as {name: (mask, over)}: the share of `mask` among the envs `over`."""
    st = probe["state"]
    n = env.num_envs
    all_ = torch.ones(n, dtype=torch.bool)
    dec = clause_decisions(cfg, probe, env)
    out = {}
    for c, m in dec.items():
        out[f"{c}: resets"] = (m, all_)
        others = torch.zeros(n, dtype=torch.bool)
        for c2, m2 in dec.items():
            if c2 != c:
                others |= m2
        out[f"{c}: the only reason"] = (m & ~others, all_)
    out["no reset"] = (~env.reset_buf, all_)
    cf = st["contact_forces"].view(n, cfg.num_bodies, 3).double()
    K = list(cfg.termination_contact_indices)
    if len(K) > 1:
        hits = cf[:, K].norm(dim=-1) > 1.0
        out["contact: one body only"] = (hits.sum(dim=1) == 1, all_)
        out["contact: the second body only"] = (hits[:, 1] & ~hits[:, 0], all_)
    ep = st["episode_length_buf"]
    out["on the resampling mark"] = (probe["mark"], all_)
    out["pre-step episode length max - 1"] = (ep == cfg.max_episode_length - 1, all_)
    out["pre-step episode length max"] = (ep == cfg.max_episode_length, all_)
    if cfg.base_vel_violate_commands:
        c0 = env.commands[:, 0]
        err = env.base_lin_vel[:, 0] - c0
        lv = env.terrain_levels
        signed = ((err > 2) & (c0 < 0)) | ((err < -2) & (c0 > 0))
        out["velocity: err > 2, cmd_x < 0"] = ((err > 2) & (c0 < 0), all_)
        out["velocity: err < -2, cmd_x > 0"] = ((err < -2) & (c0 > 0), all_)
        out["velocity: |err| > 2 with the wrong sign"] = (((err > 2) & (c0 > 0)) | ((err < -2) & (c0 < 0)), all_)
        out["velocity: |err| > 2, cmd_x == 0"] = ((err.abs() > 2) & (c0 == 0), all_)
        out["velocity: |err| < 2"] = (err.abs() < 2, all_)
        out["velocity violators: level 3"] = (lv == 3, signed)
        out["velocity violators: level 4"] = (lv == 4, signed)
        out["velocity violators: level 0"] = (lv == 0, signed)
        out["velocity violators: top level"] = (lv == cfg.num_rows - 1, signed)
        old = st["commands"][:, 0].double()
        old_err = env.base_lin_vel[:, 0] - old
        old_viol = (((old_err > 2) & (old < 0)) | ((old_err < -2) & (old > 0))) & (lv > 3)
        mk = probe["mark"]
        out["mark: the old command violates, the fresh one does not"] = (old_viol & ~env.vel_violate, mk)
        out["mark: the fresh command violates, the old one does not"] = (~old_viol & env.vel_violate, mk)
    root = st["root_states"].double()
    xl, yl = limits(cfg)
    x, y = root[:, 0], root[:, 1]
    out["border: x < 0"] = (x < 0, all_)
    out["border: y < 0"] = (y < 0, all_)
    out["border: x >= x_limit"] = (x >= xl, all_)
    out["border: y >= y_limit"] = (y >= yl, all_)
    out["border: x in the strip [x_size, x_limit)"] = ((x >= cfg.x_size) & (x < xl), all_)
    out["border: y in the strip [y_size, y_limit)"] = ((y >= cfg.y_size) & (y < yl), all_)
    out["fall-down: v_z < -5"] = (root[:, 9] < -5.0, all_)
    if cfg.heading_command:
        d = env.commands[:, 3] - heading64(root)
        for name, m in (("< -pi", d < -math.pi), ("in (-pi, 0)", (d > -math.pi) & (d < 0)),
                        ("in (0, pi)", (d > 0) & (d < math.pi)), ("> pi", d > math.pi)):
            out[f"heading: cmd[3] - heading {name}"] = (m, all_)
    out["upside down (projected gravity z > 0)"] = (env.projected_gravity[:, 2] > 0, all_)
    out["foot Fz > 1 (per foot)"] = (cf[:, cfg.feet_indices, 2] > 1.0, torch.ones(n, 4, dtype=torch.bool))
    out["last_contacts (per foot)"] = (st["last_contacts"], torch.ones(n, 4, dtype=torch.bool))
    return out


def heading64(root):
    """atan2 of the forward vector (LR:616-620) in float64 from the fp32 quaternion."""
    n = root.shape[0]
    fwd = O.quat_apply(root[:, 3:7].double(), torch.tensor([[1.0, 0.0, 0.0]], dtype=torch.float64).expand(n, 3))
    return torch.atan2(fwd[:, 1], fwd[:, 0])


def exact_slices(cfg, probe):
    """{name: bool (N,)} of the envs on an exact slice (fp32 computes the decided value exactly)."""
    st = probe["state"]
    n = st["root_states"].shape[0]
    cf = st["contact_forces"].view(n, cfg.num_bodies, 3)
    root = st["root_states"]
    xl, yl = limits(cfg)
    nx = lambda v: float(np.nextafter(np.float32(v), np.float32(-np.inf)))
    out = {}
    K = list(cfg.termination_contact_indices)
    if K:
        on_z = (cf[:, K, 0] == 0) & (cf[:, K, 1] == 0)
        out["body F = (0, 0, 1)"] = (on_z & (cf[:, K, 2] == 1.0)).any(dim=1)
        out["body F = (0, 0, nextafter(1, inf))"] = (on_z & (cf[:, K, 2] == ONE_UP)).any(dim=1)
    fz = cf[:, cfg.feet_indices, 2]
    out["foot Fz = 1"] = (fz == 1.0).any(dim=1)
    out["foot Fz = nextafter(1, inf)"] = (fz == ONE_UP).any(dim=1)
    for a, lim in ((0, xl), (1, yl)):
        ax = "xy"[a]
        out[f"{ax} = 0"] = root[:, a] == 0.0
        out[f"{ax} = {ax}_limit"] = root[:, a] == lim
        out[f"{ax} = nextafter({ax}_limit, -inf)"] = root[:, a] == nx(lim)
    out["v_z = -5"] = root[:, 9] == -5.0
    out["v_z = nextafter(-5, -inf)"] = root[:, 9] == FIVE_DOWN
    return out


def margins_ok(cfg, probe, env):
    """Envs whose decided values sit within MARGIN of a threshold without being exact in fp32: [] when the probe is
    clean."""
    st = probe["state"]
    n = env.num_envs
    cf = st["contact_forces"].view(n, cfg.num_bodies, 3).double()
    root = st["root_states"].double()
    bad = []

    def near(name, v, thr, exact=(), m=MARGIN):
        close = (v - thr).abs() < m
        for x in exact:
            close &= v != x
        idx = close.nonzero(as_tuple=False)
        bad.extend(f"{name}: env {tuple(int(i) for i in e)} value {float(v[tuple(e)])!r}" for e in idx[:20])

    K = list(cfg.termination_contact_indices)
    if K:
        near("termination-body |F|", cf[:, K].norm(dim=-1), 1.0, (1.0, ONE_UP))
    near("foot Fz", cf[:, cfg.feet_indices, 2], 1.0, (1.0, ONE_UP))
    xl, yl = limits(cfg)
    for a, lim in ((0, xl), (1, yl)):
        nx = float(np.nextafter(np.float32(lim), np.float32(-np.inf)))
        near("xy"[a], root[:, a], 0.0, (0.0,))
        near("xy"[a], root[:, a], lim, (lim, nx))
    near("root v_z", root[:, 9], -5.0, (-5.0, FIVE_DOWN))
    if cfg.base_vel_violate_commands:
        c0 = env.commands[:, 0]
        err = env.base_lin_vel[:, 0] - c0
        near("|v_x - cmd_x|", err.abs(), 2.0)
        near("cmd_x", c0, 0.0, (0.0,))
    if cfg.heading_command:
        h = heading64(root)
        d = env.commands[:, 3] - h
        for thr in (-2 * math.pi, -math.pi, 0.0, math.pi, 2 * math.pi):
            near("cmd[3] - heading", d, thr, m=1e-3)
        near("|heading| (atan2 cut)", h.abs(), math.pi, m=1e-3)
    return bad


def frame_fields(env, cmd2=True):
    """{name: (N, C)} of the frame stage (and commands[:, 2]), any precision."""
    out = dict(base_lin_vel=env.base_lin_vel, base_ang_vel=env.base_ang_vel, projected_gravity=env.projected_gravity)
    if cmd2:
        out["commands[:, 2]"] = env.commands[:, 2:3]
    return out


def check_frame(got, ref, rows, what, cmd2=True):
    """The bound on the frame fields (and, with cmd2, commands[:, 2]) of the envs `rows` (bool (N,))."""
    g, r = frame_fields(got, cmd2), frame_fields(ref, cmd2)
    rows = rows.cpu()
    for k in g:
        a, b = g[k].detach().cpu()[rows], r[k].detach().cpu()[rows]
        if len(b):
            check_bound(a.T, b.T, [f"{k}[{c}]" for c in range(b.shape[1])], f"{what}: {k}")
