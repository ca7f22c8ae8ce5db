"""-m gpu: keyed domain randomisation (ResetCfg.keyed_domain_rand): the action delay, the disturbances and the pushes
drawn from Philox streams 4-6 in the kernel chain (hl_delay_actions, hl_uniform_rows).

* Arithmetic: fed the same draws, each launch equals the torch expressions of the hooks bit for bit (torch.clamp and
  the body of _delay_actions; the two torch_rand_float forms), on clipped, NaN, +-inf and +-0 actions, aliased or not.
* Philox: the draws are the counter-based Philox4x32-10 blocks of (seed, step, global env id, stream) -- recomputed
  here on the host -- so they are uniform, independent across steps, columns and streams, and a captured launch
  draws what an eager one does.
* Two shards equal one big env for whole public step()s with the delay, disturbances and pushes.
* A replayed rollout with the real hooks equals the eager public-step() loop, and two replays draw differently.
* The gym call order is unchanged, and overriding a hook (instance or subclass) replaces the kernel.
"""
import ctypes
import weakref

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

M32 = 0xFFFFFFFF


def _bits(t):
    return t.contiguous().view(torch.int32)


def _philox_block(seed, step, env_ids, stream, block=0):
    """Philox4x32-10 of hl_noise_block (hl_common.cuh) on the host: the 4 words of (block, stream) for every env."""
    e = np.asarray(env_ids, dtype=np.uint64)
    c0 = np.full(e.shape, (block | (stream << 24)) & M32, dtype=np.uint64)
    c1 = e & M32
    c2 = (e >> np.uint64(32)) ^ np.uint64((step >> 32) & M32)
    c3 = np.full(e.shape, step & M32, dtype=np.uint64)
    k0, k1 = seed & M32, (seed >> 32) & M32
    for _ in range(10):
        p0 = c0 * np.uint64(0xD2511F53)
        p1 = c2 * np.uint64(0xCD9E8D57)
        hi0, lo0 = p0 >> np.uint64(32), p0 & np.uint64(M32)
        hi1, lo1 = p1 >> np.uint64(32), p1 & np.uint64(M32)
        c0, c1, c2, c3 = hi1 ^ c1 ^ np.uint64(k0), lo1, hi0 ^ c3 ^ np.uint64(k1), lo0
        k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
    return [c.astype(np.uint64) for c in (c0, c1, c2, c3)]


def _u01(x):
    return ((x >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)).astype(np.float32)


def _bufs(last=None, seed=0, offset=0, step_base=None):
    from isaacgymloco_b200 import _lib as L
    b = L.HlEnvBuffers()
    b.struct_bytes = ctypes.sizeof(L.HlEnvBuffers)
    b.last_actions = L.ptr(last)
    b.philox_seed, b.philox_offset = seed, offset
    b.step_base = L.ptr(step_base)
    return b


def _cfg(n, offset=0):
    from isaacgymloco_b200 import config as C
    return C.aliengo("flat", num_envs=n, env_id_offset=offset).to_c()


def _delay(c, b, a_in, a_out, delayed, dec, delay, clip, d_in, n):
    from isaacgymloco_b200 import _lib as L
    L.check(L.lib.hl_delay_actions(ctypes.byref(c), ctypes.byref(b), L.ptr(a_in), L.ptr(a_out), L.ptr(delayed), dec, delay,
                                   clip, L.ptr(d_in), n, L.stream()))


def _rows(c, b, dst, stride, cols, lo, hi, u_in, stream_id, n):
    from isaacgymloco_b200 import _lib as L
    L.check(L.lib.hl_uniform_rows(ctypes.byref(c), ctypes.byref(b), dst, stride, cols, lo, hi, L.ptr(u_in), stream_id, n,
                                  L.stream()))


def _torch_delay(actions_in, last, d, dec, delay, clip):
    """torch.clamp of step() and the body of FusedLeggedRobot._delay_actions, run on a stand-in whose torch.randint
    returns the given delays."""
    from types import SimpleNamespace
    from isaacgymloco_b200 import config as C
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    n = actions_in.shape[0]
    cfg = C.aliengo("flat", num_envs=n, decimation=dec)
    cfg.reset.delay = delay
    ns = SimpleNamespace(cfg_hot=cfg, num_envs=n, device=actions_in.device, last_actions=last,
                         actions=torch.empty_like(actions_in), delayed_actions=torch.empty(n, dec, 12, device=actions_in.device))
    torch.clamp(actions_in, -clip, clip, out=ns.actions)
    randint = torch.randint
    torch.randint = lambda lo, hi, shape, device=None: d.view(shape)
    try:
        FusedLeggedRobot._delay_actions(ns)
    finally:
        torch.randint = randint
    return ns.actions, ns.delayed_actions


def _special(x, g):
    """Sprinkle +-0, +-inf, NaN and values beyond the clip into x."""
    n = x.numel()
    flat = x.view(-1)
    for v in (0.0, -0.0, float("inf"), float("-inf"), float("nan"), 250.0, -250.0, 100.0, -100.0):
        idx = torch.randint(0, n, (max(n // 50, 1),), generator=g).to(x.device)
        flat[idx] = v
    return x


# ---------------------------------------------------------------------------------------------------- 1. arithmetic
@pytest.mark.parametrize("n", [1, 4099, 65536])
def test_delay_arithmetic_bit_for_bit(n):
    dev = "cuda:0"
    clip = 100.0
    g = torch.Generator().manual_seed(n)
    c = _cfg(n)
    for dec in (1, 2, 4):
        for delay in (True, False):
            a = _special(200.0 * torch.randn(n, 12, generator=g), g).to(dev)
            last = _special(200.0 * torch.randn(n, 12, generator=g), g).to(dev)
            d = torch.randint(0, dec, (n,), generator=g).to(dev)
            want_a, want_d = _torch_delay(a, last, d, dec, delay, clip)
            b = _bufs(last)
            out, delayed = torch.full_like(a, 7.0), torch.full((n, dec, 12), 7.0, device=dev)
            _delay(c, b, a, out, delayed, dec, int(delay), clip, d, n)
            assert torch.equal(_bits(out), _bits(want_a)), (dec, delay)
            assert torch.equal(_bits(delayed), _bits(want_d)), (dec, delay)
            alias = a.clone()                                 # actions_out aliasing actions_in
            delayed2 = torch.full_like(delayed, 7.0)
            _delay(c, b, alias, alias, delayed2, dec, int(delay), clip, d, n)
            assert torch.equal(_bits(alias), _bits(want_a)) and torch.equal(_bits(delayed2), _bits(want_d)), (dec, delay)
            assert n == 1 or torch.isnan(want_d).any()


@pytest.mark.parametrize("n", [1, 4099, 65536])
def test_uniform_rows_arithmetic_bit_for_bit(n):
    from isaacgymloco_b200 import _lib as L
    dev = "cuda:0"
    g = torch.Generator().manual_seed(7 + n)
    c, b = _cfg(n), _bufs()
    u3 = torch.rand(n, 3, generator=g)
    u3.view(-1)[:2] = torch.tensor([0.0, 1.0 - 2.0 ** -24])
    u3 = u3.to(dev)
    for lo, hi in ((-30.0, 30.0), (-30.1, 29.7), (0.0, 5.0)):
        dist = torch.full((n, 17, 3), 3.0, device=dev)
        want = dist.clone()
        want[:, 0, :] = (hi - lo) * u3 + lo                       # _disturbance_robots, LR:838-844
        _rows(c, b, L.ptr(dist), 17 * 3, 3, lo, hi, u3, 5, n)
        assert torch.equal(_bits(dist), _bits(want)), (lo, hi)
    u2 = u3[:, :2].contiguous()
    for mv in (1.0, 0.7, 1.3, 1e-3):
        root = torch.full((n, 13), 5.0, device=dev)
        want_lr = root.clone()
        want_lr[:, 7:9] = (mv - (-mv)) * u2 + (-mv)               # torch_rand_float(-mv, mv), LR:822-828
        want_here = root.clone()
        want_here[:, 7:9] = (2 * mv) * u2 - mv                    # the torch form of _push_robots
        assert torch.equal(_bits(want_lr), _bits(want_here)), mv
        _rows(c, b, L.ptr(root) + 7 * 4, 13, 2, -mv, mv, u2, 6, n)
        assert torch.equal(_bits(root), _bits(want_lr)), mv


def test_launches_reject_bad_arguments():
    from isaacgymloco_b200 import _lib as L
    n = 8
    c = _cfg(n)
    a, last = torch.zeros(n, 12, device="cuda"), torch.zeros(n, 12, device="cuda")
    b = _bufs(last)
    for dec in (0, 17):
        with pytest.raises(RuntimeError, match="decimation"):
            _delay(c, b, a, a, torch.zeros(n, 16, 12, device="cuda"), dec, 1, 100.0, None, n)
    for sid in (0, 1, 2, 3, 256):
        with pytest.raises(RuntimeError, match="stream_id"):
            _rows(c, b, L.ptr(a), 12, 3, 0.0, 1.0, None, sid, n)
    with pytest.raises(RuntimeError, match="cols"):
        _rows(c, b, L.ptr(a), 12, 5, 0.0, 1.0, None, 5, n)


# ---------------------------------------------------------------------------------------------------- 2. Philox
def test_philox_draws_statistics_and_keys():
    from scipy import stats
    from isaacgymloco_b200 import _lib as L
    n, dec, seed, off = 65536, 4, 0x1234_5678_9ABC, 4096
    dev = "cuda:0"
    c = _cfg(1 << 20, offset=off)                      # a shard whose global ids start at `off`
    gid = np.arange(n, dtype=np.uint64) + np.uint64(off)
    ones, zeros = torch.ones(n, 12, device=dev), torch.zeros(n, 12, device=dev)
    draws = {}
    for s in (5, 6, (1 << 33) + 5):
        b = _bufs(zeros, seed=seed, offset=s)
        delayed = torch.empty(n, dec, 12, device=dev)
        _delay(c, b, ones, torch.empty_like(ones), delayed, dec, 1, 100.0, None, n)
        d = dec - delayed[:, :, 0].sum(dim=1).to(torch.int64).cpu().numpy()      # actions 1, last 0: k >= d is 1
        assert (delayed[:, :, 1:] == delayed[:, :, :1]).all()
        x = _philox_block(seed, s, gid, 4)[0]
        assert np.array_equal(d, ((x * np.uint64(dec)) >> np.uint64(32)).astype(np.int64)), s   # __umulhi(x, dec)
        dist = torch.zeros(n, 17, 3, device=dev)
        _rows(c, b, L.ptr(dist), 51, 3, -30.0, 30.0, None, 5, n)
        root = torch.zeros(n, 13, device=dev)
        _rows(c, b, L.ptr(root) + 28, 13, 2, -1.0, 1.0, None, 6, n)
        w5, w6 = _philox_block(seed, s, gid, 5), _philox_block(seed, s, gid, 6)
        u5 = np.stack([_u01(w) for w in w5[:3]], 1)
        u6 = np.stack([_u01(w) for w in w6[:2]], 1)
        want5 = torch.from_numpy(np.float32(60.0) * u5).to(dev) + np.float32(-30.0)
        want6 = torch.from_numpy(np.float32(2.0) * u6).to(dev) + np.float32(-1.0)
        assert torch.equal(_bits(dist[:, 0, :]), _bits(want5)) and (dist[:, 1:, :] == 0).all(), s
        assert torch.equal(_bits(root[:, 7:9]), _bits(want6)) and (root[:, :7] == 0).all() and (root[:, 9:] == 0).all(), s
        draws[s] = dict(d=d, u5=u5, u6=u6, u0=_u01(_philox_block(seed, s, gid, 0)[0]))
    # uniformity: chi-square of the delays over {0..dec-1}, KS of every column
    for s, dr in draws.items():
        cnt = np.bincount(dr["d"], minlength=dec)
        assert len(cnt) == dec and stats.chisquare(cnt).pvalue > 1e-4, (s, cnt)
        for name, u in (("disturbance", dr["u5"]), ("push", dr["u6"])):
            for k in range(u.shape[1]):
                assert stats.kstest(u[:, k], "uniform").pvalue > 1e-4, (s, name, k)
                assert u[:, k].min() >= 0.0 and u[:, k].max() < 1.0
    # independence across steps, columns and streams 4/5/6 against stream 0
    a, b2 = draws[5], draws[6]
    cols = [a["d"] / dec, a["u5"][:, 0], a["u5"][:, 1], a["u5"][:, 2], a["u6"][:, 0], a["u6"][:, 1], a["u0"],
            b2["d"] / dec, b2["u5"][:, 0], b2["u6"][:, 0], draws[(1 << 33) + 5]["u5"][:, 0]]
    m = np.corrcoef(np.stack(cols))
    assert np.abs(m - np.eye(len(cols))).max() < 0.03, m
    assert not np.array_equal(a["d"], b2["d"]) and not np.array_equal(a["u5"], draws[(1 << 33) + 5]["u5"])


def test_captured_launch_draws_the_eager_keys():
    """Keyed by the device counter in a captured graph (step_base) = keyed by value in an eager launch."""
    from isaacgymloco_b200 import _lib as L
    n, dec, seed = 4099, 4, 99
    dev = "cuda:0"
    c = _cfg(n)
    base = torch.zeros(1, dtype=torch.long, device=dev)
    last = torch.randn(n, 12, device=dev)
    a = torch.randn(n, 12, device=dev)
    out_g, del_g = torch.empty_like(a), torch.empty(n, dec, 12, device=dev)
    dist_g, root_g = torch.zeros(n, 17, 3, device=dev), torch.zeros(n, 13, device=dev)
    bg = _bufs(last, seed=seed, offset=3, step_base=base)          # step = *step_base + 3
    _delay(c, bg, a, out_g, del_g, dec, 1, 100.0, None, n)          # eager first: the kernels are loaded before capture
    _rows(c, bg, L.ptr(dist_g), 51, 3, -30.0, 30.0, None, 5, n)
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.graph(gr, stream=s):
        _delay(c, bg, a, out_g, del_g, dec, 1, 100.0, None, n)
        _rows(c, bg, L.ptr(dist_g), 51, 3, -30.0, 30.0, None, 5, n)
        _rows(c, bg, L.ptr(root_g) + 28, 13, 2, -1.0, 1.0, None, 6, n)
    torch.cuda.current_stream().wait_stream(s)
    prev = None
    for counter in (0, 40, 41):
        base.fill_(counter)
        gr.replay()
        be = _bufs(last, seed=seed, offset=counter + 3)
        out_e, del_e = torch.empty_like(a), torch.empty(n, dec, 12, device=dev)
        dist_e, root_e = torch.zeros(n, 17, 3, device=dev), torch.zeros(n, 13, device=dev)
        _delay(c, be, a, out_e, del_e, dec, 1, 100.0, None, n)
        _rows(c, be, L.ptr(dist_e), 51, 3, -30.0, 30.0, None, 5, n)
        _rows(c, be, L.ptr(root_e) + 28, 13, 2, -1.0, 1.0, None, 6, n)
        for x, y in ((out_g, out_e), (del_g, del_e), (dist_g, dist_e), (root_g, root_e)):
            assert torch.equal(x, y), counter
        if prev is not None:
            assert not torch.equal(prev[0], del_g) and not torch.equal(prev[1], dist_g) and not torch.equal(prev[2], root_g)
        prev = (del_g.clone(), dist_g.clone(), root_g.clone())


# ---------------------------------------------------------------------------------------------------- 3. sharding
def _phys(e, k):
    e.dof_state.view(e.num_envs, 12, 2)[..., 0].add_(0.001 * e.torques)
    e.dof_state.view(e.num_envs, 12, 2)[..., 1].add_(0.01 * e.torques)


def _policy(obs):
    return 120.0 * torch.tanh(obs[:, :12] + obs[:, 45:57])     # beyond the clip for some envs


def _keyed_env(cfg, state, hf, seed=5, push_interval=5):
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    cfg.reset.keyed_domain_rand = True
    env = FusedLeggedRobot(cfg, state, hf, device="cuda:0", physics_step_fn=_phys, seed=seed)
    env.custom_origins = True
    env.push_interval = push_interval
    return env


def test_two_shards_equal_one_big_env_for_the_whole_step():
    """Shards [0, split) and [split, n) with env_id_offset 0 / split, stepped through the public step() for 20 steps
    (the delay every step, disturbances at counters 8 and 16, pushes every 5): delayed_actions, torques, the drawn
    disturbance, root_states, the snapshot and the reset ids equal the one big env's row for row."""
    from isaacgymloco_b200 import config as C, synthetic as S
    n, split = 8192, 3000
    cfg = C.aliengo("flat", num_envs=n)
    assert cfg.reset.delay and cfg.reset.disturbance and cfg.reset.push_robots
    hf = S.make_terrain(cfg, seed=3)
    state = S.make_state(cfg, n, hf, seed=41)
    envs = [_keyed_env(cfg, state, hf)]
    for lo, hi in ((0, split), (split, n)):
        st = {}
        for k, v in state.items():
            if k == "episode_sums":
                st[k] = v[:, lo:hi].contiguous()
            elif isinstance(v, torch.Tensor) and v.dim() > 0 and v.shape[0] in (n, n * 12, n * cfg.num_bodies):
                per = v.shape[0] // n
                st[k] = v[lo * per:hi * per].contiguous()
            else:
                st[k] = v
        envs.append(_keyed_env(C.aliengo("flat", num_envs=n, env_id_offset=lo), st, hf))
    drawn = []
    for e in envs:
        rec = torch.zeros(e.num_envs, 3, device=e.device)
        drawn.append(rec)
        e._disturbance_robots = (lambda e=e, rec=rec: (type(e)._disturbance_robots(e), rec.copy_(e.disturbance[:, 0, :])))
    cat = lambda xs: torch.cat(xs, dim=0)
    total = 0
    for step in range(20):
        outs = [e.step(_policy(e.obs_buf)) for e in envs]
        big, s0, s1 = envs
        for name in ("delayed_actions", "torques", "actions", "root_states", "dof_state", "disturbance"):
            assert torch.equal(_bits(getattr(big, name)), _bits(cat([getattr(s0, name), getattr(s1, name)]))), (step, name)
        sb, ss = big.snapshot(), [s0.snapshot(), s1.snapshot()]
        for key in sb:
            got = torch.cat([x[key] for x in ss], dim=1 if key == "episode_sums" else 0)
            assert torch.equal(sb[key], got), (step, key)
        ids = [o[5] for o in outs]
        assert torch.equal(ids[0], torch.cat([ids[1], ids[2] + split])), step
        total += ids[0].numel()
    assert torch.equal(drawn[0], cat(drawn[1:])) and drawn[0].abs().max() > 20.0
    assert total > 0 and envs[0].common_step_counter == 20


# ---------------------------------------------------------------------------------------------------- 4. replay == eager
def _rollout_env(task, n, seed=11):
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    from oracle.make_goldens import reset_inputs
    cfg, hf, state, _, ter, _ = reset_inputs(dict(task=task, n=n, seed=seed))
    cfg.reset.keyed_domain_rand = True
    assert cfg.reset.delay and cfg.reset.disturbance and cfg.reset.push_robots and cfg.reset.commands_curriculum
    state["episode_length_buf"][: n // 16] = 490
    env = FusedLeggedRobot(cfg, state, hf, device="cuda:0", physics_step_fn=_phys, seed=seed)
    env.custom_origins = True
    env.env_origins = ter["env_origins"].to(env.device).contiguous()
    env.terrain_origins = ter["origins"].to(env.device).contiguous()
    env.terrain_types = ter["types"].to(env.device).contiguous()
    env.max_terrain_level = cfg.num_rows
    env.refresh_buffers()
    return env


@pytest.mark.parametrize("task,n", [("flat", 4096), ("stairs", 16385)])
def test_replay_equals_eager_with_the_real_hooks(task, n):
    """capture_schedule=True, T = 20, the delay every step, a disturbance every 8, a push every 30 and the command
    curriculum every 50 (host interval): after the warm-up every window replays and equals the eager public step()."""
    from test_gpu_rollout_schedule import _Runner, _compare
    from isaacgymloco_b200.rollout_graph import env_schedule, rollout_window
    tt = 20
    a, b = _Runner(_rollout_env(task, n), eager=True, t_len=tt), _Runner(_rollout_env(task, n), eager=False, t_len=tt)
    for e in (a.env, b.env):
        e.push_interval = 30
        e.max_episode_length = 50
    rg = b.env.capture_rollout(b.body, tt, storage=b.st, finish=b.finish, capture_schedule=True)
    boost = {2: 1e3, 4: -1e3}                  # curriculum steps at counters 50 and 100
    keys = set()
    for r in range(7):
        for run in (a, b):
            run.keep.fill_(0.0 if r in boost else 1.0)
            run.boost.fill_(boost.get(r, 0.0))
        keys.add(rollout_window(b.env.common_step_counter, tt, **env_schedule(b.env), in_graph=True)[0])
        ra = a.rollout_eager()
        rb = rg.run()
        _compare(a, b, ra, rb, f"rollout {r}")
        assert torch.equal(_bits(a.env.delayed_actions), _bits(b.env.delayed_actions)), r
        assert rg.last_mode == "eager" if r == 0 else rg.last_mode in ("replay", "capture+replay"), (r, rg.last_mode)
        a.st.clear()
        b.st.clear()
    assert rg.stats["eager"] == 1 and rg.stats["replays"] == 6
    assert any(k[0] for k in keys) and any(k[1] for k in keys) and any(k[2] for k in keys)


def test_two_replays_draw_different_delays_disturbances_and_pushes():
    """One captured graph replayed twice from the same state, at counters 0 and 8: the delays, the disturbance and the
    pushes differ (the keys come from the device counter)."""
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    n, tt = 4096, 8
    env = _rollout_env("flat", n)
    env.push_interval = 4               # windows 1-8 and 9-16: pushes at steps 3 and 7, a disturbance at step 7 in both
    rec = dict(delayed=torch.zeros(tt, n, 4, 12, device=env.device), vel=torch.zeros(tt, n, 2, device=env.device),
               dist=torch.zeros(n, 3, device=env.device))
    env._disturbance_robots = lambda: (FusedLeggedRobot._disturbance_robots(env), rec["dist"].copy_(env.disturbance[:, 0, :]))

    def body(k):
        env.step_device(_policy(env.obs_buf))
        rec["delayed"][k].copy_(env.delayed_actions)
        rec["vel"][k].copy_(env.root_states[:, 7:9])

    state = {k: v.clone() for k, v in vars(env).items() if isinstance(v, torch.Tensor) and not k.endswith("_ws")
             and k != "_step_base"}
    rg = env.capture_rollout(body, tt, warmup=0, capture_schedule=True)
    outs = []
    for r in range(2):
        for k, v in state.items():
            getattr(env, k).copy_(v)
        rg.run()
        outs.append({k: v.clone() for k, v in rec.items()})
    assert rg.stats == {"replays": 2, "captures": 1, "eager": 0}
    o1, o2 = outs
    assert not torch.equal(o1["delayed"][0], o2["delayed"][0])          # delays of step 0 (stream 4)
    assert not torch.equal(o1["dist"], o2["dist"]) and o1["dist"].abs().max() > 20.0     # counters 8 / 16 (stream 5)
    assert not torch.equal(o1["vel"][3], o2["vel"][3])                  # the pushes at counters 4 / 12 (stream 6)
    mv = env.cfg_hot.reset.max_push_vel_xy
    assert o1["vel"][3].abs().max() <= mv


# ---------------------------------------------------------------------------------------------------- 5. hooks and gym calls
def test_step_drives_the_gym_like_the_reference_with_the_flag_on():
    """The recording FakeGym of test_step_drives_the_gym_like_the_reference: the same calls in the same order with
    keyed domain randomisation, the draws on the same steps, and two envs with one seed agree without any torch seed."""
    from test_gpu_reset import FakeGym
    from isaacgymloco_b200 import config as C, synthetic as S
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    n = 2048
    cfg = C.aliengo("amp", num_envs=n)
    cfg.reset.keyed_domain_rand = True
    hf = S.make_terrain(cfg, seed=1)
    state = S.make_state(cfg, n, hf, seed=9)
    env = FusedLeggedRobot(cfg, state, hf, device="cuda:0")
    env.custom_origins = True
    env.push_interval = 3
    env.gym, env.sim = FakeGym(weakref.ref(env)), object()
    pushes, dists = [], []
    orig_push, orig_dist = env._push_robots, env._disturbance_robots
    env._push_robots = lambda: (pushes.append(env.common_step_counter), orig_push())
    env._disturbance_robots = lambda: (dists.append(env.common_step_counter), orig_dist())
    ref = FusedLeggedRobot(cfg, state, hf, device="cuda:0")
    ref.custom_origins = True
    ref.push_interval = 3
    ref.physics_step_fn = _phys
    torch.manual_seed(0)
    acts = [0.3 * torch.randn(n, 12, device="cuda") for _ in range(8)]
    for i, a in enumerate(acts):
        env.gym.calls.clear()
        out = env.step(a)
        torch.manual_seed(1000 + i)                  # the keyed draws do not follow torch's generator
        out_ref = ref.step(a)
        assert len(out) == 8 and torch.equal(out[7], out_ref[7])
        calls = env.gym.calls
        sub = ["set_dof_actuation_force_tensor", "simulate", "fetch_results", "refresh_dof_state_tensor"]
        assert calls[:16] == sub * 4, calls[:16]
        assert calls[16:20] == ["refresh_actor_root_state_tensor", "refresh_net_contact_force_tensor", "refresh_force_sensor_tensor",
                                "refresh_rigid_body_state_tensor"]
        rest = calls[20:]
        if env.common_step_counter % 8 == 0:
            assert "apply_rigid_body_force_tensors" in rest
        if env.common_step_counter % 3 == 0:
            assert "set_actor_root_state_tensor" in rest
        if len(out[5]):
            assert rest[-2:] == ["set_dof_state_tensor_indexed", "set_actor_root_state_tensor_indexed"]
        for x, y in zip(out[:4], out_ref[:4]):
            assert torch.equal(x, y)
        assert torch.equal(out[5], out_ref[5]) and torch.equal(out[6], out_ref[6])
        assert torch.equal(env.delayed_actions, ref.delayed_actions) and torch.equal(env.root_states, ref.root_states)
    assert pushes == [3, 6] and dists == [8] and env.common_step_counter == 8


@pytest.mark.parametrize("how", ["instance", "subclass"])
def test_overridden_hooks_replace_the_kernel(how):
    """With the flag on, an override of _delay_actions (instance attribute or subclass method) runs after torch.clamp
    instead of hl_delay_actions, and overrides of _disturbance_robots / _push_robots run instead of hl_uniform_rows."""
    from isaacgymloco_b200 import config as C, synthetic as S
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    n = 1024
    cfg = C.aliengo("flat", num_envs=n)
    cfg.reset.keyed_domain_rand = True
    hf = S.make_terrain(cfg, seed=1)
    state = S.make_state(cfg, n, hf, seed=9)
    calls = []

    def delay(self):
        calls.append("delay")
        self.delayed_actions.copy_(self.actions.unsqueeze(1) + 0.5)

    def dist(self):
        calls.append(("dist", self.common_step_counter))
        self.disturbance[:, 0, :] = 1.25

    def push(self):
        calls.append(("push", self.common_step_counter))
        self.root_states[:, 7:9] = 0.125

    if how == "subclass":
        Env = type("Env", (FusedLeggedRobot,), dict(_delay_actions=delay, _disturbance_robots=dist, _push_robots=push))
        env = Env(cfg, state, hf, device="cuda:0", physics_step_fn=_phys)
    else:
        env = FusedLeggedRobot(cfg, state, hf, device="cuda:0", physics_step_fn=_phys)
        env._delay_actions = delay.__get__(env)
        env._disturbance_robots = dist.__get__(env)
        env._push_robots = push.__get__(env)
    env.custom_origins = True
    env.push_interval = 4
    for i in range(8):
        a = 150.0 * torch.randn(n, 12, device="cuda")
        out = env.step(a)
        want = torch.clamp(a, -100.0, 100.0)
        assert torch.equal(env.actions, want), i
        assert torch.equal(env.delayed_actions, (want.unsqueeze(1) + 0.5).expand_as(env.delayed_actions)), i
        if env.common_step_counter % 4 == 0:
            kept = torch.ones(n, dtype=torch.bool, device="cuda")
            kept[out[5]] = False
            assert (env.root_states[kept, 7:9] == 0.125).all(), i
    assert calls.count("delay") == 8 and [c for c in calls if c != "delay"] == [("push", 4), ("dist", 8), ("push", 8)]


def test_parity_draws_drive_the_step():
    """set_domain_rand_draws: the pre-drawn delays / uniforms are what the step uses, on every step while set."""
    from isaacgymloco_b200 import config as C, synthetic as S
    n = 1024
    cfg = C.aliengo("flat", num_envs=n)
    hf = S.make_terrain(cfg, seed=1)
    state = S.make_state(cfg, n, hf, seed=9)
    env = _keyed_env(cfg, state, hf, push_interval=2)
    g = torch.Generator().manual_seed(3)
    d = torch.randint(0, 4, (n,), generator=g)
    u_push = torch.rand(n, 2, generator=g, dtype=torch.float64)
    env.set_domain_rand_draws(delay=d, push=u_push)
    mv = cfg.reset.max_push_vel_xy
    for i in range(4):
        last = env.last_actions.clone()
        a = torch.randn(n, 12, device="cuda")
        out = env.step(a)
        _, want = _torch_delay(a, last, d.cuda(), 4, True, cfg.clip_actions)
        assert torch.equal(_bits(env.delayed_actions), _bits(want)), i
        if env.common_step_counter % 2 == 0:
            kept = torch.ones(n, dtype=torch.bool, device="cuda")
            kept[out[5]] = False
            want_v = (2 * mv) * u_push.float().cuda() - mv
            assert torch.equal(env.root_states[kept, 7:9], want_v[kept]), i
