"""-m gpu: the non-finite guard (hl_finite_scan, FiniteGuard) against torch, and inside replayed rollouts.

* One launch against torch's predicates (~isfinite, and ~(x > 0 & isfinite) for a scale), for every N in {1, 7, 255,
  256, 257, 4,099, 65,539} and width in {1, 3, 12, 13, 24, 51, 238}: contiguous fields at every 16-B alignment, strided
  views (a 45-column view of a 270-wide buffer, a misaligned column window) and a 16-field launch; NaN with two
  payloads and both signs, +-inf, and for the scale kind +0, -0, -1e-38, -1, placed at (0, 0), (N-1, w-1) and either
  side of a CTA boundary, plus random masks of density 1e-6 .. 0.5.  The count, the first index and the bits of the
  first element (through .view(torch.int32)) are equal; clean inputs (+-FLT_MAX, subnormals, +-0 for the finite
  kind) give zero.
* The ticket protocol: launches that alternate dirty and clean inputs give independent rows; one launch captured and
  replayed 100 times leaves the workspace re-armed.
* Inside a rollout: a NaN written into root_states[e, 7] at one step (a device op keyed to the device step counter)
  makes check() and run() raise with that step, root_states, the global env id and column 7; run() leaves the counter
  and storage.step as a clean window does, the next window returns its infos, and the replayed events equal the eager
  loop's bit for bit, also for a shard with env_id_offset > 0.  keyed_act with a NaN mean and a zero std column flags
  mu, actions and sigma while the torques and obs_buf of that step stay finite (the clamps hide it).  Clean rollouts
  of the flat, stairs and AMP presets at 4,096, 16,385 and 65,536 envs report nothing over push and curriculum
  windows with capture_schedule=True.
"""
import math
import struct

import pytest
import torch

from test_gpu_rollout_graph import GAMMA, T, _make_env, _physics, _policy, _Runner

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
NS = (1, 7, 255, 256, 257, 4099, 65539)
WIDTHS = (1, 3, 12, 13, 24, 51, 238)
CHUNK = 8192                     # elements per CTA (FS_CHUNK)


def _f(bits):
    return torch.tensor([bits], dtype=torch.int64).to(torch.int32).view(torch.float32).item()


NAN_BITS = (0x7FC00000, 0x7F800001, 0xFFC00001 - (1 << 32), 0xFF812345 - (1 << 32))   # payloads, both signs
INF_BITS = (0x7F800000, 0xFF800000 - (1 << 32))
BAD_FINITE = NAN_BITS + INF_BITS
BAD_POSITIVE = BAD_FINITE + (0x00000000, -(1 << 31), 0x80000000 + 0x006CE3EE - (1 << 32), 0xBF800000 - (1 << 32))
# ... +0, -0, -1e-38 (a negative subnormal), -1


def _bad(x, kind):
    from isaacgymloco_b200 import _lib as L
    return ~torch.isfinite(x) if kind == L.FINITE else ~((x > 0) & torch.isfinite(x))


def _expect(x, kind):
    flat = x.reshape(-1)
    mask = _bad(flat, kind)
    n = int(mask.sum())
    if n == 0:
        return [0, -1, 0]
    i = int(mask.nonzero()[0, 0])
    return [n, i, int(flat[i:i + 1].view(torch.int32).item())]


def _scan(views):
    from isaacgymloco_b200.finite_guard import finite_scan, new_workspace
    rec = torch.full((len(views), 3), -7, dtype=torch.int64, device=DEV)
    finite_scan(views, rec, new_workspace(DEV))
    return rec.tolist()


def _check(views, what):
    got = _scan(views)
    for f, (x, kind) in enumerate(views):
        assert got[f] == _expect(x, kind), (what, f, got[f], _expect(x, kind))
    return got


def _layouts(n, w, g):
    """(name, view, base) for one size: contiguous at 4 alignments, a strided column window, for n x w."""
    out = []
    base = torch.randn(n * w + 4, generator=g).abs().add_(0.5).to(DEV)
    for off in range(4):
        out.append((f"contiguous+{off}", base[off:off + n * w].view(n, w)))
    wide = torch.randn(n, 2 * w + 3, generator=g).abs().add_(0.5).to(DEV)
    out.append(("strided", wide[:, 1:1 + w]))
    return out


def _positions(n, w):
    total = n * w
    pos = {0, total - 1}
    for b in (CHUNK, 2 * CHUNK, 3 * CHUNK):
        for d in (-4, -1, 0, 1, 4):
            if 0 <= b + d < total:
                pos.add(b + d)
    return sorted(pos)


def _put(x, p, bits):
    e, c = divmod(p, x.shape[1])
    x.view(torch.int32)[e, c] = bits                  # raw bits: signalling payloads reach the device unchanged


@pytest.mark.parametrize("n", NS)
def test_launch_equals_torch(n):
    from isaacgymloco_b200 import _lib as L
    g = torch.Generator().manual_seed(n)
    for w in WIDTHS:
        pos = _positions(n, w)
        for name, x in _layouts(n, w, g):
            clean = x.clone()
            what = f"n={n} w={w} {name}"
            assert _check([(x, L.FINITE), (x, L.FINITE_POSITIVE)], what + " clean") == [[0, -1, 0]] * 2
            for kind, values in ((L.FINITE, BAD_FINITE), (L.FINITE_POSITIVE, BAD_POSITIVE)):
                for j, bits in enumerate(values):        # one value at a time, each at the next position
                    x.copy_(clean)
                    _put(x, pos[j % len(pos)], bits)
                    got = _check([(x, kind), (x, L.FINITE), (x, L.FINITE_POSITIVE)], f"{what} bits {bits:#x}")
                    assert got[0][:2] == [1, pos[j % len(pos)]]
                x.copy_(clean)
                for i, p in enumerate(pos):              # every position at once
                    _put(x, p, values[i % len(values)])
                assert _check([(x, kind)], f"{what} all positions")[0][:2] == [len(pos), 0]
                x.copy_(clean)


def test_random_masks_and_the_16_field_launch():
    from isaacgymloco_b200 import _lib as L
    g = torch.Generator().manual_seed(3)
    n = 65539
    for w in (13, 238):
        for density in (1e-6, 1e-4, 1e-2, 0.5):
            x = torch.randn(n, w, generator=g)
            u = torch.rand(n, w, generator=g)
            pick = torch.randint(0, 4, (n, w), generator=g)
            vals = torch.tensor([_f(b) for b in (0x7FC00000, 0x7F800000, 0xFF800000 - (1 << 32), 0)])
            x = torch.where(u < density, vals[pick], x).to(DEV)
            _check([(x, L.FINITE), (x, L.FINITE_POSITIVE)], f"w={w} density {density}")
    buf = torch.randn(n, 270, generator=g).to(DEV)                    # a 45-column view of a 270-wide buffer
    view = buf[:, :45]
    view[n // 3, 44] = float("nan")
    view[n // 2, 0] = float("-inf")
    buf[n // 4, 45] = float("nan")                                     # outside the view: not flagged
    got = _check([(view, L.FINITE)], "45 of 270")
    assert got[0][:2] == [2, (n // 3) * 45 + 44]
    storage = torch.rand(24, 4099, 12, generator=g).add_(0.1).to(DEV)  # storage slot views (contiguous slots)
    storage[5, 17, 3] = 0.0
    storage[6, 0, 0] = float("nan")
    got = _check([(storage[5], L.FINITE_POSITIVE), (storage[6], L.FINITE), (storage[7], L.FINITE)], "slots")
    assert [r[:2] for r in got] == [[1, 17 * 12 + 3], [1, 0], [0, -1]]
    views = []
    for f in range(16):                                               # 16 fields, all widths and kinds, 4,099 rows
        w = WIDTHS[f % len(WIDTHS)]
        x = torch.randn(4099, w + (f % 3), generator=g).abs().add_(0.25).to(DEV)[:, :w]
        if f % 4 != 3:
            m = torch.rand(4099, w, generator=g) < 10 ** -(1 + f % 4)
            x[m.to(DEV)] = _f(BAD_POSITIVE[f % len(BAD_POSITIVE)])
        views.append((x, L.FINITE_POSITIVE if f % 2 else L.FINITE))
    got = _check(views, "16 fields")
    assert sum(r[0] > 0 for r in got) >= 8
    with pytest.raises(ValueError, match="between 1 and 16"):
        _scan(views + views[:1])


def test_clean_inputs_give_zero():
    from isaacgymloco_b200 import _lib as L
    fmax, sub = 3.4028234663852886e38, 1e-40
    for n in (1, 257, 65539):
        x = torch.tensor([fmax, -fmax, sub, -sub, 0.0, -0.0, 1.0, -1.0], device=DEV).repeat(n, 1)
        pos = torch.tensor([fmax, sub, 1.4e-45, 1.0], device=DEV).repeat(n, 3)
        assert _scan([(x, L.FINITE), (pos, L.FINITE_POSITIVE)]) == [[0, -1, 0]] * 2
        assert _scan([(x, L.FINITE_POSITIVE)])[0][0] == 5 * n                # -FLT_MAX, -sub, +0, -0, -1


def test_ticket_protocol_and_replayed_launches():
    from isaacgymloco_b200 import _lib as L
    from isaacgymloco_b200.finite_guard import finite_scan, new_workspace
    n, w = 65539, 13
    clean = torch.randn(n, w, device=DEV)
    dirty = clean.clone()
    dirty[100, 3], dirty[n - 1, w - 1] = float("nan"), float("inf")
    ws = new_workspace(DEV)
    armed = ws.tolist()
    rec = torch.full((12, 1, 3), -7, dtype=torch.int64, device=DEV)
    for i in range(12):
        finite_scan([(dirty if i % 2 == 0 else clean, L.FINITE)], rec[i], ws)
    want_dirty = _expect(dirty, L.FINITE)
    for i, row in enumerate(rec.tolist()):
        assert row[0] == (want_dirty if i % 2 == 0 else [0, -1, 0]), i
    assert ws.tolist() == armed
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    gr = torch.cuda.CUDAGraph()
    one = torch.full((1, 3), -7, dtype=torch.int64, device=DEV)
    with torch.cuda.graph(gr, stream=s):
        finite_scan([(dirty, L.FINITE)], one, ws)
    torch.cuda.current_stream().wait_stream(s)
    assert one.tolist() == [[-7, -7, -7]]                          # the capture executed nothing
    for _ in range(100):
        gr.replay()
    assert one.tolist() == [want_dirty] and ws.tolist() == armed
    dirty[100, 3] = 1.0                                             # the replay reads the source's current values
    gr.replay()
    assert one.tolist()[0][:2] == [1, n * w - 1] and ws.tolist() == armed
    del gr


# ------------------------------------------------------------------------------------------------- inside a rollout
def _shard_env(task, n, offset):
    """_make_env with cfg.env_id_offset = offset (a shard of a larger env)."""
    from isaacgymloco_b200.legged_robot import FusedLeggedRobot
    from oracle.make_goldens import reset_inputs
    if offset == 0:
        return _make_env(task, n)
    cfg, hf, state, _, ter, _ = reset_inputs(dict(task=task, n=n, seed=11))
    cfg.reset.delay = False
    cfg.reset.disturbance = True
    cfg.reset.push_robots = False
    cfg.reset.commands_curriculum = False
    cfg.env_id_offset = offset
    state["episode_length_buf"][: n // 16] = 490
    env = FusedLeggedRobot(cfg, state, hf, device="cuda:0", physics_step_fn=_physics, seed=11)
    env.custom_origins = True
    env.env_origins = ter["env_origins"].to(env.device).contiguous()
    env.terrain_origins = ter["origins"].to(env.device).contiguous()
    env.terrain_types = ter["types"].to(env.device).contiguous()
    env.max_terrain_level = cfg.num_rows
    env.refresh_buffers()
    env._disturbance_robots = lambda: env.disturbance[:, 0, :].copy_(50.0 * env.base_lin_vel)
    env._push_robots = lambda: env.root_states[:, 7:9].copy_(0.5 * env.commands[:, :2])
    return env


class _GuardRunner(_Runner):
    """_Runner plus a FiniteGuard recorded after every step.  inject=(s, e): physics writes NaN into root_states[e, 7]
    at the step whose key (the device step counter + k) is s and restores 0 at s + 1 -- a device op, so eager,
    captured and replayed steps inject alike."""

    def __init__(self, env, eager, inject=None):
        from isaacgymloco_b200.finite_guard import FiniteGuard
        super().__init__(env, eager)
        self.guard = FiniteGuard(env, T, storage=self.st)
        self.inject, self.k = inject, 0
        env.physics_step_fn = self._physics

    def _physics(self, env, sub):
        _physics(env, sub)
        if self.inject is not None and sub == 0:
            s, e = self.inject
            key = env._step_base + self.k
            col = env.root_states[e:e + 1, 7]
            col.copy_(torch.where(key == s, float("nan"), torch.where(key == s + 1, 0.0, col)))

    def body(self, k):
        self.k = k
        super().body(k)
        self.guard.record(k)

    def rollout_checked(self):
        """The eager loop: T public steps, then check() once (the device counter keys the injection as run() does)."""
        self.env._step_base.fill_(self.env.common_step_counter)
        self.rollout_eager()
        self.guard.check()


def _same_events(a, b):
    assert len(a) == len(b) > 0
    for x, y in zip(a, b):
        assert {k: x[k] for k in x if k != "value"} == {k: y[k] for k in y if k != "value"}, (x, y)
        assert struct.pack("<d", x["value"]) == struct.pack("<d", y["value"]), (x, y)


@pytest.mark.parametrize("offset", [0, 3 * 4096])
def test_injected_nan_raises_in_check_and_run(offset):
    from isaacgymloco_b200.finite_guard import NonFiniteError
    n, e, k_bad = 4096, 4000, 5
    s = 2 * T + k_bad                                   # in the third rollout: a replayed window
    a = _GuardRunner(_shard_env("flat", n, offset), eager=True, inject=(s, e))
    b = _GuardRunner(_shard_env("flat", n, offset), eager=False, inject=(s, e))
    rg = b.env.capture_rollout(b.body, T, storage=b.st, finish=b.finish, finite_guard=b.guard)
    for r in range(4):
        c = b.env.common_step_counter
        if r == 2:
            with pytest.raises(NonFiniteError) as ea:
                a.rollout_checked()
            with pytest.raises(NonFiniteError) as eb:
                rg.run()
            assert rg.last_mode == "replay"
            assert b.env.common_step_counter == c + T and b.st.step == T
            assert b.env.extras["time_outs"] is b.env.time_out_buf
            _same_events(ea.value.events, eb.value.events)
            first = [ev for ev in eb.value.events if ev["k"] == k_bad]
            assert min(ev["k"] for ev in eb.value.events) == k_bad
            root = [ev for ev in first if ev["field"] == "root_states"]
            assert len(root) == 1, first
            ev = root[0]
            assert (ev["env"], ev["column"], ev["count"], ev["common_step_counter"]) == (offset + e, 7, 1, s + 1), ev
            assert math.isnan(ev["value"])
            msg = str(eb.value)
            assert f"rollout step {k_bad} (common_step_counter {s + 1})" in msg and "root_states" in msg
        else:
            a.rollout_checked()
            infos = rg.run()
            assert isinstance(infos, list)
        assert a.env.common_step_counter == b.env.common_step_counter == (r + 1) * T
        assert torch.equal(a.env.root_states, b.env.root_states) or r == 2
        a.st.clear()
        b.st.clear()
    assert rg.stats["replays"] == 3 and not b.guard.table[..., 0].any()


def test_keyed_act_nan_is_flagged_where_the_clamps_hide_it():
    from isaacgymloco_b200.finite_guard import FiniteGuard
    from isaacgymloco_b200.policy_sampling import keyed_act
    n, e, k_bad, t_len = 4096, 77, 2, 4
    env = _make_env("flat", n)
    r = _Runner(env, eager=False, t_len=t_len)
    guard = FiniteGuard(env, t_len, storage=r.st)
    std = torch.ones(12, device=env.device)
    std[3] = 0.0
    finite = torch.zeros(t_len, 2, dtype=torch.bool, device=env.device)
    for k in range(t_len):
        mean = _policy(env.obs_buf)
        if k == k_bad:
            mean[e] = float("nan")
        tr = r.tr
        act = keyed_act(env, mean, std, transition=tr, storage=r.st)
        tr.observations, tr.critic_observations, tr.values = env.obs_buf, env.privileged_obs_buf, r.values
        obs, priv, rew, done, extras, ids, n_dev, term, _ = env.step_device(act)
        r.st.record_env_step(tr, rew, done, extras, priv, ids, term, GAMMA, termination_count=n_dev)
        guard.record(k)
        finite[k, 0] = torch.isfinite(env.torques).all()
        finite[k, 1] = torch.isfinite(env.obs_buf).all()
    assert finite.all(), finite.tolist()                  # the NaN never reaches the torques or the observations
    with pytest.raises(FloatingPointError) as ei:
        guard.check()
    events = ei.value.events
    at = {ev["field"]: ev for ev in events if ev["k"] == k_bad}
    for name in ("mu", "actions"):
        assert at[name]["env"] == e and at[name]["count"] == 12 and math.isnan(at[name]["value"]), at[name]
    # sigma = mean*0. + std: column 3 of every env, and env e's other 11 columns (NaN), as the reference's scale
    assert at["sigma"]["count"] == n + 11 and (at["sigma"]["env"], at["sigma"]["column"], at["sigma"]["value"]) == (0, 3, 0.0)
    assert not any(ev["field"] in ("mu", "actions") for ev in events if ev["k"] != k_bad)
    assert not guard.table.any()                          # check() zeroed the table


@pytest.mark.parametrize("task", ["flat", "stairs", "amp"])
@pytest.mark.parametrize("n", [4096, 16385, 65536])
def test_clean_rollouts_report_nothing(task, n):
    env = _make_env(task, n, push=True, curriculum=True)
    env.push_interval = 30
    env.max_episode_length = 45
    r = _GuardRunner(env, eager=False)
    rg = env.capture_rollout(r.body, T, storage=r.st, finish=r.finish, capture_schedule=True, finite_guard=r.guard)
    for _ in range(5):
        rg.run()
        r.st.clear()
    assert rg.stats["replays"] == 4 and env.common_step_counter == 5 * T
