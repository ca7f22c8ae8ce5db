"""-m gpu: the AMP update's policy and expert minibatches drawn on the device (AMPUpdateSampler, hl_amp_update_batch).

* Draws: the rows are the Philox4x32-10 blocks of stream 8 -- recomputed on the host -- mapped to [0, n) by
  floor(u n / 2^64) of the 64-bit words (x, y) and (z, w), exactly, at every minibatch size, row count, preload size,
  row offset and seed listed; uniform (chi-square over 64 bins) and uncorrelated across the pair, calls and ranks.
* Gathers and normalisation: bit-equal to ReplayBuffer.gather, AMPLoader.gather_pairs and
  cat(normalize_torch(s), normalize_torch(s')) on the same rows, drawn or passed in, with and without a normaliser,
  var = 0 columns and values beyond +-clip.
* Key: k eager calls == one captured call replayed k times == a graph of three calls replayed; the counter counts calls.
* Device count: with ring_cursor = AMPRolloutStep._cursor the row count is the device's, before and after the ring wraps,
  and inside a graph that captures AMPRolloutStep.step() followed by sample().
* Drop-in: zipped with storage.mini_batch_generator in a HybridPPO-shaped discriminator loop, the discriminator inputs and
  the normaliser's statistics equal those of the public composition on the same rows at every minibatch.
"""
import copy

import numpy as np
import pytest
import torch

from conftest import load_golden
from test_gpu_keyed_domain_rand import _philox_block

pytestmark = pytest.mark.gpu

RING = 1_000_000


def _rows(words_hi, words_lo, n):
    """floor(((hi << 32) | lo) * n / 2^64) exactly, in uint64 limbs (n < 2^32): hi*n and lo*n stay below 2^53."""
    n = np.uint64(n)
    return ((words_hi * n + ((words_lo * n) >> np.uint64(32))) >> np.uint64(32)).astype(np.int64)


def _host_rows(seed, key, row_offset, mb, n_s, n_pre):
    x, y, z, w = _philox_block(seed, key, np.arange(mb, dtype=np.uint64) + np.uint64(row_offset), 8)
    return _rows(x, y, max(n_s, 1)), _rows(z, w, n_pre), (x, y, z, w)


def _ring(rows, dev, seed=1, scale=20.0):
    from isaacgymloco_b200.replay_buffer import ReplayBuffer
    rb = ReplayBuffer(30, rows, dev)
    g = torch.Generator(device=dev).manual_seed(seed)
    rb.states.copy_(scale * torch.randn(rows, 30, device=dev, generator=g))
    rb.next_states.copy_(scale * torch.randn(rows, 30, device=dev, generator=g))
    rb.num_samples, rb.step = rows, 0
    return rb


def _loader(n_pre, dev, seed=2, scale=20.0):
    """A real AMPLoader (golden clips) whose preload tables are then replaced by n_pre random rows."""
    from isaacgymloco_b200.motion_loader import AMPLoader
    gold = load_golden("amp.npz")
    k = len(gold["frame_durations"])
    tables = dict(frames=[gold[f"clip{i}"] for i in range(k)], frame_durations=gold["frame_durations"],
                  weights=gold["weights_raw"], names=[str(x) for x in gold["clip_names"]])
    ld = AMPLoader(dev, 0.02, preload_transitions=True, num_preload_transitions=16, clip_tables=tables)
    g = torch.Generator(device=dev).manual_seed(seed)
    ld.preloaded_s = scale * torch.randn(n_pre, 49, device=dev, generator=g)
    ld.preloaded_s_next = scale * torch.randn(n_pre, 49, device=dev, generator=g)
    return ld


def _normalizer(dev, kind):
    from isaacgymloco_b200.amp_discriminator import Normalizer
    if kind is None:
        return None
    norm = Normalizer(30, device=dev)
    g = torch.Generator().manual_seed(7)
    for _ in range(3):      # float64 statistics that fp32 cannot represent
        norm.update((torch.randn(999, 30, generator=g) * 1.7 + 0.3).to(dev))
    if kind == "var0":
        norm.var = norm.var.clone()
        norm.var[::3] = 0.0
        norm.mean = norm.mean.clone()
        norm.mean[1::4] = 0.1
    return norm


# ----------------------------------------------------------------------------- 1. draws
@pytest.mark.parametrize("mb", [1, 63, 64, 65, 4099, 102_400, 393_216])
def test_draws_equal_the_host_recomputation(mb):
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    dev = torch.device("cuda:0")
    rb = _ring(RING, dev, scale=1.0)
    for n_pre in (1, 2_000_000):
        ld = _loader(n_pre, dev, scale=1.0)
        for seed in (0, (1 << 40) + 7):
            for row_offset in (0, 3 * mb):
                sm = AMPUpdateSampler(ld, rb, None, mb, seed, row_offset=row_offset)
                for n_s in (1, 4096, 999_983, 1_000_000):
                    rb.num_samples = n_s
                    key = int(sm.draw_counter[0].item())
                    idx = sm.sample(return_indices=True).indices.cpu().numpy()
                    p, e, (x, y, z, w) = _host_rows(seed, key, row_offset, mb, n_s, n_pre)
                    what = f"mb={mb} n_pre={n_pre} seed={seed} offset={row_offset} n_s={n_s}"
                    assert np.array_equal(idx[:, 0], p), what
                    assert np.array_equal(idx[:, 1], e), what
                    assert idx[:, 0].min() >= 0 and idx[:, 0].max() < n_s and idx[:, 1].max() < n_pre, what
                    for r in range(0, mb, max(1, mb // 97)):      # the Python-integer form on a spread of rows
                        u = (int(x[r]) << 32) | int(y[r])
                        v = (int(z[r]) << 32) | int(w[r])
                        assert (idx[r, 0], idx[r, 1]) == ((u * n_s) >> 64, (v * n_pre) >> 64), (what, r)
                assert sm.draw_counter.tolist() == [4, 0]


# ----------------------------------------------------------------------------- 2. gathers + normalisation
def _composition(rb, ld, norm, idx):
    s, sn = rb.gather(idx[:, 0].cpu())
    es, esn = ld.gather_pairs(idx[:, 1])
    if norm is None:
        return s, sn, es, esn, torch.cat([s, sn], -1), torch.cat([es, esn], -1)
    return (s, sn, es, esn, torch.cat([norm.normalize_torch(s), norm.normalize_torch(sn)], -1),
            torch.cat([norm.normalize_torch(es), norm.normalize_torch(esn)], -1))


@pytest.mark.parametrize("mb", [65, 4099, 102_400])
@pytest.mark.parametrize("norm_kind", [None, "updated", "var0"])
def test_gathers_and_normalisation_bit_equal(mb, norm_kind):
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    dev = torch.device("cuda:0")
    rb, ld = _ring(150_001, dev), _loader(200_003, dev)
    rb.num_samples = 140_000
    norm = _normalizer(dev, norm_kind)
    sm = AMPUpdateSampler(ld, rb, norm, mb, 123)
    g = torch.Generator(device=dev).manual_seed(mb)
    given = torch.stack([torch.randint(0, 150_001, (mb,), device=dev, generator=g),
                         torch.randint(0, 200_003, (mb,), device=dev, generator=g)], 1)
    for mode in ("draw", "parity"):
        out = sm.sample(indices=given if mode == "parity" else None, return_indices=True)
        idx = out.indices
        if mode == "parity":
            assert torch.equal(idx, given)
        else:
            assert int(idx[:, 0].max()) < 140_000
        ref = _composition(rb, ld, norm, idx)
        for k, (a, b) in enumerate(zip(out[:6], ref)):
            assert a.shape == b.shape and a.is_contiguous(), (mode, k)
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"{mode}: output {out._fields[k]}"
        if norm is not None and mb >= 4099:
            for x in (out.x_policy, out.x_expert):
                assert (x == norm.clip_obs).any() and (x == -norm.clip_obs).any(), "no value beyond +-clip"
    assert sm.draw_counter.tolist() == [2, 0]


# ----------------------------------------------------------------------------- 3. statistics
def _chi2_ok(rows, n, bins=64):
    from scipy import stats
    edges = [(b * n + bins - 1) // bins for b in range(bins + 1)]     # bin b holds rows with floor(row * 64 / n) == b
    width = np.diff(np.array(edges, dtype=np.float64))
    obs = np.bincount((rows.astype(np.int64) * bins) // n, minlength=bins)
    exp = width / width.sum() * rows.size
    return stats.chisquare(obs, exp).pvalue


def test_draws_are_uniform_and_independent():
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    dev = torch.device("cuda:0")
    mb, n_pre = 393_216, 2_000_000
    rb, ld = _ring(RING, dev, scale=1.0), _loader(n_pre, dev, scale=1.0)
    lim = 5.0 / np.sqrt(mb)
    for n_s in (999_983, 1_000_000):
        rb.num_samples = n_s
        a = AMPUpdateSampler(ld, rb, None, mb, 99)
        b = AMPUpdateSampler(ld, rb, None, mb, 99, row_offset=mb)     # the next rank
        calls = [a.sample(return_indices=True).indices.cpu().numpy() for _ in range(4)]
        nxt = [b.sample(return_indices=True).indices.cpu().numpy() for _ in range(4)]
        pol = np.concatenate([c[:, 0] for c in calls])
        exp = np.concatenate([c[:, 1] for c in calls])
        assert _chi2_ok(pol, n_s) > 1e-4, n_s
        assert _chi2_ok(exp, n_pre) > 1e-4, n_s
        assert pol.min() >= 0 and pol.max() < n_s and exp.max() < n_pre
        u = [c[:, 0] / n_s for c in calls]
        v = [c[:, 1] / n_pre for c in calls]
        for k in range(4):
            assert abs(np.corrcoef(u[k], v[k])[0, 1]) < lim, ("pair", n_s, k)
            assert abs(np.corrcoef(u[k], nxt[k][:, 0] / n_s)[0, 1]) < lim, ("rank", n_s, k)
            assert abs(np.corrcoef(v[k], nxt[k][:, 1] / n_pre)[0, 1]) < lim, ("rank", n_s, k)
        for k in range(3):
            assert abs(np.corrcoef(u[k], u[k + 1])[0, 1]) < lim, ("calls", n_s, k)
            assert abs(np.corrcoef(v[k], v[k + 1])[0, 1]) < lim, ("calls", n_s, k)


# ----------------------------------------------------------------------------- 4. key and capture
def _capture(fn):
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.graph(g, stream=s):
        out = fn()
    torch.cuda.current_stream().wait_stream(s)
    return g, out


def test_eager_captured_and_replayed_calls_draw_alike():
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    dev = torch.device("cuda:0")
    rb, ld, norm = _ring(RING, dev), _loader(2_000_000, dev), _normalizer(dev, "updated")
    rb.num_samples = 777_777
    mb, k = 98_304, 6
    mk = lambda seed=5: AMPUpdateSampler(ld, rb, norm, mb, seed, row_offset=mb)
    eager, one, three = mk(), mk(), mk()
    want = []
    for c in range(k):
        want.append([t.clone() for t in eager.sample(return_indices=True)])
        assert eager.draw_counter.tolist() == [c + 1, 0]
    g1, out1 = _capture(lambda: one.sample(return_indices=True))
    assert one.draw_counter.tolist() == [0, 0]                 # a capture draws nothing
    got1 = []
    for c in range(k):
        g1.replay()
        got1.append([t.clone() for t in out1])
        assert one.draw_counter.tolist() == [c + 1, 0]
    g3, out3 = _capture(lambda: [three.sample(return_indices=True) for _ in range(3)])
    got3 = []
    for c in range(k // 3):
        g3.replay()
        got3 += [[t.clone() for t in o] for o in out3]
        assert three.draw_counter.tolist() == [3 * (c + 1), 0]
    for c in range(k):
        for j in range(7):
            assert torch.equal(want[c][j], got1[c][j]) and torch.equal(want[c][j], got3[c][j]), (c, j)
    assert not torch.equal(want[0][6], want[1][6])             # every call draws new rows
    other = mk(6).sample(return_indices=True).indices
    assert not torch.equal(other, want[0][6])                  # two seeds differ
    assert (other != want[0][6]).float().mean() > 0.99


# ----------------------------------------------------------------------------- 5. device count
def test_device_count_follows_the_rollout_step():
    from isaacgymloco_b200.amp_rollout import AMPRolloutStep, advance_cursor
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    from isaacgymloco_b200.replay_buffer import ReplayBuffer
    from test_gpu_amp_rollout import _amp_policy, _disc, _normalizer as _rollout_norm
    from test_gpu_rollout_graph import _make_env
    n = 4096
    env = _make_env("amp", n)
    dev = env.device
    disc, norm = _disc(dev), _rollout_norm(dev)
    size = 3 * n + 5                       # fills on the 4th step, wraps after it
    rb = ReplayBuffer(30, size, dev)
    step = AMPRolloutStep(env, disc, norm, rb)
    step.begin()
    ld = _loader(2_000_000, dev)
    mb = 1000
    on_dev = AMPUpdateSampler(ld, rb, norm, mb, 17, ring_cursor=step._cursor)
    by_val = AMPUpdateSampler(ld, rb, norm, mb, 17)
    seen_partial = seen_full = False
    for j in range(6):
        _, _, rew, _, _, ids, n_dev, _, term_amp = env.step_device(_amp_policy(env.obs_buf, step.amp_obs))
        step.step(rew, ids, n_dev, term_amp)
        a, b = on_dev.sample(return_indices=True), by_val.sample(return_indices=True)
        for k in range(7):
            assert torch.equal(a[k], b[k]), (j, k)
        assert int(a.indices[:, 0].max()) < rb.num_samples
        seen_partial |= rb.num_samples < size
        seen_full |= rb.num_samples == size and rb.step != 0
    assert seen_partial and seen_full
    # a graph of step() followed by sample(): the count it reads is the one the replayed step() left on the device
    _, _, rew, _, _, ids, n_dev, _, term_amp = env.step_device(_amp_policy(env.obs_buf, step.amp_obs))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.no_grad():
        disc.amp_linear(disc.trunk(step.x))          # cuBLAS warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    mirror = step.host_state()
    g, out = _capture(lambda: (step.step(rew, ids, n_dev, term_amp), on_dev.sample(return_indices=True))[1])
    step.set_host_state(mirror)                      # the capture ran nothing: the ring is where it was
    # start the graph from an empty-looking ring so its replays cover the partial count and the wrap
    step._cursor.copy_(torch.tensor([0, 0, 0], device=dev))
    rb.step, rb.num_samples = 0, 0
    step._cursor_mirror = (0, 0)
    for j in range(5):
        g.replay()
        step.advance(1)                              # what RolloutGraph.run() does for the host mirror
        got = [t.clone() for t in out]
        want = by_val.sample(return_indices=True)
        assert step._cursor.tolist() == [rb.step, rb.num_samples, 0], j
        for k in range(7):
            assert torch.equal(got[k], want[k]), ("graph", j, k)
        assert int(got[6][:, 0].max()) < rb.num_samples
        assert on_dev.draw_counter.tolist() == by_val.draw_counter.tolist() == [7 + j, 0]
    assert (rb.step, rb.num_samples) == advance_cursor(0, 0, size, n, 5)


# ----------------------------------------------------------------------------- 6. drop-in loop
def test_drop_in_discriminator_loop_equals_the_composition():
    from isaacgymloco_b200.amp_discriminator import AMPDiscriminator
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    from isaacgymloco_b200.rollout_storage import HIMRolloutStorage
    dev = torch.device("cuda:0")
    n, t = 64, 16
    mb = n * t // 4
    rb, ld = _ring(20_000, dev, scale=3.0), _loader(50_000, dev, scale=3.0)
    rb.num_samples = 18_000
    st = HIMRolloutStorage(n, t, [270], [238], [12], device=dev)
    torch.manual_seed(3)
    disc_a = AMPDiscriminator(60, 2.0, [256, 128], dev)
    disc_b = copy.deepcopy(disc_a)
    norm_a, norm_b = _normalizer(dev, "updated"), _normalizer(dev, "updated")
    opt_a, opt_b = torch.optim.Adam(disc_a.parameters(), lr=1e-3), torch.optim.Adam(disc_b.parameters(), lr=1e-3)
    sampler = AMPUpdateSampler(ld, rb, norm_a, mb, 42)
    twin = AMPUpdateSampler(ld, rb, norm_a, mb, 42)          # same seed: the same rows, with their indices
    mse = torch.nn.MSELoss()

    def update(disc, opt, norm, ps, es, esn, xp, xe):
        policy_d, expert_d = disc(xp), disc(xe)
        loss = (mse(expert_d, torch.ones_like(expert_d)) + mse(policy_d, -torch.ones_like(policy_d))) / 2
        loss = loss + disc.compute_grad_pen(es, esn, lambda_=10)
        opt.zero_grad()
        loss.backward()
        opt.step()
        norm.update(ps)
        norm.update(es)

    gen = st.mini_batch_generator(4, 2)
    count = 0
    for _batch, sample in zip(gen, sampler.generator(8)):
        idx = twin.sample(return_indices=True).indices
        ref = _composition(rb, ld, norm_b, idx)
        assert torch.equal(sample.x_policy, ref[4]) and torch.equal(sample.x_expert, ref[5]), count
        for k in range(4):
            assert torch.equal(sample[k], ref[k]), (count, k)
        update(disc_a, opt_a, norm_a, sample.policy_state, sample.expert_state, sample.expert_next_state,
               sample.x_policy, sample.x_expert)
        update(disc_b, opt_b, norm_b, ref[0], ref[2], ref[3], ref[4], ref[5])
        assert torch.equal(norm_a.mean, norm_b.mean) and torch.equal(norm_a.var, norm_b.var), count
        count += 1
    assert count == 8 and sampler.draw_counter.tolist() == [8, 0]


# ----------------------------------------------------------------------------- 7. argument checks
def test_argument_checks_on_the_device():
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    from isaacgymloco_b200.replay_buffer import ReplayBuffer
    dev = torch.device("cuda:0")
    rb, ld, norm = _ring(1000, dev), _loader(500, dev), _normalizer(dev, "updated")
    empty = ReplayBuffer(30, 1000, dev)
    with pytest.raises(ValueError, match="num_samples = 0"):
        AMPUpdateSampler(ld, empty, norm, 16, 0).sample()
    cpu_norm = _normalizer(dev, "updated")
    cpu_norm.mean, cpu_norm.var = cpu_norm.mean.cpu(), cpu_norm.var.cpu()
    with pytest.raises(ValueError, match="CUDA"):
        AMPUpdateSampler(ld, rb, cpu_norm, 16, 0)
    sm = AMPUpdateSampler(ld, rb, norm, 16, 0)
    norm2 = _normalizer(dev, "updated")
    norm2.mean = norm2.mean.float()
    with pytest.raises(ValueError, match="float64"):
        AMPUpdateSampler(ld, rb, norm2, 16, 0)
    for bad in (torch.zeros(16, 2, dtype=torch.long), torch.zeros(16, 2, dtype=torch.int32, device=dev),
                torch.zeros(15, 2, dtype=torch.long, device=dev), torch.zeros(16, 3, dtype=torch.long, device=dev)):
        with pytest.raises(ValueError):
            sm.sample(indices=bad)
    for bad in (torch.zeros(3, dtype=torch.long), torch.zeros(3, dtype=torch.int32, device=dev),
                torch.zeros(2, dtype=torch.long, device=dev)):
        with pytest.raises(ValueError):
            AMPUpdateSampler(ld, rb, norm, 16, 0, ring_cursor=bad)
    cpu_loader = _loader(500, dev)
    cpu_loader.preloaded_s_next = cpu_loader.preloaded_s_next.cpu()
    with pytest.raises(ValueError, match="CUDA"):
        AMPUpdateSampler(cpu_loader, rb, norm, 16, 0)
    if torch.cuda.device_count() > 1:            # a tensor on another GPU
        other = _loader(500, torch.device("cuda:1"))
        with pytest.raises(ValueError, match="cuda:0"):
            AMPUpdateSampler(other, rb, norm, 16, 0)
    assert sm.draw_counter.tolist() == [0, 0]     # nothing above launched
