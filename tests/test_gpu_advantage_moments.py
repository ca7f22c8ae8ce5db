"""-m gpu: the rollout statistics kernels against float64 references at the shapes where they branch.

hl_gae_scan_kernel<8>: T in {1, 7, 8, 9, 17, 100} (T % 8 remainder loop, T = 1) x N in {1, 3, 255, 256, 257, 4099}
(partial last block behind full ones), plus all-done, no-done and reward scales 1e3 / 1e-3.  `returns` equal the fp32
oracle bit for bit; the three float64 moments equal float64 sums of the kernel's own raw advantages within 1e-12.

hl_adv_normalize, called directly with host-made moments (n % 4 in {0, 1, 2, 3}, and a view one float into the
buffer so every thread takes the scalar branch), and after the scan with the kernel's moments: within
    |got - ref| <= 2^-23 (|mean| / std + 2 |ref|) + 1e-7
of ref = (a - mean) / (std + 1e-8) in float64 with the unbiased std.  Derivation, u = 2^-24: fl(mean) is off by
<= u |mean|, which moves the result by u |mean| / std; the subtraction a - fl(mean), fl(sqrt(var)), the + 1e-8 and the
division each round once, <= u |ref| apiece, 4 u |ref| together; 2^-23 (|mean| / std + 2 |ref|) = 2u |mean| / std +
4u |ref| leaves a factor 2 on the mean term for the float64 error of the one-pass variance and the second-order
terms, and 1e-7 absorbs fl(1e-8) vs 1e-8 and entries near 0.  The biased std (dividing by n) violates it at n = 48
and at n = 98,304.  Constant advantages give exactly 0; one element gives NaN, as torch's std() of one element.

hl_column_moments (directly and through Normalizer.update): rows in {1, 7, 8, 9, 1183, 1184, 1185, 262147} (below and
around the 148 x 8 grid stride) x dim in {1, 30, 31, 32, 33, 60, 97} (one and several 32-column chunks), with
columns of |mean| / std = 1e3 and constant columns.  Reference: two-pass float64 mean and population variance;
bounds 1e-12 max|x| (mean) and 1e-12 E[x^2] (variance).  A chain of Normalizer.update calls of mixed batch sizes,
one of them a single row, follows a float64 numpy RunningMeanStd (UT:90-110)."""
import math

import numpy as np
import pytest
import torch

import stats_reference as SR
from oracle import torch_oracle as O

pytestmark = pytest.mark.gpu

GAMMA, LAM = 0.99, 0.95


def _L():
    from isaacgymloco_b200 import _lib as L
    return L


# ----------------------------------------------------------------------------- GAE
def _rollout(t, n, seed, dones="some", scale=1.0):
    g = torch.Generator().manual_seed(seed)
    r = scale * torch.randn(t, n, 1, generator=g)
    v = torch.randn(t, n, 1, generator=g)
    if dones == "all":
        d = torch.ones(t, n, 1, dtype=torch.uint8)
    elif dones == "none":
        d = torch.zeros(t, n, 1, dtype=torch.uint8)
    else:
        d = (torch.rand(t, n, 1, generator=g) < 0.1).to(torch.uint8)
    return r, v, d, torch.randn(n, 1, generator=g)


def _gae_scan(r, v, d, lv):
    L = _L()
    t, n = r.shape[:2]
    rc, vc, dc, lc = (x.cuda().contiguous() for x in (r, v, d, lv))
    ret, adv = torch.full_like(rc, float("nan")), torch.full_like(rc, float("nan"))
    mom = torch.zeros(3, dtype=torch.float64, device="cuda")
    L.check(L.lib.hl_gae_scan(L.ptr(rc), L.ptr(vc), L.ptr(dc), L.ptr(lc), L.ptr(ret), L.ptr(adv), L.ptr(mom), t, n,
                              GAMMA, LAM, L.stream()))
    return ret, adv, mom


def _normalize(adv, moments):
    L = _L()
    L.check(L.lib.hl_adv_normalize(L.ptr(adv), L.ptr(moments), adv.numel(), L.stream()))
    torch.cuda.synchronize()
    return adv


def _norm_bound(a, ref):
    a = np.asarray(a, dtype=np.float64).ravel()
    mean = a.sum() / a.size
    std = math.sqrt(np.square(a - mean).sum() / (a.size - 1)) if a.size > 1 else float("nan")
    return 2.0 ** -23 * (abs(mean) / std + 2 * np.abs(ref)) + 1e-7


def _check_normalized(got, a, what):
    got = got.detach().cpu().double().numpy().ravel()
    ref = SR.normalize64(a)
    tol = _norm_bound(a, ref)
    err = np.abs(got - ref)
    bad = ~(err <= tol)
    if bad.any():
        i = int(np.argmax(np.where(bad, err / tol, 0)))
        raise AssertionError(f"{what}: {int(bad.sum())} of {got.size} out of bound, worst {i}: got {got[i]!r} "
                             f"ref {ref[i]!r} tol {tol[i]:.3g}")


def _check_moments(mom, adv, t, n, what):
    a = adv.detach().cpu().double().numpy().ravel()
    s1, s2 = math.fsum(a), math.fsum(a * a)
    m = mom.cpu().numpy()
    assert abs(m[0] - s1) <= 1e-12 * math.fsum(np.abs(a)), (what, m[0], s1)
    assert abs(m[1] - s2) <= 1e-12 * s2, (what, m[1], s2)
    assert m[2] == float(t * n), (what, m[2])


def _gae_case(t, n, seed, dones="some", scale=1.0):
    r, v, d, lv = _rollout(t, n, seed, dones, scale)
    ret, adv, mom = _gae_scan(r, v, d, lv)
    torch.cuda.synchronize()
    want, _ = O.compute_returns(r, v, d, lv, GAMMA, LAM)
    what = f"T={t} N={n} dones={dones} scale={scale}"
    bad = int((ret.cpu() != want).sum())
    assert bad == 0, f"{what}: {bad} returns differ from the fp32 oracle"
    assert torch.equal(adv.cpu(), want - v), f"{what}: raw advantages != returns - values"
    _check_moments(mom, adv, t, n, what)
    a = adv.cpu().numpy().copy()
    if t * n == 1:
        assert torch.isnan(_normalize(adv, mom)).all(), f"{what}: one element normalises to NaN (torch's std())"
    else:
        _check_normalized(_normalize(adv, mom), a, what)


@pytest.mark.parametrize("n", [1, 3, 255, 256, 257, 4099])
@pytest.mark.parametrize("t", [1, 7, 8, 9, 17, 100])
def test_gae_scan_shapes(t, n):
    """returns bit-equal to the fp32 oracle, the float64 moments of the raw advantages, then the normalisation."""
    _gae_case(t, n, seed=1000 * t + n)


@pytest.mark.parametrize("dones,scale", [("all", 1.0), ("none", 1.0), ("some", 1e3), ("some", 1e-3)])
@pytest.mark.parametrize("t,n", [(9, 257), (100, 4099)])
def test_gae_scan_dones_and_scales(t, n, dones, scale):
    _gae_case(t, n, seed=7 + t + n, dones=dones, scale=scale)


# ----------------------------------------------------------------------------- hl_adv_normalize
def _host_moments(a):
    a64 = np.asarray(a, dtype=np.float64).ravel()
    return torch.tensor([a64.sum(), np.square(a64).sum(), float(a64.size)], dtype=torch.float64, device="cuda")


def _normalize_host(a, offset):
    """hl_adv_normalize on a copy of `a` placed `offset` floats into a fresh buffer, with host-made moments."""
    buf = torch.full((a.size + offset,), float("nan"), device="cuda")
    view = buf[offset:]
    view.copy_(torch.from_numpy(a))
    _normalize(view, _host_moments(a))
    if offset:
        assert view.data_ptr() % 16 != 0
        assert torch.isnan(buf[:offset]).all(), "wrote before the view"
    return view


@pytest.mark.parametrize("offset", [0, 1], ids=["aligned", "offset1"])
@pytest.mark.parametrize("m", [48, 49, 50, 51, 98304, 98305, 98306, 98307])
@pytest.mark.parametrize("mean,std", [(3.0, 2.0), (-50.0, 0.5)])
def test_adv_normalize_tails_and_alignment(m, offset, mean, std):
    """Every n % 4, float4 and scalar branches: within the bound of the unbiased float64 normalisation."""
    a = np.random.default_rng(m + offset).normal(mean, std, size=m).astype(np.float32)
    _check_normalized(_normalize_host(a, offset), a, f"n={m} offset={offset}")


@pytest.mark.parametrize("m", [48, 98304])
def test_adv_normalize_bound_rejects_biased_std(m):
    """The bound separates the unbiased std from the biased one: the kernel's output is inside it for ddof 1 and
    outside it for ddof 0 (the 1 + 1/(2n) factor is 5e-6 at n = 98,304, the bound's relative part 2.4e-7)."""
    a = np.random.default_rng(m).normal(3.0, 2.0, size=m).astype(np.float32)
    got = _normalize_host(a, 0).cpu().double().numpy()
    _check_normalized(torch.from_numpy(got), a, f"n={m}")
    biased = SR.normalize64(a, ddof=0)
    assert (np.abs(got - biased) > _norm_bound(a, biased)).any(), f"n={m}: the bound does not reject the biased std"


@pytest.mark.parametrize("m", [2, 51, 98304])
@pytest.mark.parametrize("offset", [0, 1], ids=["aligned", "offset1"])
def test_adv_normalize_constant_is_zero(m, offset):
    a = np.full(m, 0.7, dtype=np.float32)
    got = _normalize_host(a, offset)
    assert torch.equal(got, torch.zeros_like(got))


@pytest.mark.parametrize("offset", [0, 1], ids=["aligned", "offset1"])
def test_adv_normalize_one_element_is_nan(offset):
    """N*T = 1: the unbiased variance is 0/0, torch's std() is NaN and so are the reference's advantages."""
    got = _normalize_host(np.array([0.25], dtype=np.float32), offset)
    assert torch.isnan(got).all()


# ----------------------------------------------------------------------------- hl_column_moments
def _batch(rows, dim, seed):
    """Columns cycle through: N(0, 1) scaled by 10^k, |mean| / std = 1e3, constant."""
    rng = np.random.default_rng(seed)
    x = np.empty((rows, dim), dtype=np.float32)
    for c in range(dim):
        kind = c % 3
        if kind == 0:
            x[:, c] = rng.normal(0.0, 10.0 ** (c % 5 - 2), size=rows)
        elif kind == 1:
            x[:, c] = rng.normal(1e3 * (1 if c % 2 else -1), 1.0, size=rows)
        else:
            x[:, c] = np.float32(0.3 + c)
    return x


def _column_moments(x):
    L = _L()
    rows, dim = x.shape
    xc = torch.from_numpy(x).cuda()
    ws = torch.zeros(int(L.lib.hl_moments_workspace_bytes(dim)), dtype=torch.uint8, device="cuda")
    out = torch.full((2 * dim,), float("nan"), dtype=torch.float64, device="cuda")
    L.check(L.lib.hl_column_moments(L.ptr(xc), rows, dim, L.ptr(out), L.ptr(ws), L.stream()))
    out = out.cpu().numpy()
    return out[:dim], out[dim:]


def _check_column_moments(mean, var, x, what):
    x64 = x.astype(np.float64)
    rm, rv = SR.moments64(x)
    mtol = 1e-12 * np.abs(x64).max(axis=0)
    vtol = 1e-12 * np.square(x64).mean(axis=0)
    bm, bv = np.abs(mean - rm) > mtol, np.abs(var - rv) > vtol
    assert not bm.any(), f"{what}: mean of columns {np.nonzero(bm)[0].tolist()}: got {mean[bm]} ref {rm[bm]}"
    assert not bv.any(), f"{what}: variance of columns {np.nonzero(bv)[0].tolist()}: got {var[bv]} ref {rv[bv]}"


@pytest.mark.parametrize("dim", [1, 30, 31, 32, 33, 60, 97])
@pytest.mark.parametrize("rows", [1, 7, 8, 9, 1183, 1184, 1185, 262147])
def test_column_moments_shapes(rows, dim):
    x = _batch(rows, dim, seed=rows * 131 + dim)
    mean, var = _column_moments(x)
    _check_column_moments(mean, var, x, f"rows={rows} dim={dim}")


@pytest.mark.parametrize("dim", [1, 33, 97])
def test_normalizer_update_chain(dim):
    """Normalizer.update's own moments (read back after each call) and its running mean/var/count after five calls of
    1185, 1, 7, 262147 and 33 rows, against the float64 numpy RunningMeanStd."""
    from isaacgymloco_b200.amp_discriminator import Normalizer
    norm = Normalizer(dim, device="cuda:0")
    rms = SR.RunningMeanStd64(dim)
    for k, rows in enumerate((1185, 1, 7, 262147, 33)):
        x = _batch(rows, dim, seed=17 * k + dim)
        norm.update(torch.from_numpy(x).cuda())
        rms.update(x)
        mv = norm._mv.cpu().numpy()
        _check_column_moments(mv[:dim], mv[dim:], x, f"update {k} ({rows} rows)")
        # the batch moments differ from two-pass float64 by up to 1e-12 of the second moment (above); the merge is
        # float64 on both sides, so the running statistics are held to 1e-11 of the running second moment
        got_mean, got_var = norm.mean.cpu().numpy(), norm.var.cpu().numpy()
        second = rms.var + np.square(rms.mean)
        bm = np.abs(got_mean - rms.mean) > 1e-11 * np.sqrt(second)
        bv = np.abs(got_var - rms.var) > 1e-11 * second
        assert not bm.any(), f"mean after update {k}, columns {np.nonzero(bm)[0].tolist()}: {got_mean[bm]} vs {rms.mean[bm]}"
        assert not bv.any(), f"var after update {k}, columns {np.nonzero(bv)[0].tolist()}: {got_var[bv]} vs {rms.var[bv]}"
        assert norm.count == rms.count
