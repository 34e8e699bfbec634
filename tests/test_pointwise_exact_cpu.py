"""Pins tests/pointwise_exact.py (the references of the memory-bound kernels) without a GPU: ``fma32`` against exact
rational arithmetic, the dropout mask against a pure-Python-int transcription of the CUDA source, the forward,
finalize and backward against torch's own norm / LeakyReLU in float64, and every comparison the GPU suite applies
against planted kernel errors it must detect."""
import random
from fractions import Fraction

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import pointwise_exact as R

M = 0xFFFFFFFF


# ---------------------------------------------------------------------------------------------------
# fma32
# ---------------------------------------------------------------------------------------------------
def _round_fraction_to_f32(x):
    """The fp32 nearest to the rational x, ties to even (exact: the candidates are compared as fractions)."""
    f = np.float32(float(x))
    cands = {f, np.nextafter(f, np.float32(np.inf)), np.nextafter(f, np.float32(-np.inf))}
    best = min(cands, key=lambda c: (abs(Fraction(float(c)) - x), int(np.array(c).view(np.int32)) & 1))
    if best == 0 and x == 0:
        return None                      # the sign of an exact zero is IEEE's, checked separately
    return best


def _check_fma(a, b, c):
    got = R.fma32(torch.from_numpy(a), torch.from_numpy(b), torch.from_numpy(c)).numpy()
    bad = []
    for i in range(a.size):
        x = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        want = _round_fraction_to_f32(x)
        if want is None:
            continue
        if np.array(got[i]).view(np.int32) != np.array(np.float32(want)).view(np.int32):
            bad.append((a[i], b[i], c[i], got[i], want))
    return bad


def test_fma32_equals_exact_rational_rounding_on_random_triples():
    rng = np.random.default_rng(0)
    n = 100_000
    a = (rng.standard_normal(n) * np.exp2(rng.integers(-20, 20, n))).astype(np.float32)
    b = (rng.standard_normal(n) * np.exp2(rng.integers(-20, 20, n))).astype(np.float32)
    c = (rng.standard_normal(n) * np.exp2(rng.integers(-40, 40, n))).astype(np.float32)
    # a third of the triples cancel nearly: c = -fl(a b) (+ a few units), where the low product bits decide the result
    near = rng.random(n) < 0.33
    c[near] = (-(a[near].astype(np.float64) * b[near])).astype(np.float32) * (1 + rng.integers(-3, 4, near.sum()) * 2.0 ** -23)
    assert _check_fma(a, b, c) == []


def test_fma32_hard_cases():
    e = 2.0 ** -12
    cases = [
        (1 + e, 1 + e, 0.0),                     # 1 + 2^-11 + 2^-24: an fp32 midpoint, ties to even
        (1 + e, 1 + e, 2.0 ** -60),              # just above the midpoint: rounds up (naive fp64 would tie)
        (1 + e, 1 + e, -(2.0 ** -60)),           # just below: rounds down
        (-(1 + e), 1 + e, 2.0 ** -60),
        (1 + 3 * e, 1 + e, 2.0 ** -70),
        (2.0 ** -24 * 3, 1.375, -0.5),           # fp16 subnormal y times a constant
        (2.0 ** -24, 0.7, 1e-8),
        (-(2.0 ** -14) * 1023 / 1024, 1.1, 2.0 ** -30),
        (65504.0, 1.0526316, -1.5),
        (-65504.0, 1.0526316, 1.5),
    ]
    a, b, c = (np.array(v, dtype=np.float32) for v in zip(*cases))
    assert _check_fma(a, b, c) == []
    # exact cancellation: +0 for x + (-x), -0 only for (-0) + (-0)
    z = R.fma32(torch.tensor([3.0, -3.0, 0.0, -0.0, 0.0, 2.0 ** -24]), torch.tensor([5.0, 5.0, 1.0, 1.0, -1.0, 4.0]),
                torch.tensor([-15.0, 15.0, -0.0, -0.0, -0.0, -(2.0 ** -22)]))
    assert R.bits(z).tolist() == R.bits(torch.tensor([0.0, 0.0, 0.0, -0.0, -0.0, 0.0])).tolist()


# ---------------------------------------------------------------------------------------------------
# dropout
# ---------------------------------------------------------------------------------------------------
def _py_keep(e, seed, t15):
    """pointwise.cuh dropout_bits8 / dropout_maskw with Python ints, for element index e."""
    def mulfold(x, y):
        m = (x & M) * (y & M)
        return (m & M) ^ (m >> 32)
    e0 = e & ~7
    idx = (e0 >> 3) & M
    salt = (seed ^ (((e0 >> 35) * 0x7FEB352D) & M)) & M
    m = mulfold(idx ^ 0x9E3779B9, 0x85EBCA6B ^ (((salt << 1) | 1) & M)) ^ salt
    p0 = (m ^ 0xC2B2AE35) * 0x27D4EB2F
    p1 = (m ^ 0x165667B1) * 0x9E3779B1
    q = mulfold((m + 0x632BE5AB) & M, 0xD2B74407)
    rot = lambda x, r: ((x >> r) | (x << (32 - r))) & M
    u = [(p0 & M) ^ q, (p0 >> 32) ^ rot(q, 7), (p1 & M) ^ rot(q, 13), (p1 >> 32) ^ rot(q, 21)]
    lane = e & 7
    word = u[lane >> 1]
    # the lane compare of dropout_maskw: bit 15 of ((u15 | 0x8000) - t15)
    d = ((word >> (16 * (lane & 1))) & 0x7FFF | 0x8000) - t15
    return bool(d & 0x8000)


def test_dropout_keep_equals_python_transcription():
    rng = random.Random(0)
    idx = [rng.randrange(0, 1 << 26) for _ in range(1500)]
    idx += [(1 << 31) + rng.randrange(-4096, 4096) for _ in range(500)]           # past 2^31 elements
    idx += [(1 << 35) * rng.randrange(1, 40) + rng.randrange(0, 1 << 20) for _ in range(500)]   # salted by e0 >> 35
    seeds = [0, 1234, 0x80000000, 0x9E3779B1, 0xFFFFFFFF]
    for p in (0.05, 0.5):
        t15 = R.drop_thresh(p)
        for seed in seeds:
            got = R.dropout_keep(torch.tensor(idx), seed, p).tolist()
            assert got == [_py_keep(e, seed, t15) for e in idx], (p, seed)


def test_drop_thresh_is_the_hosts_rounding():
    assert R.drop_thresh(0.05) == 1638 and R.drop_thresh(0.5) == 16384 and R.drop_thresh(0.999999) == 32767
    assert R.drop_thresh(0.0) == 0


@pytest.mark.parametrize("p", [0.05, 0.5])
def test_dropout_keep_rate(p):
    n = 1 << 24
    keep = R.dropout_keep(torch.arange(n, dtype=torch.int64) + (3 << 30), 0x9E3779B1, p)
    rate = keep.double().mean().item()
    want = 1 - R.drop_thresh(p) / 32768
    sigma = (want * (1 - want) / n) ** 0.5
    assert abs(rate - want) < 4 * sigma, (rate, want, sigma)


# ---------------------------------------------------------------------------------------------------
# forward, finalize and backward against torch in float64
# ---------------------------------------------------------------------------------------------------
def _sample_block(mode, n=3, c=24, cp=32, dims=(4, 6, 8), seed=0):
    g = torch.Generator().manual_seed(seed)
    y = (torch.randn((n, *dims, c), generator=g) * 1.7 + 0.3).to(torch.float16)
    gamma = torch.rand(c, generator=g) + 0.5
    beta = torch.randn(c, generator=g) * 0.2
    rm, rv = torch.randn(c, generator=g) * 0.1, torch.rand(c, generator=g) + 0.5
    yp = torch.zeros((n, *dims, cp), dtype=torch.float16)
    yp[..., :c] = y
    s = yp.double().sum((1, 2, 3))
    q = (yp.double() ** 2).sum((1, 2, 3))
    return yp, y, gamma, beta, rm, rv, s, q


def _torch_norm(y, gamma, beta, mode, rm, rv):
    x = y.double().permute(0, 4, 1, 2, 3)
    if mode == R.INSTANCE:
        z = F.instance_norm(x, weight=gamma.double(), bias=beta.double(), eps=1e-5)
    else:
        z = F.batch_norm(x, rm, rv, gamma.double(), beta.double(), training=mode == R.BATCH_TRAIN, momentum=0.1,
                         eps=1e-5)
    return z.permute(0, 2, 3, 4, 1)


@pytest.mark.parametrize("mode", [R.INSTANCE, R.BATCH_TRAIN, R.BATCH_EVAL])
def test_finalize_and_act_fwd_match_torch(mode):
    yp, y, gamma, beta, rm, rv, s, q = _sample_block(mode)
    n, c = y.shape[0], y.shape[-1]
    vox = y[0, ..., 0].numel()
    ref = R.finalize(s, q, vox, gamma, beta, 1e-5, mode, 0.1, rm, rv)
    rm64, rv64 = rm.double().clone(), rv.double().clone()
    z = _torch_norm(y, gamma, beta, mode, rm64, rv64)
    if mode == R.BATCH_TRAIN:       # running statistics (unbiased variance), to the fp32 cast of momentum / eps
        assert torch.allclose(ref["running_mean"], rm64, rtol=1e-7, atol=1e-9)
        assert torch.allclose(ref["running_var"], rv64, rtol=1e-7, atol=0)
    sc, sh = ref["scale"].float(), ref["shift"].float()
    # normalised value from the fp32 constants: two fp32 roundings of the constants, eps as fp32
    zr = y.double() * sc[:, None, None, None, :c].double() + sh[:, None, None, None, :c].double()
    scale_mag = (y.double().abs() + ref["mean"][:, None, None, None, :c].abs()) * ref["scale"][:, None, None, None, :c].abs()
    assert bool(((zr - z).abs() <= 4e-7 * (scale_mag + beta.double().abs()) + 1e-12).all())
    # the forward: LeakyReLU(fmaf) rounded to bf16 / fp16 within half a unit of the float64 value
    slope = 0.2
    a, a16 = R.act_fwd(yp, sc, sh, slope)
    want = F.leaky_relu(z, slope)
    tol = 2.0 ** -23 * (scale_mag + beta.double().abs()) + 1e-30
    for got, half_unit in ((a, 2.0 ** -8), (a16, 2.0 ** -11)):
        assert bool(((got[..., :c].double() - want).abs() <= half_unit * want.abs() + tol * 2).all())
    assert bool((R.bits(a[..., c:]) == 0).all())


@pytest.mark.parametrize("mode", [R.INSTANCE, R.BATCH_TRAIN, R.BATCH_EVAL])
def test_norm_bwd_matches_float64_autograd(mode):
    yp, y, gamma, beta, rm, rv, s, q = _sample_block(mode, seed=1)
    n, c, cp = y.shape[0], y.shape[-1], yp.shape[-1]
    vox = y[0, ..., 0].numel()
    ref = R.finalize(s, q, vox, gamma, beta, 1e-5, mode, 0.1, rm, rv)
    sc, sh, mean, rstd = (ref[k].float() for k in ("scale", "shift", "mean", "rstd"))
    slope, p, seed = 0.2, 0.3, 77
    g = torch.Generator().manual_seed(2)
    dA = torch.zeros(yp.shape, dtype=torch.bfloat16)
    dA[..., :c] = torch.randn((n, *y.shape[1:4], c), generator=g).to(torch.bfloat16)
    out = R.norm_bwd(dA, yp, mode, mean, rstd, sc, sh, slope, p, seed, c)
    # the same graph in float64 autograd, from the fp32 statistics and with the mask fixed
    keep = R.dropout_keep(R.element_index(tuple(yp.shape), "cpu"), seed, p)[..., :c]
    pos = (R.pre_activation(yp, sc, sh, p) > 0)[..., :c]
    yd = y.double().requires_grad_(True)
    gd = gamma.double().requires_grad_(True)
    bd = beta.double().requires_grad_(True)
    ref64 = R.finalize(s, q, vox, gamma, beta, 1e-5, mode, 0.1, rm, rv)
    m64, r64 = ref64["mean"][:, :c], ref64["rstd"][:, :c]
    if mode == R.BATCH_EVAL:
        xhat = (yd - m64[:, None, None, None]) * r64[:, None, None, None]
    else:
        dims = (1, 2, 3) if mode == R.INSTANCE else (0, 1, 2, 3)
        mu = yd.mean(dims, keepdim=True)
        var = ((yd - mu) ** 2).mean(dims, keepdim=True)
        xhat = (yd - mu) / torch.sqrt(var + R.f32(1e-5).double())
    zz = xhat * gd + bd
    inv = R.fold_inv(p)
    fac = torch.where(pos, inv, R.f32(slope) * inv).double()       # the kernels' fp32 factors
    act = zz * fac * keep
    act.backward(dA[..., :c].double())
    # the autograd graph differentiates through its own float64 statistics; the kernels use the fp32 ones
    rel = lambda a_, b_: float((a_ - b_).abs().max() / b_.abs().max())
    assert rel(out["dy"][..., :c], yd.grad) < 1e-6
    assert rel(out["dgamma"], gd.grad) < 1e-6 and rel(out["dbeta"], bd.grad) < 1e-12       # dbeta = sum dz
    # with the float64 statistics the restatement is float64 autograd to rounding
    out64 = R.norm_bwd(dA, yp, mode, ref64["mean"], ref64["rstd"], ref64["scale"], sh, slope, p, seed, c,
                       dz=out["dz"])
    assert rel(out64["dy"][..., :c], yd.grad) < 1e-12
    assert rel(out64["dgamma"], gd.grad) < 1e-12 and rel(out64["dbeta"], bd.grad) < 1e-12
    if mode == R.BATCH_EVAL:
        assert rel(out["dbias"], (gamma.double() * r64[0] * bd.grad)) < 1e-6
    else:
        assert bool((out["dbias"] == 0).all())


# ---------------------------------------------------------------------------------------------------
# planted errors: every comparison of the GPU suite must fail on them
# ---------------------------------------------------------------------------------------------------
def _fwd_data(seed=3, p=0.05):
    g = torch.Generator().manual_seed(seed)
    n, d, h, w, cp = 2, 4, 6, 8, 32
    y = torch.randn((n, d, h, w, cp), generator=g) * 2
    y[torch.rand(y.shape, generator=g) < 0.2] = 0.0
    y[torch.rand(y.shape, generator=g) < 0.1] = -0.0
    y = y.to(torch.float16)
    scale = torch.rand((n, cp), generator=g) + 0.5
    shift = torch.randn((n, cp), generator=g) * 0.3
    shift[:, ::4] = -0.0
    return y, scale, shift, p


def test_planted_unbiased_variance_fails_the_finalize_comparison():
    g = torch.Generator().manual_seed(4)
    n, cp, c, vox = 8, 32, 32, 128 ** 3
    s = torch.randint(-5000, 5000, (n, cp), generator=g).double()
    q = torch.randint(vox, 2 * vox, (n, cp), generator=g).double()
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g)
    for mode in (R.INSTANCE, R.BATCH_TRAIN):
        ref = R.finalize(s, q, vox, gamma, beta, 1e-5, mode)
        planted = R.finalize(s, q, vox, gamma, beta, 1e-5, mode, unbiased_norm=True)
        good = {k: v.float() for k, v in ref.items()}
        assert R.check_finalize(good, ref, c, mode)[0] == []
        fails, _ = R.check_finalize({k: v.float() for k, v in planted.items()}, ref, c, mode)
        assert any(f.startswith("rstd") for f in fails) and any(f.startswith("scale") for f in fails)


def test_planted_dropout_counter_off_by_one_vector_fails_the_forward_comparison():
    y, scale, shift, p = _fwd_data()
    a, a16 = R.act_fwd(y, scale, shift, 0.2, p, 99)
    assert R.check_act_fwd(y, scale, shift, 0.2, p, 99, 32, a=a, a16=a16) == []
    # the kernel's counter one vector (8 elements) ahead: the mask of the neighbouring vector
    x = R.leaky(R.pre_activation(y, scale, shift, p), 0.2)
    keep = R.dropout_keep(R.element_index(tuple(y.shape), "cpu") + 8, 99, p)
    bad = torch.where(keep, x.to(torch.bfloat16), torch.zeros((), dtype=torch.bfloat16))
    fails = R.check_act_fwd(y, scale, shift, 0.2, p, 99, 32, a=bad)
    assert fails and fails[0].startswith("a:")


def test_planted_zero_c2_fails_the_dy_comparison():
    y, scale, shift, p = _fwd_data(seed=5)
    g = torch.Generator().manual_seed(6)
    n, cp = y.shape[0], y.shape[-1]
    mean = torch.randn((n, cp), generator=g) * 0.1
    rstd = torch.rand((n, cp), generator=g) + 0.5
    dA = (torch.randn(y.shape, generator=g)).to(torch.bfloat16)
    ref = R.norm_bwd(dA, y, R.INSTANCE, mean, rstd, scale, shift, 0.2, p, 9, cp)
    planted = R.norm_bwd(dA, y, R.INSTANCE, mean, rstd, scale, shift, 0.2, p, 9, cp, zero_c2=True)
    good = ref["dy"].to(torch.bfloat16)
    assert R.check_dy(good, ref, y, mean, rstd, scale, 8, cp)[0] == []
    fails, _ = R.check_dy(planted["dy"].float().to(torch.bfloat16), ref, y, mean, rstd, scale, 8, cp)
    assert fails and fails[0].startswith("dy:")


def test_planted_last_maximum_fails_the_pooling_comparisons():
    y, scale, shift, p = _fwd_data(seed=7, p=0.5)        # many +0 (dropped) and -0 activations: ties in the windows
    a, _ = R.act_fwd(y, scale, shift, 0.2, p, 5)
    g = torch.Generator().manual_seed(8)
    dP = torch.randn((2, 2, 3, 4, 32), generator=g).to(torch.bfloat16)
    assert R.check_maxpool_bwd(a, dP, None, R.maxpool_bwd(a, dP)) == []
    assert R.check_maxpool_bwd(a, dP, None, R.maxpool_bwd(a, dP, last=True))
    assert R.check_act_fwd(y, scale, shift, 0.2, p, 5, 32, pooled=R.pool_first_max(a, last=True)[0])


def test_planted_ge_in_the_sign_test_fails_the_backward_comparison():
    g = torch.Generator().manual_seed(9)
    shape = (2, 4, 4, 8, 32)
    a = torch.randn(shape, generator=g).to(torch.bfloat16)
    a[torch.rand(shape, generator=g) < 0.1] = 0.0           # a pre-activation of exactly 0
    dA = torch.randn(shape, generator=g).to(torch.bfloat16)
    good = R.ref_bwd_none(dA, a, 0.2, 0.0, 0)
    assert R.check_bwd_none(dA, a, 0.2, 0.0, 0, good) == []
    assert R.check_bwd_none(dA, a, 0.2, 0.0, 0, R.ref_bwd_none(dA, a, 0.2, 0.0, 0, ge=True))
    # and in the statistics path: the dz of the sums
    y, scale, shift, p = _fwd_data(seed=10, p=0.0)
    dA2 = torch.ones(y.shape, dtype=torch.bfloat16)
    pre = R.pre_activation(y, scale, shift, p)
    assert bool((pre == 0).any())
    d_gt = R.dz_of(dA2, y, scale, shift, 0.2, p, 0)
    d_ge = R.dz_of(dA2, y, scale, shift, 0.2, p, 0, ge=True)
    assert not torch.equal(d_gt, d_ge)
