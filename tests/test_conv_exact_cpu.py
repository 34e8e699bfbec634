"""The exact convolution references of tests/conv_exact.py, pinned on the CPU: the float64 tap sums against
torch's own float64 convolutions and autograd, the integer operand generator and its exactness precondition, and
the rounding of the expected kernel output."""
import pytest
import torch
import torch.nn.functional as F

from tests.conv_exact import (DECONV_K2S2, F16_MAX, K1, K3S1P1, K4S2P1, K4S2P1_S2D, check_exact_bound, epilogue_fp32,
                              granularity, int_operand, ref_dgrad, ref_fwd, ref_wgrad, round_out, to_s2d, weight_shape)

def _torch_conv(kind, x, w):
    if kind == K3S1P1:
        return F.conv3d(x, w, padding=1)
    if kind == K1:
        return F.conv3d(x, w)
    if kind in (K4S2P1, K4S2P1_S2D):
        return F.conv3d(x, w, stride=2, padding=1)
    return F.conv_transpose3d(x, w, stride=2)


def _cl(t):
    return t.permute(0, 2, 3, 4, 1)


@pytest.mark.parametrize("kind,c0,c1,co,shape", [
    (K3S1P1, 5, 0, 3, (2, 5, 7, 6)),
    (K3S1P1, 3, 4, 2, (1, 4, 3, 5)),        # two sources: the dgrad is split at c0
    (K1, 6, 0, 4, (2, 3, 5, 4)),
    (K4S2P1, 3, 0, 5, (2, 6, 8, 4)),
    (K4S2P1_S2D, 4, 0, 3, (1, 4, 6, 8)),
    (DECONV_K2S2, 5, 0, 3, (2, 3, 2, 5)),
])
def test_reference_matches_torch_float64(kind, c0, c1, co, shape):
    g = torch.Generator().manual_seed(kind * 17 + c0)
    n, d, h, w = shape
    ci = c0 + c1
    x = torch.randn((n, ci, d, h, w), generator=g, dtype=torch.float64, requires_grad=True)
    wt = torch.randn(weight_shape(kind, ci, co), generator=g, dtype=torch.float64, requires_grad=True)
    y = _torch_conv(kind, x, wt)
    dy = torch.randn(y.shape, generator=g, dtype=torch.float64)
    dx, dw = torch.autograd.grad(y, (x, wt), dy)
    got = ref_fwd(kind, _cl(x.detach()), wt.detach())
    torch.testing.assert_close(got, _cl(y.detach()), rtol=1e-12, atol=1e-12)
    gdx = ref_dgrad(kind, _cl(dy), wt.detach(), (d, h, w))
    # split into the two sources' channel ranges, as the kernels write them
    torch.testing.assert_close(gdx[..., :c0], _cl(dx)[..., :c0], rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(gdx[..., c0:], _cl(dx)[..., c0:], rtol=1e-12, atol=1e-12)
    gdw = ref_wgrad(kind, _cl(x.detach()), _cl(dy), tuple(wt.shape))
    torch.testing.assert_close(gdw, dw, rtol=1e-12, atol=1e-12)


def test_reference_detects_a_wrong_tap():
    """A reference whose tap (0, 0, 1) reads one voxel too far must not pass the pin above."""
    import tests.conv_exact as CE
    g = torch.Generator().manual_seed(3)
    x = torch.randn((1, 3, 4, 5, 6), generator=g, dtype=torch.float64)
    wt = torch.randn((2, 3, 3, 3, 3), generator=g, dtype=torch.float64)
    good = CE._window

    def shifted(t, kd, kh, kw, s, od, oh, ow):
        if (kd, kh, kw) == (0, 0, 1):
            t = F.pad(t, (0, 0, 0, 1))[:, :, 1:]
        return good(t, kd, kh, kw, s, od, oh, ow)

    CE._window = shifted
    try:
        bad = ref_fwd(K3S1P1, _cl(x), wt)
    finally:
        CE._window = good
    assert not torch.allclose(bad, _cl(F.conv3d(x, wt, padding=1)))


def test_s2d_layout():
    t = torch.arange(2 * 4 * 6 * 2 * 3, dtype=torch.float32).view(2, 4, 6, 2, 3)
    s = to_s2d(t)
    assert s.shape == (2, 8, 2, 3, 1, 3)
    for pd in range(2):
        for ph in range(2):
            for pw in range(2):
                assert torch.equal(s[:, (pd * 2 + ph) * 2 + pw], t[:, pd::2, ph::2, pw::2])


def test_int_operand_is_seeded_sparse_and_integer():
    a = int_operand((64, 64, 64), 0.25, [-3, -1, 2, 5], torch.Generator().manual_seed(1), "cpu")
    b = int_operand((64, 64, 64), 0.25, [-3, -1, 2, 5], torch.Generator().manual_seed(1), "cpu")
    assert torch.equal(a, b)
    nz = a[a != 0]
    assert abs(nz.numel() / a.numel() - 0.25) < 0.01
    assert set(nz.unique().tolist()) == {-3.0, -1.0, 2.0, 5.0}
    s = int_operand((1000,), 1.0, [3], torch.Generator().manual_seed(2), "cpu", scale_pow2=-4)
    assert torch.equal(s, torch.full((1000,), 3 / 16))


def test_granularity():
    assert granularity(torch.tensor([0.0, 3.0, -5.0, 7.0])) == 1.0
    assert granularity(torch.tensor([0.75, 2.0])) == 0.25
    assert granularity(torch.tensor([3 * 2.0 ** 14, -2.0 ** 16])) == 2.0 ** 14
    assert granularity(torch.tensor([-2.0 ** -30])) == 2.0 ** -30
    assert granularity(torch.zeros(4)) == 1.0


def test_exact_bound_accepts_and_rejects():
    g = torch.Generator().manual_seed(4)
    x = _cl(int_operand((1, 96, 6, 6, 6), 0.5, [-7, -3, 1, 4], g, "cpu"))
    w = int_operand((32, 96, 3, 3, 3), 1.0, [-2, -1, 1, 2], g, "cpu")
    bound = ref_fwd(K3S1P1, x.abs(), w.abs())
    assert 0 < check_exact_bound(bound, granularity(x) * granularity(w)) < 2.0 ** 22
    # one operand of 2^-12 makes the unit 2^12 times finer: the same sums no longer fit fp32's significand
    x2 = x.clone()
    x2[0, 0, 0, 0, 0] = 2.0 ** -12
    assert float(bound.max()) * 2 ** 12 >= 2.0 ** 22
    with pytest.raises(ValueError):
        check_exact_bound(ref_fwd(K3S1P1, x2.abs(), w.abs()), granularity(x2) * granularity(w))
    # and a sum of 2^22 units is rejected
    with pytest.raises(ValueError):
        check_exact_bound(torch.tensor([2.0 ** 22]), 1.0)
    assert check_exact_bound(torch.tensor([2.0 ** 22 - 1]), 1.0) == 2.0 ** 22 - 1


def _bits16(t):
    return t.view(torch.int16).tolist()


def test_rounding_bf16_ties_to_even():
    one = 1.0
    v = torch.tensor([one + 2 ** -8, one + 3 * 2 ** -8, 257.0, 259.0, -257.0, one + 2 ** -8 + 2 ** -20])
    got = round_out(v, torch.bfloat16).float().tolist()
    assert got == [1.0, one + 2 ** -6, 256.0, 260.0, -256.0, one + 2 ** -7]


def test_rounding_fp16_saturates():
    v = torch.tensor([65504.0, 65519.0, 65520.0, 70000.0, -70000.0, 1e30, 2049.0, 2051.0])
    got = round_out(v, torch.float16)
    assert not torch.isinf(got).any()
    assert got.float().tolist() == [65504.0, 65504.0, 65504.0, 65504.0, -65504.0, 65504.0, 2048.0, 2052.0]
    assert F16_MAX == float(torch.finfo(torch.float16).max)


def test_negative_zero_survives():
    z = torch.tensor([-0.0])
    for dtype in (torch.bfloat16, torch.float16):
        assert _bits16(round_out(z, dtype)) == [-32768]
    # LeakyReLU keeps the sign of a zero: -0 * slope = -0
    assert _bits16(round_out(epilogue_fp32(z, None, act=1, slope=0.2), torch.bfloat16)) == [-32768]


def test_epilogue_fp32_bias_and_leaky_relu():
    acc = torch.tensor([[3.0, -5.0], [16777217.0, -1.0]], dtype=torch.float64)
    bias = torch.tensor([0.5, 1.0])
    v = epilogue_fp32(acc, bias, act=1, slope=0.2)
    assert v.dtype == torch.float32
    s = torch.tensor(0.2, dtype=torch.float32)
    # fp32 rounding of the exact sum first (2^24 + 1 -> 2^24), then the fp32 bias add, then the fp32 product
    assert v.tolist() == [[3.5, (torch.tensor(-4.0) * s).item()], [16777216.0, 0.0]]
    assert epilogue_fp32(acc, bias).tolist() == [[3.5, -4.0], [16777216.0, 0.0]]
