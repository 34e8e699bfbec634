"""Exact references for the convolution kernels (test plumbing only).

With every operand a small integer (times a power of two) that bf16 / fp16 represent exactly, every product is
exact in fp32, and while sum |x| |w| stays below 2^22 units of the operands' granularity every partial sum is exact
in any order and on any split (two bits of fp32's 24-bit significand are left for the tensor cores' alignment). The
kernel's fp32 accumulator must then equal the mathematical sum, and its rounded output equals the reference rounded
the same way, bit for bit.

The reference is a plain float64 tap sum: for each filter tap, the shifted (stride 2: strided) slice of the
zero-padded channel-last input times that tap's (ci, co) weight matrix, one sample at a time. It uses neither cuDNN
nor any transform algorithm. Tensors are channel-last (N, D, H, W, C) with the real channel count; weights are in
the torch layout: (co, ci, k, k, k), the transposed conv (ci, co, 2, 2, 2).
"""
import itertools

import torch
import torch.nn.functional as F

K3S1P1, K1, K4S2P1, DECONV_K2S2, K4S2P1_S2D = 0, 1, 2, 3, 4     # ub_api.h conv kinds
EXACT_LIMIT = 2.0 ** 22
F16_MAX = 65504.0

_GEOM = {K3S1P1: (3, 1, 1), K1: (1, 1, 0), K4S2P1: (4, 2, 1), K4S2P1_S2D: (4, 2, 1)}   # kernel, stride, padding


def weight_shape(kind, ci, co):
    if kind == DECONV_K2S2:
        return (ci, co, 2, 2, 2)
    k = _GEOM[kind][0]
    return (co, ci, k, k, k)


def out_dims(kind, d, h, w):
    if kind == DECONV_K2S2:
        return 2 * d, 2 * h, 2 * w
    k, s, p = _GEOM[kind]
    return tuple((e + 2 * p - k) // s + 1 for e in (d, h, w))


def _taps(k):
    return itertools.product(range(k), repeat=3)


def _window(t, kd, kh, kw, s, od, oh, ow):
    """The (od, oh, ow) positions of a padded (D, H, W, C) sample that tap (kd, kh, kw) reads, stride s."""
    return t[kd:kd + s * (od - 1) + 1:s, kh:kh + s * (oh - 1) + 1:s, kw:kw + s * (ow - 1) + 1:s]


def _pad(t, p):
    return F.pad(t, (0, 0, p, p, p, p, p, p)) if p else t


def ref_fwd(kind, x, w):
    """Convolution (no bias) of channel-last x (N, D, H, W, ci) -> float64 (N, Do, Ho, Wo, co)."""
    n, d, h, wd, ci = x.shape
    w = w.double()
    od, oh, ow = out_dims(kind, d, h, wd)
    co = w.shape[1] if kind == DECONV_K2S2 else w.shape[0]
    out = torch.zeros((n, od, oh, ow, co), dtype=torch.float64, device=x.device)
    for i in range(n):
        xi = x[i].double()
        if kind == DECONV_K2S2:
            for a, b, c in _taps(2):
                out[i, a::2, b::2, c::2] = xi @ w[:, :, a, b, c]
            continue
        k, s, p = _GEOM[kind]
        xp = _pad(xi, p)
        for kd, kh, kw in _taps(k):
            out[i] += _window(xp, kd, kh, kw, s, od, oh, ow) @ w[:, :, kd, kh, kw].t()
    return out


def ref_dgrad(kind, dy, w, in_dhw):
    """Input gradient of ``ref_fwd`` for the output gradient dy (N, Do, Ho, Wo, co) -> float64 (N, D, H, W, ci)."""
    n = dy.shape[0]
    d, h, wd = in_dhw
    w = w.double()
    ci = w.shape[0] if kind == DECONV_K2S2 else w.shape[1]
    out = torch.zeros((n, d, h, wd, ci), dtype=torch.float64, device=dy.device)
    od, oh, ow = out_dims(kind, d, h, wd)
    for i in range(n):
        gi = dy[i].double()
        if kind == DECONV_K2S2:
            for a, b, c in _taps(2):
                out[i] += gi[a::2, b::2, c::2] @ w[:, :, a, b, c].t()
            continue
        k, s, p = _GEOM[kind]
        acc = torch.zeros((d + 2 * p, h + 2 * p, wd + 2 * p, ci), dtype=torch.float64, device=dy.device)
        for kd, kh, kw in _taps(k):
            _window(acc, kd, kh, kw, s, od, oh, ow).add_(gi @ w[:, :, kd, kh, kw])
        out[i] = acc[p:p + d, p:p + h, p:p + wd]
    return out


def ref_wgrad(kind, x, dy, wshape):
    """Weight gradient of ``ref_fwd``: float64 in the torch weight layout ``wshape``."""
    n, d, h, wd, ci = x.shape
    dw = torch.zeros(wshape, dtype=torch.float64, device=x.device)
    od, oh, ow = out_dims(kind, d, h, wd)
    for i in range(n):
        xi, gi = x[i].double(), dy[i].double()
        if kind == DECONV_K2S2:
            x2 = xi.reshape(-1, ci)
            for a, b, c in _taps(2):
                dw[:, :, a, b, c] += x2.t() @ gi[a::2, b::2, c::2].reshape(-1, gi.shape[-1])
            continue
        k, s, p = _GEOM[kind]
        xp = _pad(xi, p)
        g2 = gi.reshape(-1, gi.shape[-1])
        for kd, kh, kw in _taps(k):
            dw[:, :, kd, kh, kw] += g2.t() @ _window(xp, kd, kh, kw, s, od, oh, ow).reshape(-1, ci)
    return dw


# ---------------------------------------------------------------------------------------------------
# operands and the exactness precondition
# ---------------------------------------------------------------------------------------------------
def int_operand(shape, density, values, gen, device, scale_pow2=0):
    """Seeded float32 tensor: each element is nonzero with probability ``density``, then drawn uniformly from
    ``values`` (integers), times 2^scale_pow2."""
    vals = torch.tensor(values, dtype=torch.float32, device=device)
    keep = torch.rand(shape, generator=gen, device=device) < density
    idx = torch.randint(0, len(values), shape, generator=gen, device=device)
    return torch.where(keep, vals[idx], torch.zeros((), device=device)) * (2.0 ** scale_pow2)


def granularity(t):
    """Largest power of two every element of t is an integer multiple of (1.0 for an all-zero tensor)."""
    v = t[t != 0].double()
    if v.numel() == 0:
        return 1.0
    m, e = torch.frexp(v)
    mant = (m.abs() * 2.0 ** 53).to(torch.int64)
    low = torch.log2((mant & -mant).double()).round().to(torch.int64)
    return 2.0 ** int((e.to(torch.int64) - 53 + low).min())


def check_exact_bound(abs_sum, unit, what="sum |x| |w|"):
    """Raise ValueError unless every entry of ``abs_sum`` is below 2^22 units ``unit`` (the granularity of its
    terms): otherwise a fp32 partial sum could round and a bitwise comparison would not be sound."""
    worst = float(abs_sum.max()) / unit if abs_sum.numel() else 0.0
    if not worst < EXACT_LIMIT:
        raise ValueError(f"{what} reaches {worst:.4g} units of {unit:g}: not exact in fp32 (limit 2^22)")
    return worst


# ---------------------------------------------------------------------------------------------------
# what the kernels store
# ---------------------------------------------------------------------------------------------------
def epilogue_fp32(acc, bias=None, act=0, slope=0.0):
    """The fp32 value the forward epilogue holds: fp32(exact sum) + fp32 bias, then LeakyReLU in fp32 if act."""
    v = acc.float()
    if bias is not None:
        v = v + bias.float()
    if act:
        v = torch.where(v > 0, v, v * torch.tensor(slope, dtype=torch.float32, device=v.device))
    return v


def round_out(v, dtype):
    """Round fp32 to the stored dtype to nearest even; fp16 saturates at +-65504 (cvt.rn.satfinite)."""
    if dtype == torch.float16:
        return v.clamp(-F16_MAX, F16_MAX).to(torch.float16)
    return v.to(dtype)


# ---------------------------------------------------------------------------------------------------
# layouts the kernels read
# ---------------------------------------------------------------------------------------------------
def pad_channels(x, dtype):
    """(N, D, H, W, c) -> (N, D, H, W, pad32(c)) of ``dtype`` with zero channel padding."""
    c = x.shape[-1]
    cp = (c + 31) // 32 * 32
    out = torch.zeros(x.shape[:-1] + (cp,), dtype=dtype, device=x.device)
    out[..., :c] = x.to(dtype)
    return out


def to_s2d(t):
    """(N, D, H, W, C) -> the parity-planar space-to-depth layout (N, 8 = (pd, ph, pw), D/2, H/2, W/2, C)."""
    n, d, h, w, c = t.shape
    return t.view(n, d // 2, 2, h // 2, 2, w // 2, 2, c).permute(0, 2, 4, 6, 1, 3, 5, 7).reshape(
        n, 8, d // 2, h // 2, w // 2, c).contiguous()
