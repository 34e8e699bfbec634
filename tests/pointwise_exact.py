"""Exact references for the memory-bound kernels of csrc/pointwise.cuh and csrc/head_mma.cuh (test plumbing only).

Each function takes torch tensors on any device and restates, in float64 or exact integer arithmetic, what the kernel
source defines: where the kernel rounds to fp32 (an explicit ``fmaf``, a multiply, a cast from double) the reference
rounds at the same point, so the stored bits can be compared bit for bit. Tensors are channel-last (N, D, H, W, Cp)
with the padded channel count, per-(n, c) constants are (N, Cp) fp32, as the kernels take them.

* ``fma32``: a correctly rounded fp32 fused multiply-add (exact fp64 product, TwoSum, round-to-odd, one fp32 cast).
* ``drop_thresh`` / ``dropout_keep``: the host's 15-bit threshold and ``dropout_bits8`` / ``dropout_maskw``.
* ``act_fwd`` / ``pool_first_max`` / ``maxpool_bwd``: ``deferred_act8`` (the one definition of a block's activations),
  the max-pool's first-maximum rule and the routed (optionally accumulated) gradient.
* ``finalize``: ``stats_finalize_kernel`` / ``bn_stats_stage2_kernel``, term for term in float64.
* ``norm_bwd``: dz, S1, S2, c1, c2, dgamma, dbeta, dbias and dy of the norm / dropout / LeakyReLU backward, in float64.
"""
import torch

M32 = 0xFFFFFFFF
INSTANCE, BATCH_TRAIN, BATCH_EVAL, NONE = 0, 1, 2, 3      # ub_api.h UB_NORM_*


def f32(v, device=None):
    """The fp32 value of a Python float (what crosses the C ABI as ``float``), as a 0-d float32 tensor."""
    return torch.tensor(v, dtype=torch.float32, device=device)


# ---------------------------------------------------------------------------------------------------
# fp32 fused multiply-add
# ---------------------------------------------------------------------------------------------------
def fma32(a, b, c):
    """fp32 fma(a, b, c), correctly rounded to nearest even, for float32 tensors (broadcasting).

    The product of two fp32 values has at most 48 significant bits: exact in fp64. s = fl64(p + c) with its exact error
    e from TwoSum; when e != 0 the fp64 result is rounded to odd (moved one unit towards e if its last bit is even), which
    keeps the sticky information, so the single cast to fp32 (24 <= 53 - 2 bits) rounds as the exact sum would. The sign
    of an exact zero is IEEE's: x + (-x) = +0 under round-to-nearest, (-0) + (-0) = -0 -- fp64 and fp32 agree."""
    p = a.double() * b.double()
    cd = c.double()
    s = p + cd
    bb = s - p
    err = (p - (s - bb)) + (cd - bb)
    bits = s.view(torch.int64)
    even = (bits & 1) == 0
    toward_larger = (err > 0) == (s > 0)          # |s| grows when e has the sign of s
    adj = torch.where(toward_larger, torch.ones_like(bits), -torch.ones_like(bits))
    bits = torch.where((err != 0) & even, bits + adj, bits)
    return bits.view(torch.float64).float()


# ---------------------------------------------------------------------------------------------------
# dropout mask
# ---------------------------------------------------------------------------------------------------
def drop_thresh(p):
    """The host's 15-bit threshold: (uint32_t)(p * 32768.0f + 0.5f), clamped to 32767, p a C float."""
    t = int((f32(p) * f32(32768.0) + f32(0.5)).item())
    return min(t, 32767)


def _mul64(a, b):
    """(lo, hi) 32-bit halves of the 64-bit product of two uint32 values held in int64 tensors; every intermediate
    stays below 2^49 (b split into 16-bit halves)."""
    b0, b1 = b & 0xFFFF, b >> 16
    x0, x1 = a * b0, a * b1
    t = x0 + ((x1 & 0xFFFF) << 16)
    return t & M32, (t >> 32) + (x1 >> 16)


def _mulfold(a, b):
    lo, hi = _mul64(a, b)
    return lo ^ hi


def _rotr(x, r):
    return ((x >> r) | (x << (32 - r))) & M32


def dropout_bits(e0, seed):
    """dropout_bits8: the four 32-bit words u[0..3] of the vector whose first element index is e0 (int64 tensor,
    multiple of 8). seed: uint32 Python int."""
    e0 = e0.to(torch.int64)
    seed_t = torch.full_like(e0, seed & M32)
    idx = (e0 >> 3) & M32
    salt = seed_t ^ (((e0 >> 35) * 0x7FEB352D) & M32)
    m = _mulfold(idx ^ 0x9E3779B9, 0x85EBCA6B ^ (((salt << 1) | 1) & M32)) ^ salt
    lo0, hi0 = _mul64(m ^ 0xC2B2AE35, torch.full_like(m, 0x27D4EB2F))
    lo1, hi1 = _mul64(m ^ 0x165667B1, torch.full_like(m, 0x9E3779B1))
    q = _mulfold((m + 0x632BE5AB) & M32, torch.full_like(m, 0xD2B74407))
    return lo0 ^ q, hi0 ^ _rotr(q, 7), lo1 ^ _rotr(q, 13), hi1 ^ _rotr(q, 21)


def dropout_keep(elem_index, seed, p):
    """Keep decision of the elements with these global element indices (int64 tensor: n * D*H*W*Cp + voxel * Cp + c):
    element 2i / 2i+1 of its 8-element vector is kept when the low 15 bits of the low / high 16-bit lane of u[i] are
    >= drop_thresh(p). p == 0: everything is kept (the kernels skip the mask)."""
    e = elem_index.to(torch.int64)
    if p <= 0:
        return torch.ones_like(e, dtype=torch.bool)
    u = torch.stack(dropout_bits(e & ~7, seed), 0)
    lane = e & 7
    word = torch.gather(u, 0, (lane >> 1).unsqueeze(0)).squeeze(0)
    v = (word >> (16 * (lane & 1))) & 0x7FFF
    return v >= drop_thresh(p)


def element_index(shape, device, n0=0):
    """Global element indices of a (N, D, H, W, Cp) tensor, optionally of samples n0 .. n0+N-1 of a larger batch."""
    numel = 1
    for s in shape:
        numel *= s
    return torch.arange(numel, dtype=torch.int64, device=device).view(shape) + n0 * (numel // shape[0])


# ---------------------------------------------------------------------------------------------------
# forward: activations, pooling, max-pool backward
# ---------------------------------------------------------------------------------------------------
def fold_inv(p, device=None):
    """1 / (1 - p) in fp32 as the kernels form it (1.f / (1.f - p)); 1 without dropout."""
    if p <= 0:
        return f32(1.0, device)
    return f32(1.0, device) / (f32(1.0, device) - f32(p, device))


def folded_constants(scale, shift, p, n, cp, device):
    """(sc, sh): fl(scale * inv), fl(shift * inv) as (N, 1, 1, 1, Cp) fp32 (scale None: the identity)."""
    inv = fold_inv(p, device)
    if scale is None:
        scale = torch.ones((n, cp), dtype=torch.float32, device=device)
        shift = torch.zeros((n, cp), dtype=torch.float32, device=device)
    sc = (scale.float() * inv).view(n, 1, 1, 1, cp)
    sh = (shift.float() * inv).view(n, 1, 1, 1, cp)
    return sc, sh


def pre_activation(y, scale, shift, p):
    """fmaf(y, sc, sh): the fp32 value whose sign every forward and backward pass takes."""
    n, cp = y.shape[0], y.shape[-1]
    sc, sh = folded_constants(scale, shift, p, n, cp, y.device)
    return fma32(y.float(), sc, sh)


def leaky(hi, slope):
    """max(hi, fl(hi * slope)) for slope <= 1, else the select (the kernels' two forms)."""
    lo = hi * f32(slope, hi.device)
    return torch.maximum(hi, lo) if slope <= 1 else torch.where(hi > 0, hi, lo)


def act_fwd(y, scale, shift, slope, p=0.0, seed=0, n0=0):
    """deferred_act8 over a (N, D, H, W, Cp) fp16 tensor -> (a bf16, a16 fp16): fp32 x = LeakyReLU(fmaf(y, sc, sh)),
    a = RNE bf16(x), a16 = saturating RNE fp16(x), dropped elements cleared to +0 in both. ``n0``: index of the first
    sample in the batch the dropout counter runs over."""
    x = leaky(pre_activation(y, scale, shift, p), slope)
    a = x.to(torch.bfloat16)
    a16 = x.clamp(-65504.0, 65504.0).to(torch.float16)
    if p > 0:
        keep = dropout_keep(element_index(tuple(y.shape), y.device, n0), seed, p)
        a = torch.where(keep, a, torch.zeros_like(a))
        a16 = torch.where(keep, a16, torch.zeros_like(a16))
    return a, a16


def _windows(t):
    """(N, D, H, W, C) -> (N, D/2, H/2, W/2, C, 8), window index j = 4 jd + 2 jh + jw (the kernels' scan order)."""
    n, d, h, w, c = t.shape
    return t.view(n, d // 2, 2, h // 2, 2, w // 2, 2, c).permute(0, 1, 3, 5, 7, 2, 4, 6).reshape(
        n, d // 2, h // 2, w // 2, c, 8)


def _unwindows(t):
    n, dp, hp, wp, c, _ = t.shape
    return t.view(n, dp, hp, wp, c, 2, 2, 2).permute(0, 1, 5, 2, 6, 3, 7, 4).reshape(n, 2 * dp, 2 * hp, 2 * wp, c)


def pool_first_max(a, last=False):
    """-> (pooled bf16, arg int64 (N, D/2, H/2, W/2, C)): the first maximum of each 2x2x2 window under a strict ``>``
    in (d, h, w) order, starting from -inf; the pooled value carries that element's bits (the sign of a zero included).
    ``last``: the last maximum instead (a planted error for the tests)."""
    v = _windows(a)
    vf = v.float()
    is_max = vf == vf.max(-1, keepdim=True).values
    j = torch.arange(8, device=a.device)
    arg = torch.where(is_max, j, -1).max(-1).values if last else torch.where(is_max, j, 8).min(-1).values
    pooled = torch.gather(v, -1, arg.unsqueeze(-1)).squeeze(-1)
    return pooled, arg


def maxpool_bwd(a, dP, dA=None, last=False):
    """Route dP to the first maximum of each window of ``a``: o = (dA if accumulating else 0) + (routed ? g : 0) in fp32,
    rounded to bf16 (so an unrouted -0 of dA becomes +0, as the kernel's fp32 add makes it)."""
    _, arg = pool_first_max(a, last)
    j = torch.arange(8, device=a.device)
    g = torch.where(arg.unsqueeze(-1) == j, dP.float().unsqueeze(-1), torch.zeros((), device=a.device))
    base = _windows(dA).float() if dA is not None else torch.zeros_like(g)
    return _unwindows((base + g).to(torch.bfloat16))


# ---------------------------------------------------------------------------------------------------
# statistics finalisation
# ---------------------------------------------------------------------------------------------------
def finalize(s, q, count_per_sample, gamma, beta, eps, mode, momentum=0.1, running_mean=None, running_var=None,
             unbiased_norm=False):
    """stats_finalize_kernel / bn_stats_stage2_kernel in float64. s, q: (N, Cp) float64 sums of the records of each
    sample (exact: the tests feed integer-valued records); gamma, beta: (C,) fp32; eps, momentum: Python floats that
    cross the ABI as fp32. -> dict of float64 (N, Cp) scale, shift, mean, rstd and, in train-mode BatchNorm with
    buffers, the (C,) running_mean / running_var the kernel stores. ``unbiased_norm``: normalise with the unbiased
    variance (a planted error for the tests)."""
    n, cp = s.shape
    c = gamma.shape[0]
    dev = s.device
    eps64 = f32(eps, dev).double()
    mom64 = f32(momentum, dev).double()
    g = torch.zeros(cp, dtype=torch.float64, device=dev)
    b = torch.zeros(cp, dtype=torch.float64, device=dev)
    g[:c], b[:c] = gamma.double(), beta.double()
    out = {}
    if mode == BATCH_EVAL:
        mean = torch.zeros(cp, dtype=torch.float64, device=dev)
        var = torch.ones(cp, dtype=torch.float64, device=dev)
        mean[:c], var[:c] = running_mean.double(), running_var.double()
        mean, var = mean.expand(n, cp), var.expand(n, cp)
    else:
        cnt = float(count_per_sample) * (1 if mode == INSTANCE else n)
        if mode == BATCH_TRAIN:
            s, q = s.sum(0, keepdim=True).expand(n, cp), q.sum(0, keepdim=True).expand(n, cp)
        mean = s / cnt
        var = (q / cnt - mean * mean).clamp_min(0.0)
        if unbiased_norm and cnt > 1:
            var = var * cnt / (cnt - 1.0)
        if mode == BATCH_TRAIN and running_mean is not None:
            unbiased = var[0, :c] * cnt / (cnt - 1.0) if cnt > 1 else var[0, :c]
            out["running_mean"] = (1.0 - mom64) * running_mean.double() + mom64 * mean[0, :c]
            out["running_var"] = (1.0 - mom64) * running_var.double() + mom64 * unbiased
    rstd = 1.0 / torch.sqrt(var + eps64)
    out["scale"] = g * rstd
    out["shift"] = b - mean * g * rstd
    out["mean"] = mean.clone()
    out["rstd"] = rstd
    return out


# ---------------------------------------------------------------------------------------------------
# norm / dropout / LeakyReLU backward
# ---------------------------------------------------------------------------------------------------
def dz_of(dA, y, scale, shift, slope, p, seed, n0=0, from_a=None, ge=False):
    """float64 dz = dA * keep * (pre-activation > 0 ? inv : fl(slope * inv)) (the fp32 factors of the kernels, the
    product unrounded). The sign is that of fmaf(y, sc, sh) (folded constants), or with ``from_a`` (mode NONE) that of
    the stored activation. ``ge``: ``>=`` instead of ``>`` in the sign test (a planted error for the tests)."""
    dev = dA.device
    inv = fold_inv(p, dev)
    sinv = f32(slope, dev) * inv
    pre = from_a.float() if from_a is not None else pre_activation(y, scale, shift, p)
    pos = pre >= 0 if ge else pre > 0
    fac = torch.where(pos, inv, sinv).double()
    dz = dA.double() * fac
    if p > 0:
        dz = torch.where(dropout_keep(element_index(tuple(dA.shape), dev, n0), seed, p), dz, torch.zeros_like(dz))
    return dz


def norm_bwd(dA, y, mode, mean, rstd, scale, shift, slope, p, seed, c, n0=0, dz=None, zero_c2=False):
    """The backward of (norm -> dropout -> LeakyReLU) in float64 from the kernels' fp32 inputs. mean, rstd, scale
    (= gamma * rstd), shift: (N, Cp) fp32. -> dict: dz, xhat, S1, S2 ((N, Cp) per sample), c1, c2, dgamma, dbeta,
    dbias ((C,)) and dy, with
      S1 = sum dz, S2 = sum dz * xhat, xhat = (y - mean) * rstd         (sums over the voxels of a sample)
      c1 = S1 / cnt, c2 = S2 / cnt       (InstanceNorm: per sample; train BatchNorm: over the batch; eval: 0)
      dgamma = sum_n S2, dbeta = sum_n S1, dbias = gscale * sum_n S1 in eval BatchNorm, else 0
      dy = gscale * (dz - c1 - xhat * c2).
    ``zero_c2``: c2 = 0 (a planted error for the tests)."""
    n, cp = dA.shape[0], dA.shape[-1]
    vox = dA[0, ..., 0].numel()
    if dz is None:
        dz = dz_of(dA, y, scale, shift, slope, p, seed, n0)
    v = lambda t: t.double().view(n, 1, 1, 1, cp)
    xhat = (y.double() - v(mean)) * v(rstd)
    s1 = dz.sum((1, 2, 3))
    s2 = (dz * xhat).sum((1, 2, 3))
    if mode == INSTANCE:
        c1, c2 = s1 / vox, s2 / vox
    elif mode == BATCH_TRAIN:
        c1 = (s1.sum(0, keepdim=True) / (vox * n)).expand(n, cp)
        c2 = (s2.sum(0, keepdim=True) / (vox * n)).expand(n, cp)
    else:
        c1 = c2 = torch.zeros_like(s1)
    if zero_c2:
        c2 = torch.zeros_like(c2)
    g = scale.double()
    dy = v(g) * (dz - v(c1) - xhat * v(c2))
    dbias = g[0, :c] * s1.sum(0)[:c] if mode == BATCH_EVAL else torch.zeros(c, dtype=torch.float64, device=dA.device)
    return {"dz": dz, "xhat": xhat, "S1": s1, "S2": s2, "c1": c1, "c2": c2, "dgamma": s2.sum(0)[:c],
            "dbeta": s1.sum(0)[:c], "dbias": dbias, "dy": dy}


# ---------------------------------------------------------------------------------------------------
# comparison helpers
# ---------------------------------------------------------------------------------------------------
def bits(t):
    """Bit patterns of a tensor (int16 / int32 view): torch.equal on values treats -0 and +0 as equal."""
    return t.contiguous().view({2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


def bit_mismatch(what, got, want):
    """None when got and want are bit-identical, else a description of the first difference."""
    gb, wb = bits(got), bits(want.to(got.dtype))
    if torch.equal(gb, wb):
        return None
    bad = (gb != wb).nonzero()
    i = tuple(bad[0].tolist())
    return (f"{what}: {bad.shape[0]} of {gb.numel()} differ in bits, first at {i}: {got[i].item()!r} vs "
            f"{want.to(got.dtype)[i].item()!r}")


def _neighbours(r, mant_bits):
    """(lo, hi, mid) float64: the two values of a binary format with ``mant_bits`` significant bits around r (r itself
    when representable), and their midpoint. Normal range only (|r| >= 2^-120 or r == 0)."""
    m, e = torch.frexp(r)
    ulp = torch.ldexp(torch.ones_like(r), e.to(torch.int32) - mant_bits)
    lo = torch.floor(r / ulp) * ulp
    hi = lo + ulp
    return lo, hi, lo + ulp / 2


def fp32_rounding_mismatch(what, got, ref64, rel_slack=2.0 ** -50):
    """got (fp32) must equal RNE fp32(ref64) bit for bit, except where ref64 lies within ``rel_slack`` |ref64| of a
    midpoint between two fp32 values (the float64 restatement and the kernel's float64 may differ in their last bits:
    contraction of a * b + c into one fma), and there got must be one of the two neighbours. -> (failure | None,
    number of elements that needed the midpoint exception)."""
    want = ref64.float()
    same = bits(got) == bits(want)
    if bool(same.all()):
        return None, 0
    lo, hi, mid = _neighbours(ref64, 24)
    near = (ref64 - mid).abs() <= rel_slack * ref64.abs()
    g = got.double()
    ok = same | (near & ((g == lo) | (g == hi)))
    if not bool(ok.all()):
        i = tuple((~ok).nonzero()[0].tolist())
        return (f"{what}: {int((~ok).sum())} of {got.numel()} differ, first at {i}: {got[i].item()!r} vs "
                f"{ref64[i].item()!r} (not an fp32 midpoint)"), 0
    return None, int((~same).sum())


def rne_bf16(r):
    """Round float64 to the nearest bf16 value, ties to even, directly (no double rounding through fp32); float64."""
    lo, hi, mid = _neighbours(r, 8)
    lo_even = (torch.frexp(lo)[0].abs() * 2.0 ** 8).remainder(2) == 0
    out = torch.where(r < mid, lo, torch.where(r > mid, hi, torch.where(lo_even, lo, hi)))
    return torch.where(r == lo, lo, out)


def bf16_near_midpoint_check(got, ref64, tol):
    """The criterion of a bf16 output computed in fp32 with compiler-contractable steps: the kernel's fp32 value lies
    within ``tol`` (a float64 tensor: the fp32 error bound of the computation) of the float64 value r, so the stored bf16
    must be the round-to-nearest-even of some value in [r - tol, r + tol]: RNE(r - tol) <= got <= RNE(r + tol) (RNE is
    monotone). Where tol is below half a bf16 unit that is RNE(r) itself, except where r lies within tol of a bf16
    midpoint, where it is one of r's two bf16 neighbours. Values are compared (a zero's sign is not specified by a
    bound). -> (number of violations, number of elements whose interval holds two or more bf16 values, first
    violation index)."""
    lo, hi = rne_bf16(ref64 - tol), rne_bf16(ref64 + tol)
    g = got.double()
    ok = (g >= lo) & (g <= hi)
    near = lo != hi
    bad = (~ok).nonzero()
    first = tuple(bad[0].tolist()) if bad.shape[0] else None
    return int(bad.shape[0]), int(near.sum()), first


# ---------------------------------------------------------------------------------------------------
# the comparisons the GPU suite applies (kernel output against the reference); each returns a list of failures
# ---------------------------------------------------------------------------------------------------
def check_act_fwd(y, scale, shift, slope, p, seed, c, a=None, a16=None, pooled=None, n0=0):
    """ub_norm_act_fwd outputs against ``act_fwd`` / ``pool_first_max``: bit for bit, padded channels +0."""
    ra, ra16 = act_fwd(y, scale, shift, slope, p, seed, n0)
    fails = []
    for what, got, want in (("a", a, ra), ("a16", a16, ra16)):
        if got is not None:
            fails.append(bit_mismatch(what, got, want))
            fails.append(bit_mismatch(f"{what} padded channels", got[..., c:], torch.zeros_like(got[..., c:])))
    if pooled is not None:
        fails.append(bit_mismatch("pooled", pooled, pool_first_max(ra)[0]))
    return [f for f in fails if f]


def check_maxpool_bwd(a, dP, dA_in, got):
    """ub_maxpool_bwd against ``maxpool_bwd`` on the (materialised or recomputed) bf16 activations ``a``: bit for bit."""
    f = bit_mismatch("maxpool_bwd dA", got, maxpool_bwd(a, dP, dA_in))
    return [f] if f else []


def check_finalize(got, ref, c, mode):
    """ub_norm_finalize outputs ((N, Cp) fp32 scale, shift, mean, rstd; (C,) running statistics) against ``finalize``:
    the float64 restatement cast to fp32, bit for bit; a difference is accepted only at an fp32 midpoint of the
    float64 value (reported). -> (failures, midpoint count)."""
    fails, mids = [], 0
    keys = ["scale", "shift", "mean", "rstd"] + (["running_mean", "running_var"] if "running_mean" in ref else [])
    for k in keys:
        f, m = fp32_rounding_mismatch(k, got[k], ref[k])
        mids += m
        if f:
            fails.append(f)
    return fails, mids


def ref_bwd_none(dA, a, slope, p, seed, n0=0, ge=False):
    """mode NONE (a conv with the LeakyReLU fused, no norm): dy = bf16(fl32(dA * keep * (a > 0 ? inv : fl(slope inv))))
    -- one fp32 multiply, then the bf16 rounding; a dropped element gives +0."""
    dev = dA.device
    inv = fold_inv(p, dev)
    fac = torch.where(a.float() >= 0 if ge else a.float() > 0, inv, f32(slope, dev) * inv)
    da = dA.float()
    if p > 0:
        da = torch.where(dropout_keep(element_index(tuple(dA.shape), dev, n0), seed, p), da, torch.zeros_like(da))
    return (da * fac).to(torch.bfloat16)


def check_bwd_none(dA, a, slope, p, seed, got):
    f = bit_mismatch("norm_act_bwd (mode NONE) dy", got, ref_bwd_none(dA, a, slope, p, seed))
    return [f] if f else []


def apply_tolerance(ref, y, mean, rstd, scale, chain):
    """First-order fp32 error bound of the apply pass o = fmaf(ka, dz, fmaf(kc, y, kb)) against the float64 dy:
      ka = g (exact), kc = fl(fl(-g r) c2) (2 roundings), kb = -g c1 - kc m (<= 2 roundings, contractable),
      c1, c2 = fp32 casts of S1 / cnt, S2 / cnt whose sums carry <= ``chain`` roundings relative to their (non-negative)
      terms; dz = fl(dA * factor) (1 rounding), the inner and the outer fma (1 each).
    -> 2^-24 (2 |ka dz| + (chain + 6) (|kc y| + |kc m| + |g c1|)) with 1 % slack, float64 of dy's shape. The outer fma's
    own rounding is covered by the first term's second unit (|o| <= |ka dz| + the rest)."""
    n, cp = y.shape[0], y.shape[-1]
    v = lambda t: t.double().view(n, 1, 1, 1, cp)
    g, r, m = v(scale), v(rstd), v(mean)
    kc = (g * r * v(ref["c2"])).abs()
    rest = kc * y.double().abs() + kc * m.abs() + (g * v(ref["c1"])).abs()
    return 1.01 * 2.0 ** -24 * (2 * (g * ref["dz"]).abs() + (chain + 6) * rest)


def check_dy(got, ref, y, mean, rstd, scale, chain, c, what="dy"):
    """``got`` (bf16 dy of a norm backward) against ref["dy"] (float64) with ``bf16_near_midpoint_check`` under
    ``apply_tolerance``; padded channels must be zero. -> (failures, near-midpoint count)."""
    tol = apply_tolerance(ref, y, mean, rstd, scale, chain)
    nbad, near, first = bf16_near_midpoint_check(got[..., :c], ref["dy"][..., :c], tol[..., :c])
    fails = []
    if nbad:
        fails.append(f"{what}: {nbad} of {got[..., :c].numel()} elements outside the rounding of [dy - tol, dy + tol], "
                     f"first at {first}: {got[first].item()!r} vs {ref['dy'][first].item()!r}, tol {tol[first].item():.3g}")
    if not bool((got[..., c:].float() == 0).all()):      # +0 or -0: gscale = 0 there
        fails.append(f"{what}: nonzero padded channels")
    return fails, near
