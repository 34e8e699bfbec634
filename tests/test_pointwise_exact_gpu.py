"""Exact tests of the memory-bound kernels (norm statistics, norm + dropout + LeakyReLU (+ max-pool) forward, the norm
backward, max-pool backward, bias column sums, the warp-MMA output head) at the training step's own shapes.

The census: one GanTrainer step (config 2: bssfp, 8 x 128^3) runs with recording wrappers around ``ops.norm_finalize``,
``ops.norm_act_fwd``, ``ops.norm_act_bwd``, ``ops.maxpool_bwd``, ``ops.colsum``, ``ops.conv1x1_to_ncdhw`` and
``ops.head_bwd_fused``; every distinct call is rerun at its real shape against tests/pointwise_exact.py. Which criterion
applies to which output, and why it is sound:

* bit for bit (bit patterns, so -0 != +0): the forward activations, their fp16 copy and the pooled values (the
  reference restates deferred_act8's explicit fmaf, the fp32 multiply and the RNE casts); the max-pool backward (fp32
  add of two bf16 values, RNE); the mode-NONE backward (one fp32 multiply, RNE); ``norm_finalize`` fed integer-valued
  records (its fp64 sums are then exact in any order; the rest is a float64 formula cast to fp32, where only a value at
  an fp32 midpoint may differ, and is shown to be one); ``colsum`` with sparse integer operands below 2^22 units.
* a derived first-order fp32 bound, with sensitivity (every partial record exceeds it): the norm backward's sums S1 / S2
  (through dgamma / dbeta), the output head's weight gradient and its block sums; the output head's forward, whose
  bound must also be beaten by the error of dropping the ``lo`` term of its hi + mid + lo weight split.
* the RNE bf16 of a value within the fp32 bound of the float64 value (where the bound is below half a bf16 unit: the
  RNE of the float64 value, or one of its two neighbours near a midpoint): the dy of the norm backward (``ka / kb /
  kc`` are compiler-contractable) and of the fused head backward. The count of elements whose band holds two bf16
  values is printed; it is asserted small where c1 / c2 are known to one rounding (external records).

The default step materialises every pooled block, so the pooled-only forward and the max-pool backward on a deferred
source are added beside the census at the step's shape (SYNTHETIC).
"""
from collections import namedtuple

import pytest
import torch

from tests import pointwise_exact as R
from tests.conv_exact import check_exact_bound, granularity, int_operand
from tests.step_census import run_step

pytestmark = pytest.mark.gpu
DEV = "cuda"

Fwd = namedtuple("Fwd", "n d h w cp c slope p pool materialize f16")
Fin = namedtuple("Fin", "n cp c mode tiles voxels running")
Bwd = namedtuple("Bwd", "n d h w cp c mode slope p records")           # records: per sample of partial= (0: none)
PoolB = namedtuple("PoolB", "n d h w cp deferred acc slope p")
Col = namedtuple("Col", "rows cp c")
HeadF = namedtuple("HeadF", "n d h w co ci deferred slope p")
HeadB = namedtuple("HeadB", "n d h w co ci mode c slope p")
NAMES = {Fwd: "norm_act_fwd", Fin: "norm_finalize", Bwd: "norm_act_bwd", PoolB: "maxpool_bwd", Col: "colsum",
         HeadF: "conv1x1_to_ncdhw", HeadB: "head_bwd_fused"}


def _ops():
    from unet_bssfp_b200 import ops
    return ops


def record_census(modality, batch, size):
    """One GanTrainer step with recording wrappers -> sorted list of distinct entries (namedtuples above)."""
    ops = _ops()
    seen = set()

    def finalize(f0):
        def w(stats, n, voxels, cp, c, gamma, beta, eps, mode, momentum=0.1, running_mean=None, running_var=None):
            tiles = 0 if stats is None else stats.shape[0] // n
            seen.add(Fin(n, cp, c, mode, tiles, int(voxels), running_mean is not None))
            return f0(stats, n, voxels, cp, c, gamma, beta, eps, mode, momentum, running_mean, running_var)
        return w

    def act_fwd(f0):
        def w(y, scale, shift, slope, drop_p=0.0, drop_seed=0, pool=False, materialize=True, f16_copy=False):
            seen.add(Fwd(*y.shape[:4], y.shape[4], y.shape[4], float(slope), float(drop_p), bool(pool),
                         bool(materialize), bool(f16_copy)))
            return f0(y, scale, shift, slope, drop_p, drop_seed, pool=pool, materialize=materialize, f16_copy=f16_copy)
        return w

    def act_bwd(f0):
        def w(dA, a, y, mode, mean, rstd, scale, slope, drop_p, drop_seed, c, want_param_grads=True,
              want_bias_grad=True, shift=None, partial=None):
            recs = 0 if partial is None else partial.shape[0] // dA.shape[0]
            seen.add(Bwd(*dA.shape, c, mode, float(slope), float(drop_p), recs))
            return f0(dA, a, y, mode, mean, rstd, scale, slope, drop_p, drop_seed, c, want_param_grads,
                      want_bias_grad, shift=shift, partial=partial)
        return w

    def pool_bwd(f0):
        def w(a, dP, dA=None):
            d = isinstance(a, ops.DeferredAct)
            seen.add(PoolB(*a.shape, d, dA is not None, float(a.slope) if d else 0.0, float(a.drop_p) if d else 0.0))
            return f0(a, dP, dA)
        return w

    def colsum(f0):
        def w(x, c):
            seen.add(Col(x.numel() // x.shape[-1], x.shape[-1], c))
            return f0(x, c)
        return w

    def head_fwd(f0):
        def w(u, weight, bias):
            d = isinstance(u, ops.DeferredAct)
            seen.add(HeadF(*u.shape[:4], weight.shape[0], weight.shape[1], d, float(u.slope) if d else 0.0,
                           float(u.drop_p) if d else 0.0))
            return f0(u, weight, bias)
        return w

    def head_bwd(f0):
        def w(dout, fuse, weight, mode, c, need_params=True, want_block_grads=True):
            seen.add(HeadB(*fuse.y.shape[:4], weight.shape[0], weight.shape[1], mode, c, float(fuse.slope),
                           float(fuse.drop_p)))
            return f0(dout, fuse, weight, mode, c, need_params, want_block_grads)
        return w

    run_step(modality, batch, size, {"norm_finalize": finalize, "norm_act_fwd": act_fwd, "norm_act_bwd": act_bwd,
                                     "maxpool_bwd": pool_bwd, "colsum": colsum, "conv1x1_to_ncdhw": head_fwd,
                                     "head_bwd_fused": head_bwd})
    order = list(NAMES)
    return sorted(seen, key=lambda e: (order.index(type(e)), tuple(str(v) for v in e)))


@pytest.fixture(scope="module")
def census():
    return record_census("bssfp", 8, 128)


def _label(e):
    return f"{NAMES[type(e)]}{tuple(e)}"


# ---------------------------------------------------------------------------------------------------
# operands
# ---------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _nextafter32(x, k):
    """x moved k fp32 units (k may be negative; same sign region)."""
    b = x.view(torch.int32) + torch.where(x >= 0, k, -k).to(torch.int32)
    return b.view(torch.float32)


def constants_with_zero_preactivation(n, cp, c, p, g, positive=False, narrow=False):
    """(scale, shift, y0): per-(n, c) fp32 constants, all different, and a power of two y0 (fp16-exact) per (n, c) with
    fmaf(y0, sc, sh) == 0 exactly for the folded sc = fl(scale inv), sh = fl(shift inv). A quarter of the channels have
    shift = -0 (there y0 = +-0, and y = +-0 gives pre-activations of +0 or -0). Padded channels: scale = shift = 0.
    ``positive``: scale > 0 and y0 > 0 (then shift < 0). ``narrow``: scale in [0.9, 1.1) (samples of similar weight)."""
    inv = R.fold_inv(p, DEV)
    scale = torch.rand((n, cp), device=DEV, generator=g) * (0.2 if narrow else 1.5) + (0.9 if narrow else 0.25)
    shift = (torch.rand((n, cp), device=DEV, generator=g) * 0.8 + 0.1) * (-1 if positive else
                                                                          torch.where(torch.rand((n, cp), device=DEV, generator=g) < 0.5, -1.0, 1.0))
    if not positive:
        scale = scale * torch.where(torch.rand((n, cp), device=DEV, generator=g) < 0.2, -1.0, 1.0)
    k = torch.randint(-3, 3, (n, cp), device=DEV, generator=g).float()
    if narrow:      # |shift| = |scale| 2^k: the search below then keeps scale at its start, in [0.9, 1.1)
        shift = torch.sign(shift) * scale.abs() * torch.exp2(k)
    todo = torch.ones((n, cp), dtype=torch.bool, device=DEV)
    y0 = torch.zeros((n, cp), device=DEV)
    for _ in range(64):
        sh = shift * inv
        sc_sign = torch.sign(scale)
        y0_try = -torch.sign(sh) * sc_sign * torch.exp2(k)           # sc = -sh / y0 keeps the sign of scale
        target = -sh / y0_try                                        # exact: division by a power of two
        base = target / inv
        found = torch.zeros_like(todo)
        for dk in (0, -1, 1, -2, 2):
            cand = _nextafter32(base, dk)
            ok = (cand * inv == target) & ~found & todo
            scale = torch.where(ok, cand, scale)
            y0 = torch.where(ok, y0_try, y0)
            found |= ok
        todo &= ~found
        if not bool(todo.any()):
            break
        shift = torch.where(todo, _nextafter32(shift, 1), shift)
    assert not bool(todo.any())
    negz = torch.rand((n, cp), device=DEV, generator=g) < 0.25
    if positive:
        negz[:] = False
    shift = torch.where(negz, torch.full_like(shift, -0.0), shift)
    y0 = torch.where(negz, torch.zeros_like(y0), y0)
    scale[:, c:] = 0.0
    shift[:, c:] = 0.0
    y0[:, c:] = 0.0
    assert bool((R.fma32(y0.to(torch.float16).float(), scale * inv, shift * inv) == 0).all())
    return scale.contiguous(), shift.contiguous(), y0


def special_y(shape, y0, g, positive=False):
    """fp16 y (N, D, H, W, Cp) for sample-wise use: N(0, 2) values, a small discrete set (ties inside pooling windows),
    and the edges: +-65504 (saturated), +-0, fp16 subnormals and y0 (exact zero pre-activation) per (n, c).
    ``positive``: |values| + 2^-10 instead, y0 kept, no negative edges."""
    n, cp = shape[0], shape[-1]
    y = torch.randn(shape, device=DEV, generator=g) * 2.0
    sel = torch.rand(shape, device=DEV, generator=g)
    disc = torch.tensor([-2.0, -1.0, 1.0, 2.0], device=DEV)[torch.randint(0, 4, shape, device=DEV, generator=g)]
    sub = torch.randint(1, 1024, shape, device=DEV, generator=g).float() * 2.0 ** -24
    sgn = torch.where(torch.rand(shape, device=DEV, generator=g) < 0.5, -1.0, 1.0)
    y0b = y0.view(n, 1, 1, 1, cp).expand(shape)
    if positive:
        y = y.abs() + 2.0 ** -10
        y = torch.where(sel < 0.01, sub, y)
        y = torch.where((sel >= 0.01) & (sel < 0.03), y0b, y)
        return y.to(torch.float16)
    y = torch.where(sel < 0.15, disc, y)
    y = torch.where((sel >= 0.15) & (sel < 0.16), sgn * 65504.0, y)
    y = torch.where((sel >= 0.16) & (sel < 0.18), sgn * 0.0, y)
    y = torch.where((sel >= 0.18) & (sel < 0.20), sgn * sub, y)
    y = torch.where((sel >= 0.20) & (sel < 0.23), y0b, y)
    return y.to(torch.float16)


def bf16_operand(shape, g, neg_zero=True):
    """Random bf16 values with -0 and +0 among them."""
    t = (torch.randn(shape, device=DEV, generator=g) * 1.5).to(torch.bfloat16)
    z = torch.rand(shape, device=DEV, generator=g)
    t = torch.where(z < 0.03, torch.zeros((), dtype=torch.bfloat16, device=DEV), t)
    if neg_zero:
        t = torch.where((z >= 0.03) & (z < 0.06), torch.full((), -0.0, dtype=torch.bfloat16, device=DEV), t)
    return t


# ---------------------------------------------------------------------------------------------------
# bit-exact: forward, max-pool backward, mode-NONE backward, finalize, colsum
# ---------------------------------------------------------------------------------------------------
SEED = 0x9E3779B1            # bit 31 set: exercises the seed's full 32 bits


def run_fwd(e, seed=5):
    ops = _ops()
    g = _gen(seed)
    c = e.c
    scale, shift, y0 = constants_with_zero_preactivation(e.n, e.cp, c, e.p, g)
    y = special_y((e.n, e.d, e.h, e.w, e.cp), y0, g)
    y[..., c:] = 0
    res = ops.norm_act_fwd(y, scale, shift, e.slope, e.p, SEED, pool=e.pool, materialize=e.materialize,
                           f16_copy=e.f16)
    a, pooled = res[0], res[1]
    a16 = res[2] if e.f16 else None
    fails = []
    for i in range(e.n):
        s = slice(i, i + 1)
        fails += [f"sample {i}: {f}" for f in R.check_act_fwd(
            y[s], scale[s], shift[s], e.slope, e.p, SEED, c, a=None if a is None else a[s],
            a16=None if a16 is None else a16[s], pooled=None if pooled is None else pooled[s], n0=i)]
    return fails


def run_pool_bwd(e, seed=6):
    ops = _ops()
    g = _gen(seed)
    scale, shift, y0 = constants_with_zero_preactivation(e.n, e.cp, e.cp, e.p, g)
    y = special_y((e.n, e.d, e.h, e.w, e.cp), y0, g)
    a = torch.cat([R.act_fwd(y[i:i + 1], scale[i:i + 1], shift[i:i + 1], e.slope, e.p, SEED, i)[0]
                   for i in range(e.n)])
    dP = bf16_operand((e.n, e.d // 2, e.h // 2, e.w // 2, e.cp), g)
    base = bf16_operand(tuple(a.shape), g) if e.acc else None
    src = ops.DeferredAct(y, scale, shift, e.slope, e.p, SEED) if e.deferred else a
    got = ops.maxpool_bwd(src, dP, base.clone() if e.acc else None)
    fails = []
    for i in range(e.n):
        s = slice(i, i + 1)
        fails += [f"sample {i}: {f}" for f in R.check_maxpool_bwd(a[s], dP[s], None if base is None else base[s], got[s])]
    return fails


def run_bwd_none(e, seed=7):
    ops = _ops()
    g = _gen(seed)
    shape = (e.n, e.d, e.h, e.w, e.cp)
    fails = []
    for p in sorted({e.p, 0.05}):
        a = bf16_operand(shape, g)
        dA = bf16_operand(shape, g)
        dy, *_ = ops.norm_act_bwd(dA, a, None, R.NONE, None, None, None, e.slope, p, SEED, e.c)
        for i in range(e.n):
            s = slice(i, i + 1)
            want = R.ref_bwd_none(dA[s], a[s], e.slope, p, SEED, n0=i)
            f = R.bit_mismatch(f"p={p} sample {i} dy", dy[s], want)
            if f:
                fails.append(f)
    return fails


def run_finalize(e, seed=8):
    """Integer-valued records: every fp64 sum of the kernels is exact whatever its order."""
    ops = _ops()
    g = _gen(seed)
    n, cp, c = e.n, e.cp, e.c
    tiles = max(e.tiles, 1)
    stats = torch.zeros((n * tiles, 2, cp), device=DEV)
    stats[:, 0, :c] = torch.randint(-256, 257, (n * tiles, c), device=DEV, generator=g).float()
    stats[:, 1, :c] = torch.randint(0, 1 << 16, (n * tiles, c), device=DEV, generator=g).float() + float(2 * e.voxels // tiles)
    gamma = torch.rand(c, device=DEV, generator=g) + 0.5
    beta = torch.randn(c, device=DEV, generator=g) * 0.3
    rm = torch.randn(c, device=DEV, generator=g) * 0.2
    rv = torch.rand(c, device=DEV, generator=g) + 0.5
    eps, mom = 1e-5, 0.1
    has_run = e.mode != R.INSTANCE          # train BatchNorm: also the running-statistics update
    rm_k, rv_k = (rm.clone(), rv.clone()) if has_run else (None, None)
    st = None if e.mode == R.BATCH_EVAL else stats
    scale, shift, mean, rstd = ops.norm_finalize(st, n, e.voxels, cp, c, gamma, beta, eps, e.mode, mom, rm_k, rv_k)
    rec = stats.double().view(n, tiles, 2, cp).sum(1)
    ref = R.finalize(rec[:, 0], rec[:, 1], e.voxels, gamma, beta, eps, e.mode, mom, rm if has_run else None,
                     rv if has_run else None)
    got = {"scale": scale, "shift": shift, "mean": mean, "rstd": rstd}
    if "running_mean" in ref:
        got.update(running_mean=rm_k, running_var=rv_k)
    fails, mids = R.check_finalize(got, ref, c, e.mode)
    if mids:
        print(f"  {_label(e)}: {mids} value(s) at an fp32 midpoint of the float64 result")
    return fails


def run_colsum(e, seed=9):
    ops = _ops()
    g = _gen(seed)
    dens = min(0.5, 2.0 ** 20 / (e.rows * 1.5))
    x = int_operand((e.rows, e.c), dens, [-2, -1, 1, 2], g, DEV)
    xp = torch.zeros((e.rows, e.cp), dtype=torch.bfloat16, device=DEV)
    xp[:, :e.c] = x.to(torch.bfloat16)
    got = ops.colsum(xp, e.c)
    check_exact_bound(x.abs().double().sum(0), granularity(x), "sum |dy|")
    f = R.bit_mismatch("colsum", got, x.double().sum(0).float())
    return [f] if f else []


# ---------------------------------------------------------------------------------------------------
# bounds: the norm backward's reduction and apply passes
# ---------------------------------------------------------------------------------------------------
def _reduce_plan(n, cp, vox):
    """ub_norm_act_bwd's reduce launch: (blocks per sample, threads, vps)."""
    c8 = cp // 8
    vps = vox * c8
    bps_max = max(128, (1184 + n - 1) // n)
    threads = max(256, cp)
    bps = bps_max
    if bps * threads * 4 > vps:
        bps = max(1, (vps + 4 * threads - 1) // (4 * threads))
    return bps, threads, vps


def reduce_records(t, bps, threads):
    """The per-block records of norm_act_bwd_reduce_kernel for one sample: t (1, D, H, W, Cp) float64 terms ->
    (bps, Cp) sums. Block b, thread x takes vectors idx = b * threads + x + k * (bps * threads)."""
    cp = t.shape[-1]
    v = t.reshape(-1, 8)
    stride = bps * threads
    rounds = -(-v.shape[0] // stride)
    pad = torch.zeros((rounds * stride - v.shape[0], 8), dtype=t.dtype, device=t.device)
    v = torch.cat([v, pad]).view(rounds, bps, threads // (cp // 8), cp)
    return v.sum((0, 2))


def bwd_operands(e, g):
    """dA >= 0 (small integers) and y > 0 > mean: every term of S1 and S2 is non-negative."""
    n, cp, c = e.n, e.cp, e.c
    shape = (n, e.d, e.h, e.w, cp)
    scale, shift, y0 = constants_with_zero_preactivation(n, cp, c, e.p, g, positive=True)
    y = special_y(shape, y0, g, positive=True)
    y[..., c:] = 0
    dA = int_operand(shape, 0.7, [1, 2, 3], g, DEV).to(torch.bfloat16)
    dA[..., c:] = 0
    mean = -(torch.rand((n, cp), device=DEV, generator=g) * 0.5 + 0.05)
    rstd = torch.rand((n, cp), device=DEV, generator=g) * 1.5 + 0.5
    if e.mode == R.BATCH_EVAL:      # one set of per-channel constants for the whole batch
        scale, shift, mean, rstd = (t[:1].expand(n, cp).contiguous() for t in (scale, shift, mean, rstd))
    return dA, y, scale, shift, mean, rstd


def run_bwd_bounds(e, seed=10, report=None):
    """dgamma / dbeta / dbias and dy of ``norm_act_bwd`` with its own reduce (e.records == 0) or with external records.

    Bound of the reduce (norm_act_bwd_reduce_kernel): per channel a thread adds its T = ceil(vps / (bps threads)) terms
    in one fp32 chain, then one thread adds the lanes_v = threads / (Cp / 8) lane sums in sequence; S2's term carries
    dz = fl(dA * factor), moff = fl(-mean rstd) and the fma forming xhat (3 roundings). The finalize adds the records in
    fp64 and rounds once. So |error| <= (T + lanes_v + 4) 2^-24 sum |terms| (first order, 1 % slack). External records
    (rounded once each to fp32 here): (2 + 1) 2^-24. The terms are non-negative, so sum |terms| is the sum itself and
    every record (computed in float64 with the kernel's own partition) must exceed the bound of the total it enters:
    a lost, zeroed or doubled record fails. dbias (eval BatchNorm): one more product, fl(tot1 * gscale)."""
    ops = _ops()
    g = _gen(seed)
    n, cp, c = e.n, e.cp, e.c
    vox = e.d * e.h * e.w
    dA, y, scale, shift, mean, rstd = bwd_operands(e, g)
    bps, threads, vps = _reduce_plan(n, cp, vox)
    if e.records:
        chain = 3
    else:
        chain = -(-vps // (bps * threads)) + threads // (cp // 8) + 4
    k = 1.01 * chain * 2.0 ** -24
    s1 = torch.zeros((n, cp), dtype=torch.float64, device=DEV)
    s2 = torch.zeros_like(s1)
    dz = torch.empty(dA.shape, dtype=torch.float64, device=DEV)
    min_rec = [float("inf"), float("inf")]
    partial = torch.zeros((n * max(e.records, 1), 2, cp), device=DEV) if e.records else None
    for i in range(n):
        s = slice(i, i + 1)
        dz[s] = R.dz_of(dA[s], y[s], scale[s], shift[s], e.slope, e.p, SEED, n0=i)
        xhat = (y[s].double() - mean[s].double().view(1, 1, 1, 1, cp)) * rstd[s].double().view(1, 1, 1, 1, cp)
        t2 = dz[s] * xhat
        s1[i], s2[i] = dz[s].sum((0, 1, 2, 3)), t2.sum((0, 1, 2, 3))
        if e.records:       # external records: contiguous voxel ranges, each rounded once to fp32
            rid = torch.arange(vox, device=DEV) * e.records // vox
            r1 = torch.zeros((e.records, cp), dtype=torch.float64, device=DEV).index_add_(0, rid, dz[s].reshape(-1, cp))
            r2 = torch.zeros((e.records, cp), dtype=torch.float64, device=DEV).index_add_(0, rid, t2.reshape(-1, cp))
            partial[i * e.records:(i + 1) * e.records, 0] = r1.float()
            partial[i * e.records:(i + 1) * e.records, 1] = r2.float()
        else:
            r1, r2 = reduce_records(dz[s], bps, threads), reduce_records(t2, bps, threads)
        min_rec[0] = min(min_rec[0], float(r1[:, :c].min()))
        min_rec[1] = min(min_rec[1], float(r2[:, :c].min()))
        del xhat, t2
    if e.records:            # the reference is the sum of the records the kernel reads
        pr = partial.double().view(n, e.records, 2, cp).sum(1)
        s1, s2 = pr[:, 0], pr[:, 1]
    dy, dgamma, dbeta, dbias = ops.norm_act_bwd(dA, None, y, e.mode, mean, rstd, scale, e.slope, e.p, SEED, c,
                                                shift=shift, partial=partial)
    ref = R.norm_bwd(dA, y, e.mode, mean, rstd, scale, shift, e.slope, e.p, SEED, c, dz=dz)
    ref["S1"], ref["S2"] = s1, s2
    ref = _recombine(ref, e.mode, vox, n, scale, c)
    fails = []
    ratios = {}
    tot1, tot2 = s1.sum(0)[:c], s2.sum(0)[:c]
    for what, got, want, bound in (("dbeta", dbeta, tot1, k * tot1), ("dgamma", dgamma, tot2, k * tot2)):
        r = float(((got.double() - want).abs() / bound).max())
        ratios[what] = r
        if not r <= 1:
            fails.append(f"{what}: error / bound {r:.3g}")
    sens = min(min_rec[0] / float((k * tot1).max()), min_rec[1] / float((k * tot2).max()))
    if not sens > 1:
        fails.append(f"sensitivity: smallest record / bound {sens:.3g} <= 1")
    if e.mode == R.BATCH_EVAL:
        bound = (k + 2.0 ** -23) * tot1 * scale[0, :c].double()
        r = float(((dbias.double() - ref["dbias"]).abs() / bound).max())
        ratios["dbias"] = r
        if not r <= 1:
            fails.append(f"dbias: error / bound {r:.3g}")
    else:
        f = R.bit_mismatch("dbias (analytically zero)", dbias, torch.zeros_like(dbias))
        if f:
            fails.append(f)
    near = 0
    for i in range(n):
        s = slice(i, i + 1)
        refi = {"dz": dz[s], "dy": ref["dy"][s], "c1": ref["c1"][s], "c2": ref["c2"][s]}
        f, m = R.check_dy(dy[s], refi, y[s], mean[s], rstd[s], scale[s], chain, c, f"sample {i} dy")
        fails += f
        near += m
    if report is not None:
        report.append(f"    error / bound: " + ", ".join(f"{k_} {v:.3g}" for k_, v in ratios.items())
                      + f"; smallest record / bound {sens:.3g}; dy near a bf16 midpoint: {near} of {dy[..., :c].numel()}")
    # with external records c1 / c2 carry one rounding each and the band is narrow; with the kernel's own reduce they
    # carry the whole chain bound, and the band is reported, not asserted
    if e.records and near > 1e-3 * dy[..., :c].numel():
        fails.append(f"dy: {near} elements near a bf16 midpoint (expected a handful)")
    return fails


def _recombine(ref, mode, vox, n, scale, c):
    """c1, c2, dy of ``R.norm_bwd`` from the sums in ref["S1"] / ref["S2"] (the reduce's own or the records' totals)."""
    s1, s2 = ref["S1"], ref["S2"]
    cp = s1.shape[-1]
    if mode == R.INSTANCE:
        c1, c2 = s1 / vox, s2 / vox
    elif mode == R.BATCH_TRAIN:
        c1 = (s1.sum(0, keepdim=True) / (vox * n)).expand(n, cp)
        c2 = (s2.sum(0, keepdim=True) / (vox * n)).expand(n, cp)
    else:
        c1 = c2 = torch.zeros_like(s1)
    v = lambda t: t.double().view(n, 1, 1, 1, cp)
    ref = dict(ref, c1=c1, c2=c2)
    ref["dy"] = v(scale) * (ref["dz"] - v(c1) - ref["xhat"] * v(c2))
    ref["dbias"] = scale[0, :c].double() * s1.sum(0)[:c] if mode == R.BATCH_EVAL else ref["dbias"]
    return ref


# ---------------------------------------------------------------------------------------------------
# the output head (warp-level MMAs)
# ---------------------------------------------------------------------------------------------------
def _split3(w):
    """The kernel's hi + mid + lo bf16 split of fp32 weights."""
    hi = w.to(torch.bfloat16).float()
    r = w - hi
    mid = r.to(torch.bfloat16).float()
    lo = (r - mid).to(torch.bfloat16).float()
    return hi, mid, lo


def head_fwd_bound(u, hi, mid, lo, bias):
    """Bound of head_fwd_mma_kernel for out[n, co, v] against the exact sum. Six MMAs in order lo(k-step 0), lo(1),
    mid(0), mid(1), hi(0), hi(1), each adding 16 exact bf16 products to the fp32 accumulator C. Model of one MMA:
    every addend aligned to the largest of |C| and the products and truncated to 24 bits (< 1 unit 2^-23 of that
    largest each, 17 addends), then one rounding of the result: err <= 2^-23 (17 max(|C|, max |p|) + |D|). The bias
    adds one fp32 rounding. Magnitudes are taken from the exact partial sums of |terms| (first order, 1 % slack)."""
    step0 = (torch.arange(32, device=u.device) % 8) < 4
    ua = u.double().abs()
    bound = torch.zeros(u.shape[:-1] + (hi.shape[0],), dtype=torch.float64, device=u.device)
    acc = torch.zeros_like(bound)
    for part in (lo, mid, hi):
        for sel in (step0, ~step0):
            wa = (part.double().abs() * sel).t()           # (32, co)
            terms = ua @ wa
            mx = (ua.unsqueeze(-1) * wa).amax(-2)
            bound += 2.0 ** -23 * 17 * torch.maximum(acc, mx)
            acc = acc + terms
            bound += 2.0 ** -23 * acc
    bound += 2.0 ** -24 * (acc + bias.double().abs())
    return 1.01 * bound


def run_head_fwd(e, seed=11, report=None):
    """conv1x1_to_ncdhw on a deferred source with weights of full 24-bit significands (hi + mid + lo all nonzero and
    positive, u >= 0 mostly): within ``head_fwd_bound``, and that bound is smaller than the error of dropping ``lo``."""
    ops = _ops()
    g = _gen(seed)
    n, cp = e.n, 32
    scale, shift, y0 = constants_with_zero_preactivation(n, cp, cp, e.p, g, positive=True)
    shift = shift.abs()                                          # mostly positive pre-activations: coherent sums
    y = special_y((n, e.d, e.h, e.w, cp), y0, g, positive=True)
    # w = hi + mid + lo in [1/2, 1): hi of 8 bits, mid = k 2^-17 (k in [128, 256)) below half of hi's unit, lo = k 2^-24
    # (k in [32, 64)) below half of mid's unit -- 24 significant bits, the kernel's split returns the three terms
    ri = lambda a, b: torch.randint(a, b, (e.co, e.ci), device=DEV, generator=g).float()
    hi = ri(128, 256) * 2.0 ** -8
    mid = ri(128, 256) * 2.0 ** -17
    lo = ri(32, 64) * 2.0 ** -24
    w = hi + mid + lo
    h2, m2, l2 = _split3(w)
    assert torch.equal(h2, hi) and torch.equal(m2, mid) and torch.equal(l2, lo) and bool((lo != 0).all())
    bias = torch.randn(e.co, device=DEV, generator=g)
    src = ops.DeferredAct(y, scale, shift, e.slope, e.p, SEED) if e.deferred else None
    fails, worst, sens = [], 0.0, 1.0
    for i in range(n):
        s = slice(i, i + 1)
        u = R.act_fwd(y[s], scale[s], shift[s], e.slope, e.p, SEED, n0=i)[0].float()
        if i == 0:
            out = ops.conv1x1_to_ncdhw(src if e.deferred else R.act_fwd(y, scale, shift, e.slope, e.p, SEED)[0],
                                       w.view(e.co, e.ci, 1, 1, 1), bias)
        ud = u.double().reshape(-1, 32)
        exact = ud @ w.double().t() + bias.double()
        nolo = ud @ (hi + mid).double().t() + bias.double()
        bound = head_fwd_bound(u.reshape(-1, 32), hi, mid, lo, bias)
        got = out[i].reshape(e.co, -1).t().double()
        worst = max(worst, float(((got - exact).abs() / bound).max()))
        sens = min(sens, float(((nolo - exact).abs() > bound).double().mean()))
    if not worst <= 1:
        fails.append(f"head forward: error / bound {worst:.3g}")
    if not sens > 0.5:
        fails.append(f"head forward: dropping lo exceeds the bound on only {sens:.1%} of the outputs")
    if report is not None:
        report.append(f"    forward error / bound {worst:.3g}; dropping lo exceeds the bound on {sens:.1%} of the outputs")
    return fails


def run_head_bwd(e, seed=12, report=None):
    """head_bwd_fused with dout >= 0 (small integers) and weights >= 0 (multiples of 1/8): du = bf16(dout)^T bf16(W) is
    exact, dz >= 0, y > 0 > mean, so every term of S1, S2 and dW is non-negative.

    Bounds (first order, 1 % slack). Kernel 1: a warp lane takes T = ceil(units / (blocks * 8)) units of 16 voxels, two
    voxels per unit per chain, so S1 / s2 chains are 2T long; dz = fl(du * factor) (1), S2 = fma(r, s2, fl(fl(-m r)
    s1)) (3), a 3-level lane tree, the 8-warp sum (8), the fp64 finalize and one cast: (2T + 16) 2^-24 sum |terms|.
    dW: T MMAs per warp, each within 2^-23 (17 + 1) of the warp's (growing, non-negative) accumulator, then the 8-warp
    sum and the fp64 finish: (36 T + 10) 2^-24 dW. db sums integers: exact. Every record (a block of a sample) exceeds
    the bound of its total. dy: the apply criterion with chain = 2T + 16."""
    ops = _ops()
    g = _gen(seed)
    n, cp, c = e.n, 32, e.c
    vox = e.d * e.h * e.w
    shape = (n, e.d, e.h, e.w, cp)
    scale, shift, y0 = constants_with_zero_preactivation(n, cp, c, e.p, g, positive=True, narrow=True)
    # y >= y0 per channel: every pre-activation >= 0 (u >= 0, so dW's terms are non-negative); y == y0 at 2 % of the
    # voxels takes the slope branch at a pre-activation of exactly 0
    y0b = y0.view(n, 1, 1, 1, cp).expand(shape)
    y = (y0b + torch.randn(shape, device=DEV, generator=g).abs() * 2 + 2.0 ** -10).to(torch.float16)
    y = torch.where(torch.rand(shape, device=DEV, generator=g) < 0.02, y0b.to(torch.float16), y)
    mean = -(torch.rand((n, cp), device=DEV, generator=g) * 0.5 + 0.05)
    rstd = torch.rand((n, cp), device=DEV, generator=g) * 1.5 + 0.5
    if e.mode == R.BATCH_EVAL:
        scale, shift, mean, rstd = (t[:1].expand(n, cp).contiguous() for t in (scale, shift, mean, rstd))
    dout = int_operand((n, e.co, e.d, e.h, e.w), 0.8, [1, 2, 3], g, DEV)
    w = int_operand((e.co, e.ci), 1.0, [1, 2, 3], g, DEV, scale_pow2=-3)
    fuse = ops.NormBwdFusion(y, scale, shift, mean, rstd, e.slope, e.p, SEED)
    dy, dgamma, dbeta, dbias, dw, db = ops.head_bwd_fused(dout, fuse, w.view(e.co, e.ci, 1, 1, 1), e.mode, c)
    units = vox // 16
    bps = min(-(-296 // n), -(-units // 8))
    T = -(-units // (bps * 8))
    chain = 2 * T + 16
    k = 1.01 * chain * 2.0 ** -24
    kw = 1.01 * (36 * T + 10) * 2.0 ** -24
    dz = torch.empty(shape, dtype=torch.float64, device=DEV)
    dw_ref = torch.zeros((e.co, e.ci), dtype=torch.float64, device=DEV)
    s1 = torch.zeros((n, cp), dtype=torch.float64, device=DEV)
    s2 = torch.zeros_like(s1)
    min_rec = [float("inf")] * 2
    min_wrec = torch.full((e.co, e.ci), float("inf"), dtype=torch.float64, device=DEV)
    for i in range(n):
        s = slice(i, i + 1)
        go = dout[i].reshape(e.co, -1).t().double()                       # (V, co)
        du = (go @ w.double()).view(1, e.d, e.h, e.w, e.ci)
        dz[s] = R.dz_of(du, y[s], scale[s], shift[s], e.slope, e.p, SEED, n0=i)
        xhat = (y[s].double() - mean[s].double().view(1, 1, 1, 1, cp)) * rstd[s].double().view(1, 1, 1, 1, cp)
        s1[i], s2[i] = dz[s].sum((0, 1, 2, 3)), (dz[s] * xhat).sum((0, 1, 2, 3))
        u = R.act_fwd(y[s], scale[s], shift[s], e.slope, e.p, SEED, n0=i)[0].double().reshape(-1, cp)
        dw_ref += go.t() @ u[:, :e.ci]
        # records: block b of the sample takes units b * 8 + warp + j * bps * 8
        unit_of = torch.arange(vox, device=DEV) // 16
        blk = (unit_of // 8) % bps
        oh = torch.nn.functional.one_hot(blk, bps).double()              # (V, bps)
        min_rec[0] = min(min_rec[0], float((oh.t() @ dz[s].reshape(-1, cp))[:, :c].min()))
        min_rec[1] = min(min_rec[1], float((oh.t() @ (dz[s] * xhat).reshape(-1, cp))[:, :c].min()))
        wrec = (oh.t() @ (go.unsqueeze(-1) * u[:, :e.ci].unsqueeze(1)).reshape(vox, -1)).view(bps, e.co, e.ci)
        min_wrec = torch.minimum(min_wrec, wrec.amin(0))
        del xhat, u, oh, wrec
    ref = R.norm_bwd(y, y, e.mode, mean, rstd, scale, shift, e.slope, e.p, SEED, c, dz=dz)
    ref["S1"], ref["S2"] = s1, s2
    ref = _recombine(ref, e.mode, vox, n, scale, c)
    fails, ratios = [], {}
    tot1, tot2 = s1.sum(0)[:c], s2.sum(0)[:c]
    for what, got, want, bound in (("dbeta", dbeta, tot1, k * tot1), ("dgamma", dgamma, tot2, k * tot2),
                                   ("dW", dw, dw_ref, kw * dw_ref)):
        r = float(((got.double().reshape(want.shape) - want).abs() / bound).max())
        ratios[what] = r
        if not r <= 1:
            fails.append(f"{what}: error / bound {r:.3g}")
    f = R.bit_mismatch("db", db, dout.double().sum((0, 2, 3, 4)).float())
    if f:
        fails.append(f)
    sens = min(min_rec[0] / float((k * tot1).max()), min_rec[1] / float((k * tot2).max()))
    sens_w = float((min_wrec / (kw * dw_ref)).min())
    if not (sens > 1 and sens_w > 1):
        fails.append(f"sensitivity: smallest record / bound S {sens:.3g}, dW {sens_w:.3g}")
    if e.mode != R.BATCH_EVAL:
        f = R.bit_mismatch("dbias (analytically zero)", dbias, torch.zeros_like(dbias))
        if f:
            fails.append(f)
    near = 0
    for i in range(n):
        s = slice(i, i + 1)
        refi = {"dz": dz[s], "dy": ref["dy"][s], "c1": ref["c1"][s], "c2": ref["c2"][s]}
        f, m = R.check_dy(dy[s], refi, y[s], mean[s], rstd[s], scale[s], chain, c, f"sample {i} dy")
        fails += f
        near += m
    if report is not None:
        report.append("    error / bound: " + ", ".join(f"{k_} {v:.3g}" for k_, v in ratios.items())
                      + f"; smallest record / bound S {sens:.3g}, dW {sens_w:.3g}; dy near a bf16 midpoint: {near}")
    # kernel 1's per-(n, c) sums are not observable, so dy's band carries their whole chain bound (2T + 16 units): the
    # count is reported, not asserted small (norm_act_bwd with external records checks the same apply arithmetic with
    # a narrow band)
    return fails


# ---------------------------------------------------------------------------------------------------
# running the census
# ---------------------------------------------------------------------------------------------------
def _run(e, report):
    t = type(e)
    if t is Fwd:
        return run_fwd(e)
    if t is PoolB:
        return run_pool_bwd(e)
    if t is Fin:
        return run_finalize(e)
    if t is Col:
        return run_colsum(e)
    if t is HeadF:
        return run_head_fwd(e, report=report)
    if t is HeadB:
        return run_head_bwd(e, report=report)
    if e.mode == R.NONE:
        return run_bwd_none(e)
    fails = run_bwd_bounds(e, report=report)
    if not e.records:
        # the same pass fed records of the reduce's own partition (rounded once each): c1 / c2 are then known to one
        # rounding and dy's near-midpoint band is narrow
        report.append("    with external records:")
        fails += [f"external records: {f}" for f in
                  run_bwd_bounds(e._replace(records=_reduce_plan(e.n, e.cp, e.d * e.h * e.w)[0]), report=report)]
    return fails


def _run_entries(entries, report):
    failures = []
    for e in entries:
        sub = []
        fails = _run(e, sub)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        report.append(f"{_label(e)} {'ok' if not fails else 'FAIL'}")
        report += sub
        failures += [f"{_label(e)}: {f}" for f in fails]
    return failures


# beside the census: eval-mode BatchNorm, the non-FIXED forward kernel (Cp / 8 = 12 does not divide 256), a ragged
# voxel count, and channel padding (c < Cp)
SYNTHETIC = [
    Fin(4, 64, 48, R.BATCH_EVAL, 0, 8 * 8 * 8, True),
    Bwd(4, 8, 8, 8, 64, 48, R.BATCH_EVAL, 0.2, 0.05, 0),
    Fwd(2, 6, 10, 12, 96, 80, 0.2, 0.05, False, True, True),
    Fwd(2, 6, 10, 14, 96, 80, 0.2, 0.05, True, True, False),
    Bwd(3, 5, 7, 9, 32, 24, R.INSTANCE, 0.2, 0.05, 0),
    Fwd(3, 5, 7, 9, 32, 24, 0.2, 0.05, False, True, True),
    HeadB(2, 8, 8, 8, 6, 32, R.BATCH_TRAIN, 32, 0.2, 0.05),
    # at step shape, paths the default step does not take: the pooled-only forward (a deferred block feeding a pool),
    # the max-pool backward on a deferred source, and a non-accumulating one
    Fwd(8, 128, 128, 128, 32, 32, 0.1, 0.05, True, False, False),
    PoolB(8, 128, 128, 128, 32, True, True, 0.1, 0.05),
    PoolB(2, 16, 16, 32, 64, False, False, 0.2, 0.0),
]

GROUPS = {"forward": (Fwd, PoolB), "norm_backward": (Bwd,), "finalize_colsum": (Fin, Col), "head": (HeadF, HeadB)}


@pytest.mark.parametrize("group", list(GROUPS))
def test_census_exact(census, group):
    entries = [e for e in census + SYNTHETIC if type(e) in GROUPS[group]]
    report = []
    failures = _run_entries(entries, report)
    print(f"\n{group}: {len(entries)} entries\n" + "\n".join(report))
    assert not failures, "\n".join(failures)


def test_census_contents_and_coverage(census):
    """The census reaches the paths the suite is meant to test."""
    print(f"\ncensus: {len(census)} entries\n" + "\n".join(_label(e) for e in census))
    has = lambda pred: any(pred(e) for e in census)
    fin = [e for e in census if type(e) is Fin]
    two_stage = [e for e in fin if e.mode == R.BATCH_TRAIN and e.n > 1 and e.tiles * e.n >= 2048]
    single = [e for e in fin if not (e.mode == R.BATCH_TRAIN and e.n > 1 and e.tiles * e.n >= 2048)]
    assert two_stage and single
    assert has(lambda e: type(e) is Fwd and e.d == 128 and e.cp == 32)
    assert has(lambda e: type(e) is Fin and e.mode == R.INSTANCE and e.voxels == 128 ** 3 and e.c == 32)
    assert has(lambda e: type(e) is Fwd and e.cp == 512)
    assert has(lambda e: type(e) is Fwd and e.f16 and not e.materialize)                          # fp16 copy only
    assert has(lambda e: type(e) is PoolB and not e.deferred and e.acc)
    # the default step materialises every pooled block (UB_POOL_FUSE and the deferred pooling are opt-in), so the
    # pooled-only forward and the deferred max-pool backward come from SYNTHETIC, at the step's 8 x 128^3 x 32 shape
    synth = lambda pred: any(pred(e) for e in SYNTHETIC if e.n == 8 and e.d == 128)
    assert synth(lambda e: type(e) is Fwd and e.pool and not e.materialize and not e.f16)
    assert synth(lambda e: type(e) is PoolB and e.deferred and e.acc)
    assert has(lambda e: type(e) is Bwd and e.mode != R.NONE and e.records)
    assert has(lambda e: type(e) is Bwd and e.mode != R.NONE and not e.records)
    assert has(lambda e: type(e) is Bwd and e.mode == R.NONE)
    assert has(lambda e: type(e) is HeadB) and has(lambda e: type(e) is HeadF and e.deferred)
    multi = [(e, _reduce_plan(e.n, e.cp, e.d * e.h * e.w)[0]) for e in census
             if type(e) is Bwd and e.mode != R.NONE and not e.records]
    assert any(b > 1 for _, b in multi)
    print("two-stage BatchNorm finalize:", [tuple(e) for e in two_stage])
    print("reduce blocks per sample:", sorted({b for _, b in multi}))


# ---------------------------------------------------------------------------------------------------
# config 4 (t1w, batch 16): tensors of 2^31 bytes
# ---------------------------------------------------------------------------------------------------
def _bytes(e):
    t = type(e)
    if t in (Fwd, Bwd, PoolB):
        return e.n * e.d * e.h * e.w * e.cp * 2
    if t in (HeadF, HeadB):
        return e.n * e.d * e.h * e.w * 32 * 2
    if t is Col:
        return e.rows * e.cp * 2
    return 0


def test_config4_batch16_beyond_2gib():
    """Every entry of a t1w batch-16 step whose tensors reach 2^31 bytes, rerun on all 16 samples (dropout counters
    past 2^31 elements, 64-bit sample bases): the bit-exact criteria, and the bounds on the norm backward entries."""
    entries = [e for e in record_census("t1w", 16, 128) if _bytes(e) >= 2 ** 31]
    assert any(type(e) is Fwd for e in entries) and any(type(e) is Bwd and e.mode != R.NONE for e in entries)
    report = []
    failures = _run_entries(entries, report)
    print(f"\nconfig 4 entries at >= 2^31 bytes: {len(entries)}\n" + "\n".join(report))
    assert not failures, "\n".join(failures)
