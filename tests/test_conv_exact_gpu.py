"""Bit-exact tests of the tcgen05 convolutions at the training step's own layer shapes.

The census: one GanTrainer step (config 2: bssfp, 8 x 128^3) runs with thin wrappers around ``ops.conv_fwd``,
``ops.conv_dgrad`` and ``ops.conv_wgrad`` that record every distinct convolution the step issues. Each entry is then
rerun at its real shape with integer operands (tests/conv_exact.py): the fp32 accumulators must equal the exact sums,
so forward outputs (bias, fused LeakyReLU, bf16 / saturating fp16 rounding), per-sample statistics, split dgrad
outputs and weight gradients are compared bit for bit with a float64 tap-sum reference. At these shapes the persistent
generic kernel runs many tiles per CTA (both accumulator sets, ring phases across tiles, ragged last rounds, statistics
carried across a sample boundary) and the marching kernels march whole 128-plane volumes; the test asserts that.
"""
import ctypes as C
import math
from collections import namedtuple

import pytest
import torch

from tests.conv_exact import (DECONV_K2S2, K1, K3S1P1, K4S2P1, K4S2P1_S2D, check_exact_bound, epilogue_fp32,
                              granularity, int_operand, pad_channels, ref_dgrad, ref_fwd, ref_wgrad, round_out, to_s2d,
                              weight_shape)

pytestmark = pytest.mark.gpu
DEV = "cuda"

# one distinct convolution call of the step
Entry = namedtuple("Entry", "dir kind c0 c1 co dims stats act slope f16 fuse bias drop", defaults=(0.0,))
DIRS = {"fwd": 0, "dgrad": 1, "wgrad": 2}
NTAPS = {K3S1P1: 27, K1: 1, K4S2P1: 64, K4S2P1_S2D: 64, DECONV_K2S2: 8}
BIG_F16 = [-2047, -1023, -257, 257, 1023, 2047]      # fp16-exact, not bf16-exact: they must reach the MMA unrounded


def _ops():
    from unet_bssfp_b200 import ops
    return ops


def _lib():
    from unet_bssfp_b200 import _lib
    return _lib.load()


def _spec(e):
    return _ops().ConvSpec(e.kind, e.c0, e.co, e.c1)


def _pad32(c):
    return (c + 31) // 32 * 32


def _label(e):
    n, d, h, w = e.dims
    src = f"{e.c0}+{e.c1}" if e.c1 else f"{e.c0}"
    extra = "".join([" stats" if e.stats else "", f" act({e.slope:g})" if e.act else "", " f16-src0" if e.f16 else "",
                     f" fused(p={e.drop:g})" if e.fuse else ""])
    return f"{e.dir} kind{e.kind} {src}->{e.co} @{n}x{d}x{h}x{w}{extra}"


def record_census(modality, batch, size):
    """Run one GanTrainer step with recording wrappers; -> sorted list of distinct Entry."""
    import unet_bssfp_b200 as ub
    from unet_bssfp_b200.train_step import GanTrainer
    ops = _ops()
    seen = set()
    fwd0, dgrad0, wgrad0 = ops.conv_fwd, ops.conv_dgrad, ops.conv_wgrad

    def fwd(spec, src0, src1, w_packed, bias, act=0, slope=0.0, want_stats=False):
        assert not isinstance(src0, ops.DeferredAct), "the census records the default (materialised) operand paths"
        seen.add(Entry("fwd", spec.kind, spec.c0, spec.c1, spec.co, spec.in_dims(src0), bool(want_stats), int(act),
                       float(slope) if act else 0.0, src0.dtype == torch.float16, False, bias is not None))
        return fwd0(spec, src0, src1, w_packed, bias, act=act, slope=slope, want_stats=want_stats)

    def dgrad(spec, dy, w_packed_dgrad, in_dhw, fuse=None):
        seen.add(Entry("dgrad", spec.kind, spec.c0, spec.c1, spec.co, (dy.shape[0],) + tuple(in_dhw), False, 0,
                       float(fuse.slope) if fuse is not None else 0.0, False, fuse is not None, False,
                       float(fuse.drop_p) if fuse is not None else 0.0))
        return dgrad0(spec, dy, w_packed_dgrad, in_dhw, fuse=fuse)

    def wgrad(spec, src0, src1, dy, weight_shape):
        assert not isinstance(src0, ops.DeferredAct)
        seen.add(Entry("wgrad", spec.kind, spec.c0, spec.c1, spec.co, spec.in_dims(src0), False, 0, 0.0, False, False,
                       False))
        return wgrad0(spec, src0, src1, dy, weight_shape)

    cin = 24 if modality == "bssfp" else 6
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(ops, "conv_fwd", fwd)
        mp.setattr(ops, "conv_dgrad", dgrad)
        mp.setattr(ops, "conv_wgrad", wgrad)
        torch.manual_seed(0)
        g, d = ub.Generator(modality).to(DEV), ub.Discriminator(modality).to(DEV)
        tr = GanTrainer(g, d)
        torch.manual_seed(1)
        x = torch.rand(batch, cin, size, size, size, device=DEV)
        y = torch.rand(batch, 6, size, size, size, device=DEV)
        tr.step(x, y)
        torch.cuda.synchronize()
        del tr, g, d, x, y
    torch.cuda.empty_cache()
    return sorted(seen, key=lambda e: (list(DIRS).index(e.dir), e.kind, e.c0, e.c1, e.co, e.dims, e.stats, e.f16, e.fuse))


@pytest.fixture(scope="module")
def census():
    return record_census("bssfp", 8, 128)


# ---------------------------------------------------------------------------------------------------
# coverage: which kernel serves an entry and how much of its persistent / marching loop it runs
# ---------------------------------------------------------------------------------------------------
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def expected_class(e):
    """The kernel class (ub_conv_kernel_class) this suite expects: 0 generic, 1 marching, 2 marching wgrad, 3 wgrad."""
    c0p, c1p, cop = _pad32(e.c0), _pad32(e.c1) if e.c1 else 0, _pad32(e.co)
    n, d, h, w = e.dims
    if e.dir == "wgrad":
        if e.kind == K4S2P1_S2D:
            return 2 if h >= 32 and w >= 16 and c0p * cop <= 64 * 64 else 3
        return 2 if e.kind == K3S1P1 and h >= 16 and w >= 8 and (c0p + c1p) * cop <= 128 * 256 else 3
    if e.kind != K3S1P1:
        return 0
    if e.dir == "fwd":
        return 1 if cop == 32 and c0p + c1p <= 96 else 0
    return 1 if c1p == 0 and c0p == 32 and cop <= 96 else 0


def coverage(e):
    """-> dict of the launch facts of this entry."""
    lib = _lib()
    desc = _spec(e).desc(*e.dims)
    cls = lib.ub_conv_kernel_class(C.byref(desc), DIRS[e.dir])
    assert cls == expected_class(e), (_label(e), cls)
    out = {"class": cls}
    n, d, h, w = e.dims
    c0p, c1p, cop = _pad32(e.c0), _pad32(e.c1) if e.c1 else 0, _pad32(e.co)
    if e.dir == "wgrad":
        nbytes = lib.ub_conv_wgrad_workspace_bytes(C.byref(desc))
        out["splits"] = nbytes // (NTAPS[e.kind] * (c0p + c1p) * cop * 4)
        return out
    if cls == 1:
        tiles_w = math.ceil(w / 8)
        columns = n * math.ceil(h / 16) * tiles_w
        ns = max(1, min(math.ceil(4 * _sms() / columns), max(d // 8, 1)))
        out["segment"] = math.ceil(d / ns)
        # launch_march: CTA pairs (cta_group::2) when the w tiles pair up and a plane has >= 2 K chunks -- the sources'
        # chunks for a forward, dy's for a dgrad
        chunks = (c0p + c1p) // 32 if e.dir == "fwd" else cop // 32
        out["pair"] = tiles_w % 2 == 0 and chunks >= 2
        return out
    if e.dir != "fwd":
        return out
    total = lib.ub_conv_num_tiles(C.byref(desc))
    n_ntiles = 4 if (e.kind == DECONV_K2S2 and cop == 64) else math.ceil(cop / 128) * (8 if e.kind == DECONV_K2S2 else 1)
    grid = min(max(_sms() // n_ntiles, 1), total)
    out.update(tiles=total, grid=grid, per_cta=math.ceil(total / grid), ragged=total % grid != 0,
               mma2=e.kind == K3S1P1 and cop <= 64 and d >= 4)
    if e.stats and cop == 32:
        # one 32-column chunk: sums carried across a CTA's consecutive tiles of a sample (tiles are sample-major)
        per_sample = total // n
        t = torch.arange(max(total - grid, 0))
        out["carry_cross"] = bool(((t // per_sample) != ((t + grid) // per_sample)).any())
    return out


# ---------------------------------------------------------------------------------------------------
# the three directions at one shape
# ---------------------------------------------------------------------------------------------------
def _mismatch(what, got, want):
    if torch.equal(got, want):
        return None
    bad = (got != want).nonzero()
    i = tuple(bad[0].tolist())
    return f"{what}: {bad.shape[0]} of {want.numel()} differ, first at {i}: {got[i].item()} vs {want[i].item()}"


def _fwd_operands(e, g, big_src0):
    n, d, h, w = e.dims
    ci, kt = e.c0 + e.c1, NTAPS[e.kind]
    if e.stats and not big_src0:
        # per-(n, c) sums of y and y^2 over a sample must stay exact: E[acc^2] * voxels ~ 2^20 (the bias adds at most
        # one per voxel), i.e. sparse x at 128^3 and dense x (capped at 1/2) at the deep levels
        od, oh, ow = _spec(e).out_dims(d, h, w)
        x = int_operand((n, d, h, w, ci), min(0.5, 2.0 ** 21 / (od * oh * ow * kt * ci)), [-1, 1], g, DEV)
        wt = int_operand(weight_shape(e.kind, ci, e.co), 0.5, [-1, 1], g, DEV)
        bias = int_operand((e.co,), 1.0, [-1, 0, 1], g, DEV)
    else:
        x = int_operand((n, d, h, w, ci), 0.5, [-3, -2, -1, 1, 2, 3], g, DEV)
        wt = int_operand(weight_shape(e.kind, ci, e.co), 0.5, [-2, -1, 1, 2], g, DEV)
        bias = int_operand((e.co,), 1.0, [-3, -2, -1, 0, 1, 2, 3], g, DEV)
    if big_src0:
        x[..., :e.c0] = int_operand((n, d, h, w, e.c0), 1 / 16, BIG_F16 + [-3, -1, 1, 3], g, DEV)
    return x, wt, bias


def run_fwd(e, seed=0, big_src0=False, operands=None):
    """Forward of entry e with integer operands; -> list of failure strings (empty = bit-exact)."""
    ops = _ops()
    spec = _spec(e)
    g = torch.Generator(device=DEV).manual_seed(seed)
    x, wt, bias = operands if operands is not None else _fwd_operands(e, g, big_src0)
    if not e.bias:
        bias = None
    s0 = pad_channels(x[..., :e.c0], torch.float16 if e.f16 else torch.bfloat16)
    if e.kind == K4S2P1_S2D:
        s0 = to_s2d(s0)
    s1 = pad_channels(x[..., e.c0:], torch.bfloat16) if e.c1 else None
    wpk = ops.pack_conv_weights(spec, wt, ops.UB_PACK_F16_SRC0 if e.f16 else 0)
    out, stats = ops.conv_fwd(spec, s0, s1, wpk, bias, act=e.act, slope=e.slope, want_stats=e.stats)
    del s0, s1, wpk
    check_exact_bound(ref_fwd(e.kind, x.abs(), wt.abs()), granularity(x) * granularity(wt))
    v = epilogue_fp32(ref_fwd(e.kind, x, wt), bias, e.act, e.slope)
    del x
    fails = []
    want = round_out(v, out.dtype)
    fails.append(_mismatch("output", out[..., :e.co], want))
    del want
    fails.append(_mismatch("padded output channels", out[..., e.co:], torch.zeros_like(out[..., e.co:])))
    if e.stats and not big_src0:       # the large fp16 values break the exactness of sum y^2: output bits only
        n = e.dims[0]
        vd = v.double()
        del v
        gv = granularity(vd)
        s_exact = vd.sum((1, 2, 3))
        q_exact = (vd * vd).sum((1, 2, 3))
        check_exact_bound(vd.abs().sum((1, 2, 3)), gv, "sum |y|")
        check_exact_bound(q_exact, gv * gv, "sum y^2")
        rec = stats.double().view(n, -1, 2, stats.shape[-1]).sum(1)
        fails.append(_mismatch("statistics sum", rec[:, 0, :e.co], s_exact))
        fails.append(_mismatch("statistics sum of squares", rec[:, 1, :e.co], q_exact))
        fails.append(_mismatch("padded statistics", rec[:, :, e.co:], torch.zeros_like(rec[:, :, e.co:])))
    return [f for f in fails if f]


def run_dgrad(e, seed=1):
    ops = _ops()
    spec = _spec(e)
    n, d, h, w = e.dims
    g = torch.Generator(device=DEV).manual_seed(seed)
    ci = e.c0 + e.c1
    od, oh, ow = spec.out_dims(d, h, w)
    dy = int_operand((n, od, oh, ow, e.co), 0.5, [-3, -2, -1, 1, 2, 3], g, DEV)
    wt = int_operand(weight_shape(e.kind, ci, e.co), 0.5, [-2, -1, 1, 2], g, DEV)
    d0, d1 = ops.conv_dgrad(spec, pad_channels(dy, torch.bfloat16), ops.pack_conv_weights(spec, wt, 1), (d, h, w))
    check_exact_bound(ref_dgrad(e.kind, dy.abs(), wt.abs(), (d, h, w)), granularity(dy) * granularity(wt))
    want = round_out(ref_dgrad(e.kind, dy, wt, (d, h, w)).float(), torch.bfloat16)
    fails = [_mismatch("dsrc0", d0[..., :e.c0], want[..., :e.c0]),
             _mismatch("dsrc0 padding", d0[..., e.c0:], torch.zeros_like(d0[..., e.c0:]))]
    if e.c1:
        fails += [_mismatch("dsrc1", d1[..., :e.c1], want[..., e.c0:]),
                  _mismatch("dsrc1 padding", d1[..., e.c1:], torch.zeros_like(d1[..., e.c1:]))]
    return [f for f in fails if f]


def run_wgrad(e, seed=2):
    ops = _ops()
    spec = _spec(e)
    n, d, h, w = e.dims
    g = torch.Generator(device=DEV).manual_seed(seed)
    ci = e.c0 + e.c1
    od, oh, ow = spec.out_dims(d, h, w)
    # each weight sums over every output voxel: keep sum |x| |dy| near 2^20
    vox = n * (d * h * w if e.kind == DECONV_K2S2 else od * oh * ow)
    p = min(0.5, math.sqrt(2.0 ** 20 / (vox * 2.25)))
    x = int_operand((n, d, h, w, ci), p, [-2, -1, 1, 2], g, DEV)
    dy = int_operand((n, od, oh, ow, e.co), p, [-2, -1, 1, 2], g, DEV)
    s0 = pad_channels(x[..., :e.c0], torch.bfloat16)
    if e.kind == K4S2P1_S2D:
        s0 = to_s2d(s0)
    s1 = pad_channels(x[..., e.c0:], torch.bfloat16) if e.c1 else None
    wshape = weight_shape(e.kind, ci, e.co)
    dw = ops.conv_wgrad(spec, s0, s1, pad_channels(dy, torch.bfloat16), wshape)
    del s0, s1
    check_exact_bound(ref_wgrad(e.kind, x.abs(), dy.abs(), wshape), granularity(x) * granularity(dy))
    return [f for f in [_mismatch("dw", dw, ref_wgrad(e.kind, x, dy, wshape).float())] if f]


RUN = {"fwd": run_fwd, "dgrad": run_dgrad, "wgrad": run_wgrad}


def _run_entries(entries, report):
    failures = []
    for e in entries:
        cov = coverage(e)
        fails = RUN[e.dir](e)
        if e.dir == "fwd" and e.f16:
            fails += [f"big fp16 source 0: {f}" for f in run_fwd(e, seed=3, big_src0=True)]
        torch.cuda.synchronize()
        report.append(f"{_label(e):64s} {cov} {'ok' if not fails else 'FAIL'}")
        failures += [f"{_label(e)}: {f}" for f in fails]
    return failures


# a moderate synthetic case beside the census: the input head's carried statistics with ~5 tiles per CTA and
# sample changes inside a CTA's tile sequence
SYNTHETIC = [Entry("fwd", K1, 24, 0, 32, (3, 16, 128, 64), True, 0, 0.0, False, False, True)]


@pytest.mark.parametrize("direction", ["fwd", "dgrad", "wgrad"])
def test_census_bit_exact(census, direction):
    entries = [e for e in census if e.dir == direction] + [e for e in SYNTHETIC if e.dir == direction]
    report = []
    failures = _run_entries(entries, report)
    print(f"\n{direction}: {len(entries)} entries ({len(census)} census entries in all)\n" + "\n".join(report))
    assert not failures, "\n".join(failures)


def test_census_contents_and_coverage(census):
    """The census holds the layers the suite is meant to reach, and those reach the kernels' multi-tile code."""
    labels = "\n".join(_label(e) for e in census)
    print(f"\ncensus: {len(census)} entries\n{labels}")
    has = lambda pred: any(pred(e) for e in census)
    assert has(lambda e: e.dir == "fwd" and e.kind == K1 and e.c0 == 24 and e.stats)       # input head DownSampleConv
    assert has(lambda e: e.dir == "fwd" and e.f16)                                                       # fp16 copies
    assert has(lambda e: e.kind == K3S1P1 and e.c0 == 32 and e.c1 == 64 and e.co == 32 and e.dir == "dgrad")
    assert has(lambda e: e.kind == DECONV_K2S2 and e.c0 == 64 and e.co == 64)
    assert has(lambda e: e.kind == K4S2P1_S2D and e.c0 < 32)                                             # the stem
    assert has(lambda e: e.kind == K4S2P1_S2D and e.c0 >= 32 and e.dir == "fwd")                        # d2 .. d5
    assert has(lambda e: e.act == 1)                                                                     # d1 + LeakyReLU
    assert has(lambda e: e.co >= 512 or e.c0 >= 512)                                                     # the 8^3 level
    assert has(lambda e: e.dir == "fwd" and e.kind == K1 and e.c0 == 512 and e.co == 1)                 # final 1x1 conv
    assert has(lambda e: e.dir == "dgrad" and e.fuse)
    covs = [(e, coverage(e)) for e in census + SYNTHETIC]
    # the full-resolution 32-output-channel layers: 32 -> 32 (three layers, one entry each with / without the fp16
    # source 0) and upcat_1.conv_0 [32 | 64] -> 32, all marching 128 planes deep
    march_fwd = {(e.c0, e.c1) for e, c in covs if e.dir == "fwd" and c["class"] == 1 and e.dims[1] == 128}
    assert {(32, 0), (32, 64)} <= march_fwd, march_fwd
    for direction in ("fwd", "dgrad"):                # CTA-pair and single-CTA marching variants, both directions
        assert any(c.get("pair") is True for e, c in covs if e.dir == direction), direction
        assert any(c.get("pair") is False for e, c in covs if e.dir == direction), direction
    gen = [(e, c) for e, c in covs if "tiles" in c]
    assert any(c["per_cta"] >= 3 and c["ragged"] for e, c in gen)
    assert any(c["per_cta"] >= 2 and c["mma2"] for e, c in gen) and any(c["per_cta"] >= 2 and not c["mma2"] for e, c in gen)
    assert any(c.get("carry_cross") for e, c in gen)
    assert max(c.get("segment", 0) for e, c in covs) >= 64
    assert max(c.get("splits", 0) for e, c in covs) > 1
    print("max tiles per CTA (generic forward):", max(c["per_cta"] for e, c in gen),
          "| marching segments:", sorted({c["segment"] for e, c in covs if "segment" in c}),
          "| wgrad splits:", sorted({c["splits"] for e, c in covs if "splits" in c}))


# ---------------------------------------------------------------------------------------------------
# fp16 saturation of a conv -> norm block's raw output
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,c0,dims", [(K1, 24, (2, 8, 32, 16)), (K3S1P1, 32, (2, 16, 32, 16))])
def test_fp16_output_saturates_and_statistics_do_not(kind, c0, dims):
    """Exact outputs beyond 65504 are stored as +-65504 (never inf); the statistics records hold the unsaturated fp32
    values. Operands are multiples of 2^10 and 2^4, so every sum, square and statistic is a multiple of 2^14 / 2^28
    far below 2^22 units: exact in fp32."""
    e = Entry("fwd", kind, c0, 0, 32, dims, True, 0, 0.0, False, False, True)
    g = torch.Generator(device=DEV).manual_seed(11)
    n, d, h, w = dims
    x = int_operand((n, d, h, w, c0), 0.1 if kind == K1 else 0.01, [-5, -1, 1, 5], g, DEV, scale_pow2=10)
    wt = int_operand(weight_shape(kind, c0, 32), 0.5, [-1, 1], g, DEV, scale_pow2=4)
    bias = int_operand((32,), 1.0, [-1, 0, 1], g, DEV, scale_pow2=14)
    v = epilogue_fp32(ref_fwd(kind, x, wt), bias)
    assert (v.abs() > 65504).sum() > 100 and (v.abs() < 65504).sum() > 100
    assert run_fwd(e, operands=(x, wt, bias)) == []
    ops = _ops()
    out, stats = ops.conv_fwd(_spec(e), pad_channels(x, torch.bfloat16), None, ops.pack_conv_weights(_spec(e), wt, 0),
                              bias, want_stats=True)
    assert not torch.isinf(out).any()
    big = v.abs() > 65504
    assert torch.equal(out[..., :32][big].float(), torch.sign(v[big]) * 65504)
    # the records differ from the statistics of the stored (saturated) values
    rec = stats.double().view(n, -1, 2, 32).sum(1)
    stored = out.double()
    assert not torch.equal(rec[:, 1], (stored * stored).sum((1, 2, 3)))


# ---------------------------------------------------------------------------------------------------
# the fused norm-backward dgrad at step shape
# ---------------------------------------------------------------------------------------------------
def test_fused_dgrad_at_step_shape(census):
    """ub_conv_dgrad_fused at every fused dgrad of the step, with the step's dropout p: the gradient is bit-identical
    to the unfused call, and the per-(n, c) sums of the partial records agree with a float64 recomputation from the
    same y, dropout mask and (rounded) dA.

    Bound, from the epilogue's summation (igemm_march.cuh): per channel a thread adds its voxel row's seg terms in
    one fp32 chain (seg = the CTA's depth segment), forms S2 = fma(rstd, sum dz y, fl(-mean rstd) * sum dz), then a
    5-level lane transpose-reduce and a 4-term sum over the lane quarters write the record. Every term therefore
    passes at most seg + 9 additions, and carries at most 2 roundings of its own (dz = dA * fl(inv * slope)) plus 3
    in forming S2, so |record error| <= (seg + 16) 2^-24 * sum |terms| (first order, with 1 % slack): sum |dz| for S1,
    rstd sum |dz y| + |mean rstd| sum |dz| for S2. Operands make every term non-negative (dA >= 0, y > 0 > mean), so
    the bound is ~(seg + 16) 2^-24 of the sums themselves, and the test asserts that every single record exceeds it:
    a record that is lost, zeroed or written twice fails."""
    ops = _ops()
    fused = [e for e in census if e.dir == "dgrad" and e.fuse]
    assert any(e.drop > 0 for e in fused)      # the U-Net blocks' Dropout(p) in training (the input head has none)
    for e in fused:
        spec = _spec(e)
        n, d, h, w = e.dims
        g = torch.Generator(device=DEV).manual_seed(21)
        dy = pad_channels(int_operand((n, d, h, w, e.co), 0.5, [1, 2, 3], g, DEV), torch.bfloat16)
        wpk = ops.pack_conv_weights(spec, int_operand(weight_shape(e.kind, e.c0, e.co), 0.5, [1, 2], g, DEV), 1)
        y = (torch.randn((n, d, h, w, 32), device=DEV, generator=g).abs() * 1.5 + 0.1).to(torch.float16)
        scale = torch.rand((n, 32), device=DEV, generator=g) + 0.5
        shift = torch.randn((n, 32), device=DEV, generator=g) * 0.5 - 0.8       # both signs of the pre-activation
        mean = -torch.randn((n, 32), device=DEV, generator=g).abs() * 0.3
        rstd = torch.rand((n, 32), device=DEV, generator=g) * 1.5 + 0.5
        seed = 4242
        fuse = ops.NormBwdFusion(y, scale, shift, mean, rstd, e.slope, e.drop, seed)
        d0, _ = ops.conv_dgrad(spec, dy, wpk, (d, h, w))
        f0, _, partial = ops.conv_dgrad(spec, dy, wpk, (d, h, w), fuse=fuse)
        assert torch.equal(d0.view(torch.int16), f0.view(torch.int16)), _label(e)
        del d0, dy
        # the dropout mask of (y, p, seed): ub_norm_act_fwd with scale 1, shift 0, slope 1 keeps y * inv (y > 0)
        ones = torch.ones((n, 32), device=DEV)
        kept, _ = ops.norm_act_fwd(y, ones, torch.zeros_like(ones), 1.0, e.drop, seed)
        keep = kept != 0
        del kept
        f32 = lambda v: torch.tensor(v, dtype=torch.float32, device=DEV)
        inv = f32(1.0) / (f32(1.0) - f32(e.drop))
        slope = f32(e.slope)
        sc = (scale * inv).double()[:, None, None, None]           # the kernel's folded constants (fold_inv)
        sh = (shift * inv).double()[:, None, None, None]
        yd = y.double()
        factor = torch.where(yd * sc + sh > 0, inv.double(), (inv * slope).double()) * keep
        del keep
        dz = f0.double() * factor
        del factor, f0
        assert (dz >= 0).all() and bool((yd * sc + sh <= 0).any())
        rs, mu = rstd.double(), mean.double()
        dzy = dz * yd
        s1, sdzy = dz.sum((1, 2, 3)), dzy.sum((1, 2, 3))
        s2 = sdzy * rs - mu * rs * s1
        del dz, dzy, yd
        records = partial.shape[0] // n
        ns = records // (math.ceil(h / 16) * math.ceil(w / 8))
        seg = math.ceil(d / ns)
        k = (seg + 16) * 2.0 ** -24 * 1.01
        b1 = k * s1                                                  # terms >= 0: sum |t| = sum t
        b2 = k * (rs * sdzy + (mu * rs).abs() * s1)
        rec = partial.double().view(n, records, 2, 32)
        got = rec.sum(1)
        c = e.c0                                                     # real channels (the rest are padding: all zero)
        r1 = ((got[:, 0, :c] - s1[:, :c]).abs() / b1[:, :c]).max().item()
        r2 = ((got[:, 1, :c] - s2[:, :c]).abs() / b2[:, :c]).max().item()
        assert r1 <= 1 and r2 <= 1, (_label(e), r1, r2)
        assert torch.equal(got[:, :, c:], torch.zeros_like(got[:, :, c:]))
        # sensitivity: every record alone is larger than the whole sample's bound
        m1 = (rec[:, :, 0, :c].amin(1) / b1[:, :c]).min().item()
        m2 = (rec[:, :, 1, :c].amin(1) / b2[:, :c]).min().item()
        assert m1 > 1 and m2 > 1, (_label(e), m1, m2)
        print(f"{_label(e)}: seg = {seg}, {records} records per sample; worst error / bound: S1 {r1:.3g}, S2 {r2:.3g}; "
              f"smallest record / bound: S1 {m1:.3g}, S2 {m2:.3g}")


# ---------------------------------------------------------------------------------------------------
# config 4 (t1w, batch 16): tensors of 2^31 elements
# ---------------------------------------------------------------------------------------------------
def _tensor_sizes(e):
    """Element counts of the tensors an entry reads or writes (16-bit elements: bytes are twice these)."""
    n, d, h, w = e.dims
    od, oh, ow = _spec(e).out_dims(d, h, w)
    ins = [n * d * h * w * _pad32(e.c0)] + ([n * d * h * w * _pad32(e.c1)] if e.c1 else [])
    return ins + [n * od * oh * ow * _pad32(e.co)]


def test_config4_batch16_beyond_2gib_bit_exact():
    """Every convolution of a t1w batch-16 step whose source, destination or gradient reaches 2^31 elements or bytes,
    rerun bit-exactly on all 16 samples (an int byte offset or index + extent would corrupt samples 8 .. 15)."""
    entries = [e for e in record_census("t1w", 16, 128) if max(_tensor_sizes(e)) * 2 >= 2 ** 31]
    big = [e for e in entries if max(_tensor_sizes(e)) >= 2 ** 31]
    assert any(e.kind == DECONV_K2S2 and e.c0 == 64 for e in big)
    assert any(e.kind == K3S1P1 and e.c1 == 64 and e.dir == "dgrad" for e in big)
    report = []
    failures = _run_entries(entries, report)
    print(f"\nconfig 4 entries at >= 2^31 bytes: {len(entries)}\n" + "\n".join(report))
    assert not failures, "\n".join(failures)
