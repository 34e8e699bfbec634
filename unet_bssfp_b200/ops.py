"""Tensor-level wrappers over the C ABI (``include/ub_api.h``).

torch is plumbing here: device memory (caching allocator), the current CUDA stream, dtype tags.
Every function enqueues hand-written sm_100a kernels through ``libubssfp.so`` and never falls back
to a torch / cuDNN op. Internal activations and gradients are ``(N, D, H, W, Cp)`` bf16 tensors, ``Cp`` =
channel count padded to a multiple of 32; the raw output ``y`` of a conv that feeds a normalisation is a
``float16`` tensor of the same shape (never a tensor-core operand; see ``include/ub_api.h``).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch

from . import _lib
from ._lib import (ConvDesc, UB_PACK_F16_SRC0, UB_CONV_K1, UB_CONV_K3S1P1, UB_CONV_K4S2P1, UB_CONV_K4S2P1_S2D, UB_DECONV_K2S2,
                   UB_NORM_BATCH_EVAL, UB_NORM_BATCH_TRAIN, UB_NORM_INSTANCE, UB_NORM_NONE)

__all__ = [
    "ConvSpec", "DeferredAct", "UB_PACK_F16_SRC0", "deferred_src0_ok", "pad32", "pack_conv_weights", "pack_conv_weights_multi", "conv_fwd", "conv_dgrad", "conv_wgrad", "conv1x1_to_ncdhw", "conv1x1_from_ncdhw_bwd", "pack_ncdhw", "unpack_ncdhw",
    "pack_patches", "unpack_patch", "paste_patch", "blend_patches", "blend_finish",
    "norm_finalize", "bn_running_update", "norm_act_fwd", "norm_act_bwd", "maxpool_bwd", "colsum", "l1_fwd", "l1_bwd", "bce_logits",
    "scale_by", "relerr_map_reduce", "dti_scalar_maps", "denorm_to_nifti",
]


def pad32(c: int) -> int:
    return (c + 31) // 32 * 32


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require_dtype(t, dtype, what):
    if t is not None and t.dtype != dtype:
        raise RuntimeError(f"{what} must be {dtype}, got {t.dtype}")


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("unet_bssfp_b200 kernels run on CUDA tensors only (there is no CPU fallback)")


@dataclass
class DeferredAct:
    """The activations ``LeakyReLU(Dropout(y * scale + shift))`` of a conv -> norm -> dropout -> LeakyReLU block,
    kept as the block's raw fp16 output and its per-(n, c) constants (``ub_deferred_act``). Consumers apply it on
    their operand path; the activation tensor itself is never materialised."""
    y: torch.Tensor          # (N, D, H, W, 32) float16
    scale: torch.Tensor      # [N][32] fp32
    shift: torch.Tensor
    slope: float
    drop_p: float = 0.0
    drop_seed: int = 0
    f16_operand: bool = False   # conv_fwd only: evaluate in packed fp16 and multiply with fp16-packed weights (no backward)

    @property
    def shape(self):
        return self.y.shape

    @property
    def device(self):
        return self.y.device

    @property
    def is_cuda(self):
        return self.y.is_cuda

    def struct(self):
        if self.y.dtype != torch.float16 or self.y.shape[-1] != 32:
            raise RuntimeError("a deferred activation needs a (N, D, H, W, 32) float16 conv output")
        return _lib.DeferredAct(self.scale.data_ptr(), self.shift.data_ptr(), self.slope, self.drop_p,
                                self.drop_seed & 0xFFFFFFFF, 1 if self.f16_operand else 0)


def _split_deferred(src):
    """-> (tensor whose pointer crosses the ABI, byref(ub_deferred_act) | None, keep-alive)."""
    if isinstance(src, DeferredAct):
        st = src.struct()
        return src.y, C.byref(st), st
    return src, None, None


@dataclass(frozen=True)
class ConvSpec:
    """Static description of one convolution of the hot path (mirrors ``ub_conv_desc``)."""
    kind: int
    c0: int
    co: int
    c1: int = 0

    @property
    def c0p(self):
        return pad32(self.c0)

    @property
    def c1p(self):
        return pad32(self.c1) if self.c1 else 0

    @property
    def cop(self):
        return pad32(self.co)

    def desc(self, n, d, h, w) -> ConvDesc:
        return ConvDesc(self.kind, n, d, h, w, self.c0, self.c0p, self.c1, self.c1p, self.co, self.cop)

    def in_dims(self, src0):
        """(n, d, h, w) of the ORIGINAL input of this conv given its source tensor."""
        if self.kind == UB_CONV_K4S2P1_S2D:      # parity-planar space-to-depth source (n, 8, d/2, h/2, w/2, c0p)
            n, _, d, h, w, _ = src0.shape
            return n, 2 * d, 2 * h, 2 * w
        n, d, h, w, _ = src0.shape
        return n, d, h, w

    def out_dims(self, d, h, w):
        if self.kind in (UB_CONV_K4S2P1, UB_CONV_K4S2P1_S2D):
            return d // 2, h // 2, w // 2
        if self.kind == UB_DECONV_K2S2:
            return d * 2, h * 2, w * 2
        return d, h, w


# ---------------------------------------------------------------------------------------------------
# convolution family
# ---------------------------------------------------------------------------------------------------
def pack_conv_weights(spec: ConvSpec, w: torch.Tensor, direction: int) -> torch.Tensor:
    """fp32 torch-layout weight -> packed bf16 [tap][rows_pad][cols_pad]; direction 0 fwd, 1 dgrad, optionally
    OR-ed with ``UB_PACK_F16_SRC0`` (source-0 columns as fp16, for ``DeferredAct(f16_operand=True)`` sources)."""
    _require_cuda(w)
    lib = _lib.load()
    d = spec.desc(1, 32, 32, 32)
    n = lib.ub_packed_weight_elems(C.byref(d), direction & 1)
    if n < 0:
        _lib.check(-1, "ub_packed_weight_elems")
    out = torch.empty(n, dtype=torch.bfloat16, device=w.device)
    w32 = w.detach().contiguous().float()
    _lib.check(lib.ub_pack_conv_weights(C.byref(d), direction, _p(w32), _p(out), _stream()), "ub_pack_conv_weights")
    return out


def deferred_src0_ok(spec: ConvSpec, n, d, h, w) -> bool:
    """True when source 0 of this convolution may be a ``DeferredAct`` (forward and weight gradient)."""
    desc = spec.desc(n, d, h, w)
    r = _lib.load().ub_conv_deferred_src0_ok(C.byref(desc))
    if r < 0:
        _lib.check(-1, "ub_conv_deferred_src0_ok")
    return r == 1


def pack_conv_weights_multi(items):
    """``items``: list of (spec, fp32 weight, direction). One multi-tensor launch (per 32 weights) -> list of packed
    bf16 tensors, read from the live parameter memory."""
    if not items:
        return []
    lib = _lib.load()
    table = (_lib.WeightPackItem * len(items))()
    outs, keep = [], []
    for k, (spec, w, direction) in enumerate(items):
        _require_cuda(w)
        d = spec.desc(1, 32, 32, 32)
        n = lib.ub_packed_weight_elems(C.byref(d), direction & 1)
        if n < 0:
            _lib.check(-1, "ub_packed_weight_elems")
        w32 = w.detach()
        if w32.dtype != torch.float32 or not w32.is_contiguous():
            w32 = w32.contiguous().float()
        keep.append(w32)
        out = torch.empty(n, dtype=torch.bfloat16, device=w.device)
        outs.append(out)
        table[k].desc = d
        table[k].dir = direction
        table[k].w = w32.data_ptr()
        table[k].packed = out.data_ptr()
    _lib.check(lib.ub_pack_conv_weights_multi(table, len(items), _stream()), "ub_pack_conv_weights_multi")
    return outs


def conv_fwd(spec: ConvSpec, src0, src1, w_packed, bias, act=0, slope=0.0, want_stats=False):
    """-> (out (N,Do,Ho,Wo,cop), stats_partial [tiles][2][cop] fp32 | None). ``out`` is bf16, or -- with
    ``want_stats``, where it is the raw input ``y`` of a normalisation -- float16. ``src0`` may be a
    ``DeferredAct`` where ``deferred_src0_ok``."""
    _require_cuda(src0, src1, w_packed, bias)
    lib = _lib.load()
    n, d, h, w = spec.in_dims(src0)
    desc = spec.desc(n, d, h, w)
    od, oh, ow = spec.out_dims(d, h, w)
    s0, act0, _keep = _split_deferred(src0)
    src0_f16 = 1 if (act0 is None and s0.dtype == torch.float16) else 0     # a materialised fp16 operand copy
    if act0 is None and not src0_f16:
        _require_dtype(s0, torch.bfloat16, "conv_fwd: src0")
    _require_dtype(src1, torch.bfloat16, "conv_fwd: src1")
    out = torch.empty((n, od, oh, ow, spec.cop), dtype=torch.float16 if want_stats else torch.bfloat16, device=s0.device)
    stats = None
    if want_stats:
        tiles = lib.ub_conv_num_tiles(C.byref(desc))
        stats = torch.empty((tiles, 2, spec.cop), dtype=torch.float32, device=s0.device)
    _lib.check(lib.ub_conv_fwd(C.byref(desc), _p(s0), _p(src1), _p(w_packed), _p(bias), act, slope, _p(out),
                               _p(stats), act0, src0_f16, _stream()), "ub_conv_fwd")
    return out, stats


@dataclass
class NormBwdFusion:
    """Saved tensors of the block that PRODUCED a conv's input: lets that conv's dgrad epilogue
    accumulate the block's norm-backward reductions (``ub_norm_bwd_fuse``)."""
    y: torch.Tensor
    scale: torch.Tensor
    shift: torch.Tensor
    mean: torch.Tensor
    rstd: torch.Tensor
    slope: float
    drop_p: float
    drop_seed: int


def dgrad_fuse_records(spec: ConvSpec, n, d, h, w) -> int:
    """Number of partial records ``conv_dgrad(..., fuse=)`` would emit; 0 when the fusion is unavailable."""
    desc = spec.desc(n, d, h, w)
    r = _lib.load().ub_conv_dgrad_fuse_records(C.byref(desc))
    if r < 0:
        _lib.check(-1, "ub_conv_dgrad_fuse_records")
    return r


def conv_dgrad(spec: ConvSpec, dy, w_packed_dgrad, in_dhw, fuse: NormBwdFusion | None = None):
    """dy (N,Do,Ho,Wo,cop) -> (dsrc0, dsrc1|None), each (N,d,h,w,c*p) bf16.
    With ``fuse`` -> (dsrc0, dsrc1, partial [records][2][32] fp32): norm-backward sums of the producer block."""
    _require_cuda(dy, w_packed_dgrad)
    lib = _lib.load()
    n = dy.shape[0]
    d, h, w = in_dhw
    desc = spec.desc(n, d, h, w)
    d0 = torch.empty((n, d, h, w, spec.c0p), dtype=torch.bfloat16, device=dy.device)
    d1 = torch.empty((n, d, h, w, spec.c1p), dtype=torch.bfloat16, device=dy.device) if spec.c1 else None
    if fuse is None:
        _lib.check(lib.ub_conv_dgrad(C.byref(desc), _p(dy), _p(w_packed_dgrad), _p(d0), _p(d1), _stream()), "ub_conv_dgrad")
        return d0, d1
    records = lib.ub_conv_dgrad_fuse_records(C.byref(desc))
    if records <= 0:
        raise RuntimeError("conv_dgrad: the norm-backward fusion is not available for this convolution")
    partial = torch.empty((records, 2, 32), dtype=torch.float32, device=dy.device)
    f = _lib.NormBwdFuse(fuse.y.data_ptr(), fuse.scale.data_ptr(), fuse.shift.data_ptr(), fuse.mean.data_ptr(),
                         fuse.rstd.data_ptr(), fuse.slope, fuse.drop_p, fuse.drop_seed & 0xFFFFFFFF, partial.data_ptr())
    _lib.check(lib.ub_conv_dgrad_fused(C.byref(desc), _p(dy), _p(w_packed_dgrad), _p(d0), _p(d1), C.byref(f), _stream()),
               "ub_conv_dgrad_fused")
    return d0, d1, partial


def conv_wgrad(spec: ConvSpec, src0, src1, dy, weight_shape):
    """-> dw fp32 in the torch weight layout ``weight_shape``."""
    _require_cuda(src0, src1, dy)
    lib = _lib.load()
    n, d, h, w = spec.in_dims(src0)
    desc = spec.desc(n, d, h, w)
    nbytes = lib.ub_conv_wgrad_workspace_bytes(C.byref(desc))
    if nbytes < 0:
        _lib.check(-1, "ub_conv_wgrad_workspace_bytes")
    s0, act0, _keep = _split_deferred(src0)
    if act0 is None:
        _require_dtype(s0, torch.bfloat16, "conv_wgrad: src0")
    _require_dtype(dy, torch.bfloat16, "conv_wgrad: dy")
    ws = torch.empty(nbytes // 4, dtype=torch.float32, device=dy.device)
    dw = torch.zeros(weight_shape, dtype=torch.float32, device=dy.device)
    _lib.check(lib.ub_conv_wgrad(C.byref(desc), _p(s0), _p(src1), _p(dy), _p(ws), _p(dw), act0, _stream()),
               "ub_conv_wgrad")
    return dw


def conv1x1_to_ncdhw(u, weight, bias):
    """Generator output head: u (N,D,H,W,32) bf16 (or a ``DeferredAct``), weight (co, ci, 1,1,1) fp32, bias (co)
    -> (N,co,D,H,W) fp32."""
    _require_cuda(u, weight, bias)
    lib = _lib.load()
    u, act0, _keep = _split_deferred(u)
    n, d, h, w, cp = u.shape
    co, ci = weight.shape[0], weight.shape[1]
    ws = torch.empty(lib.ub_conv1x1_workspace_bytes() // 4, dtype=torch.float32, device=u.device)
    out = torch.empty((n, co, d, h, w), dtype=torch.float32, device=u.device)
    wt = weight.detach().contiguous().float()
    _lib.check(lib.ub_conv1x1_to_ncdhw(_p(u), cp, _p(wt), ci, _p(bias), co, n, d * h * w, _p(ws), _p(out), act0,
                                       _stream()), "ub_conv1x1_to_ncdhw")
    return out


def conv1x1_from_ncdhw_bwd(dout, u, weight, need_input=True, need_params=True):
    """Backward of ``conv1x1_to_ncdhw`` in one pass: -> (du (N,D,H,W,32) bf16 | None, dweight | None, dbias | None)."""
    _require_cuda(dout, u, weight)
    lib = _lib.load()
    u, act0, _keep = _split_deferred(u)
    n, d, h, w, cp = u.shape
    co, ci = weight.shape[0], weight.shape[1]
    dout = dout.contiguous().float()
    ws = torch.empty(lib.ub_conv1x1_workspace_bytes() // 4, dtype=torch.float32, device=u.device)
    du = torch.empty(u.shape, dtype=torch.bfloat16, device=u.device) if need_input else None
    dw = torch.empty(tuple(weight.shape), dtype=torch.float32, device=u.device) if need_params else None
    db = torch.empty(co, dtype=torch.float32, device=u.device) if need_params else None
    wt = weight.detach().contiguous().float()
    _lib.check(lib.ub_conv1x1_from_ncdhw_bwd(_p(dout), co, _p(u), cp, _p(wt), ci, n, d * h * w, _p(ws), _p(du), _p(dw),
                                             _p(db), act0, _stream()), "ub_conv1x1_from_ncdhw_bwd")
    return du, dw, db


def head_bwd_fused_ok(dout, fuse) -> bool:
    """``head_bwd_fused`` serves this call: 32-channel block, voxels per sample a multiple of 16, <= 8 outputs."""
    n, co = dout.shape[0], dout.shape[1]
    vox = dout.shape[2] * dout.shape[3] * dout.shape[4]
    return fuse is not None and fuse.y.shape[-1] == 32 and vox % 16 == 0 and co <= 8


def head_bwd_fused(dout, fuse: NormBwdFusion, weight, mode, c, need_params=True, want_block_grads=True):
    """Backward of ``conv1x1_to_ncdhw`` on the DEFERRED activations of the block described by ``fuse``, fused with that
    block's norm backward (``ub_head_bwd_fused``): -> (dy of the block (N,D,H,W,32) bf16, dgamma, dbeta, dbias of the
    block | None, dweight, dbias of the head | None). ``du`` is never materialised."""
    _require_cuda(dout, weight)
    lib = _lib.load()
    y = fuse.y
    _require_dtype(y, torch.float16, "head_bwd_fused: y")
    n, d, h, w, cp = y.shape
    co, ci = weight.shape[0], weight.shape[1]
    dev = y.device
    dout = dout.contiguous().float()
    ws = torch.empty(lib.ub_head_bwd_fused_workspace_bytes(n) // 4, dtype=torch.float32, device=dev)
    dy = torch.empty(y.shape, dtype=torch.bfloat16, device=dev)
    dgamma = dbeta = dbias = dw = db = None
    if want_block_grads:
        dgamma = torch.empty(c, dtype=torch.float32, device=dev)
        dbeta = torch.empty(c, dtype=torch.float32, device=dev)
        dbias = torch.empty(c, dtype=torch.float32, device=dev)
    if need_params:
        dw = torch.empty(tuple(weight.shape), dtype=torch.float32, device=dev)
        db = torch.empty(co, dtype=torch.float32, device=dev)
    wt = weight.detach().contiguous().float()
    f = _lib.NormBwdFuse(y.data_ptr(), fuse.scale.data_ptr(), fuse.shift.data_ptr(), fuse.mean.data_ptr(),
                         fuse.rstd.data_ptr(), fuse.slope, fuse.drop_p, fuse.drop_seed & 0xFFFFFFFF, None)
    _lib.check(lib.ub_head_bwd_fused(_p(dout), co, _p(wt), ci, n, d * h * w, C.byref(f), mode, c, _p(ws), _p(dy),
                                     _p(dgamma), _p(dbeta), _p(dbias), _p(dw), _p(db), _stream()), "ub_head_bwd_fused")
    return dy, dgamma, dbeta, dbias, dw, db


# ---------------------------------------------------------------------------------------------------
# layout
# ---------------------------------------------------------------------------------------------------
class _WidenedInput:
    """fp32 image of the most recent bf16 module input (opt-in, ``UB_WIDEN_BF16=1``). A bf16 ``x`` is a transport format
    (half the host-to-device bytes of the conditioning input); one training step packs it four times (generator
    input + the three PatchGAN calls). Round 2 first widened it once per tensor version because the two-voxels-per-
    thread bf16 pack kernel ran at 2.25 ms against 0.41 ms for the fp32 kernel; that was a code-generation problem
    (loads in separate basic blocks, then funnelled through one register -- see pack_ncdhw_a16_kernel), fixed since:
    0.45 / 0.68 ms plain / space-to-depth, and a whole step is ~1 ms faster without the 1.6 GB widened copy. Kept for
    A/B. Held through a weak reference: the cache never extends the life of a batch."""

    def __init__(self):
        self._ref = self._key = self._wide = None

    def get(self, x):
        key = (x.data_ptr(), x._version, tuple(x.shape), x.device)
        if self._ref is not None and self._ref() is x and self._key == key:
            return self._wide
        import weakref
        wide = x.float()
        self._key, self._wide = key, wide
        self._ref = weakref.ref(x, lambda _: self.clear())
        return wide

    def clear(self):
        self._ref = self._key = self._wide = None


_widened_input = _WidenedInput()
import os as _os
_WIDEN_BF16_INPUT = _os.environ.get("UB_WIDEN_BF16", "0") == "1"      # default: bf16 inputs go to the pack kernels as they are


def pack_ncdhw(a: torch.Tensor, b: torch.Tensor | None = None, s2d: bool = False) -> torch.Tensor:
    """cat[a, b] NCDHW fp32 -> (N,D,H,W,Cp) bf16; ``s2d``: parity-planar space-to-depth layout
    (N, 8 = (pd,ph,pw), D/2, H/2, W/2, Cp) -- the input layout of the stride-2 PatchGAN stem."""
    _require_cuda(a, b)
    lib = _lib.load()
    if a.dtype == torch.bfloat16 and _WIDEN_BF16_INPUT and a.is_contiguous():
        a = _widened_input.get(a)
    a16 = 1 if a.dtype == torch.bfloat16 else 0          # a bf16 input is read as it is (bit-identical pack)
    a = a.contiguous() if a16 else a.contiguous().float()
    n, ca, d, h, w = a.shape
    cb = 0
    if b is not None:
        b = b.contiguous().float()
        cb = b.shape[1]
    cp = pad32(ca + cb)
    if s2d:
        out = torch.empty((n, 8, d // 2, h // 2, w // 2, cp), dtype=torch.bfloat16, device=a.device)
        _lib.check(lib.ub_pack_ncdhw_s2d(_p(a), a16, ca, _p(b), cb, n, d, h, w, cp, _p(out), _stream()),
                   "ub_pack_ncdhw_s2d")
        return out
    out = torch.empty((n, d, h, w, cp), dtype=torch.bfloat16, device=a.device)
    _lib.check(lib.ub_pack_ncdhw(_p(a), a16, ca, _p(b), cb, n, d * h * w, cp, _p(out), _stream()), "ub_pack_ncdhw")
    return out


def to_s2d(a: torch.Tensor) -> torch.Tensor:
    """(N,D,H,W,Cp) bf16 -> (N, 8 = (pd,ph,pw), D/2, H/2, W/2, Cp): the parity-planar space-to-depth layout a
    ``UB_CONV_K4S2P1_S2D`` conv reads (a permuting copy)."""
    _require_cuda(a)
    _require_dtype(a, torch.bfloat16, "to_s2d")
    n, d, h, w, cp = a.shape
    out = torch.empty((n, 8, d // 2, h // 2, w // 2, cp), dtype=torch.bfloat16, device=a.device)
    _lib.check(_lib.load().ub_to_s2d(_p(a.contiguous()), n, d, h, w, cp, _p(out), _stream()), "ub_to_s2d")
    return out


def pack_patches(volume: torch.Tensor, origins, patch, out: torch.Tensor | None = None) -> torch.Tensor:
    """Gather ``len(origins)`` patches of an NCDHW fp32 volume (1,C,D,H,W) or (C,D,H,W) into one
    (n, pd, ph, pw, Cp) bf16 batch. ``origins``: (z, y, x) starts; ``patch``: (pd, ph, pw). ``out``: write into the
    first ``len(origins)`` samples of this existing batch tensor (the static input of a captured CUDA graph)."""
    _require_cuda(volume)
    lib = _lib.load()
    vol = volume if volume.dim() == 4 else volume[0]
    if vol.dtype != torch.float32 or vol.stride(-1) != 1:
        vol = vol.float().contiguous()
    c, D, H, W = vol.shape
    pd, ph, pw = patch
    sc, sd, sh, _ = vol.stride()
    n = len(origins)
    offs = (C.c_longlong * n)(*[z * sd + y * sh + x for (z, y, x) in origins])
    for (z, y, x) in origins:
        if z < 0 or y < 0 or x < 0 or z + pd > D or y + ph > H or x + pw > W:
            raise RuntimeError(f"patch at {(z, y, x)} of size {patch} leaves the volume {(D, H, W)}")
    cp = pad32(c)
    if out is None:
        out = torch.empty((n, pd, ph, pw, cp), dtype=torch.bfloat16, device=vol.device)
    elif (out.dtype != torch.bfloat16 or not out.is_contiguous() or out.shape[0] < n
          or tuple(out.shape[1:]) != (pd, ph, pw, cp)):
        raise RuntimeError("pack_patches: `out` must be a contiguous (>= n, pd, ph, pw, Cp) bf16 tensor")
    _lib.check(lib.ub_pack_patches(_p(vol), c, n, offs, pd, ph, pw, sc, sd, sh, cp, _p(out), _stream()), "ub_pack_patches")
    return out


def unpack_patch(batch: torch.Tensor, sample: int, c: int, volume: torch.Tensor, origin, c_begin: int = 0):
    """Write channels [c_begin, c_begin+c) of ``batch[sample]`` (NDHWC bf16) into the (c,D,H,W) fp32
    ``volume`` at ``origin``; the later call wins where patches overlap."""
    _require_cuda(batch, volume)
    lib = _lib.load()
    if volume.dtype != torch.float32 or volume.dim() != 4 or volume.stride(-1) != 1:
        raise RuntimeError("unpack_patch writes into a (C,D,H,W) fp32 tensor with contiguous rows")
    _, pd, ph, pw, cp = batch.shape
    z, y, x = origin
    sc, sd, sh, _ = volume.stride()
    _, D, H, W = volume.shape
    if z < 0 or y < 0 or x < 0 or z + pd > D or y + ph > H or x + pw > W or volume.shape[0] < c:
        raise RuntimeError(f"patch at {origin} of size {(pd, ph, pw)} leaves the volume {(D, H, W)}")
    _lib.check(lib.ub_unpack_patch(_p(batch), cp, c_begin, c, sample, pd, ph, pw, _p(volume), z * sd + y * sh + x, sc, sd,
                                   sh, _stream()), "ub_unpack_patch")


def paste_patch(patch: torch.Tensor, volume: torch.Tensor, origin):
    """Write an NCDHW fp32 patch (c, pd, ph, pw) into the (c, D, H, W) fp32 ``volume`` at ``origin`` (later wins)."""
    _require_cuda(patch, volume)
    lib = _lib.load()
    if patch.dtype != torch.float32 or not patch.is_contiguous():
        patch = patch.float().contiguous()
    if volume.dtype != torch.float32 or volume.dim() != 4 or volume.stride(-1) != 1:
        raise RuntimeError("paste_patch writes into a (C,D,H,W) fp32 tensor with contiguous rows")
    c, pd, ph, pw = patch.shape
    z, y, x = origin
    sc, sd, sh, _ = volume.stride()
    _, D, H, W = volume.shape
    if z < 0 or y < 0 or x < 0 or z + pd > D or y + ph > H or x + pw > W or volume.shape[0] < c:
        raise RuntimeError(f"patch at {origin} of size {(pd, ph, pw)} leaves the volume {(D, H, W)}")
    _lib.check(lib.ub_paste_patch(_p(patch), c, pd, ph, pw, _p(volume), z * sd + y * sh + x, sc, sd, sh, _stream()),
               "ub_paste_patch")


BLEND_MODES = ("crop", "average", "hann")


def blend_patches(patches: torch.Tensor, volume: torch.Tensor, origins, mode: str = "crop", boxes=None,
                  weight: torch.Tensor | None = None, window: torch.Tensor | None = None):
    """Aggregate a batch of NCDHW fp32 patches (n, c, pd, ph, pw), in sampler order, into the contiguous (c, D, H, W)
    fp32 ``volume`` in one launch (torchio ``GridAggregator.add_batch``). ``origins``: (z, y, x) per patch; ``boxes``:
    (z0, y0, x0, z1, y1, x1) volume region each patch writes (default: the whole patch). ``mode``: "crop" (the later
    patch wins), "average" (``volume += p``, ``weight += 1``) or "hann" (``volume += p * w``, ``weight += w``,
    ``w = (wz * wy) * wx`` from ``window`` = cat[wz, wy, wx], fp32 on the device). ``weight``: contiguous (D, H, W) fp32,
    needed by the accumulating modes; ``blend_finish`` divides once after the last batch."""
    _require_cuda(patches, volume, weight, window)
    lib = _lib.load()
    if mode not in BLEND_MODES:
        raise ValueError(f"overlap mode must be one of {BLEND_MODES}, got {mode!r}")
    if patches.dtype != torch.float32 or not patches.is_contiguous() or patches.dim() != 5:
        raise RuntimeError("blend_patches reads a contiguous (n, c, pd, ph, pw) fp32 tensor")
    if volume.dtype != torch.float32 or volume.dim() != 4 or not volume.is_contiguous():
        raise RuntimeError("blend_patches writes into a contiguous (C, D, H, W) fp32 tensor")
    n, c, pd, ph, pw = patches.shape
    _, D, H, W = volume.shape
    if volume.shape[0] != c or len(origins) != n:
        raise RuntimeError(f"blend_patches: {n} patches of {c} channels, {len(origins)} origins, volume {tuple(volume.shape)}")
    if mode != "crop" and (weight is None or weight.dtype != torch.float32 or tuple(weight.shape) != (D, H, W)
                           or not weight.is_contiguous()):
        raise RuntimeError(f"blend_patches: mode {mode!r} needs a contiguous ({D}, {H}, {W}) fp32 weight volume")
    if mode == "hann" and (window is None or window.dtype != torch.float32 or window.numel() != pd + ph + pw):
        raise RuntimeError(f"blend_patches: hann mode needs the {pd} + {ph} + {pw} fp32 window values")
    orgs = (C.c_int * (3 * n))(*[v for o in origins for v in o])
    bx = None if boxes is None else (C.c_int * (6 * n))(*[v for b in boxes for v in b])
    _lib.check(lib.ub_blend_patches(_p(patches), n, c, pd, ph, pw, orgs, bx, BLEND_MODES.index(mode),
                                    _p(window.contiguous()) if mode == "hann" else None, _p(volume),
                                    _p(weight) if mode != "crop" else None, D, H, W, _stream()), "ub_blend_patches")


def blend_finish(volume: torch.Tensor, weight: torch.Tensor):
    """``volume /= weight`` in place over every channel: the end of an accumulating ``blend_patches`` sequence."""
    _require_cuda(volume, weight)
    if (volume.dtype != torch.float32 or volume.dim() != 4 or not volume.is_contiguous() or weight.dtype != torch.float32
            or tuple(weight.shape) != tuple(volume.shape[1:]) or not weight.is_contiguous()):
        raise RuntimeError("blend_finish: a contiguous (C, D, H, W) fp32 volume and its (D, H, W) fp32 weight")
    _lib.check(_lib.load().ub_blend_finish(_p(volume), _p(weight), volume.shape[0], weight.numel(), _stream()),
               "ub_blend_finish")


def unpack_ncdhw(x: torch.Tensor, c: int, c_begin: int = 0) -> torch.Tensor:
    """(N,D,H,W,Cp) bf16 -> NCDHW fp32 of channels [c_begin, c_begin + c)."""
    _require_cuda(x)
    lib = _lib.load()
    n, d, h, w, cp = x.shape
    out = torch.empty((n, c, d, h, w), dtype=torch.float32, device=x.device)
    _lib.check(lib.ub_unpack_ncdhw(_p(x), cp, c_begin, c, n, d * h * w, _p(out), _stream()), "ub_unpack_ncdhw")
    return out


# ---------------------------------------------------------------------------------------------------
# norm / dropout / activation
# ---------------------------------------------------------------------------------------------------
def norm_finalize(stats, n, voxels, cp, c, gamma, beta, eps, mode, momentum=0.1, running_mean=None,
                  running_var=None):
    """-> (scale, shift, mean, rstd), each [n][cp] fp32."""
    lib = _lib.load()
    dev = gamma.device
    scale = torch.empty((n, cp), dtype=torch.float32, device=dev)
    shift = torch.empty_like(scale)
    mean = torch.empty_like(scale)
    rstd = torch.empty_like(scale)
    tiles_per_sample = 0 if stats is None else stats.shape[0] // n
    _lib.check(lib.ub_norm_finalize(_p(stats), tiles_per_sample, n, cp, c, float(voxels), _p(gamma), _p(beta), eps,
                                    mode, momentum, _p(running_mean), _p(running_var), _p(scale), _p(shift), _p(mean),
                                    _p(rstd), _stream()), "ub_norm_finalize")
    return scale, shift, mean, rstd


def bn_running_update(mean, rstd, c, count, eps, momentum, running_mean, running_var):
    """Deferred BatchNorm running-statistics update from saved batch statistics (``norm_finalize`` without buffers)."""
    _lib.check(_lib.load().ub_bn_running_update(_p(mean), _p(rstd), c, float(count), eps, momentum, _p(running_mean),
                                                _p(running_var), _stream()), "ub_bn_running_update")


def norm_act_fwd(y, scale, shift, slope, drop_p=0.0, drop_seed=0, pool=False, materialize=True, f16_copy=False):
    """y (float16) -> (a bf16 | None, pooled bf16 | None), or with ``f16_copy`` -> (a, pooled, a16): ``a16`` holds the
    same fp32 values rounded to float16 -- the operand copy a marching forward conv takes as source 0 (fp16 x fp16
    MMAs). ``materialize=False`` (needs ``pool`` or ``f16_copy``): the bf16 tensor is not written."""
    lib = _lib.load()
    _require_dtype(y, torch.float16, "norm_act_fwd: y")
    if not materialize and not pool and not f16_copy:
        raise RuntimeError("norm_act_fwd: nothing to compute (materialize=False without pool / f16_copy)")
    n, d, h, w, cp = y.shape
    a = torch.empty(y.shape, dtype=torch.bfloat16, device=y.device) if materialize else None
    a16 = torch.empty(y.shape, dtype=torch.float16, device=y.device) if f16_copy else None
    pooled = torch.empty((n, d // 2, h // 2, w // 2, cp), dtype=torch.bfloat16, device=y.device) if pool else None
    _lib.check(lib.ub_norm_act_fwd(_p(y), _p(scale), _p(shift), slope, drop_p, drop_seed & 0xFFFFFFFF, n, d, h, w, cp,
                                   _p(a), _p(a16), _p(pooled), _stream()), "ub_norm_act_fwd")
    return (a, pooled, a16) if f16_copy else (a, pooled)


def norm_act_bwd(dA, a, y, mode, mean, rstd, scale, slope, drop_p, drop_seed, c, want_param_grads=True,
                 want_bias_grad=True, shift=None, partial=None):
    """-> (dy, dgamma|None, dbeta|None, dbias|None). With ``shift`` (norm modes) the activation sign is
    recomputed from ``y`` and ``a`` is not read (may be None). ``partial``: reduction records already
    accumulated by ``conv_dgrad(..., fuse=)`` -- the reduction pass is skipped."""
    lib = _lib.load()
    _require_dtype(dA, torch.bfloat16, "norm_act_bwd: dA")
    _require_dtype(y, torch.float16, "norm_act_bwd: y")
    n, d, h, w, cp = dA.shape
    voxels = d * h * w
    dev = dA.device
    dy = torch.empty_like(dA)
    ws = None
    dgamma = dbeta = dbias = None
    if mode != UB_NORM_NONE:
        ws = torch.empty(lib.ub_norm_act_bwd_workspace_bytes(n, cp) // 4, dtype=torch.float32, device=dev)
        if want_param_grads:
            dgamma = torch.empty(c, dtype=torch.float32, device=dev)
            dbeta = torch.empty(c, dtype=torch.float32, device=dev)
        if want_bias_grad:
            dbias = torch.empty(c, dtype=torch.float32, device=dev)
    _lib.check(lib.ub_norm_act_bwd(_p(dA), _p(a), _p(y), mode, _p(mean), _p(rstd), _p(scale), _p(shift), slope, drop_p,
                                   drop_seed & 0xFFFFFFFF, n, voxels, cp, c, _p(ws), _p(dy), _p(dgamma), _p(dbeta),
                                   _p(dbias), _p(partial), 0 if partial is None else partial.shape[0] // n, _stream()),
               "ub_norm_act_bwd")
    return dy, dgamma, dbeta, dbias


def maxpool_bwd(a, dP, dA=None):
    """Route dP to the arg-max voxels of ``a`` (bf16 tensor or ``DeferredAct``); accumulates onto ``dA`` if given,
    else creates it."""
    lib = _lib.load()
    a, act0, _keep = _split_deferred(a)
    n, d, h, w, cp = a.shape
    acc = 1
    if dA is None:
        dA = torch.empty(a.shape, dtype=torch.bfloat16, device=a.device)
        acc = 0
    _lib.check(lib.ub_maxpool_bwd(_p(a), _p(dP), _p(dA), acc, n, d, h, w, cp, act0, _stream()), "ub_maxpool_bwd")
    return dA


def maxpool_bwd_fuse_records(n, d, h, w, cp) -> int:
    """Partial records ``maxpool_bwd_fused`` emits for an (n, d, h, w, cp) activation tensor; 0 = unsupported."""
    return _lib.load().ub_maxpool_bwd_fuse_records(n, d, h, w, cp)


def maxpool_bwd_fused(dP, dA, fuse: NormBwdFusion):
    """Max-pool backward of a conv -> norm block whose dA is complete after this pass, fused with that block's
    norm-backward reduction: routes ``dP`` onto the arg-max voxels of the activations recomputed from ``fuse.y``
    (accumulating onto ``dA`` if given) -> (dA, partial [records][2][cp]) for ``norm_act_bwd(partial=)``."""
    lib = _lib.load()
    y = fuse.y
    _require_dtype(y, torch.float16, "maxpool_bwd_fused: y")
    n, d, h, w, cp = y.shape
    records = lib.ub_maxpool_bwd_fuse_records(n, d, h, w, cp)
    if records <= 0:
        raise RuntimeError("maxpool_bwd_fused: unsupported shape")
    acc = 1
    if dA is None:
        dA = torch.empty(y.shape, dtype=torch.bfloat16, device=y.device)
        acc = 0
    partial = torch.empty((records, 2, cp), dtype=torch.float32, device=y.device)
    f = _lib.NormBwdFuse(y.data_ptr(), fuse.scale.data_ptr(), fuse.shift.data_ptr(), fuse.mean.data_ptr(),
                         fuse.rstd.data_ptr(), fuse.slope, fuse.drop_p, fuse.drop_seed & 0xFFFFFFFF, partial.data_ptr())
    _lib.check(lib.ub_maxpool_bwd_fused(_p(dP), _p(dA), acc, n, d, h, w, cp, C.byref(f), _stream()),
               "ub_maxpool_bwd_fused")
    return dA, partial


def colsum(x, c):
    lib = _lib.load()
    cp = x.shape[-1]
    rows = x.numel() // cp
    ws = torch.empty(lib.ub_colsum_workspace_bytes(cp) // 4, dtype=torch.float32, device=x.device)
    out = torch.empty(c, dtype=torch.float32, device=x.device)
    _lib.check(lib.ub_colsum(_p(x), rows, cp, c, _p(ws), _p(out), _stream()), "ub_colsum")
    return out


# ---------------------------------------------------------------------------------------------------
# losses
# ---------------------------------------------------------------------------------------------------
_l1_ws = {}


def _l1_workspace(dev):
    ws = _l1_ws.get(dev)
    if ws is None:
        ws = torch.zeros(_lib.load().ub_l1_workspace_bytes() // 8 + 1, dtype=torch.float64, device=dev)
        _l1_ws[dev] = ws
    return ws


def l1_fwd(a, b):
    lib = _lib.load()
    loss = torch.empty((), dtype=torch.float32, device=a.device)
    _lib.check(lib.ub_l1_fwd(_p(a), _p(b), a.numel(), _p(_l1_workspace(a.device)), _p(loss), _stream()), "ub_l1_fwd")
    return loss


def l1_bwd(a, b, grad_out):
    lib = _lib.load()
    da = torch.empty_like(a)
    _lib.check(lib.ub_l1_bwd(_p(a), _p(b), _p(grad_out), a.numel(), _p(da), _stream()), "ub_l1_bwd")
    return da


def bce_logits(x, target, want_grad=True):
    """target: python float (constant) or a tensor shaped like x."""
    lib = _lib.load()
    loss = torch.empty((), dtype=torch.float32, device=x.device)
    dx = torch.empty_like(x) if want_grad else None
    tptr, tconst = (None, float(target)) if not torch.is_tensor(target) else (_p(target), 0.0)
    _lib.check(lib.ub_bce_logits(_p(x), tptr, tconst, x.numel(), _p(loss), _p(dx), _stream()), "ub_bce_logits")
    return loss, dx


def scale_by(x, scalar):
    lib = _lib.load()
    y = torch.empty_like(x)
    _lib.check(lib.ub_scale(_p(x), _p(scalar), x.numel(), _p(y), _stream()), "ub_scale")
    return y


# ---------------------------------------------------------------------------------------------------
# evaluation
# ---------------------------------------------------------------------------------------------------
def relerr_map_reduce(pred, target, mask=None, probseg=None, angular=False, want_map=True):
    """pred/target: (..., C) fp32 channel-last. -> (diff|None, sums [R][C] f64|None, norms [R] f64|None)."""
    _require_cuda(pred, target, mask, probseg)
    lib = _lib.load()
    c = pred.shape[-1]
    voxels = pred.numel() // c
    diff = torch.empty_like(pred) if want_map else None
    sums = norms = None
    r = 0
    if probseg is not None:
        r = probseg.shape[-1]
        sums = torch.empty((r, c), dtype=torch.float64, device=pred.device)
        norms = torch.empty((r,), dtype=torch.float64, device=pred.device)
    _lib.check(lib.ub_relerr_map_reduce(_p(pred), _p(target), _p(mask), _p(probseg), c, r, voxels, int(angular),
                                        _p(diff), _p(sums), _p(norms), _stream()), "ub_relerr_map_reduce")
    return diff, sums, norms


def dti_scalar_maps(tensor6: torch.Tensor):
    """(..., 6) fp32 channel-last diffusion tensors -> dict of fp32 maps: fa, md, ad, rd, azimuth,
    inclination (shape ...) and rgb (..., 3). ref:src/eval.py:73-116."""
    _require_cuda(tensor6)
    lib = _lib.load()
    t = tensor6.contiguous().float()
    if t.shape[-1] != 6:
        raise RuntimeError("dti_scalar_maps expects the 6 unique tensor components in the last dimension")
    shape = t.shape[:-1]
    out = {k: torch.empty(shape, dtype=torch.float32, device=t.device) for k in ("fa", "md", "ad", "rd", "azimuth", "inclination")}
    out["rgb"] = torch.empty(tuple(shape) + (3,), dtype=torch.float32, device=t.device)
    _lib.check(lib.ub_dti_scalar_maps(_p(t), t.numel() // 6, _p(out["fa"]), _p(out["md"]), _p(out["ad"]), _p(out["rd"]),
                                      _p(out["azimuth"]), _p(out["inclination"]), _p(out["rgb"]), _stream()),
               "ub_dti_scalar_maps")
    return out


def denorm_to_nifti(volume: torch.Tensor, scale: float = 1.0, offset: float = 0.0):
    """(C,X,Y,Z) fp32 -> (C,Z,Y,X) fp32 = NIfTI storage order of the channel-last array, values
    ``v * scale + offset`` evaluated in fp64 (ref:src/eval.py:39-47, ref:src/model.py:344-346)."""
    _require_cuda(volume)
    if volume.dim() != 4:
        raise RuntimeError("denorm_to_nifti expects one (C,X,Y,Z) volume")
    v = volume.contiguous().float()
    c, x, y, z = v.shape
    out = torch.empty((c, z, y, x), dtype=torch.float32, device=v.device)
    _lib.check(_lib.load().ub_denorm_to_nifti(_p(v), c, x, y, z, float(scale), float(offset), _p(out), _stream()),
               "ub_denorm_to_nifti")
    return out
