"""Whole-volume sliding-window inference and its evaluation, on device.

Mirrors what ``predict_step`` / ``test_step`` of the reference do with torchio (ref:src/model.py:291-333,
ref:src/data_module.py:168-183; torchio==0.19.6 ``GridSampler(subject, patch_size, patch_overlap)`` and
``GridAggregator(sampler, overlap_mode)``; the reference uses the defaults, overlap 0 and ``'crop'``): the volume
is covered by a grid of patches whose last patch per axis is shifted back to end at the border, every patch goes
through the generator, and ``add_batch`` aggregates each prediction into the output volume in sampler order --
in ``'crop'`` mode the later patch wins where the cropped patches overlap; ``'average'`` and ``'hann'`` blend them.

Here the sampler and aggregator are index arithmetic inside the kernels (``ub_pack_patches`` gathers a batch,
``ub_blend_patches`` aggregates it in one launch): no host round trip and no host-side patch tensors.
``relative_error`` then runs the fused error-map + ROI reduction of ref:src/eval.py:154-166,217-258.
"""
from __future__ import annotations

import itertools
import os

import torch

from . import ops

__all__ = ["grid_locations", "crop_boxes", "hann_window", "shard_indices", "predict_volume", "relative_error"]

_USE_GRAPH = os.environ.get("UB_INFER_GRAPH", "0") == "1"


class _GraphedForward:
    """``gen.forward_packed`` on one batch shape, captured once as a CUDA graph and replayed per batch (one launch
    instead of ~110). Measured on B200 at config 5 (160 x 192 x 160, 27 patches of 64^3): 5.9 ms per volume either
    way -- the eager path is already GPU-bound there -- so it is opt-in, for small patches / slow hosts.
    Valid while nothing the graph baked in has moved: the storage of the parameters and buffers (the captured
    forward re-packs its bf16 weight operands from the live parameter memory on every replay, so weight VALUES may
    change freely) and eval mode."""

    def __init__(self, gen, shape, device):
        self.gen = gen
        self.inp = torch.zeros(shape, dtype=torch.bfloat16, device=device)
        self.fingerprint = self._fingerprint(gen)
        main = torch.cuda.current_stream(device)
        side = torch.cuda.Stream(device=device)
        side.wait_stream(main)
        with torch.cuda.stream(side):               # eager warm-up: packs weights, sets kernel attributes
            gen.forward_packed(self.inp)
        main.wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = gen.forward_packed(self.inp)

    @staticmethod
    def _fingerprint(gen):
        return tuple(t.data_ptr() for t in itertools.chain(gen.parameters(), gen.buffers()))

    def valid(self):
        return (not self.gen.training) and self.fingerprint == self._fingerprint(self.gen)

    def __call__(self):
        self.graph.replay()
        return self.out


def _graphed_forward(gen, shape, device):
    cache = gen.__dict__.setdefault("_infer_graphs", {})
    key = (tuple(shape), str(device))
    g = cache.get(key)
    if g is None or not g.valid():
        g = _GraphedForward(gen, shape, device)
        cache[key] = g
    return g


def _triple(v):
    return (v,) * 3 if isinstance(v, int) else tuple(v)


def grid_locations(shape, patch, patch_overlap=0):
    """Patch origins of torchio's GridSampler, in sampler order (lexicographic in (axis0, axis1, axis2)): per axis,
    with ``step = patch - patch_overlap``, ``range(0, size + 1 - patch, step)`` plus a last origin at
    ``size - patch`` when the grid does not end at the border. ``patch_overlap``: an even int or 3-tuple, smaller
    than the patch."""
    patch, overlap = _triple(patch), _triple(patch_overlap)
    for size, p, o in zip(shape, patch, overlap):
        if p > size:
            raise ValueError(f"patch size {p} larger than the volume ({size})")
        if o < 0 or o >= p:
            raise ValueError(f"patch overlap {o} must be at least 0 and smaller than the patch size {p}")
        if o % 2:
            raise ValueError(f"patch overlap must be a tuple of even integers, got {overlap}")
    per_axis = []
    for size, p, o in zip(shape, patch, overlap):
        idx = list(range(0, size + 1 - p, p - o))
        if idx[-1] != size - p:
            idx.append(size - p)
        per_axis.append(idx)
    return list(itertools.product(*per_axis))


def crop_boxes(shape, patch, patch_overlap, origins):
    """The volume region each patch writes in torchio's ``'crop'`` overlap mode, (z0, y0, x0, z1, y1, x1) half-open:
    half the overlap comes off each side, except a side where the patch touches the volume border."""
    patch, half = _triple(patch), [o // 2 for o in _triple(patch_overlap)]
    boxes = []
    for org in origins:
        lo = [o if o == 0 else o + h for o, h in zip(org, half)]
        hi = [o + p if o + p == s else o + p - h for o, p, h, s in zip(org, patch, half, shape)]
        boxes.append(tuple(lo + hi))
    return boxes


def hann_window(patch):
    """The three 1-D factors (wz, wy, wx), concatenated, of torchio's Hann window: per axis
    ``torch.hann_window(p + 2, periodic=False)[1:-1]``, computed on the CPU as torchio computes it (the fp32 values are
    not exactly symmetric, so they are used as they are)."""
    return torch.cat([torch.hann_window(p + 2, periodic=False)[1:-1] for p in _triple(patch)])


def shard_indices(n: int, rank: int, world: int):
    """Round-robin share of ``n`` independent work items (patches of one volume, or volumes of a test set)."""
    return list(range(rank, n, world))


@torch.no_grad()
def predict_volume(gen, volume: torch.Tensor, patch=64, batch: int = 8, use_graph: bool | None = None,
                   group=None, shard: bool | None = None, patch_overlap=0, overlap_mode: str = "crop") -> torch.Tensor:
    """``volume``: (C,D,H,W) or (1,C,D,H,W) fp32 CUDA tensor. Returns the aggregated prediction
    (6,D,H,W) fp32 on the same device. ``gen`` is a ``unet_bssfp_b200.Generator`` (its train/eval mode is
    respected, as in the reference where ``predict_step`` runs under ``model.eval()``).
    ``patch_overlap`` / ``overlap_mode``: those of torchio's ``GridSampler`` / ``GridAggregator`` -- an even overlap
    per axis (int or 3-tuple), and ``"crop"`` (each patch loses half the overlap on every side not at the border; the
    later patch wins), ``"average"`` or ``"hann"`` (patches weighted by a separable Hann window, then normalised by
    the summed weights). The result is bit-identical to torchio's aggregator fed the same patch predictions.
    ``use_graph`` (default off; ``UB_INFER_GRAPH=1`` turns it on, eval mode only): replay the generator forward as
    a CUDA graph on a static batch buffer; a short last batch is padded by repeating its last patch, and only its
    real patches are aggregated.

    Multi-GPU (``shard``; default: on when ``torch.distributed`` is initialised with more than one rank, every rank
    holding the same volume and weights): the patches are dealt round-robin over the ranks of ``group`` -- the
    generator work, which is all of the cost, needs no exchange -- and the per-rank partial volumes are combined.
    ``"crop"``: the result is bit-identical to the single-process one, including the sampler-order rule "the later
    patch wins": every rank records which patch wrote each voxel last, an all-reduce (MAX) of that owner map decides
    the winner, and an all-reduce (SUM) of the partial volumes masked to the winners delivers it to every rank.
    ``"average"`` / ``"hann"``: every rank accumulates the weighted sum and the weight of its own patches, one
    all-reduce (SUM) of each combines them, then the division. That reorders the fp32 sums over the few patches
    covering a voxel, so the result equals the single-process one to rounding, not bit for bit. (For a test SET,
    give each rank its own volumes -- ``shard_indices`` -- and no collective is needed at all.)"""
    if overlap_mode not in ops.BLEND_MODES:
        raise ValueError(f"overlap_mode must be one of {ops.BLEND_MODES}, got {overlap_mode!r}")
    vol = volume if volume.dim() == 4 else volume[0]
    if not vol.is_cuda:
        raise RuntimeError("predict_volume runs on CUDA tensors only (there is no CPU fallback)")
    patch = _triple(patch)
    shape = tuple(vol.shape[1:])
    origins = grid_locations(shape, patch, patch_overlap)
    crop = overlap_mode == "crop"
    boxes = crop_boxes(shape, patch, patch_overlap, origins) if crop else None
    window = hann_window(patch).to(vol.device) if overlap_mode == "hann" else None
    out_c = gen.blocks["unet"].out_channels
    out = torch.zeros((out_c,) + shape, dtype=torch.float32, device=vol.device)
    weight = None if crop else torch.zeros(shape, dtype=torch.float32, device=vol.device)

    def blend(y, idx):                           # one launch per batch, in sampler order
        ops.blend_patches(y[:len(idx)], out, [origins[k] for k in idx], overlap_mode,
                          None if boxes is None else [boxes[k] for k in idx], weight, window)

    import torch.distributed as dist
    dist_on = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    if shard is None:
        shard = dist_on
    if shard and dist_on:
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        mine = shard_indices(len(origins), rank, world)
        owner = torch.full(shape, -1, dtype=torch.int32, device=vol.device) if crop else None
        for i in range(0, len(mine), batch):
            idx = mine[i:i + batch]
            blend(gen.forward_packed(ops.pack_patches(vol, [origins[k] for k in idx], patch)), idx)
            if crop:
                for k in idx:                    # increasing sampler index: locally the later patch wins
                    z0, y0, x0, z1, y1, x1 = boxes[k]
                    owner[z0:z1, y0:y1, x0:x1] = k
        if crop:
            winner = owner.clone()
            dist.all_reduce(winner, op=dist.ReduceOp.MAX, group=group)
            out.mul_((owner == winner).unsqueeze(0))
            dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
            return out
        dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(weight, op=dist.ReduceOp.SUM, group=group)
        ops.blend_finish(out, weight)
        return out
    from .modules import _precision_of
    if use_graph is None:
        use_graph = _USE_GRAPH
    if use_graph and not gen.training and _precision_of(gen) == "bf16":
        n = min(batch, len(origins))
        fwd = _graphed_forward(gen, (n,) + patch + (ops.pad32(vol.shape[0]),), vol.device)
        for i in range(0, len(origins), n):
            idx = list(range(i, min(i + n, len(origins))))
            padded = idx + [idx[-1]] * (n - len(idx))
            ops.pack_patches(vol, [origins[k] for k in padded], patch, out=fwd.inp)
            blend(fwd(), idx)                    # (n, 6, pd, ph, pw) fp32, the graph's static output: real patches only
    else:
        for i in range(0, len(origins), batch):
            idx = list(range(i, min(i + batch, len(origins))))
            blend(gen.forward_packed(ops.pack_patches(vol, [origins[k] for k in idx], patch)), idx)
    if weight is not None:
        ops.blend_finish(out, weight)
    return out


def relative_error(pred: torch.Tensor, target: torch.Tensor, mask=None, probseg=None, angular: bool = False):
    """``pred`` / ``target``: (C,D,H,W) fp32 volumes (module layout). Returns ``(diff (D,H,W,C), errs [R][C] |
    None)``: the map of ``do_calc_diff_maps`` (channel-last, as the reference stores NIfTI volumes) and the
    per-ROI probseg-weighted means of ``do_calc_error_avg``."""
    # module layout (C,D,H,W) -> the channel-last layout of the reference's NIfTI volumes (one strided copy each)
    p = pred.permute(1, 2, 3, 0).contiguous().float()
    t = target.permute(1, 2, 3, 0).contiguous().float()
    diff, sums, norms = ops.relerr_map_reduce(p, t, mask, probseg, angular=angular)
    errs = None if sums is None else sums / norms[:, None]
    return diff, errs
