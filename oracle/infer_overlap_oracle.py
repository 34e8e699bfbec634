"""ORACLE (test infrastructure only) -- restatement of torchio 0.19.6's sliding-window sampler and aggregator with
``patch_overlap`` and every ``overlap_mode``: what ``inference.predict_volume(..., patch_overlap, overlap_mode)``
reproduces. ``oracle/infer_oracle.py`` restates the reference's own call (overlap 0, ``'crop'``); with those
arguments this module gives the same locations and volume (tests/test_inference_overlap_cpu.py).

Only ``tests/`` may import this. torchio is not installable here (no network); its published algorithm is restated
line by line:

* ``grid_locations``   torchio/data/sampler/grid.py ``GridSampler._parse_sizes`` + ``_get_patches_locations``:
                       per axis ``range(0, size + 1 - patch, patch - overlap)``; if the last index is not
                       ``size - patch`` it is appended; the Cartesian product is de-duplicated and sorted
                       lexicographically (``np.unique(..., axis=0)``). ValueError for a patch larger than the image,
                       an overlap not smaller than the patch, or an odd overlap.
* ``hann_window``      torchio/data/inference/aggregator.py ``GridAggregator._get_hann_window``.
* ``_crop_patch``      ``GridAggregator._crop_patch``.
* ``aggregate``        ``GridAggregator.add_batch``: ``'crop'`` assigns each cropped patch in sampler order -- the
                       later patch wins; ``'average'`` adds the patch and 1 into the average mask; ``'hann'`` adds
                       ``patch * window`` and the window.
* ``finish``           ``GridAggregator.get_output_tensor``: ``true_divide`` by the mask in the accumulating modes.
* ``predict_volume``   ref:src/model.py:315-327 ``predict_step`` with both arguments passed through. torchio
                       aggregates on the CPU (``batch_tensor.cpu()``), and so does this restatement.

PARITY PIN: the known answers of tests/test_inference_overlap_cpu.py (location counts and per-axis origins at
config 5 with overlap 16 and 32; the 1 x 1 x 6 volume with two patches in each mode, Hann values in fp32).
"""
import numpy as np
import torch


def _triple(v):
    return (v,) * 3 if isinstance(v, int) else tuple(v)


def grid_locations(shape, patch, overlap=(0, 0, 0)):
    image_size, patch_size, patch_overlap = np.array(shape), np.array(patch), np.array(_triple(overlap))
    if np.any(patch_size > image_size):
        raise ValueError(f"patch size {patch} larger than the image {shape}")
    if np.any(patch_overlap >= patch_size):
        raise ValueError(f"patch overlap {overlap} must be smaller than the patch size {patch}")
    if np.any(patch_overlap % 2):
        raise ValueError(f"Patch overlap must be a tuple of even integers, not {overlap}")
    indices = []
    for size, p, o in zip(shape, patch, _triple(overlap)):
        end = size + 1 - p
        step = p - o
        idx = list(range(0, end, step))
        if idx[-1] != size - p:
            idx.append(size - p)
        indices.append(idx)
    ini = np.array(np.meshgrid(*indices)).reshape(len(shape), -1).T
    ini = np.unique(ini, axis=0)
    return [tuple(int(v) for v in row) for row in ini]


def hann_window(patch_size):
    """(pd, ph, pw) fp32, ``((1 * wz) * wy) * wx`` by broadcasting."""
    hann_window_3d = torch.as_tensor([1])
    for spatial_dim, size in enumerate(patch_size):
        window_shape = np.ones_like(patch_size)
        window_shape[spatial_dim] = size
        hann_window_1d = torch.hann_window(size + 2, periodic=False)
        hann_window_1d = hann_window_1d[1:-1].view(*[int(s) for s in window_shape])
        hann_window_3d = hann_window_3d * hann_window_1d
    return hann_window_3d


def _crop_patch(patch, location, overlap, spatial_shape):
    """``location``: the patch origin. Returns the cropped patch and its box (z0, y0, x0, z1, y1, x1)."""
    half_overlap = np.array(_triple(overlap)) // 2
    patch_size = np.array(patch.shape[-3:])
    index_ini = np.array(location)
    index_fin = index_ini + patch_size
    crop_ini = half_overlap.copy()
    crop_fin = half_overlap.copy()
    crop_ini[index_ini == 0] = 0
    crop_fin[index_fin == np.array(spatial_shape)] = 0
    new_index_ini = index_ini + crop_ini
    new_index_fin = index_fin - crop_fin
    i_ini, j_ini, k_ini = crop_ini
    i_fin, j_fin, k_fin = patch_size - crop_fin
    return patch[:, i_ini:i_fin, j_ini:j_fin, k_ini:k_fin], tuple(int(v) for v in new_index_ini) + \
        tuple(int(v) for v in new_index_fin)


def aggregate(out, patches, locations, mode="crop", overlap=(0, 0, 0), avgmask=None):
    """One ``add_batch``. out (C,D,H,W); patches: iterable of (C,pd,ph,pw) in sampler order; locations: their
    origins. ``'average'`` / ``'hann'`` also accumulate into ``avgmask`` (C,D,H,W); ``finish`` divides."""
    if mode == "crop":
        for p, loc in zip(patches, locations):
            cropped, (i0, j0, k0, i1, j1, k1) = _crop_patch(p, loc, overlap, out.shape[1:])
            out[:, i0:i1, j0:j1, k0:k1] = cropped
    elif mode == "average":
        for p, (z, y, x) in zip(patches, locations):
            out[:, z:z + p.shape[1], y:y + p.shape[2], x:x + p.shape[3]] += p
            avgmask[:, z:z + p.shape[1], y:y + p.shape[2], x:x + p.shape[3]] += 1
    elif mode == "hann":
        window = None
        for p, (z, y, x) in zip(patches, locations):
            if window is None:
                window = hann_window(tuple(p.shape[1:])).to(p.device)
            p = p * window
            out[:, z:z + p.shape[1], y:y + p.shape[2], x:x + p.shape[3]] += p
            avgmask[:, z:z + p.shape[1], y:y + p.shape[2], x:x + p.shape[3]] += window
    else:
        raise ValueError(f'Overlap mode must be "crop", "average" or "hann" but "{mode}" was passed')
    return out


def finish(out, avgmask, mode):
    return torch.true_divide(out, avgmask) if mode in ("average", "hann") else out


@torch.no_grad()
def predict_volume(gen, volume, patch=(64, 64, 64), batch=8, out_channels=6, overlap=(0, 0, 0), mode="crop"):
    """gen: any callable (N,C,pd,ph,pw) -> (N,6,pd,ph,pw); volume (C,D,H,W) torch tensor. The aggregation runs on
    the CPU, as torchio's does; the result is returned on the volume's device."""
    shape = tuple(volume.shape[1:])
    locs = grid_locations(shape, patch, overlap)
    out = torch.zeros((out_channels,) + shape, dtype=torch.float32)
    avgmask = torch.zeros((out_channels,) + shape, dtype=torch.float32) if mode != "crop" else None
    for i in range(0, len(locs), batch):
        group = locs[i:i + batch]
        x = torch.stack([volume[:, z:z + patch[0], y:y + patch[1], w:w + patch[2]] for (z, y, w) in group])
        y_hat = gen(x).float().cpu()
        aggregate(out, list(y_hat), group, mode, overlap, avgmask)
    return finish(out, avgmask, mode).to(volume.device)
