"""Overlapping sliding-window inference without a GPU: torchio 0.19.6 GridSampler locations with ``patch_overlap``
(known answers, and the product against the oracle restatement), the argument checks, the crop boxes of the
product against the oracle's ``_crop_patch``, and known answers of the oracle aggregator in its three modes."""
import numpy as np
import pytest
import torch

from oracle import infer_oracle as I0
from oracle import infer_overlap_oracle as I
from unet_bssfp_b200 import inference


def _axes(locs):
    return [sorted({loc[a] for loc in locs}) for a in range(3)]


def test_sampler_known_answers():
    shape = (160, 192, 160)
    locs = inference.grid_locations(shape, 64, 16)
    assert len(locs) == 36 and _axes(locs) == [[0, 48, 96], [0, 48, 96, 128], [0, 48, 96]]
    locs = inference.grid_locations(shape, (64, 64, 64), (32, 32, 32))
    assert len(locs) == 80 and _axes(locs) == [[0, 32, 64, 96], [0, 32, 64, 96, 128], [0, 32, 64, 96]]
    assert len(inference.grid_locations((96, 128, 128), 64, 32)) == 18
    assert inference.grid_locations(shape, 64) == inference.grid_locations(shape, 64, 0) == \
        I.grid_locations(shape, (64, 64, 64)) == I0.grid_locations(shape, (64, 64, 64))


def test_overlap_oracle_at_overlap_zero_is_the_reference_oracle():
    """With the reference's own arguments (overlap 0, 'crop') the overlap restatement gives the locations and the
    volume of the restatement of the reference's call, later patch winning where the shifted last patches overlap."""
    shape, patch = (20, 36, 28), (16, 16, 16)
    locs = I.grid_locations(shape, patch)
    assert locs == I0.grid_locations(shape, patch)
    g = torch.Generator().manual_seed(0)
    patches = list(torch.randn((len(locs), 6) + patch, generator=g))
    want = I0.aggregate(torch.zeros((6,) + shape), patches, locs)
    got = I.finish(I.aggregate(torch.zeros((6,) + shape), patches, locs), None, "crop")
    assert torch.equal(got, want)


@pytest.mark.parametrize("shape,patch,overlap", [
    ((160, 192, 160), (64, 64, 64), (0, 0, 0)),
    ((160, 192, 160), (64, 64, 64), (16, 16, 16)),
    ((160, 192, 160), (64, 64, 64), (32, 32, 32)),
    ((96, 128, 128), (64, 64, 64), (32, 32, 32)),
    ((11, 13, 17), (4, 6, 8), (2, 2, 4)),          # anisotropic, ragged last origins
    ((20, 36, 28), (16, 16, 16), (0, 8, 14)),
    ((7, 9, 5), (7, 4, 2), (0, 2, 0)),             # one patch spans an axis
    ((33, 47, 65), (16, 32, 16), (6, 30, 10)),
])
def test_sampler_matches_oracle(shape, patch, overlap):
    locs = inference.grid_locations(shape, patch, overlap)
    assert locs == I.grid_locations(shape, patch, overlap)
    assert locs == sorted(set(locs))
    boxes = inference.crop_boxes(shape, patch, overlap, locs)
    p = torch.zeros((1,) + patch)
    assert boxes == [I._crop_patch(p, loc, overlap, shape)[1] for loc in locs]


@pytest.mark.parametrize("overlap", [1, (0, 0, 3), 64, (0, 66, 0), -2])
def test_sampler_rejects_bad_overlap(overlap):
    with pytest.raises(ValueError):
        inference.grid_locations((160, 192, 160), 64, overlap)
    if overlap != -2:
        with pytest.raises(ValueError):
            I.grid_locations((160, 192, 160), (64, 64, 64), overlap)
    with pytest.raises(ValueError):
        inference.grid_locations((32, 32, 32), 64)


def test_predict_volume_rejects_unknown_mode():
    with pytest.raises(ValueError, match="overlap_mode"):
        inference.predict_volume(None, torch.zeros(24, 32, 32, 32), patch=32, overlap_mode="gaussian")


def _kat(mode):
    out = torch.zeros(1, 1, 1, 6)
    avgmask = torch.zeros(1, 1, 1, 6)
    patches = [torch.tensor([1., 2., 3., 4.]).view(1, 1, 1, 4), torch.tensor([10., 20., 30., 40.]).view(1, 1, 1, 4)]
    locs = I.grid_locations((1, 1, 6), (1, 1, 4), (0, 0, 2))
    assert locs == [(0, 0, 0), (0, 0, 2)]
    I.aggregate(out, patches, locs, mode, (0, 0, 2), avgmask)
    return I.finish(out, avgmask, mode).flatten()


def test_aggregator_known_answers():
    assert torch.equal(_kat("crop"), torch.tensor([1., 2., 3., 20., 30., 40.]))
    assert torch.equal(_kat("average"), torch.tensor([1., 2., 6.5, 12., 30., 40.]))
    want = torch.tensor(np.array([1, 2, 4.93475246, 15.5777102, 30, 40], dtype=np.float32))
    assert torch.equal(_kat("hann"), want)
    w = torch.hann_window(6, periodic=False)[1:-1]
    assert torch.equal(w, torch.tensor(np.array([0.345491529, 0.904508471, 0.904508471, 0.345491439], dtype=np.float32)))
    assert torch.equal(inference.hann_window((1, 1, 4))[2:], w)
    assert torch.equal(I.hann_window((1, 1, 4)).flatten(), w)
    with pytest.raises(ValueError):
        _kat("gaussian")


def test_blend_rejects_bad_arguments():
    import ctypes as C
    from unet_bssfp_b200 import _lib
    lib = _lib.load()
    fake = C.c_void_p(256)                 # never dereferenced: every check below fails before a launch

    def call(n=1, c=6, origin=(0, 0, 0), box=None, mode=0, weight=fake, window=fake):
        orgs = (C.c_int * (3 * n))(*(list(origin) * n))
        bx = None if box is None else (C.c_int * (6 * n))(*(list(box) * n))
        return lib.ub_blend_patches(fake, n, c, 4, 4, 4, orgs, bx, mode, window, fake, weight, 8, 8, 8, None)

    for kw, msg in [(dict(mode=3), b"unknown mode"), (dict(n=65), b"at most 64 patches"), (dict(c=9), b"at most 8 channels"),
                    (dict(mode=1, weight=None), b"weight volume"), (dict(mode=2, window=None), b"window"),
                    (dict(origin=(0, 5, 0)), b"leaves"), (dict(box=(0, 0, 0, 4, 4, 5)), b"leaves"),
                    (dict(box=(2, 0, 0, 2, 4, 4)), b"leaves")]:
        assert call(**kw) < 0, kw
        assert msg in lib.ub_last_error(), (kw, lib.ub_last_error())
    assert lib.ub_blend_finish(None, fake, 6, 10, None) < 0


def test_hann_window_factors_match_oracle():
    for patch in ((4, 6, 8), (64, 64, 64), (1, 5, 2)):
        f = inference.hann_window(patch)
        wz, wy, wx = f.split(patch)
        assert torch.equal(I.hann_window(patch), ((1 * wz.view(-1, 1, 1)) * wy.view(1, -1, 1)) * wx.view(1, 1, -1))
