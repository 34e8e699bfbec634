"""Overlapping sliding-window inference on the GPU: ``ub_blend_patches`` against the oracle restatement of torchio
0.19.6's GridAggregator (bit for bit, every overlap mode), ``predict_volume`` with ``patch_overlap`` /
``overlap_mode`` against the oracle driving the same generator, the defaults, the CUDA-graph path, two ranks, and
config 5 at overlap 32 with the Hann window."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import infer_overlap_oracle as I
from tests.util import rel_l2, strict_fp32

pytestmark = pytest.mark.gpu
DEV = "cuda"
MODES = ("crop", "average", "hann")


def _blend_volume(patches, shape, locs, overlap, mode, split):
    """The product's aggregation of (n, c, pd, ph, pw) patches in launches of ``split`` patches."""
    from unet_bssfp_b200 import inference, ops
    n, c, *patch = patches.shape
    out = torch.zeros((c,) + shape, device=DEV)
    weight = None if mode == "crop" else torch.zeros(shape, device=DEV)
    window = inference.hann_window(patch).to(DEV) if mode == "hann" else None
    boxes = inference.crop_boxes(shape, patch, overlap, locs) if mode == "crop" else None
    for i in range(0, n, split):
        ops.blend_patches(patches[i:i + split], out, locs[i:i + split], mode,
                          None if boxes is None else boxes[i:i + split], weight, window)
    unfinished = out.clone()
    if weight is not None:
        ops.blend_finish(out, weight)
    return out, unfinished, weight


@pytest.mark.parametrize("shape,patch,overlap", [
    ((11, 13, 17), (4, 6, 8), (2, 2, 4)),          # odd extents, anisotropic patches, ragged last origins
    ((12, 12, 12), (8, 8, 8), (4, 4, 4)),          # 8 patches, all of them over the centre voxels
    ((12, 10, 14), (8, 8, 8), (6, 6, 6)),          # up to 4 x 4 x 4 patches over one voxel
])
@pytest.mark.parametrize("mode", MODES)
def test_blend_kernel_matches_oracle_aggregator(shape, patch, overlap, mode):
    locs = I.grid_locations(shape, patch, overlap)
    g = torch.Generator(device=DEV).manual_seed(len(locs))
    patches = torch.randn((len(locs), 6) + patch, device=DEV, generator=g)
    ref = torch.zeros((6,) + shape)
    avgmask = torch.zeros((6,) + shape)
    I.aggregate(ref, list(patches.cpu()), locs, mode, overlap, avgmask)
    ref_unfinished = ref.clone()
    ref = I.finish(ref, avgmask, mode)
    for split in (1, 5, len(locs)):
        got, unfinished, weight = _blend_volume(patches, shape, locs, overlap, mode, split)
        assert torch.equal(got.cpu(), ref), (split, (got.cpu() - ref).abs().max().item())
        assert torch.equal(unfinished.cpu(), ref_unfinished), split
        if weight is not None:
            assert all(torch.equal(weight.cpu(), avgmask[k]) for k in range(6)), split


def _generator(modality="bssfp"):
    import unet_bssfp_b200 as ub
    from oracle import model_oracle as O
    torch.manual_seed(0)
    og = O.Generator(modality).to(DEV).eval()
    g = ub.Generator(modality).to(DEV).eval()
    g.load_state_dict(og.state_dict())
    return g, og


@pytest.mark.parametrize("overlap", [16, (16, 8, 0)])
@pytest.mark.parametrize("mode", MODES)
def test_predict_volume_with_overlap_matches_oracle(overlap, mode):
    """predict_volume == the oracle sampler/aggregator driving the same generator patch by patch with the same
    batch size (bit-exact), and close to the fp32 oracle generator (bf16 bar)."""
    strict_fp32()
    import unet_bssfp_b200 as ub
    g, og = _generator()
    torch.manual_seed(3)
    vol = torch.rand((24, 48, 80, 40), device=DEV)
    ov = (overlap,) * 3 if isinstance(overlap, int) else overlap
    got = ub.inference.predict_volume(g, vol, patch=32, batch=5, patch_overlap=overlap, overlap_mode=mode)
    same = I.predict_volume(lambda x: g(x), vol, patch=(32, 32, 32), batch=5, overlap=ov, mode=mode)
    assert torch.equal(got, same), (got - same).abs().max().item()
    ref = I.predict_volume(og, vol, patch=(32, 32, 32), batch=5, overlap=ov, mode=mode)
    assert rel_l2(got, ref) < 2e-2


def test_defaults_are_overlap_zero_crop_and_the_per_patch_paste():
    """The explicit defaults equal the default call, and both equal pasting each patch in sampler order."""
    import unet_bssfp_b200 as ub
    from unet_bssfp_b200 import ops
    g, _ = _generator()
    torch.manual_seed(3)
    vol = torch.rand((24, 48, 80, 40), device=DEV)
    default = ub.inference.predict_volume(g, vol, patch=32, batch=5)
    explicit = ub.inference.predict_volume(g, vol, patch=32, batch=5, patch_overlap=0, overlap_mode="crop")
    assert torch.equal(default, explicit)
    locs = ub.inference.grid_locations(tuple(vol.shape[1:]), (32, 32, 32))
    pasted = torch.zeros_like(default)
    for i in range(0, len(locs), 5):
        y = g.forward_packed(ops.pack_patches(vol, locs[i:i + 5], (32, 32, 32)))
        for k, org in enumerate(locs[i:i + 5]):
            ops.paste_patch(y[k], pasted, org)
    assert torch.equal(default, pasted)


@pytest.mark.parametrize("mode", MODES)
def test_graph_replay_equals_eager_with_overlap(mode):
    """16 patches in batches of 5: the padded last batch of one real patch must be blended once."""
    import unet_bssfp_b200 as ub
    torch.manual_seed(0)
    g = ub.Generator("t1w").to(DEV).eval()
    torch.manual_seed(3)
    vol = torch.rand((6, 48, 80, 40), device=DEV)
    assert len(ub.inference.grid_locations(tuple(vol.shape[1:]), 32, 16)) == 16
    kw = dict(patch=32, batch=5, patch_overlap=16, overlap_mode=mode)
    eager = ub.inference.predict_volume(g, vol, use_graph=False, **kw)
    graph = ub.inference.predict_volume(g, vol, use_graph=True, **kw)
    assert torch.equal(eager, graph)


def test_config5_overlap32_hann():
    import unet_bssfp_b200 as ub
    shape = (160, 192, 160)
    assert len(ub.inference.grid_locations(shape, 64, 32)) == 80
    torch.manual_seed(0)
    g = ub.Generator("bssfp").to(DEV).eval()
    torch.manual_seed(5)
    vol = torch.rand((24,) + shape, device=DEV)
    pred = ub.inference.predict_volume(g, vol, patch=64, batch=8, patch_overlap=32, overlap_mode="hann")
    assert pred.shape == (6,) + shape and torch.isfinite(pred).all()


# ---------------- two ranks on one GPU (gloo): the spawn harness of tests/test_ddp_gpu.py ----------------

def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
        torch.cuda.set_device(0)
        dev = torch.device("cuda", 0)
        import unet_bssfp_b200 as ub
        res = {}
        torch.manual_seed(0)                                           # the same weights on every rank
        g = ub.Generator("t1w").to(dev).eval()
        torch.manual_seed(5)                                           # ... and the same volume
        vol = torch.rand((6, 48, 80, 40), device=dev)                 # 16 patches of 32^3 at overlap 16
        for mode in MODES:
            # one patch per launch: the same generator launch geometry whoever runs the patch
            kw = dict(patch=32, batch=1, patch_overlap=16, overlap_mode=mode)
            whole = ub.inference.predict_volume(g, vol, shard=False, **kw)
            sharded = ub.inference.predict_volume(g, vol, **kw)           # shards: dist is initialised
            if mode == "crop":
                ok = bool(torch.equal(whole, sharded))
            else:                                                      # the fp32 sums of a voxel are reordered
                ok = bool((whole - sharded).abs().max().item() <= 1e-6 * whole.abs().max().item())
            res[f"sharded_{mode}"] = ok if ok else (
                f"max |diff| {(whole - sharded).abs().max().item():.3e}, max |out| {whole.abs().max().item():.3e}")
        q.put((rank, res))
        dist.destroy_process_group()
    except Exception:   # surface the failure in the parent instead of a queue timeout
        import traceback
        q.put((rank, {"exception": traceback.format_exc()[-1500:]}))


def test_sharded_overlap_two_ranks_on_the_gpu():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=120)
    for rank in (0, 1):
        assert "exception" not in res[rank], res[rank]["exception"]
        for k, v in res[rank].items():
            assert v is True, (rank, k, v)
