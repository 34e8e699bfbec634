"""Config 5: whole-volume sliding-window inference (160 x 192 x 160, 64^3 patches) + relative-error evaluation:
eager launches vs CUDA-graph replay of the generator forward; then the overlap settings (0 / crop: 27 patches,
32 / average and 32 / hann: 80 patches) with the blend kernel's own time from CUDA events, and the A/B of the
overlap-0 aggregation: one ub_blend_patches launch per batch against one ub_paste_patch launch per patch.
python tools/bench_inference.py"""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import unet_bssfp_b200 as ub  # noqa: E402

dev = "cuda"
shape = (160, 192, 160)
P = (64, 64, 64)
torch.manual_seed(0)
g = ub.Generator("bssfp").to(dev).eval()
vol = torch.rand((24,) + shape, device=dev)
tgt = torch.rand((6,) + shape, device=dev) * 0.95 + 0.05
mask = (torch.rand(shape, device=dev) > 0.3).to(torch.uint8)
probseg = torch.rand(shape + (3,), device=dev)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit not readable"
    return f"{torch.cuda.get_device_name()}, {q}"


def timed(fn, iters=5):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / iters * 1e3


print(f"card: {card()}")
vox = shape[0] * shape[1] * shape[2]
for batch in (8, 9, 27):
    e = timed(lambda: ub.inference.predict_volume(g, vol, patch=64, batch=batch, use_graph=False))
    c = timed(lambda: ub.inference.predict_volume(g, vol, patch=64, batch=batch, use_graph=True))
    print(f"predict_volume batch {batch:2d}: eager {e:7.2f} ms ({vox / e / 1e3:7.1f} Mvox/s)   graph {c:7.2f} ms ({vox / c / 1e3:7.1f} Mvox/s)")
pred = ub.inference.predict_volume(g, vol, patch=64, batch=9)
r = timed(lambda: ub.inference.relative_error(pred, tgt, mask, probseg))
print(f"relative_error (map + ROI means): {r:.3f} ms")
m = timed(lambda: ub.ops.dti_scalar_maps(pred.permute(1, 2, 3, 0).contiguous()))
print(f"dti_scalar_maps: {m:.3f} ms")
n = timed(lambda: ub.nifti.volume_to_nifti_order(pred, (-0.003, 0.004)))
print(f"denorm_to_nifti: {n:.3f} ms")


# ---- overlap settings: predict_volume per volume, and the aggregation kernels alone ----
BATCH = 8


def predict_paste():
    """The overlap-0 aggregation as one ub_paste_patch launch per patch (the A arm of the A/B)."""
    locs = ub.inference.grid_locations(shape, P)
    out = torch.zeros((6,) + shape, device=dev)
    for i in range(0, len(locs), BATCH):
        y = g.forward_packed(ub.ops.pack_patches(vol, locs[i:i + BATCH], P))
        for k, org in enumerate(locs[i:i + BATCH]):
            ub.ops.paste_patch(y[k], out, org)
    return out


def batches(overlap):
    """Per batch: origins, crop boxes and the generator's (n, 6, 64, 64, 64) fp32 output."""
    locs = ub.inference.grid_locations(shape, P, overlap)
    boxes = ub.inference.crop_boxes(shape, P, overlap, locs)
    return locs, [(locs[i:i + BATCH], boxes[i:i + BATCH], g.forward_packed(ub.ops.pack_patches(vol, locs[i:i + BATCH], P)))
                  for i in range(0, len(locs), BATCH)]


def event_ms(fn, reps=20):
    """Device time of fn's launches alone: the volumes it writes are zeroed outside the timed window, and the
    launches are queued behind a device-side sleep, so the host's launch cost does not open gaps between them."""
    total = 0.0
    for i in range(reps + 1):
        fn(zero=True)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(20_000_000)
        a.record()
        fn(zero=False)
        b.record()
        b.synchronize()
        if i > 0:
            total += a.elapsed_time(b)
    return total / reps


def blend_launches(mode, todo):
    out = torch.zeros((6,) + shape, device=dev)
    weight = torch.zeros(shape, device=dev)
    window = ub.inference.hann_window(P).to(dev)

    def run(zero):
        if zero:
            out.zero_(); weight.zero_()
            return
        for locs, boxes, y in todo:
            ub.ops.blend_patches(y, out, locs, mode, boxes if mode == "crop" else None, weight, window)
        if mode != "crop":
            ub.ops.blend_finish(out, weight)
    return run


def paste_launches(todo):
    out = torch.zeros((6,) + shape, device=dev)

    def run(zero):
        if zero:
            out.zero_()
            return
        for locs, _, y in todo:
            for k, org in enumerate(locs):
                ub.ops.paste_patch(y[k], out, org)
    return run


assert torch.equal(predict_paste(), ub.inference.predict_volume(g, vol, patch=64, batch=BATCH)), "overlap-0 A/B arms differ"
print(f"\noverlap settings, batch {BATCH} (predict_volume per volume; aggregation = the blend launches of one volume "
      f"from CUDA events, generator outputs precomputed, 20 repetitions)")
for overlap, mode in ((0, "crop"), (32, "average"), (32, "hann")):
    locs, todo = batches(overlap)
    t = timed(lambda: ub.inference.predict_volume(g, vol, patch=64, batch=BATCH, patch_overlap=overlap, overlap_mode=mode))
    k = event_ms(blend_launches(mode, todo))
    gb = len(locs) * 6 * P[0] * P[1] * P[2] * 4 / 1e9
    print(f"overlap {overlap:2d} / {mode:7s}: {len(locs):2d} patches  predict_volume {t:7.2f} ms  "
          f"aggregation {k:6.3f} ms ({gb:.3f} GB of patch predictions read, {gb / k:5.2f} TB/s)")
    del todo

locs, todo = batches(0)
print("\nA/B overlap 0 / crop, alternating: one blend launch per batch (B) against one paste launch per patch (A)")
for rnd in range(3):
    a = timed(predict_paste)
    b = timed(lambda: ub.inference.predict_volume(g, vol, patch=64, batch=BATCH))
    ka = event_ms(paste_launches(todo))
    kb = event_ms(blend_launches("crop", todo))
    print(f"round {rnd}: predict_volume A {a:7.2f} ms  B {b:7.2f} ms   aggregation A {ka:6.3f} ms ({len(locs)} launches)  "
          f"B {kb:6.3f} ms ({len(todo)} launches)")
print(f"card: {card()}")
