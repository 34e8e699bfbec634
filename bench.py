#!/usr/bin/env python
"""bench.py -- G+D train-step voxels/s of the sm_100a hot path (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference          # the reference arithmetic (oracle) on the host cores
    python bench.py --dump-outputs DIR        # also write the last timed step's outputs, to compare two builds

One "step" = one ``training_step`` of ref:src/model.py:259-281 (G phase + AdamW, D phase on a fresh G
forward + AdamW; L1 + adversarial losses, perceptual term out of scope) on one synthetic batch:
config[1] of BASELINE.json -- ``bssfp`` (24 input channels), batch 8 per GPU, 128^3 patches, bf16
tensor-core math with fp32 accumulate. Data-parallel over ranks (weak scaling, per-rank batch fixed),
gradient all-reduce on NCCL. Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "G+D train-step voxels/sec"
UNIT = "voxels/s"
# conv/deconv MACs x 2 per input voxel per train step, reference semantics (SURVEY.md section 8d)
FLOP_PER_VOXEL = {"bssfp": 2369152, "pc-bssfp": 2369152, "t1w": 2311264, "dwi-tensor": 2311264}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"bf16_burst": p["bf16_tflops"], "bf16_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "hbm": p["hbm_gbs"], "src": "measured"}
    except Exception:
        return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                try:
                    pw.append(float(r[2]))
                except Exception:
                    pass
                for k, nme in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        # median under load: ignore idle samples far below the busiest
        hot = [v for v in sm if v >= 0.5 * max(sm)] if sm else []
        hot_pw = [p for p, v in zip(pw, sm) if v >= 0.5 * max(sm)] if (sm and len(pw) == len(sm)) else pw
        return {"sm_mhz": statistics.median(hot) if hot else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": statistics.median(hot_pw) if hot_pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_run(steps, warmup, size=64, modality="bssfp", threads=None):
    """The reference arithmetic (oracle restatement of ref:src/model.py) on the host cores: full GAN
    step at batch 1, size^3 (a bounded sample of the workload). -> (voxels/s, ms/step, cores)."""
    from oracle import model_oracle as O
    torch.set_num_threads(threads or os.cpu_count() or 1)
    torch.manual_seed(0)
    og, od = O.Generator(modality), O.Discriminator(modality)
    opt_g, opt_d = O.make_optimizers(og, od)
    cin = O.in_channels_of(modality)
    torch.manual_seed(1234)
    x, y = torch.rand(1, cin, size, size, size), torch.rand(1, 6, size, size, size)
    for _ in range(warmup):
        O.gan_step(og, od, opt_g, opt_d, x, y)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.gan_step(og, od, opt_g, opt_d, x, y)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return size ** 3 / dt, dt * 1e3, torch.get_num_threads()


def cpu_config1_run(steps, warmup, threads=None, size=64):
    """BASELINE config 1: U-Net generator forward + backward on one 64^3 bSSFP patch, batch 1, fp32, train mode,
    L1 loss (the oracle restatement of ref:src/model.py:15-39,126). -> (voxels/s, ms, cores)."""
    from oracle import model_oracle as O
    torch.set_num_threads(threads or os.cpu_count() or 1)
    torch.manual_seed(0)
    og = O.Generator("bssfp").train()
    torch.manual_seed(1234)
    x, y = torch.rand(1, 24, size, size, size), torch.rand(1, 6, size, size, size)

    def one():
        for p in og.parameters():
            p.grad = None
        torch.nn.functional.l1_loss(og(x), y).backward()

    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return size ** 3 / dt, dt * 1e3, torch.get_num_threads()


def cpu_eval_run(shape=(160, 192, 160)):
    """NumPy restatement of ref:src/eval.py:154-166,217-258 on one float64 volume of config 5's size, single
    process (relative-error map + masked, probseg-weighted ROI means). -> (voxels/s, ms)."""
    import numpy as np
    from oracle import eval_oracle as E
    rng = np.random.default_rng(0)
    pred = rng.random(shape + (6,))
    tgt = rng.random(shape + (6,)) * 0.95 + 0.05
    mask = (rng.random(shape) > 0.3).astype(np.uint8)
    probseg = rng.random(shape + (3,))
    t0 = time.perf_counter()
    diff = E.rel_error_map(pred, tgt)
    E.roi_error_avg(diff, mask, probseg)
    dt = time.perf_counter() - t0
    return shape[0] * shape[1] * shape[2] / dt, dt * 1e3


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(1, min(args.warmup, 1))
    v, ms, cores = cpu_reference_run(steps, warmup, size=64, modality=args.modality)
    sample = f"full GAN step, batch 1 x 64^3 ({args.modality}), fp32 torch CPU, {steps} timed steps after {warmup} warm-up"
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic",
        "config": {"workload": f"full GAN step (U-Net G + PatchGAN D, L1+adversarial), {args.modality}, "
                               f"batch {args.batch} x {args.size}^3 per GPU", "sampled_as": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


TENSOR_CLASSES = ("igemm_fwd_kernel", "igemm_march_kernel", "wgrad_march_kernel", "igemm_wgrad_kernel")


def roofline_table(trainer, batches, peaks, flop_step, ms_step, profile_steps=2):
    """Per-kernel-class roofline of the step, measured IN THIS RUN: ``profile_steps`` further steps run under the
    per-op CUDA-event profiler (unet_bssfp_b200/profiler.py; serial times, weight gradients on the main stream).
    Tensor-core classes: algorithmic conv FLOPs / time against the SUSTAINED bf16 peak (kernels timed inside a long
    step); memory-bound ops: tensor bytes (inputs once + outputs once) / time against the measured HBM copy peak.
    ``kernel`` names the class with the largest share of the step time."""
    from unet_bssfp_b200 import profiler
    with profiler.profile() as records:
        for i in range(profile_steps):
            trainer.step(*batches[i % len(batches)])
        torch.cuda.synchronize()
    per_class, per_op = profiler.summarize(records, steps=profile_steps)
    covered = sum(v["ms"] for v in per_class.values())
    classes = {}
    for cls, v in sorted(per_class.items(), key=lambda kv: -kv[1]["ms"]):
        if v["ms"] < 0.05:
            continue
        e = {"ms_per_step": round(v["ms"], 3), "share": round(v["ms"] / covered, 4), "calls_per_step": v["calls"]}
        if cls in TENSOR_CLASSES:
            tf = v["flops"] / (v["ms"] * 1e-3) / 1e12
            e.update({"bound": "tensor", "flops": v["flops"], "achieved": round(tf, 1), "unit": "TFLOP/s",
                      "frac": round(tf / peaks["bf16_sustained"], 4)})
        else:
            gb = v["bytes"] / (v["ms"] * 1e-3) / 1e9
            e.update({"bound": "hbm", "bytes": v["bytes"], "achieved": round(gb, 1), "unit": "GB/s",
                      "frac": round(gb / peaks["hbm"], 4)})
        classes[cls] = e
    dom = max(classes, key=lambda c: classes[c]["ms_per_step"])
    # the longest single launch of the dominant class
    tops = [(k, v) for k, v in per_op.items() if k[1] == dom]
    (op, _, label), tv = max(tops, key=lambda kv: kv[1]["ms"] / kv[1]["calls"])
    top_ms = tv["ms"] / tv["calls"]
    top = {"op": op, "shape": label, "ms_per_launch": round(top_ms, 4)}
    if tv["flops"]:
        top["achieved"] = round(tv["flops"] / tv["calls"] / (top_ms * 1e-3) / 1e12, 1)
        top["unit"] = "TFLOP/s"
    d = classes[dom]
    step_tf = flop_step / (ms_step * 1e-3) / 1e12
    conv_ms = sum(classes[c]["ms_per_step"] for c in classes if c in TENSOR_CLASSES)
    conv_fl = sum(classes[c]["flops"] for c in classes if c in TENSOR_CLASSES)
    return {
        "bound": d["bound"], "kernel": dom + " (time-dominant kernel class of the step)",
        "achieved": d["achieved"], "peak": peaks["bf16_sustained"] if d["bound"] == "tensor" else peaks["hbm"],
        "peak_src": peaks["src"] + (" (sustained: kernels timed inside a long step)" if d["bound"] == "tensor" else ""),
        "unit": d["unit"], "frac": d["frac"], "share_of_step": d["share"], "longest_launch": top,
        "traffic": None,
        "traffic_note": "per-launch DRAM traffic is in the committed ncu summaries (profiles/r02_*_ncu_summary.txt)",
        "how": f"{profile_steps} profiled steps, CUDA events around every op on its launching stream",
        "profiled_ms_per_step_serial": round(covered, 3),
        "classes": classes,
        "all_conv_kernels": {"ms_per_step": round(conv_ms, 3), "achieved": round(conv_fl / (conv_ms * 1e-3) / 1e12, 1),
                             "unit": "TFLOP/s", "frac_of_sustained": round(conv_fl / (conv_ms * 1e-3) / 1e12 / peaks["bf16_sustained"], 4)},
        "step_tflops": step_tf, "step_frac_of_burst_peak": step_tf / peaks["bf16_burst"],
        "step_frac_of_sustained_peak": step_tf / peaks["bf16_sustained"],
        "flop_per_step": flop_step,
    }


def secondary_configs(dev, skip4=False):
    """BASELINE configs 4 and 5 as secondary, driver-run numbers (N = 1 only; a few steps each)."""
    import unet_bssfp_b200 as ub
    from unet_bssfp_b200.train_step import GanTrainer
    out = {}
    if not skip4:
        try:
            torch.manual_seed(0)
            g, d = ub.Generator("t1w").to(dev), ub.Discriminator("t1w").to(dev)
            tr = GanTrainer(g, d)
            B, S = 16, 128
            torch.manual_seed(99)
            bs = [(torch.rand(B, 6, S, S, S, device=dev), torch.rand(B, 6, S, S, S, device=dev)) for _ in range(2)]
            for i in range(3):
                tr.step(*bs[i % 2])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            K = 6
            e0.record()
            for i in range(K):
                tr.step(*bs[i % 2])
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / K
            fl = FLOP_PER_VOXEL["t1w"] * B * S ** 3
            out["config4_t1w_batch16_128"] = {"ms_per_step": ms, "value": B * S ** 3 / (ms * 1e-3), "unit": UNIT, "steps": K,
                                              "warmup": 3, "step_tflops": fl / (ms * 1e-3) / 1e12,
                                              "workload": "full GAN step, t1w (6 input channels, D sees 12), batch 16 x 128^3"}
            del tr, g, d, bs
            torch.cuda.empty_cache()
        except Exception as ex:   # reported, never fatal for the headline line
            out["config4_t1w_batch16_128"] = {"error": repr(ex)[:300]}
    try:
        shape = (160, 192, 160)
        torch.manual_seed(0)
        g = ub.Generator("bssfp").to(dev).eval()
        vol = torch.rand((24,) + shape, device=dev)
        tgt = torch.rand((6,) + shape, device=dev) * 0.95 + 0.05
        mask = (torch.rand(shape, device=dev) > 0.3).to(torch.uint8)
        probseg = torch.rand(shape + (3,), device=dev)

        def timed(fn, iters=5):
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                r = fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / iters, r

        vox = shape[0] * shape[1] * shape[2]
        ms_p, pred = timed(lambda: ub.inference.predict_volume(g, vol, patch=64, batch=9, use_graph=False))
        ms_r, _ = timed(lambda: ub.inference.relative_error(pred, tgt, mask, probseg))
        ms_m, _ = timed(lambda: ub.ops.dti_scalar_maps(pred.permute(1, 2, 3, 0).contiguous()))
        out["config5_inference_160x192x160"] = {
            "predict_volume_ms": ms_p, "value": vox / (ms_p * 1e-3), "unit": "output voxels/s", "patches": 27, "patch": 64,
            "relative_error_ms": ms_r, "dti_scalar_maps_ms": ms_m,
            "workload": "sliding-window inference (27 patches of 64^3, later patch wins) + relative-error map and ROI means + DTI maps"}
    except Exception as ex:
        out["config5_inference_160x192x160"] = {"error": repr(ex)[:300]}
    return out


DUMP_SAMPLE = 1 << 22    # parameters written per network by --dump-outputs (16 MB of float32 each)


def dump_outputs(out_dir, trainer, g_loss, d_loss):
    """Write what the last timed step hands its caller as ``out_dir/<name>.npy``: the two losses, and the state of the
    two networks it updated -- a fixed sample of the parameters (indices drawn by ``numpy.random.default_rng(0)`` from
    the concatenation of ``parameters()`` in order, ascending) and every buffer (BatchNorm statistics, as float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"g_loss": g_loss, "d_loss": d_loss}
    for name, net in (("gen", trainer.gen), ("discr", trainer.discr)):
        flat = torch.cat([p.detach().reshape(-1) for p in net.parameters()])
        idx = np.sort(np.random.default_rng(0).choice(flat.numel(), min(DUMP_SAMPLE, flat.numel()), replace=False))
        arrays[f"{name}_params_sample"] = flat[torch.from_numpy(idx).to(flat.device)]
        arrays[f"{name}_buffers"] = torch.cat([b.detach().reshape(-1).double() for b in net.buffers()])
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v.cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="per-GPU batch (BASELINE config 2: 8)")
    ap.add_argument("--size", type=int, default=128, help="patch edge (BASELINE config 2: 128)")
    ap.add_argument("--modality", default="bssfp")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the config-4 / config-5 secondary numbers")
    ap.add_argument("--e2e-x-dtype", default="bf16", choices=["bf16", "fp32"],
                    help="host dtype of the conditioning input x in the end-to-end loop (bf16: same packed bits, "
                         "half the H2D bytes of x)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the losses and the updated network state of the last one to "
                         "DIR/<name>.npy (inputs and initial weights are seeded: the same arguments give the same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; it is not available with --impl reference")
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries ONE JSON line (rank 0): everything else that writes to fd 1 while the bench runs (NCCL's
    # version banner, library chatter) is sent to stderr; the line itself goes to the saved descriptor.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import unet_bssfp_b200 as ub
    from unet_bssfp_b200 import _lib, hostmem
    from unet_bssfp_b200.train_step import GanTrainer
    lib = _lib.load()
    peaks = load_peaks()
    # one process per GPU: stage the pinned input batch on the NUMA node of this rank's GPU (before allocating it)
    numa_cpus = hostmem.bind_to_gpu(local) if (world > 1 and os.environ.get("UB_BIND_NUMA", "1") != "0") else None

    torch.manual_seed(1000 + rank)    # DIFFERENT initial weights per rank: GanTrainer broadcasts rank 0's (as DDP does)
    gen = ub.Generator(args.modality).to(dev)
    dis = ub.Discriminator(args.modality).to(dev)
    trainer = GanTrainer(gen, dis)
    cin = 24 if args.modality in ("bssfp", "pc-bssfp") else 6
    B, S = args.batch, args.size
    # two different synthetic batches per rank, alternated step by step: every timed step packs a NEW input, as a
    # real loader would deliver one (no cross-step reuse of the packed input)
    host = []
    for k in range(2):
        torch.manual_seed(1234 + 7919 * k + rank)
        host.append((torch.rand(B, cin, S, S, S).pin_memory(), torch.rand(B, 6, S, S, S).pin_memory()))
    batches = [(xh.to(dev), yh.to(dev)) for xh, yh in host]
    voxels_per_step = B * S ** 3 * world

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput ("value") ----------------
    for i in range(args.warmup):
        trainer.step(*batches[i % 2])
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = lib.ub_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        g_loss, d_loss = trainer.step(*batches[i % 2])
    e1.record()
    barrier()
    launches = lib.ub_launch_count() - n0
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_step = ms_total.item() / args.steps
    clocks = sampler.stop() if rank == 0 else None
    value = voxels_per_step / (ms_step * 1e-3)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, trainer, g_loss, d_loss)

    # ---------------- end-to-end: host buffers, H2D + D2H inside the timed region ----------------
    e2e = None
    if not args.no_e2e:
        copy_stream = torch.cuda.Stream(device=dev)
        xdt = torch.bfloat16 if args.e2e_x_dtype == "bf16" else torch.float32
        # the loader's host batches: x in its transport dtype (bf16 packs to the same bits as fp32), y in fp32
        host_e = [(xh.to(xdt).pin_memory(), yh) for xh, yh in host]
        bufs = [(torch.empty(batches[0][0].shape, dtype=xdt, device=dev), torch.empty_like(batches[0][1])) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]
        loss_host = torch.zeros(2, 2).pin_memory()

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done[i % 2])
                bufs[i % 2][0].copy_(host_e[i % 2][0], non_blocking=True)
                bufs[i % 2][1].copy_(host_e[i % 2][1], non_blocking=True)
                ready[i % 2].record(copy_stream)

        def e2e_loop(nsteps):
            for ev in done:
                ev.record()
            prefetch(0)
            for i in range(nsteps):
                if i + 1 < nsteps:
                    prefetch(i + 1)
                torch.cuda.current_stream().wait_event(ready[i % 2])
                gl, dl = trainer.step(*bufs[i % 2])
                done[i % 2].record()
                loss_host[i % 2, 0].copy_(gl, non_blocking=True)
                loss_host[i % 2, 1].copy_(dl, non_blocking=True)
            torch.cuda.synchronize()
            return float(loss_host[(nsteps - 1) % 2, 0])

        e2e_loop(2)
        barrier()
        e0.record()
        e2e_loop(args.steps)
        e1.record()
        barrier()
        ms_e = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms_e, op=dist.ReduceOp.MAX)
        ms_e_step = ms_e.item() / args.steps
        h2d = int(host_e[0][0].numel() * host_e[0][0].element_size() + host_e[0][1].numel() * 4)
        e2e = {"value": voxels_per_step / (ms_e_step * 1e-3), "unit": UNIT, "ms_per_step": ms_e_step,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
               "x_host_dtype": args.e2e_x_dtype, "y_host_dtype": "fp32",
               "how": "pinned host batch (a new one every step) -> double-buffered H2D on a copy stream -> "
                      "GanTrainer.step (packs the input) -> losses D2H",
               "numa_bound_cpus": len(numa_cpus) if numa_cpus else None}

    roof = cpu = secondary = None
    flop_step = FLOP_PER_VOXEL[args.modality] * B * S ** 3
    if rank == 0 and not args.no_roofline:
        roof = roofline_table(trainer, batches, peaks, flop_step, ms_step)
    elif world > 1 and not args.no_roofline:
        # the other ranks run the same profiled steps (the all-reduce inside trainer.step is collective)
        for i in range(2):
            trainer.step(*batches[i % 2])
        torch.cuda.synchronize()
    if rank == 0 and roof is None:
        step_tf = flop_step / (ms_step * 1e-3) / 1e12
        roof = {"bound": "tensor", "step_tflops": step_tf, "step_frac_of_burst_peak": step_tf / peaks["bf16_burst"],
                "step_frac_of_sustained_peak": step_tf / peaks["bf16_sustained"]}
    if world > 1:
        dist.barrier()
    if rank == 0 and world == 1:
        del trainer, gen, dis, batches
        torch.cuda.empty_cache()
        if not args.no_secondary:
            secondary = secondary_configs(dev)
        if not args.no_cpu_baseline:   # reported at N = 1 only (torchrun pins OMP_NUM_THREADS=1)
            v, ms, cores = cpu_reference_run(steps=2, warmup=1, size=64, modality=args.modality)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_step": ms,
                   "sample": f"full GAN step, batch 1 x 64^3 ({args.modality}), fp32 torch CPU oracle, 2 timed steps after 1 warm-up"}
            legs = {}
            v1, ms1, _ = cpu_reference_run(steps=1, warmup=1, size=64, modality=args.modality, threads=1)
            legs["full_step_1_thread"] = {"value": v1, "unit": UNIT, "ms_per_step": ms1, "cores": 1,
                                          "note": "the reference's job script exports OMP_NUM_THREADS=1 (ref:run.sh:51)"}
            vc, msc, cc = cpu_config1_run(steps=2, warmup=1)
            legs["config1_G_fwd_bwd_64"] = {"value": vc, "unit": "voxels/s", "ms": msc, "cores": cc,
                                            "sample": "BASELINE config 1: generator fwd + bwd, 1 x 24 x 64^3, L1 loss, train mode"}
            vc1, msc1, _ = cpu_config1_run(steps=1, warmup=1, threads=1)
            legs["config1_G_fwd_bwd_64_1_thread"] = {"value": vc1, "unit": "voxels/s", "ms": msc1, "cores": 1}
            ve, mse = cpu_eval_run()
            legs["eval_relerr_roi_numpy_160x192x160"] = {"value": ve, "unit": "voxels/s", "ms": mse, "cores": 1,
                                                         "sample": "NumPy restatement of ref:eval.py:154-166,217-258, float64, single process"}
            cpu["legs"] = legs
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": f"full GAN step (U-Net G + PatchGAN D, L1+adversarial, 2x AdamW), {args.modality}, "
                                   f"batch {B} x {S}^3 per GPU", "global_batch": B * world, "patch": S,
                       "parallelism": f"dp{world}", "l2": "inputs larger than L2 (activations are GBs per step)",
                       "input_batches": "two synthetic batches alternated: every step packs a new input",
                       "intermediates": "bf16 operands, fp32 accumulate; raw conv outputs feeding a norm stored as fp16",
                       "losses": [float(g_loss), float(d_loss)]},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu,
            "secondary": secondary,
        }
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
