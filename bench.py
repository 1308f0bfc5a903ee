#!/usr/bin/env python
"""bench.py — MADM diffusion feature extraction on B200 (BASELINE.json metric: feature-extract images/s @512^2).

  python bench.py --gpus N --steps K --warmup W            # product arm (CUDA engine through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # reference arm: the fp32 oracle on the host cores

One "step" = one pass of the hot path (VAE encode -> q-sample -> UNet + taps -> GN-bottleneck projections, SURVEY §8
rows a-1..a-9) over one batch of 8 synthetic 512x512 images per GPU (BASELINE.json configs[1]; random-init weights,
seeded as SURVEY §8d).  For N > 1 the driver launches this file with torchrun: one rank per GPU, images batch-sharded,
no collective on the data path (weak scaling); timing = max over ranks of the CUDA-event time of exactly K steps,
bracketed by barrier + synchronize.  Rank 0 prints ONE JSON line.

--config selects the measured workload (default `base` = BASELINE.json configs[1], the contract's bench line):
  base         8 x 3 x 512^2 per GPU, feature extraction a-1..a-9                                   (BASELINE configs[1])
  slide1024    1024^2 sliding-window inference, 9 crops per image, images sharded over the ranks    (BASELINE configs[2])
  teacher2048  1024 x 2048 EMA-teacher pass: 21 crops per image -> EMA projections -> head -> pseudo-labels (BASELINE configs[3])
  train        LoRA training step, 2 images per GPU: forward + backward + gradient all-reduce + AdamW + EMA   (BASELINE configs[4])
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "UNet feature-extract images/s @512^2 (VAE-enc + q-sample + SD-1.4 UNet+LoRA taps + projections)"
UNIT = "images/s"
PER_GPU_BATCH = 8
# algorithmic FLOPs per 512^2 image (2*MAC), SURVEY §8d / BASELINE.md §2
GF_PER_IMG = {"vae_encoder": 1116.66, "unet_taps": 803.18, "projections": 14.35, "total": 1934.2}
# --variant s0 (not the default bench line): the vae_decoder_loss configuration of the shipped experiment files (SURVEY §8 a-11):
# + UNet conv_out, VAE decoder 2514.5, Bottleneck(3->128->128) at 512^2 instead of the s2 projection; SURVEY §8d total 4526.0
GF_PER_IMG_S0 = {"vae_encoder": 1116.66, "unet": 803.27, "vae_decoder": 2514.5, "projections": 91.6, "total": 4526.0}
DUMP_BYTES = 60_000_000  # --dump-outputs: data budget of all files together, leaves room for the .npy headers under 64 MB


def dump_outputs(out_dir, named):
    """--dump-outputs: writes each output as out_dir/<name>.npy in float32.  An output larger than its equal share of DUMP_BYTES is
    written as out_dir/<name>_sample.npy instead: its flattened values at the sorted, de-duplicated flat indices
    torch.randint(numel, (share,), generator=torch.Generator().manual_seed(0)).unique() -- the same indices in every run, so that two
    builds can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // 4 // len(named)
    for name, t in named.items():
        t = t.detach().float()
        if t.numel() > share:
            idx = torch.randint(t.numel(), (share,), generator=torch.Generator().manual_seed(0)).unique()
            t, name = t.reshape(-1)[idx.to(t.device)], name + "_sample"
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], tflops_burst=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(pw)}


def cpu_oracle_throughput(timed: int = 3, warm: int = 1, variant: str = "base"):
    """The fp32 oracle (CPU restatement of the reference path) on the host cores: config 1, 1x3x512x512."""
    import torch
    from oracle import synthetic
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ob = synthetic.build_backbone(with_ema=False, variant=variant)
    img = synthetic.synthetic_images(1)
    with torch.no_grad():
        for _ in range(warm):
            ob(img, input_modal="others")
        t0 = time.perf_counter()
        for _ in range(timed):
            ob(img, input_modal="others")
        dt = (time.perf_counter() - t0) / timed
    return dict(value=1.0 / dt, unit=UNIT, cores=torch.get_num_threads(), kind="port",
                sample=f"BASELINE config 1: 1x3x512x512 fp32 oracle forward, {warm} warm-up + {timed} timed, {dt:.2f} s/img, "
                       f"{(GF_PER_IMG if variant == 'base' else GF_PER_IMG_S0)['total'] / dt:.0f} GFLOP/s implied"), dt


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU implementation of the path = the oracle port (the reference itself cannot be
    imported here: diffusers/peft/detectron2 absent).  Rank 0 alone runs it."""
    if rank != 0:
        return
    steps = args.steps
    base, dt = cpu_oracle_throughput(timed=steps, warm=1, variant=args.variant)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": 1, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic (seeded, SURVEY §8d)",
        "config": {"workload": "MADM SD-1.4 UNet+LoRA backbone feature extraction, 8x3x512x512 per GPU in the product arm; the CPU "
                               "arm times a bounded sample of it: 1 image per step", "bounded_sample": "1x3x512x512 per step"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_product(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from helpers import build_product_backbone, set_lora_adapter

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa = None
    if world > 1:
        from madm_b200.sharding import bind_to_gpu_numa
        numa = bind_to_gpu_numa(local_rank)  # before any pinned allocation: first touch places the host buffers next to the GPU
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    torch.manual_seed(1234 + rank)
    bb = build_product_backbone(dev, compute_dtype=args.dtype, variant=args.variant)  # random-init SD-1.4 weights + 2 LoRA adapters (r16)
    gf = GF_PER_IMG if args.variant == "base" else GF_PER_IMG_S0
    ldm = bb.feature_extractor.ldm_extractor
    with torch.no_grad():  # de-degenerate the zero-init pieces like the parity fixtures do
        g = torch.Generator(device=dev).manual_seed(99)
        for _, m in ldm.unet.lora_layers():
            for a in m.lora_B:
                m.lora_B[a].weight.copy_(torch.randn(m.lora_B[a].weight.shape, device=dev, generator=g) * 0.02)
    set_lora_adapter(ldm.unet, "Depth")
    gi = torch.Generator().manual_seed(rank)
    img_host = (torch.rand(B, 3, 512, 512, generator=gi)).pin_memory()
    img_dev = img_host.to(dev, non_blocking=True)
    from madm_b200.engine import OUT_SHAPES
    outs_host = [torch.empty(B, c, s, s, dtype=torch.float32).pin_memory() for c, s in OUT_SHAPES[args.variant]]
    outs_dev = [torch.empty(B, c, s, s, dtype=torch.float32, device=dev) for c, s in OUT_SHAPES[args.variant]]

    # B <= engine.graph_max_batch (8): the backbone replays the step's ~555 launches as one CUDA graph (static input buffer,
    # results cloned out of the static output buffers); larger batches launch on the stream into `outs_dev`.
    graphed = 0 < B <= ldm.engine().graph_max_batch
    last = {}  # the feature maps of the latest step_resident call (--dump-outputs)

    def step_resident():
        last["features"] = bb._extract(img_dev, "others", False, None, out=None if graphed else outs_dev)["features"]

    def step_e2e():
        x = img_host.to(dev, non_blocking=True)               # H2D of this step's inputs from pinned memory
        res = bb._extract(x, "others", False, None, out=None if graphed else outs_dev)
        for h, d in zip(outs_host, res["features"]):           # D2H of this step's result (the feature dict)
            h.copy_(d, non_blocking=True)
        return res

    # the same end-to-end work, with the copies of neighbouring steps overlapped with compute on a second stream
    from madm_b200.pipeline import HostPipeline
    pipe = HostPipeline(lambda x: bb._extract(x, "others", False, None), dev)

    def run_e2e_pipelined(steps):  # streaming mode: `depth` pinned buffer sets, each step's result is handed over once downloaded
        return pipe.run([img_host] * steps, consume=lambda i, host: None)

    # The faithful end of MADM's eval loop: the feature dict never leaves the device -- the head consumes it (mtmadise.py:685-688)
    # and only the arg-max labels go to the host (evaluation/d2_evaluator.py:106).  Backbone + head stage + fused
    # upsample / softmax / arg-max on the device, 8 x 512 x 512 int64 labels downloaded per step.
    from madm_b200 import teacher as mteacher
    from madm_b200.head import DAFormerHead
    from test_head_gpu import HEAD_KW
    head = None
    if args.variant == "base":
        head = DAFormerHead(**HEAD_KW, device=dev, compute_dtype=args.dtype).eval()

    def seg_step(x):
        res = bb._extract(x, "others", False, None)
        logits = head({"output_features": dict(zip(("s2", "s3", "s4", "s5"), res["features"]))})
        label, _, _, _ = mteacher.pseudo_labels(logits, (512, 512), 0.0)
        return {"label": [label]}

    pipe_head = HostPipeline(seg_step, dev, select=lambda res: res["label"]) if head is not None else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, sampler=None):
        barrier()
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)  # max over ranks; the data path itself has no collective
        barrier()
        return ms.item(), clocks

    with torch.no_grad():
        for _ in range(max(3, args.warmup)):
            step_resident()
        ms, clocks = timed(step_resident, args.steps, ClockSampler(local_rank) if rank == 0 else None)
        if args.dump_outputs and rank == 0:  # before the runs below reuse the output buffers
            dump_outputs(args.dump_outputs, dict(zip(bb._out_features, last["features"])))
        for _ in range(2):
            step_e2e()
        ms_e2e_serial, _ = timed(step_e2e, args.steps)
        run_e2e_pipelined(2)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run_e2e_pipelined(args.steps)  # K steps: every step's H2D, compute and D2H inside the timed region
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        barrier()
        ms_e2e = t.item()
        # opt-in fp16 feature maps (backbone.feature_dtype = torch.float16, MADM_FLAG_OUT_FP16): the same pipelined end-to-end run with
        # half the download -- what a host-bound consumer of the feature dict would choose; `e2e` above stays on the reference's fp32 maps
        ms_e2e_f16 = None
        if args.variant == "base":
            bb.feature_dtype = torch.float16
            run_e2e_pipelined(2)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run_e2e_pipelined(args.steps)
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            barrier()
            ms_e2e_f16 = t.item()
            bb.feature_dtype = torch.float32
        ms_e2e_head = None
        if pipe_head is not None:
            pipe_head.run([img_host] * 2, consume=lambda i, host: None)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            pipe_head.run([img_host] * args.steps, consume=lambda i, host: None)
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            barrier()
            ms_e2e_head = t.item()
        # roofline inputs: per-kernel-family CUDA-event timing of instrumented steps on the launch stream
        eng = ldm.engine()
        prof = None
        if rank == 0:
            eng.set_profiling(True)
            acc, acc_unet = None, None
            psteps = 2
            from madm_b200 import _lib as mlib

            def add(dst, p):
                if dst is None:
                    return p
                for k in p:
                    for f in p[k]:
                        dst[k][f] += p[k][f]
                return dst

            for _ in range(psteps):
                bb._extract(img_dev, "others", False, None, out=outs_dev)  # stream launches: the per-launch events live there
                acc = add(acc, eng.profile())
                acc_unet = add(acc_unet, eng.profile(mlib.STAGE_UNET))
            eng.set_profiling(False)
            prof = {k: {f: v[f] / psteps for f in v} for k, v in acc.items()}
            prof_unet = {k: {f: v[f] / psteps for f in v} for k, v in acc_unet.items()}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = read_peaks()
    imgs = B * world * args.steps
    value = imgs / (ms / 1e3)
    e2e_value = imgs / (ms_e2e / 1e3)
    launches = eng.launch_count(B)
    gemm = prof["gemm_tc"]
    gemm_tflops = gemm["flops"] / (gemm["ms"] / 1e3) / 1e12
    total_ms = sum(v["ms"] for v in prof.values())
    gn = prof["groupnorm"]
    gemm_traffic = None
    try:  # measured once under ncu for this build; null if the summary is not in the tree
        with open(os.path.join(ROOT, "profiles", "r02_gemm_dram_traffic.json")) as f:
            gemm_traffic = json.load(f)["dram_bytes_per_launch"]
    except (OSError, KeyError, ValueError):
        pass
    # the north_star's target: the UNet's contractions (convs / linears AND the attention products) against the sustained tensor peak
    u_ms = prof_unet["gemm_tc"]["ms"] + prof_unet["flash_attention"]["ms"]
    u_fl = prof_unet["gemm_tc"]["flops"] + prof_unet["flash_attention"]["flops"]
    roofline_unet = {
        "kernels": "UNet stage: gemm_tc_kernel + fa_tc_kernel launches", "bound": "tensor", "unit": "TFLOP/s",
        "achieved": u_fl / (u_ms / 1e3) / 1e12, "peak": peaks["tflops_sustained"], "frac": u_fl / (u_ms / 1e3) / 1e12 / peaks["tflops_sustained"],
        "algorithmic_gflop_per_step": u_fl / 1e9, "ms_per_step": u_ms,
        "gemm": {"tflops": prof_unet["gemm_tc"]["flops"] / (prof_unet["gemm_tc"]["ms"] / 1e3) / 1e12, "ms": prof_unet["gemm_tc"]["ms"],
                 "launches": prof_unet["gemm_tc"]["launches"]},
        "attention": {"tflops": prof_unet["flash_attention"]["flops"] / (prof_unet["flash_attention"]["ms"] / 1e3) / 1e12,
                      "ms": prof_unet["flash_attention"]["ms"], "launches": prof_unet["flash_attention"]["launches"]},
        "stage_ms_by_family": {k: v["ms"] for k, v in prof_unet.items()},
    }
    roofline = {
        "kernel": "gemm_tc_kernel (tcgen05 implicit GEMM: all convs / linears)", "bound": "tensor",
        "achieved": gemm_tflops, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": gemm_tflops / peaks["tflops_sustained"],
        "flops": "algorithmic (2*MAC of the reference's convs / linears; K padding and the identity-weight residual segments of the 16-bit "
                 "VAE stream are excluded)",
        "executed_tflops": gemm["exec_flops"] / (gemm["ms"] / 1e3) / 1e12,
        "peak_source": peaks["source"] + ", sustained cuBLAS bf16 figure (kernel timed inside a long step)",
        "traffic": gemm_traffic, "traffic_unit": "bytes per launch (ncu dram read + write, profiles/r02_gemm_dram_traffic.json)",
        "algorithmic_bytes_per_launch": gemm["bytes"] / max(1, gemm["launches"]),
        "launches_per_step": gemm["launches"], "avg_launch_ms": gemm["ms"] / max(1, gemm["launches"]),
        "algorithmic_gflop_per_launch": gemm["flops"] / max(1, gemm["launches"]) / 1e9,
        "share_of_step": gemm["ms"] / total_ms,
        "families": {k: {"ms_per_step": v["ms"], "launches": v["launches"], "share": v["ms"] / total_ms} for k, v in prof.items()},
        "groupnorm_hbm": {"achieved_gbs": gn["bytes"] / (gn["ms"] / 1e3) / 1e9 if gn["ms"] > 0 else None, "peak_gbs": peaks["hbm_gbs"]},
        "whole_path_tflops": value / world * gf["total"] / 1e3,
    }
    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_base, _ = cpu_oracle_throughput(timed=3, warm=1, variant=args.variant)
    ws_gb = eng._ws.numel() / 2 ** 30
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic (seeded rand images, random-init SD-1.4 weights + r16 LoRA, SURVEY §8d)",
        "config": {"workload": (f"BASELINE configs[1]: {B}x3x512x512 per GPU, feature extraction a-1..a-9 "
                                "(VAE-enc + q-sample t=0 + UNet taps + s2..s5 projections); sem_seg_head is SURVEY §8 f-2 (next), not timed")
                   if args.variant == "base" else
                   (f"{B}x3x512x512 per GPU, vae_decoder_loss / s0 variant of the shipped experiment configs (SURVEY §8 a-11): VAE-enc + "
                    "q-sample t=0 + UNet to its final output + VAE decoder + s0/s3/s4/s5 projections"),
                   "variant": args.variant,
                   "per_gpu_batch": B, "global_batch": B * world, "input_modal": "others", "adapter": "Depth_r16_a16 (folded)",
                   "l2": f"working set (packed weights 1.8 GB + workspace {ws_gb:.1f} GB) >> 126 MB L2; no explicit flush",
                   "accumulate": "fp32", "residual_stream": "fp32 (UNet, projections); fp16 in the VAE 512^2 / 256^2 stages with fp16 operands, like the reference's fp16 VAE", "gflop_per_image": gf},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": img_host.numel() * 4, "d2h_bytes_per_step": sum(t.numel() * 4 for t in outs_host),
                "api": "madm_b200.pipeline.HostPipeline around AttentionFeatureExtractorBackbone._extract -> madm_extract (C ABI): pinned "
                       "host buffers, H2D / D2H of neighbouring steps overlapped with compute on a copy stream",
                "serial_value": imgs / (ms_e2e_serial / 1e3), "serial_ms_per_step": ms_e2e_serial / args.steps,
                "cuda_graph": bool(graphed)},
        "gpu_launches": launches * args.steps,
        "roofline": roofline,
        "roofline_unet": roofline_unet,
        "cpu_baseline": cpu_base,
    }
    if ms_e2e_head is not None:
        line["e2e_head"] = {"value": imgs / (ms_e2e_head / 1e3), "unit": UNIT, "ms_per_step": ms_e2e_head / args.steps,
                            "h2d_bytes_per_step": img_host.numel() * 4, "d2h_bytes_per_step": B * 512 * 512 * 8,
                            "api": "HostPipeline around backbone -> madm_b200.head.DAFormerHead (MADM_STAGE_HEAD) -> teacher.pseudo_labels "
                                   "(fused upsample / softmax / arg-max): the feature dict stays on the device as in MADM's eval loop "
                                   "(mtmadise.py:685-688), only the int64 label map is downloaded (d2_evaluator.py:106)"}
    if ms_e2e_f16 is not None:
        line["e2e_fp16_features"] = {"value": imgs / (ms_e2e_f16 / 1e3), "unit": UNIT, "ms_per_step": ms_e2e_f16 / args.steps,
                                     "h2d_bytes_per_step": img_host.numel() * 4, "d2h_bytes_per_step": sum(t.numel() * 2 for t in outs_host),
                                     "api": "as `e2e`, with backbone.feature_dtype = torch.float16 (opt-in extension: fp16 feature maps)"}
    if numa:
        line["config"]["numa"] = numa
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_slide(args, rank, local_rank, world):
    """BASELINE configs[2] / configs[3]: sliding-window inference over full-resolution images, crops as the engine's batch dimension
    (feature_extractor.py:199-278), images sharded over the ranks with no collective (weak scaling: --images per GPU).
      slide1024   : 1024 x 1024, 9 crops / image, input_modal 'others' -> merged feature dict (what slide_forward returns)
      teacher2048 : 1024 x 2048, 21 crops / image, 'others' + ema_forward -> EMA-projected merged features -> DAFormer head on the
                    256 x 512 grid -> fused upsample / softmax / max -> pseudo-labels + weights (mtmadise.py:335-349)"""
    import torch
    import torch.distributed as dist
    from helpers import build_product_backbone, set_lora_adapter
    from madm_b200 import teacher as mteacher
    from madm_b200.head import DAFormerHead
    from test_head_gpu import HEAD_KW

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa = None
    if world > 1:
        from madm_b200.sharding import bind_to_gpu_numa
        numa = bind_to_gpu_numa(local_rank)
        dist.init_process_group("nccl", device_id=dev)
    teacher = args.config == "teacher2048"
    H, W = (1024, 2048) if teacher else (1024, 1024)
    n_img = args.images
    torch.manual_seed(1234 + rank)
    bb = build_product_backbone(dev, compute_dtype=args.dtype)
    ldm = bb.feature_extractor.ldm_extractor
    with torch.no_grad():
        g = torch.Generator(device=dev).manual_seed(99)
        for _, m in ldm.unet.lora_layers():
            for a in m.lora_B:
                m.lora_B[a].weight.copy_(torch.randn(m.lora_B[a].weight.shape, device=dev, generator=g) * 0.02)
    set_lora_adapter(ldm.unet, "Depth")
    bb._slide_inference = True
    crops = len(bb.slide_windows(H, W))
    bb.crop_batch = 18 if not teacher else 21  # whole images per engine call: 2 x 9 or 1 x 21 crops (CUDA-graph replay per call)
    head = DAFormerHead(**HEAD_KW, device=dev, compute_dtype=args.dtype).eval() if teacher else None
    gi = torch.Generator().manual_seed(rank)
    img_host = torch.rand(n_img, 3, H, W, generator=gi).pin_memory()
    img_dev = img_host.to(dev)

    def step(x):
        out = bb.slide_forward(x, "others", ema_forward=teacher)
        if not teacher:
            return list(out["output_features"].values())
        logits = head(out)                                       # [n, 19, 256, 512]
        label, prob, weight, count = mteacher.pseudo_labels(logits, (H, W), 0.968)
        return [label, weight]

    host_out = None
    copy_stream = torch.cuda.Stream(device=dev)
    chunk = max(1, bb.crop_batch // crops)  # images per engine call

    def step_e2e():
        """Streaming: the images go through in chunks of one engine call; the upload of chunk k+1 and the download of chunk k's results run on
        a copy stream while chunk k+1 computes (pinned host buffers for the whole step, every byte inside the timed region)."""
        nonlocal host_out
        main = torch.cuda.current_stream(dev)
        keep = []
        up = {}

        def upload(i):
            with torch.cuda.stream(copy_stream):
                x = img_host[i:i + chunk].to(dev, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            up[i] = (x, ev)

        upload(0)
        for i in range(0, n_img, chunk):
            x, ev = up.pop(i)
            if i + chunk < n_img:
                upload(i + chunk)
            main.wait_event(ev)
            x.record_stream(main)
            res = step(x)
            if host_out is None:
                host_out = [torch.empty((n_img,) + tuple(t.shape[1:]), dtype=t.dtype).pin_memory() for t in res]
            done = torch.cuda.Event()
            done.record(main)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done)
                for h, d in zip(host_out, res):
                    h[i:i + d.shape[0]].copy_(d, non_blocking=True)
                    d.record_stream(copy_stream)
            keep.append(res)
        main.wait_stream(copy_stream)  # the step ends when its last result is on the host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, sampler=None):
        barrier()
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return ms.item(), clocks

    last = []  # what the latest timed step returned (--dump-outputs)

    def step_resident():
        last[:] = step(img_dev)

    with torch.no_grad():
        for _ in range(max(3, args.warmup)):
            step(img_dev)
        ms, clocks = timed(step_resident, args.steps, ClockSampler(local_rank) if rank == 0 else None)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, dict(zip(["label", "weight"] if teacher else bb._out_features, last)))
        for _ in range(2):
            step_e2e()
        ms_e2e, _ = timed(step_e2e, args.steps)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    eng = ldm.engine()
    imgs = n_img * world * args.steps
    calls = (n_img + max(1, bb.crop_batch // crops) - 1) // max(1, bb.crop_batch // crops)
    per_call = crops * max(1, bb.crop_batch // crops)
    line = {
        "metric": METRIC, "value": imgs / (ms / 1e3), "unit": "full-resolution images/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic (seeded rand images, random-init SD-1.4 weights + r16 LoRA, SURVEY §8d)",
        "crops_per_s": imgs * crops / (ms / 1e3),
        "config": {"workload": (f"BASELINE configs[3]: {n_img} x 3 x 1024 x 2048 per GPU, EMA-teacher pseudo-label pass: 21 crops / image -> "
                                "feature extraction with ema_feature_projections -> merged maps -> DAFormer head (256 x 512 grid) -> "
                                "pseudo-labels + weights (mtmadise.py:335-349)") if teacher else
                               (f"BASELINE configs[2]: {n_img} x 3 x 1024 x 1024 per GPU, sliding-window inference: 9 crops / image at stride 256 "
                                "-> merged s2..s5 maps (feature_extractor.py:199-278)"),
                   "config": args.config, "images_per_gpu": n_img, "crops_per_image": crops, "crops_per_engine_call": per_call,
                   "engine_calls_per_step": calls, "input_modal": "others", "adapter": "Depth_r16_a16 (folded)",
                   "l2": "working set >> 126 MB L2; no explicit flush", "cuda_graph": per_call <= eng.graph_max_batch},
        "clocks": clocks,
        "e2e": {"value": imgs / (ms_e2e / 1e3), "unit": "full-resolution images/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": img_host.numel() * 4, "d2h_bytes_per_step": sum(t.numel() * t.element_size() for t in host_out),
                "api": "backbone.slide_forward" + (" -> DAFormerHead -> teacher.pseudo_labels; labels + weights downloaded" if teacher else
                                                   "; merged feature dict downloaded") + " (pinned host buffers; uploads / downloads of neighbouring engine calls overlap compute on a copy stream)"},
        "gpu_launches": eng.launch_count(per_call) * calls * args.steps,
        "whole_path_tflops_per_gpu": imgs / world * crops / (ms / 1e3) * GF_PER_IMG["total"] / 1e3,
    }
    if numa:
        line["config"]["numa"] = numa
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_train(args, rank, local_rank, world):
    """BASELINE configs[4]: the LoRA training step, 2 images per GPU (SURVEY §3.2 / §8d config 5; reference MTMADISE.forward
    mtmadise.py:177-656 under AMPTrainer.run_step, engine/train_loop.py:257-311).  One step =
      source pass  : backbone(source, 'rgb', adapter default) under grad
      teacher pass : backbone(target, 'others', ema_forward=True, adapter Depth) under no_grad -> DAFormer head -> pseudo-labels / weights
      DACS mix     : class mask from the source labels, image_mix, one_mix of labels / weights (device kernels, no host sync)
      mixed pass   : backbone(mixed, 'mixed', adapter Depth) under grad
      backward     : ONE backward of the summed losses through both student passes (madm_backward x 2)
      all-reduce   : ONE NCCL all-reduce over the flat gradient buffer of the trainable set (zeros for what took no part)
      update       : FusedAdamW with folded clip_grad_norm_, EMA update of the teacher's projections
    The segmentation head + criterion of the student passes are outside SURVEY §8's path (they stay the reference's own PyTorch code in a
    real run): the bench closes the loop with a fixed linear functional of the feature dict weighted by the mixed pixel weights, so
    every gradient the engine produces is consumed.  value = source images per second over all ranks (2 per GPU per step)."""
    import torch
    import torch.distributed as dist
    from helpers import build_product_backbone, set_lora_adapter
    from madm_b200 import teacher as mteacher
    from madm_b200.head import DAFormerHead
    from madm_b200.optim import FusedAdamW, allreduce_grads, update_ema
    from test_head_gpu import HEAD_KW

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = 2
    dtype = args.train_dtype
    torch.manual_seed(1234)  # identical replicas on every rank (DDP broadcasts the weights; here the seed does)
    bb = build_product_backbone(dev, compute_dtype=dtype)
    ldm = bb.feature_extractor.ldm_extractor
    with torch.no_grad():
        g = torch.Generator(device=dev).manual_seed(99)
        for _, m in ldm.unet.lora_layers():
            for a in m.lora_B:
                m.lora_B[a].weight.copy_(torch.randn(m.lora_B[a].weight.shape, device=dev, generator=g) * 0.02)
    for n, p in bb.named_parameters():  # the LoRA training step's trainable set (BASELINE.json narrows config 5 to it)
        p.requires_grad_(("lora_" in n) or n.startswith("feature_projections.") or (n.startswith("feature_extractor.clip_project_")))
    trainable = [p for p in bb.parameters() if p.requires_grad]
    n_train = sum(p.numel() for p in trainable)
    opt = FusedAdamW(trainable, lr=1e-5, weight_decay=0.01)
    head = DAFormerHead(**HEAD_KW, device=dev, compute_dtype=dtype).eval()
    gi = torch.Generator().manual_seed(100 + rank)
    src_host = torch.rand(B, 3, 512, 512, generator=gi).pin_memory()
    tgt_host = torch.rand(B, 3, 512, 512, generator=gi).pin_memory()
    lab_host = torch.randint(0, 19, (B, 512, 512), generator=gi).pin_memory()
    src_dev, tgt_dev, lab_dev = src_host.to(dev), tgt_host.to(dev), lab_host.to(dev)
    gr = torch.Generator().manual_seed(7)
    R = [torch.randn(B, 512, s, s, generator=gr).to(dev) / 1e3 for s in (128, 64, 32, 16)]
    classes = torch.arange(0, 19, 2, device=dev)
    ev = {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for k in ("fwd", "bwd", "allreduce", "update")}
    acc_ms = {k: 0.0 for k in ev}
    it = [0]

    def functional(feats, w=None):
        tot = 0.0
        for f, r in zip(feats.values(), R):
            t = f * r
            if w is not None:
                t = t * w
            tot = tot + t.sum()
        return tot

    def step(src, tgt, lab, timed=False):
        if timed:
            ev["fwd"][0].record()
        set_lora_adapter(ldm.unet, "default")
        f_src = bb(src, input_modal="rgb")["output_features"]
        loss = functional(f_src)
        with torch.no_grad():
            set_lora_adapter(ldm.unet, "Depth")
            f_t = bb(tgt, input_modal="others", ema_forward=True)
            label, prob, weight, count = mteacher.pseudo_labels(head(f_t), (512, 512), 0.968)
            mixed, wmix = [], []
            for i in range(B):
                mask = mteacher.generate_class_mask(lab[i], classes)
                mixed.append(mteacher.image_mix(mask, torch.stack((src[i], tgt[i]))))
                _, wm = mteacher.one_mix(mask, target=torch.stack((lab[i], label[i])),
                                         weight=torch.stack((torch.ones_like(weight[i]), weight[i])))
                wmix.append(wm)
            mixed = torch.cat(mixed)
            wscalar = torch.cat(wmix).mean()
        f_mix = bb(mixed, input_modal="mixed")["output_features"]
        loss = loss + functional(f_mix) * wscalar
        if timed:
            ev["fwd"][1].record(); ev["bwd"][0].record()
        loss.backward()
        if timed:
            ev["bwd"][1].record(); ev["allreduce"][0].record()
        allreduce_grads(trainable)
        if timed:
            ev["allreduce"][1].record(); ev["update"][0].record()
        opt.step(clip_grad=1.0)
        it[0] += 1
        update_ema(list(bb.ema_feature_projections.parameters()), list(bb.feature_projections.parameters()), it[0])
        opt.zero_grad(set_to_none=True)
        if timed:
            ev["update"][1].record()
        return loss.detach()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step(src_dev, tgt_dev, lab_dev)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    prof = bool(os.environ.get("MADM_BENCH_CUDA_PROFILE"))  # bracket the timed steps for `ncu --profile-from-start off`
    if prof:
        torch.cuda.cudart().cudaProfilerStart()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step(src_dev, tgt_dev, lab_dev, timed=True)
    e1.record()
    torch.cuda.synchronize()
    if prof:
        torch.cuda.cudart().cudaProfilerStop()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:  # the step's loss and the trainable parameters it updated
        dump_outputs(args.dump_outputs, {"loss": loss, **{n: p for n, p in bb.named_parameters() if p.requires_grad}})
    for k in ev:  # (events of the LAST step: a per-phase picture, not the timed total)
        acc_ms[k] = ev[k][0].elapsed_time(ev[k][1])
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    barrier()
    # end to end: the step's inputs come from pinned host memory, its loss is read back
    loss_host = torch.zeros(1).pin_memory()

    def step_e2e():
        l = step(src_host.to(dev, non_blocking=True), tgt_host.to(dev, non_blocking=True), lab_host.to(dev, non_blocking=True))
        loss_host.copy_(l.reshape(1), non_blocking=True)
    step_e2e()
    barrier()
    e0.record()
    for _ in range(args.steps):
        step_e2e()
    e1.record()
    torch.cuda.synchronize()
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    eng = ldm.engine()
    imgs = B * world * args.steps
    fwd_l = eng.launch_count(B)
    bwd_l = int(eng.lib.madm_backward_launch_count(eng.ctx, B))
    # algorithmic FLOPs of one step per GPU: 3 forwards of the base path on 2 images + 2 backward passes through UNet + projections
    # (input gradients ~ 1x the forward contractions of the UNet, attention backward 2.5x its forward; LoRA / projection weight
    # gradients are small) -- reported as an estimate, the bench's figure of merit is images/s
    gf_fwd = 3 * B * GF_PER_IMG["total"]
    gf_bwd = 2 * B * (GF_PER_IMG["unet_taps"] * 1.25 + GF_PER_IMG["projections"] * 2)
    line = {
        "metric": METRIC, "value": imgs / (ms.item() / 1e3), "unit": "training images/s (2 source images per GPU per step)", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms.item() / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": dtype, "data": "synthetic (seeded rand images / labels, random-init SD-1.4 weights + r16 LoRA, SURVEY §8d)",
        "config": {"workload": "BASELINE configs[4]: LoRA training step, 2 images per GPU: source pass (rgb / default) + EMA-teacher pass + DACS "
                               "mix + mixed pass (mixed / Depth) under grad, one backward, one gradient all-reduce, AdamW + clip, EMA update",
                   "config": "train", "per_gpu_batch": B, "trainable_parameters": n_train, "allreduce_bytes": n_train * 4,
                   "loss": "fixed linear functional of the feature dict (the head + criterion of the student passes are outside SURVEY §8)",
                   "loss_scale": float(getattr(ldm, "train_loss_scale", None) or (1.0 if dtype == "bf16" else 4096.0)),
                   "l2": "working set >> 126 MB L2; no explicit flush"},
        "clocks": clocks,
        "e2e": {"value": imgs / (ms2.item() / 1e3), "unit": "training images/s", "ms_per_step": ms2.item() / args.steps,
                "h2d_bytes_per_step": 2 * src_host.numel() * 4 + lab_host.numel() * 8, "d2h_bytes_per_step": 4,
                "api": "backbone(...) under grad x 2 + teacher pass + loss.backward() + allreduce_grads + FusedAdamW.step + update_ema; images "
                       "and labels uploaded from pinned memory, the loss read back"},
        "phases_last_step_ms": acc_ms,
        "allreduce_exposed_ms": acc_ms["allreduce"],
        "gpu_launches": (3 * fwd_l + 2 * bwd_l) * args.steps,
        "launches_per_step": {"forward_per_pass": fwd_l, "backward_per_pass": bwd_l},
        "estimated_tflops_per_gpu": (gf_fwd + gf_bwd) / (ms.item() / args.steps),
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="madm_b200", choices=["madm_b200", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="images per GPU per step")
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"], help="GEMM operand dtype (fp32 accumulate)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="base", choices=["base", "slide1024", "teacher2048", "train"],
                    help="base = BASELINE configs[1] (the bench line); slide1024 / teacher2048 / train = BASELINE configs[2..4]")
    ap.add_argument("--train-dtype", default="fp16", choices=["fp16", "bf16"],
                    help="operand dtype of the training step: fp16 + loss scale (the reference's AMP regime, default) or bf16")
    ap.add_argument("--images", type=int, default=8, help="full-resolution images per GPU per step (slide1024 / teacher2048)")
    ap.add_argument("--variant", default="base", choices=["base", "s0"],
                    help="base = BASELINE configs[1] (the bench line); s0 = vae_decoder_loss configuration of the shipped experiment files")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rank 0) as DIR/<name>.npy in float32, "
                         "under 64 MB in all: outputs larger than their share are written as a fixed, seeded sample, DIR/<name>_sample.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the product arm (--impl madm_b200)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1 and args.gpus > 1:
        # convenience: spawn torchrun ourselves when called directly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", os.environ.get("MASTER_PORT", "29533"), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.config in ("slide1024", "teacher2048"):
        run_slide(args, rank, local_rank, world)
    elif args.config == "train":
        run_train(args, rank, local_rank, world)
    else:
        run_product(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
