"""Training step of the vae_decoder_loss / s0 variant (the configuration the shipped experiment files select), timed next to the base
variant's step of bench.py --config train in the same process, alternating the two.

One step, 2 images per GPU, as bench.py run_train:
  source pass  : backbone(source, 'rgb', adapter default, return_unet_final_output=True) under grad; the loss takes a term on
                 'before_vae.decoder' (what the meta-arch's vae_decoder_loss differentiates) next to the feature functional
  teacher pass : backbone(target, 'others', ema_forward=True, adapter Depth) under no_grad -> DAFormer head -> pseudo-labels / weights
  DACS mix     : class mask, image_mix, one_mix
  mixed pass   : backbone(mixed, 'mixed', adapter Depth) under grad
  backward     : one loss.backward(), gradient all-reduce, FusedAdamW with clip, EMA update of the teacher's projections
Afterwards one profiled s0 step (torch.profiler, its own run) gives the device time of projection 0's backward, the 512^2 Bottleneck(3 -> 128)
on the decoded image, with its two weight-gradient launches (conv2 3x3 and conv3 1x1, each a wgrad kernel + its reduce) shown separately.
Prints one JSON line.  Usage: python tools/bench_train_s0.py [--steps 10] [--warmup 3] [--rounds 3] [--dtype fp16|bf16]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

B = 2


def card():
    """Name and power limit of the GPU, read now (they belong next to every number this script prints)."""
    import torch
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip().split(",")
        info["name"], info["power_limit_w"] = q[0].strip(), float(q[1])
    except Exception:  # the limit is then reported as unknown
        pass
    return info


def make_step(variant, dtype, dev):
    """A closure running one training step of `variant` (and the objects it trains), built as bench.py run_train builds the base one."""
    import torch
    from helpers import build_product_backbone, set_lora_adapter
    from madm_b200 import teacher as mteacher
    from madm_b200.head import DAFormerHead
    from madm_b200.optim import FusedAdamW, allreduce_grads, update_ema
    from test_head_gpu import HEAD_KW
    s0 = variant == "s0"
    torch.manual_seed(1234)
    bb = build_product_backbone(dev, compute_dtype=dtype, variant=variant)
    ldm = bb.feature_extractor.ldm_extractor
    with torch.no_grad():
        g = torch.Generator(device=dev).manual_seed(99)
        for _, m in ldm.unet.lora_layers():
            for a in m.lora_B:
                m.lora_B[a].weight.copy_(torch.randn(m.lora_B[a].weight.shape, device=dev, generator=g) * 0.02)
    for n, p in bb.named_parameters():
        p.requires_grad_(("lora_" in n) or n.startswith("feature_projections.") or (n.startswith("feature_extractor.clip_project_")))
    trainable = [p for p in bb.parameters() if p.requires_grad]
    opt = FusedAdamW(trainable, lr=1e-5, weight_decay=0.01)
    kw = dict(HEAD_KW, in_channels=[128, 512, 512, 512], in_keys=["s0", "s3", "s4", "s5"]) if s0 else HEAD_KW
    head = DAFormerHead(**kw, device=dev, compute_dtype=dtype).eval()
    gi = torch.Generator().manual_seed(100)
    src = torch.rand(B, 3, 512, 512, generator=gi).to(dev)
    tgt = torch.rand(B, 3, 512, 512, generator=gi).to(dev)
    lab = torch.randint(0, 19, (B, 512, 512), generator=gi).to(dev)
    gr = torch.Generator().manual_seed(7)
    shapes = ((128, 512), (512, 64), (512, 32), (512, 16)) if s0 else ((512, 128), (512, 64), (512, 32), (512, 16))
    R = [torch.randn(B, c, s, s, generator=gr).to(dev) / 1e3 for c, s in shapes]
    R_final = torch.randn(B, 4, 64, 64, generator=gr).to(dev) / 1e3
    classes = torch.arange(0, 19, 2, device=dev)
    ev = {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for k in ("fwd", "bwd", "allreduce", "update")}
    it = [0]

    def functional(feats, w=None):
        tot = 0.0
        for f, r in zip(feats.values(), R):
            t = f * r
            tot = tot + (t * w if w is not None else t).sum()
        return tot

    def step(timed=False):
        if timed:
            ev["fwd"][0].record()
        set_lora_adapter(ldm.unet, "default")
        if s0:
            feats, final = bb(src, input_modal="rgb", return_unet_final_output=True)
            loss = functional(feats["output_features"]) + (final["before_vae.decoder"] * R_final).sum()
        else:
            loss = functional(bb(src, input_modal="rgb")["output_features"])
        with torch.no_grad():
            set_lora_adapter(ldm.unet, "Depth")
            f_t = bb(tgt, input_modal="others", ema_forward=True)
            label, prob, weight, count = mteacher.pseudo_labels(head(f_t), (512, 512), 0.968)
            mixed, wmix = [], []
            for i in range(B):
                mask = mteacher.generate_class_mask(lab[i], classes)
                mixed.append(mteacher.image_mix(mask, torch.stack((src[i], tgt[i]))))
                _, wm = mteacher.one_mix(mask, target=torch.stack((lab[i], label[i])), weight=torch.stack((torch.ones_like(weight[i]), weight[i])))
                wmix.append(wm)
            mixed = torch.cat(mixed)
            wscalar = torch.cat(wmix).mean()
        loss = loss + functional(bb(mixed, input_modal="mixed")["output_features"]) * wscalar
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

    def phases():
        return {k: ev[k][0].elapsed_time(ev[k][1]) for k in ev}

    def launches():
        eng = ldm.engine()
        return {"forward_per_pass": eng.launch_count(B, eng.stage_all), "backward_per_pass": int(eng.lib.madm_backward_launch_count(eng.ctx, B))}

    return step, phases, launches


def proj0_backward(step, out_dir):
    """Device time of projection 0's backward in each madm_backward of one profiled step, from the kernel trace: the kernels from the ReLU
    backward that precedes the first K = 3 partials kernel through the second K = 3 finish kernel.  The weight gradients inside it are the
    runs of wgrad kernels: conv3 (1x1) first, then conv2 (3x3)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    path = os.path.join(out_dir, "bench_train_s0_trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    k = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    names = [e["name"] for e in k]
    parts = [j for j, n in enumerate(names) if "c3_gn_bwd_partials" in n]
    fins = [j for j, n in enumerate(names) if "c3_gn_bwd_finish" in n]
    passes = []
    for first, end in zip(parts[0::2], fins[1::2]):  # conv1, then shortcut: two partials / finish pairs per pass
        start = max(j for j in range(first) if "relu_bwd_nchw" in names[j])
        seg = k[start:end + 1]
        runs, cur = [], None
        for e in seg:
            if "wgrad" in e["name"]:
                cur = (cur or 0.0) + e["dur"]
            elif cur is not None:
                runs.append(cur)
                cur = None
        passes.append({"total_us": sum(e["dur"] for e in seg), "launches": len(seg),
                       "wgrad_conv3_us": runs[0] if runs else None, "wgrad_conv2_us": runs[1] if len(runs) > 1 else None,
                       "k3_branches_us": sum(e["dur"] for e in seg if "c3_gn_bwd" in e["name"])})
    return passes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternating timed windows per variant")
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--out", default=None, help="directory for the profiler trace (default: a temporary directory)")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_train_s0 measures on the GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    steps = {v: make_step(v, args.dtype, dev) for v in ("s0", "base")}
    for v in steps:
        for _ in range(args.warmup):
            steps[v][0]()
    torch.cuda.synchronize()
    ms = {v: [] for v in steps}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for v in steps:
            e0.record()
            for _ in range(args.steps):
                steps[v][0](timed=True)
            e1.record()
            torch.cuda.synchronize()
            ms[v].append(e0.elapsed_time(e1) / args.steps)
    phases = {v: steps[v][1]() for v in steps}
    launches = {v: steps[v][2]() for v in steps}
    out_dir = args.out or tempfile.mkdtemp(prefix="bench_train_s0_")
    os.makedirs(out_dir, exist_ok=True)
    p0 = proj0_backward(steps["s0"][0], out_dir)
    M = B * 512 * 512
    line = {
        "metric": "training step ms, vae_decoder_loss / s0 variant vs base (2 images per GPU, 1 GPU)",
        "card": card(), "dtype": args.dtype, "steps": args.steps, "rounds": args.rounds,
        "ms_per_step": {v: min(x) for v, x in ms.items()}, "ms_per_step_all_rounds": ms,
        "images_per_s": {v: B / (min(x) / 1e3) for v, x in ms.items()},
        "phases_last_step_ms": phases,
        "launches": launches,
        "proj0_backward_per_pass": p0,
        "proj0_wgrad_gflop_per_pass": {"conv2_3x3": 2.0 * M * 128 * 1152 / 1e9, "conv3_1x1": 2.0 * M * 128 * 128 / 1e9},
        "trace": os.path.join(out_dir, "bench_train_s0_trace.json"),
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
