#!/usr/bin/env python
"""Attention backward against torch.autograd on a chosen input distribution (peaky softmax, loss-scaled dO), at the d = 40 self-attention
shape that runs on the tcgen05 kernels.  Usage: check_attn_bwd.py [qk_scale] [do_scale] [dtype]"""
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
from madm_b200 import ops  # noqa: E402

qk_scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
do_scale = float(sys.argv[2]) if len(sys.argv) > 2 else 0.1
dt = torch.bfloat16 if (len(sys.argv) > 3 and sys.argv[3] == "bf16") else torch.float16
dev = torch.device("cuda:0")
B, heads, d, N = 2, 8, 40, 1024
Cc = heads * d
g = torch.Generator(device="cuda").manual_seed(1)
qkv = torch.randn(B, N, 3 * Cc, device=dev, generator=g)
qkv[..., :2 * Cc] *= qk_scale
qkv = qkv.to(dt)
q, k, v = qkv[..., :Cc], qkv[..., Cc:2 * Cc], qkv[..., 2 * Cc:]
dqkv = torch.zeros_like(qkv)
dq, dk, dv = dqkv[..., :Cc], dqkv[..., Cc:2 * Cc], dqkv[..., 2 * Cc:]
dout = (torch.randn(B, N, Cc, device=dev, generator=g) * do_scale).to(dt)
split = lambda t: t.double().reshape(B, -1, heads, d).transpose(1, 2)  # noqa: E731
qr, kr, vr = (split(t).detach().requires_grad_(True) for t in (q, k, v))
ref_o = F.scaled_dot_product_attention(qr, kr, vr)
ref_o.backward(split(dout))
o = ref_o.transpose(1, 2).reshape(B, N, Cc).to(dt).contiguous()
ops.attention_bwd(q, 3 * Cc, k, 3 * Cc, v, 3 * Cc, o, Cc, dout, Cc, dq, 3 * Cc, dk, 3 * Cc, dv, 3 * Cc, B, heads, d, N, N, N * 3 * Cc, N * 3 * Cc, N * Cc, N * Cc,
                  N * 3 * Cc, N * 3 * Cc, 1.0 / math.sqrt(d))
torch.cuda.synchronize()
merge = lambda t: t.transpose(1, 2).reshape(B, -1, Cc)  # noqa: E731
print(f"qk_scale {qk_scale} do_scale {do_scale} {dt}")
for name, got, ref in (("dq", dq, qr.grad), ("dk", dk, kr.grad), ("dv", dv, vr.grad)):
    r = merge(ref).double().flatten(); gg = got.double().flatten()
    cos = F.cosine_similarity(gg, r, dim=0).item()
    print(f"  {name}: cosine {cos:.7f}  |got|/|ref| {(gg.norm() / r.norm()).item():.5f}  max-rel {((gg - r).abs().max() / r.abs().max()).item():.2e}  nonfinite {int((~torch.isfinite(got)).sum())}")
