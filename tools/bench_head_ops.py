import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from madm_b200 import ops
dev = torch.device('cuda:0')
def timed(fn, n=10):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3
B = 8
x = torch.randn(B, 512, 128, 128, device=dev)
t = timed(lambda: ops.nchw_to_nhwc16(x)); print(f"nchw_to_nhwc16 s2: {t:.1f} us  {x.numel()*6/t/1e6:.0f} GB/s")
e = torch.randn(B, 64, 64, 256, device=dev).half()
cat = torch.empty(B, 128, 128, 1024, device=dev, dtype=torch.float16)
t = timed(lambda: ops.bilinear_resize(e, 128, 128, out=cat[..., 256:], pitch=1024)); print(f"bilinear 64->128: {t:.1f} us  {(B*128*128*256*2 + e.numel()*2)/t/1e6:.0f} GB/s")
w9 = torch.randn(9, 1024, device=dev); sh = torch.randn(1024, device=dev)
for d in (6, 12, 18):
    t = timed(lambda: ops.depthwise3x3(cat, w9, sh, d)); print(f"depthwise dil={d}: {t:.1f} us  {cat.numel()*4/t/1e6:.0f} GB/s")
