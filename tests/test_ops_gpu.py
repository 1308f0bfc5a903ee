"""Kernel-level parity (GPU): every CUDA kernel of the hot path, called through the C ABI (madm_op_*), against a
plain PyTorch fp32 restatement of the same op on the same (bf16-rounded) inputs.

Tolerances: GEMM/conv fp32 outputs rel 2e-3 of max|ref| (fp32 accumulation order), bf16 outputs 1e-2;
norms 1e-2 (bf16 output rounding); attention 2e-2 (bf16 P).  Byte/index kernels (pack, s2d, upsample) bit-exact.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


DT = torch.float16  # operand dtype under test; the module is re-run for bf16 through the `dt` fixture


def bf(t):
    """Round to the 16-bit operand dtype under test."""
    return t.to(DT)


def relerr(a, b):
    return ((a.float() - b.float()).abs().max() / b.float().abs().max().clamp_min(1e-6)).item()


@pytest.fixture(scope="module", params=["fp16", "bf16"])
def ops(request, cuda_device):
    """The op wrappers, with the module-level operand dtype switched for the whole parametrised pass."""
    global DT
    DT = torch.float16 if request.param == "fp16" else torch.bfloat16
    from madm_b200 import ops as o
    return o


def nhwc(x):  # NCHW -> NHWC contiguous
    return x.permute(0, 2, 3, 1).contiguous()


# ---------------------------------------------------------------------------------------------- plain GEMM
@pytest.mark.parametrize("M,K,N,bn", [(300, 320, 320, 0), (300, 320, 320, 64), (1024, 1280, 640, 128), (77, 768, 1920, 192),
                                      (8, 320, 1280, 0), (256, 64, 128, 0), (512, 2560, 1280, 256), (130, 128, 96, 32),
                                      (4096, 512, 4096, 0)])
def test_gemm_plain(ops, cuda_device, M, K, N, bn):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N)
    a = bf(torch.randn(M, K, device=cuda_device, generator=g))
    w = bf(torch.randn(N, K, device=cuda_device, generator=g) / math.sqrt(K))
    bias = torch.randn(N, device=cuda_device, generator=g)
    o32 = torch.full((M, N), float("nan"), device=cuda_device)
    o16 = torch.empty(M, N, dtype=DT, device=cuda_device)
    ops.gemm([ops.make_seg(a, 1, 1, M, K)], M, N, w, bias=bias, out_f32=o32, ldo32=N, out_bf16=o16, ldo16=N, bn=bn)
    ref = a.float() @ w.float().t() + bias
    assert relerr(o32, ref) < 2e-3
    assert relerr(o16, ref) < 1e-2


@pytest.mark.parametrize("B,H,W,Cin,Cout", [(2, 32, 32, 128, 128), (1, 8, 128, 64, 128), (3, 8, 8, 128, 256), (1, 16, 16, 64, 640), (1, 16, 24, 64, 128)])
def test_conv3x3_256row_tiles(ops, cuda_device, B, H, W, Cin, Cout):
    """bn = 128 with two M sub-tiles per CTA (256-row tiles sharing each weight box), incl. ragged M and fused statistics."""
    g = torch.Generator(device="cuda").manual_seed(B * 10 + H + Cout)
    if W == 24:  # plain matrix with M not a multiple of 256
        M, K = 1000, 320
        a = bf(torch.randn(M, K, device=cuda_device, generator=g))
        w = bf(torch.randn(Cout, K, device=cuda_device, generator=g) / math.sqrt(K))
        out = torch.empty(M, Cout, device=cuda_device)
        ops.gemm([ops.make_seg(a, 1, 1, M, K)], M, Cout, w, out_f32=out, ldo32=Cout, bn=128, mt=2)
        assert relerr(out, a.float() @ w.float().t()) < 2e-3
        return
    x = bf(torch.randn(B, Cin, H, W, device=cuda_device, generator=g))
    w = torch.randn(Cout, Cin, 3, 3, device=cuda_device, generator=g) / math.sqrt(9 * Cin)
    bias = torch.randn(Cout, device=cuda_device, generator=g)
    wp = ops.pack_conv(w, dtype=DT)
    a = nhwc(x)
    M = B * H * W
    out = torch.empty(M, Cout, device=cuda_device)
    o16 = torch.empty(M, Cout, dtype=DT, device=cuda_device)
    cs = torch.full((M // 32, Cout, 2), float("nan"), device=cuda_device)
    ops.gemm([ops.make_seg(a, B, H, W, Cin, taps=ops.taps_3x3())], M, Cout, wp, bias=bias, out_f32=out, ldo32=Cout, out_bf16=o16, ldo16=Cout,
             colstats=cs, stat_rows=32, bn=128, mt=2)
    ref = nhwc(F.conv2d(x.float(), bf(w).float(), bias, padding=1)).reshape(M, Cout)
    assert relerr(out, ref) < 2e-3
    assert relerr(o16, ref) < 1e-2
    assert relerr(cs[..., 0], out.reshape(M // 32, 32, Cout).sum(1)) < 1e-4


def test_gemm_epilogue_variants(ops, cuda_device):
    g = torch.Generator(device="cuda").manual_seed(5)
    B, HW, K, N = 3, 256, 128, 320
    M = B * HW
    a = bf(torch.randn(M, K, device=cuda_device, generator=g))
    w = bf(torch.randn(N, K, device=cuda_device, generator=g) / math.sqrt(K))
    bias = torch.randn(N, device=cuda_device, generator=g)
    rowbias = torch.randn(B, 1000, device=cuda_device, generator=g)
    res = torch.randn(M, N, device=cuda_device, generator=g)
    # row bias (time embedding), residual in place, SiLU, alpha
    out = res.clone()
    ops.gemm([ops.make_seg(a, 1, 1, M, K)], M, N, w, bias=bias, rowbias=rowbias[:, 40:], rows_per_img=HW, ld_rowbias=1000,
             residual=out, ldr=N, out_f32=out, ldo32=N, alpha=0.5)
    ref = 0.5 * (a.float() @ w.float().t()) + bias + rowbias[:, 40:40 + N].repeat_interleave(HW, 0) + res
    assert relerr(out, ref) < 2e-3
    o16 = torch.empty(M, N, dtype=DT, device=cuda_device)
    ops.gemm([ops.make_seg(a, 1, 1, M, K)], M, N, w, bias=bias, out_bf16=o16, ldo16=N, act=1)
    assert relerr(o16, F.silu(a.float() @ w.float().t() + bias)) < 1e-2
    ops.gemm([ops.make_seg(a, 1, 1, M, K)], M, N, w, bias=bias, out_bf16=o16, ldo16=N, act=3)
    assert relerr(o16, F.relu(a.float() @ w.float().t() + bias)) < 1e-2
    # narrow N (latent head): N=4 of a 16-row padded weight, scalar epilogue path, pitch 4
    w16 = torch.zeros(16, K, dtype=DT, device=cuda_device)
    w16[:4] = w[:4]
    o4 = torch.empty(M, 4, device=cuda_device)
    ops.gemm([ops.make_seg(a, 1, 1, M, K)], M, 4, w16, Nw=16, bias=bias[:16].contiguous(), out_f32=o4, ldo32=4, bn=16)
    assert relerr(o4, a.float() @ w[:4].float().t() + bias[:4]) < 2e-3


def test_gemm_strided_operands(ops, cuda_device):
    """A and W read out of wider buffers (q | k halves of a fused projection), as the VAE attention does."""
    g = torch.Generator(device="cuda").manual_seed(9)
    T, Cc = 512, 128
    qk = bf(torch.randn(T, 2 * Cc, device=cuda_device, generator=g))
    S = torch.empty(T, T, device=cuda_device)
    ops.gemm([ops.make_seg(qk, 1, 1, T, Cc, ld=2 * Cc)], T, T, qk[:, Cc:], ldw=2 * Cc, out_f32=S, ldo32=T, alpha=0.125)
    ref = 0.125 * (qk[:, :Cc].float() @ qk[:, Cc:].float().t())
    assert relerr(S, ref) < 2e-3


def test_gemm_geglu(ops, cuda_device):
    g = torch.Generator(device="cuda").manual_seed(11)
    M, Cc = 384, 320
    x = bf(torch.randn(M, Cc, device=cuda_device, generator=g))
    w = torch.randn(8 * Cc, Cc, device=cuda_device, generator=g) / math.sqrt(Cc)
    b = torch.randn(8 * Cc, device=cuda_device, generator=g)
    wp, bp = ops.pack_geglu(w, b, dtype=DT)
    out = torch.empty(M, 4 * Cc, dtype=DT, device=cuda_device)
    ops.gemm([ops.make_seg(x, 1, 1, M, Cc)], M, 4 * Cc, wp, Nw=8 * Cc, bias=bp, out_bf16=out, ldo16=4 * Cc, act=2)
    p = x.float() @ bf(w).float().t() + b
    h, gate = p.chunk(2, dim=-1)
    assert relerr(out, h * F.gelu(gate)) < 1e-2


@pytest.mark.parametrize("M,K,N,bn,pair", [(300, 320, 320, 0, 0), (1000, 320, 960, 192, -1), (4096, 1280, 320, 0, 1), (32768, 320, 320, 0, 0), (520, 640, 640, 64, 0),
                                           (2048, 128, 96, 32, 0), (8192, 640, 1280, 128, 0), (8192, 512, 512, 256, 1)])
def test_gemm_tma_store_epilogue_matches_coalesced(ops, cuda_device, monkeypatch, M, K, N, bn, pair):
    """The TMA-store epilogue (bulk tensor stores of swizzled 32x32 tiles; bulk reduce-add for `hs += GEMM`) against the coalesced-store
    epilogue (MADM_GEMM_TMA_EPI=0) on the same launch: bit-identical for every mode it takes over, incl. ragged M (clipped by the
    tensor map), row bias, activation and untouched neighbours in a wider output buffer."""
    g = torch.Generator(device="cuda").manual_seed(M + N + bn)
    a = bf(torch.randn(M, K, device=cuda_device, generator=g))
    w = bf(torch.randn(N, K, device=cuda_device, generator=g) / math.sqrt(K))
    bias = torch.randn(N, device=cuda_device, generator=g)
    HW = 8 if M % 32 else 32
    nimg = (M + HW - 1) // HW
    rowbias = torch.randn(nimg, N, device=cuda_device, generator=g) if M % 32 == 0 else None
    res = torch.randn(M, N + 32, device=cuda_device, generator=g)
    seg = ops.make_seg(a, 1, 1, M, K)

    def run_all():
        outs = []
        o32 = torch.full((M, N + 32), 7.0, device=cuda_device)  # wider buffer: the last 32 columns must stay untouched
        ops.gemm([seg], M, N, w, bias=bias, rowbias=rowbias, rows_per_img=HW, out_f32=o32, ldo32=N + 32, bn=bn, pair=pair, act=1)
        outs.append(o32)
        hs = res.clone()
        ops.gemm([seg], M, N, w, bias=bias, residual=hs, ldr=N + 32, out_f32=hs, ldo32=N + 32, bn=bn, pair=pair, alpha=0.5)
        outs.append(hs)
        o16 = torch.full((M, N + 32), 3.0, device=cuda_device, dtype=DT)
        ops.gemm([seg], M, N, w, bias=bias, out_bf16=o16, ldo16=N + 32, bn=bn, pair=pair)
        outs.append(o16)
        o16r = torch.full((M, N + 32), 3.0, device=cuda_device, dtype=DT)  # out-of-place fp32 residual, 16-bit output (the FF out-projection)
        ops.gemm([seg], M, N, w, bias=bias, residual=res, ldr=N + 32, out_bf16=o16r, ldo16=N + 32, bn=bn, pair=pair)
        outs.append(o16r)
        if M % 32 == 0:  # fused GroupNorm column statistics next to either output kind
            for kind in ("f32", "h16"):
                cs = torch.full((M // 32, N, 2), float("nan"), device=cuda_device)
                o = torch.empty(M, N, device=cuda_device, dtype=torch.float32 if kind == "f32" else DT)
                kw = dict(out_f32=o, ldo32=N) if kind == "f32" else dict(out_bf16=o, ldo16=N)
                ops.gemm([seg], M, N, w, bias=bias, colstats=cs, stat_rows=32, bn=bn, pair=pair, **kw)
                outs += [o, cs]
        torch.cuda.synchronize()
        return outs

    monkeypatch.setenv("MADM_GEMM_TMA_EPI", "0")
    ref = run_all()
    monkeypatch.setenv("MADM_GEMM_TMA_EPI", "1")
    got = run_all()
    for i, (r_, g_) in enumerate(zip(ref, got)):
        if i >= 4 and i % 2 == 1:  # statistics: another (fixed) summation order
            assert relerr(g_, r_) < 1e-5
            o = got[i - 1].float() if got[i - 1].dtype == torch.float32 else None
            if o is not None:
                assert relerr(g_[..., 0], o.reshape(M // 32, 32, N).sum(1)) < 1e-4 and relerr(g_[..., 1], (o * o).reshape(M // 32, 32, N).sum(1)) < 1e-4
        else:
            assert torch.equal(r_, g_)
    assert relerr(got[0][:, :N], F.silu(a.float() @ w.float().t() + bias + (rowbias.repeat_interleave(HW, 0)[:M] if rowbias is not None else 0))) < 2e-3
    assert relerr(got[1][:, :N], 0.5 * (a.float() @ w.float().t()) + bias + res[:, :N]) < 2e-3
    assert torch.equal(got[1][:, N:], res[:, N:]) and bool((got[0][:, N:] == 7.0).all()) and bool((got[2][:, N:] == 3.0).all())
    assert relerr(got[3][:, :N], a.float() @ w.float().t() + bias + res[:, :N]) < 1e-2 and bool((got[3][:, N:] == 3.0).all())


def test_gemm_geglu_tma_store_matches_coalesced(ops, cuda_device, monkeypatch):
    g = torch.Generator(device="cuda").manual_seed(12)
    M, Cc = 1000, 320
    x = bf(torch.randn(M, Cc, device=cuda_device, generator=g))
    w = torch.randn(8 * Cc, Cc, device=cuda_device, generator=g) / math.sqrt(Cc)
    b = torch.randn(8 * Cc, device=cuda_device, generator=g)
    wp, bp = ops.pack_geglu(w, b, dtype=DT)
    outs = []
    for sw in ("0", "1"):
        monkeypatch.setenv("MADM_GEMM_TMA_EPI", sw)
        out = torch.zeros(M, 4 * Cc, dtype=DT, device=cuda_device)
        ops.gemm([ops.make_seg(x, 1, 1, M, Cc)], M, 4 * Cc, wp, Nw=8 * Cc, bias=bp, out_bf16=out, ldo16=4 * Cc, act=2)
        torch.cuda.synchronize()
        outs.append(out)
    assert torch.equal(outs[0], outs[1])


# ---------------------------------------------------------------------------------------------- implicit-GEMM convs
@pytest.mark.parametrize("B,H,W,Cin,Cout", [(2, 16, 16, 128, 192), (1, 8, 128, 64, 128), (3, 8, 8, 128, 320), (1, 64, 64, 320, 320),
                                            (2, 32, 32, 192, 640), (1, 4, 256, 64, 128)])
def test_conv3x3(ops, cuda_device, B, H, W, Cin, Cout):
    g = torch.Generator(device="cuda").manual_seed(B * 100 + H)
    x = bf(torch.randn(B, Cin, H, W, device=cuda_device, generator=g))
    w = torch.randn(Cout, Cin, 3, 3, device=cuda_device, generator=g) / math.sqrt(9 * Cin)
    bias = torch.randn(Cout, device=cuda_device, generator=g)
    wp = ops.pack_conv(w, dtype=DT)
    a = nhwc(x)
    M = B * H * W
    out = torch.empty(M, Cout, device=cuda_device)
    ops.gemm([ops.make_seg(a, B, H, W, Cin, taps=ops.taps_3x3())], M, Cout, wp, bias=bias, out_f32=out, ldo32=Cout)
    ref = nhwc(F.conv2d(x.float(), bf(w).float(), bias, padding=1)).reshape(M, Cout)
    assert relerr(out, ref) < 2e-3


@pytest.mark.parametrize("pad1", [True, False])
@pytest.mark.parametrize("B,H,W,Cc", [(2, 32, 32, 64), (1, 16, 16, 128), (2, 256, 256, 64)])
def test_conv3x3_stride2(ops, cuda_device, pad1, B, H, W, Cc):
    g = torch.Generator(device="cuda").manual_seed(H + (1 if pad1 else 0))
    x = torch.randn(B, Cc, H, W, device=cuda_device, generator=g)
    w = torch.randn(Cc, Cc, 3, 3, device=cuda_device, generator=g) / math.sqrt(9 * Cc)
    bias = torch.randn(Cc, device=cuda_device, generator=g)
    s2d = ops.space_to_depth(nhwc(x), dtype=DT)
    # space-to-depth is pure data movement: bit-exact
    xb = bf(nhwc(x))
    for ph in range(4):
        assert torch.equal(s2d[ph], xb[:, (ph // 2)::2, (ph % 2)::2, :])
    wp = ops.pack_conv(w, dtype=DT)
    Ho, Wo = H // 2, W // 2
    M = B * Ho * Wo
    out = torch.empty(M, Cc, device=cuda_device)
    ops.gemm([ops.make_seg(s2d, 4 * B, Ho, Wo, Cc, taps=ops.taps_stride2(B, pad1))], M, Cc, wp, bias=bias, out_f32=out, ldo32=Cc)
    xr = bf(x).float()
    if pad1:
        ref = F.conv2d(xr, bf(w).float(), bias, stride=2, padding=1)
    else:
        ref = F.conv2d(F.pad(xr, (0, 1, 0, 1)), bf(w).float(), bias, stride=2, padding=0)
    assert relerr(out, nhwc(ref).reshape(M, Cc)) < 2e-3


@pytest.mark.parametrize("B,H,W,Cc,bn", [(2, 16, 16, 128, 0), (1, 8, 128, 256, 128), (3, 8, 8, 320, 0)])
def test_gemm_space_to_depth_output(ops, cuda_device, B, H, W, Cc, bn):
    """The epilogue can write its 16-bit output directly in the space-to-depth layout the following stride-2 conv reads."""
    g = torch.Generator(device="cuda").manual_seed(H * W + Cc)
    M, K = B * H * W, 128
    a = bf(torch.randn(M, K, device=cuda_device, generator=g))
    w = bf(torch.randn(Cc, K, device=cuda_device, generator=g) / math.sqrt(K))
    out = torch.empty(M, Cc, device=cuda_device)
    s2d = torch.full((4, B, H // 2, W // 2, Cc), float("nan"), dtype=DT, device=cuda_device)
    ops.gemm([ops.make_seg(a, 1, 1, M, K)], M, Cc, w, out_f32=out, ldo32=Cc, out_bf16=s2d, ldo16=Cc, s2d_hw=(H, W), bn=bn)
    ref16 = bf(out).reshape(B, H, W, Cc)
    for ph in range(4):
        assert torch.equal(s2d[ph], ref16[:, (ph // 2)::2, (ph % 2)::2, :])


def test_conv_plus_shortcut_two_segments(ops, cuda_device):
    """out = conv3x3(h) + conv1x1(x) as one GEMM with K = 9*Cout + Cin (ResBlock conv2 + conv_shortcut)."""
    g = torch.Generator(device="cuda").manual_seed(21)
    B, H, W, Cin, Cout = 2, 16, 16, 192, 128
    h = bf(torch.randn(B, Cout, H, W, device=cuda_device, generator=g))
    x = bf(torch.randn(B, Cin, H, W, device=cuda_device, generator=g))
    w2 = torch.randn(Cout, Cout, 3, 3, device=cuda_device, generator=g) / math.sqrt(9 * Cout)
    ws = torch.randn(Cout, Cin, 1, 1, device=cuda_device, generator=g) / math.sqrt(Cin)
    K = 9 * Cout + Cin
    wp = torch.empty(Cout, K, dtype=DT, device=cuda_device)
    ops.pack_conv(w2, out=wp, ldo=K)
    ops.pack_conv(ws, out=wp[:, 9 * Cout:], ldo=K)
    M = B * H * W
    out = torch.empty(M, Cout, device=cuda_device)
    hn, xn = nhwc(h), nhwc(x)  # keep the NHWC copies alive: segments hold raw pointers
    ops.gemm([ops.make_seg(hn, B, H, W, Cout, taps=ops.taps_3x3()), ops.make_seg(xn, B, H, W, Cin)], M, Cout, wp,
             out_f32=out, ldo32=Cout)
    ref = F.conv2d(h.float(), bf(w2).float(), padding=1) + F.conv2d(x.float(), bf(ws).float())
    assert relerr(out, nhwc(ref).reshape(M, Cout)) < 2e-3


def test_upsample_conv(ops, cuda_device):
    g = torch.Generator(device="cuda").manual_seed(31)
    B, H, W, Cc = 2, 8, 8, 128
    x = torch.randn(B, Cc, H, W, device=cuda_device, generator=g)
    up = ops.upsample2x(nhwc(x), dtype=DT)
    assert torch.equal(up, bf(nhwc(F.interpolate(x, scale_factor=2.0, mode="nearest"))))


def test_image_im2col_first_conv(ops, cuda_device):
    g = torch.Generator(device="cuda").manual_seed(41)
    B, H, W = 2, 64, 128
    img = torch.rand(B, 3, H, W, device=cuda_device, generator=g)
    w = torch.randn(128, 3, 3, 3, device=cuda_device, generator=g) / math.sqrt(27)
    bias = torch.randn(128, device=cuda_device, generator=g)
    flag = torch.zeros(1, dtype=torch.int32, device=cuda_device)
    col = ops.image_im2col(img, flag, dtype=DT)
    wp = ops.pack_conv(w, Cpad=3, dtype=DT)  # K = 27 -> padded to 64 by the packer
    wp64 = torch.zeros(128, 64, dtype=DT, device=cuda_device)
    wp64[:, :27] = wp[:, :27]
    M = B * H * W
    out = torch.empty(M, 128, device=cuda_device)
    ops.gemm([ops.make_seg(col, 1, 1, M, 64)], M, 128, wp64, bias=bias, out_f32=out, ldo32=128)
    xn = bf((img - 0.5) / 0.5).float()
    ref = nhwc(F.conv2d(xn, bf(w).float(), bias, padding=1)).reshape(M, 128)
    assert relerr(out, ref) < 2e-3
    assert flag.item() == 0
    ops.image_im2col(img * 1.5, flag, dtype=DT)
    assert flag.item() == 1  # out-of-range input is reported (reference asserts, ldm_diffusers.py:147)


# ---------------------------------------------------------------------------------------------- norms
@pytest.mark.parametrize("B,HW,C0,C1,act", [(2, 4096, 320, 0, 1), (2, 256, 1280, 640, 1), (1, 64, 1280, 1280, 1), (3, 1024, 128, 0, 3),
                                            (1, 16384, 512, 0, 0), (2, 1024, 640, 320, 1)])
def test_groupnorm(ops, cuda_device, B, HW, C0, C1, act):
    g = torch.Generator(device="cuda").manual_seed(C0 + C1)
    x0 = torch.randn(B, HW, C0, device=cuda_device, generator=g) * 2 + 0.5
    x1 = torch.randn(B, HW, C1, device=cuda_device, generator=g) - 0.3 if C1 else None
    Cc = C0 + C1
    gamma = torch.randn(Cc, device=cuda_device, generator=g)
    beta = torch.randn(Cc, device=cuda_device, generator=g)
    y = torch.empty(B, HW, Cc, dtype=DT, device=cuda_device)
    raw = torch.empty_like(y)
    ops.groupnorm(x0, x1, B, HW, gamma, beta, 1e-5, act, y, raw)
    x = torch.cat([x0, x1], -1) if C1 else x0
    ref = F.group_norm(x.permute(0, 2, 1), 32, gamma, beta, 1e-5).permute(0, 2, 1)
    ref = {0: ref, 1: F.silu(ref), 3: F.relu(ref)}[act]
    assert relerr(y, ref) < 1e-2
    assert torch.equal(raw, bf(x))


@pytest.mark.parametrize("B,HW,Cc", [(2, 4096, 320), (1, 16384, 128), (3, 64, 1280)])
def test_groupnorm_16bit_input(ops, cuda_device, B, HW, Cc):
    """GroupNorm over a 16-bit intermediate (conv1 output feeding norm2)."""
    g = torch.Generator(device="cuda").manual_seed(Cc + HW)
    x = bf(torch.randn(B, HW, Cc, device=cuda_device, generator=g) * 1.5 + 0.25)
    gamma = torch.randn(Cc, device=cuda_device, generator=g)
    beta = torch.randn(Cc, device=cuda_device, generator=g)
    y = torch.empty(B, HW, Cc, dtype=DT, device=cuda_device)
    ops.groupnorm(x, None, B, HW, gamma, beta, 1e-6, 1, y)
    ref = F.silu(F.group_norm(x.float().permute(0, 2, 1), 32, gamma, beta, 1e-6).permute(0, 2, 1))
    assert relerr(y, ref) < 1e-2


@pytest.mark.parametrize("B,H,W,Cin,Cout,bn", [(2, 32, 32, 128, 320, 0), (3, 8, 8, 128, 1280, 0), (1, 64, 64, 64, 128, 0), (2, 16, 16, 128, 640, 128),
                                                (2, 16, 16, 64, 512, 256)])
def test_gemm_fused_groupnorm_statistics(ops, cuda_device, B, H, W, Cin, Cout, bn):
    """The GEMM epilogue emits per-column (sum, sumsq) of its outputs; GroupNorm of the consumer uses them instead of a
    statistics pass.  Checked against F.group_norm on the GEMM's own fp32 output, and for bit-exact repeatability."""
    g = torch.Generator(device="cuda").manual_seed(Cout + H)
    x = bf(torch.randn(B, Cin, H, W, device=cuda_device, generator=g))
    w = torch.randn(Cout, Cin, 3, 3, device=cuda_device, generator=g) / math.sqrt(9 * Cin)
    bias = torch.randn(Cout, device=cuda_device, generator=g)
    res = torch.randn(B * H * W, Cout, device=cuda_device, generator=g)
    wp = ops.pack_conv(w, dtype=DT)
    a = nhwc(x)
    M, HW = B * H * W, H * W
    sr = 32
    out = torch.empty(M, Cout, device=cuda_device)
    cs = torch.full((M // sr, Cout, 2), float("nan"), device=cuda_device)
    ops.gemm([ops.make_seg(a, B, H, W, Cin, taps=ops.taps_3x3())], M, Cout, wp, bias=bias, residual=res, ldr=Cout, out_f32=out, ldo32=Cout,
             colstats=cs, stat_rows=sr, bn=bn)
    blocks = out.reshape(M // sr, sr, Cout)
    assert relerr(cs[..., 0], blocks.sum(1)) < 1e-4
    assert relerr(cs[..., 1], (blocks * blocks).sum(1)) < 1e-4
    gamma = torch.randn(Cout, device=cuda_device, generator=g)
    beta = torch.randn(Cout, device=cuda_device, generator=g)
    y = torch.empty(B, HW, Cout, dtype=DT, device=cuda_device)
    ops.groupnorm_from_colstats(out.reshape(B, HW, Cout), B, HW, cs, sr, gamma, beta, 1e-5, 1, y)
    ref = F.silu(F.group_norm(out.reshape(B, HW, Cout).permute(0, 2, 1), 32, gamma, beta, 1e-5).permute(0, 2, 1))
    assert relerr(y, ref) < 1e-2
    cs2 = torch.empty_like(cs)
    ops.gemm([ops.make_seg(a, B, H, W, Cin, taps=ops.taps_3x3())], M, Cout, wp, bias=bias, residual=res, ldr=Cout, out_f32=out, ldo32=Cout,
             colstats=cs2, stat_rows=sr, bn=bn)
    assert torch.equal(cs, cs2)


@pytest.mark.parametrize("M,Cc", [(4096, 320), (1000, 640), (77, 1280)])
def test_layernorm(ops, cuda_device, M, Cc):
    g = torch.Generator(device="cuda").manual_seed(Cc)
    x = torch.randn(M, Cc, device=cuda_device, generator=g) * 3 + 1
    gamma = torch.randn(Cc, device=cuda_device, generator=g)
    beta = torch.randn(Cc, device=cuda_device, generator=g)
    y = torch.empty(M, Cc, dtype=DT, device=cuda_device)
    ops.layernorm(x, gamma, beta, 1e-5, y)
    assert relerr(y, F.layer_norm(x, (Cc,), gamma, beta, 1e-5)) < 1e-2
    x16 = x.to(DT)  # 16-bit input stream (the transformer blocks' hidden states with fp16 operands)
    y16 = torch.empty(M, Cc, dtype=DT, device=cuda_device)
    ops.layernorm(x16, gamma, beta, 1e-5, y16)
    assert relerr(y16, F.layer_norm(x16.float(), (Cc,), gamma, beta, 1e-5)) < 1e-2


@pytest.mark.parametrize("B,H,W,Cin,Cout,taps,bn,mt", [
    (1, 1, 640, 320, 320, 1, 160, 0),     # 5 row tiles: the last pair has an empty second CTA
    (1, 1, 1000, 256, 416, 1, 0, 0),      # ragged M and an N that is not a multiple of the tile (W rows past N are TMA zero fill)
    (2, 64, 64, 320, 320, 9, 0, 0),       # 3x3 conv, 160-wide pair tiles
    (2, 128, 128, 128, 128, 9, 128, 2),   # 512-row pair tiles (two M sub-tiles per CTA)
    (3, 32, 32, 640, 1280, 1, 0, 0),
])
def test_gemm_cta_pairs_match_single_cta(ops, cuda_device, B, H, W, Cin, Cout, taps, bn, mt):
    """tcgen05 cta_group::2 pairs (256-row MMAs, each CTA staging half of the W tile) must reproduce the single-CTA kernel bit for
    bit: same MMA k-order, same epilogue; also against a torch reference."""
    g = torch.Generator(device="cuda").manual_seed(B * H + Cout)
    M = B * H * W
    x = bf(torch.randn(B, H, W, Cin, device=cuda_device, generator=g) * 0.5)
    w = bf(torch.randn(Cout, taps * Cin, device=cuda_device, generator=g) / math.sqrt(taps * Cin))
    bias = torch.randn(Cout, device=cuda_device, generator=g)
    res = torch.randn(M, Cout, device=cuda_device, generator=g)
    seg = ops.make_seg(x, B, H, W, Cin, taps=ops.taps_3x3()) if taps == 9 else ops.make_seg(x.reshape(M, Cin), 1, 1, M, Cin)
    outs = {}
    for pair in (-1, 1):
        o32 = torch.empty(M, Cout, device=cuda_device)
        o16 = torch.empty(M, Cout, device=cuda_device, dtype=DT) if Cout % 8 == 0 else None
        kw = dict(out_bf16=o16, ldo16=Cout) if o16 is not None else {}
        ops.gemm([seg], M, Cout, w, bias=bias, residual=res, ldr=Cout, out_f32=o32, ldo32=Cout, bn=bn, mt=mt, pair=pair, **kw)
        outs[pair] = (o32, o16)
    assert torch.equal(outs[-1][0], outs[1][0])
    if outs[1][1] is not None:
        assert torch.equal(outs[-1][1], outs[1][1])
    if taps == 1:
        ref = x.reshape(M, Cin).float() @ w.float().t() + bias + res
    else:
        wc = w.float().reshape(Cout, 3, 3, Cin).permute(0, 3, 1, 2)
        ref = F.conv2d(x.float().permute(0, 3, 1, 2), wc, padding=1).permute(0, 2, 3, 1).reshape(M, Cout) + bias + res
    assert relerr(outs[1][0], ref) < 2e-3


@pytest.mark.parametrize("M,N,K,pair", [(4096, 320, 320, 0), (1000, 640, 2560, -1), (8192, 320, 1280, 1)])
def test_gemm_16bit_residual_in_place(ops, cuda_device, M, N, K, pair):
    """hs += A W^T + bias on a 16-bit stream, in place (residual and output are the same 16-bit tensor): the update the
    transformer blocks' attention out-projections perform with fp16 operands."""
    g = torch.Generator(device="cuda").manual_seed(M + N)
    a = bf(torch.randn(M, K, device=cuda_device, generator=g))
    w = bf(torch.randn(N, K, device=cuda_device, generator=g) / math.sqrt(K))
    bias = torch.randn(N, device=cuda_device, generator=g)
    hs = bf(torch.randn(M, N, device=cuda_device, generator=g))
    ref = hs.float() + a.float() @ w.float().t() + bias
    ops.gemm([ops.make_seg(a, 1, 1, M, K)], M, N, w, bias=bias, residual=hs, ldr=N, out_bf16=hs, ldo16=N, pair=pair)
    assert relerr(hs, ref) < 1e-2


def test_softmax_rows(ops, cuda_device):
    g = torch.Generator(device="cuda").manual_seed(3)
    s = torch.randn(300, 4096, device=cuda_device, generator=g) * 4
    p = torch.empty(300, 4096, dtype=DT, device=cuda_device)
    ops.softmax_rows(s, p)
    assert relerr(p, torch.softmax(s, -1)) < 1e-2


def test_gn_add_relu_nchw(ops, cuda_device):
    g = torch.Generator(device="cuda").manual_seed(13)
    B, HW, Cc = 2, 1024, 512
    a = torch.randn(B, HW, Cc, device=cuda_device, generator=g)
    s = torch.randn(B, HW, Cc, device=cuda_device, generator=g) * 2
    ga, ba, gs, bs = (torch.randn(Cc, device=cuda_device, generator=g) for _ in range(4))
    out = ops.gn_add_relu_nchw(a, ga, ba, s, gs, bs, 1e-5, B, HW, Cc)
    gn = lambda t, w, b: F.group_norm(t.permute(0, 2, 1), 32, w, b, 1e-5)  # noqa: E731
    ref = F.relu(gn(a, ga, ba) + gn(s, gs, bs))
    assert relerr(out, ref) < 1e-4
    out2 = ops.gn_add_relu_nchw(a, ga, ba, s, None, None, 1e-5, B, HW, Cc)
    assert relerr(out2, F.relu(gn(a, ga, ba) + s.permute(0, 2, 1))) < 1e-4


# ---------------------------------------------------------------------------------------------- attention
@pytest.mark.parametrize("impl", [0])  # the tcgen05/TMEM kernel (the round-1 mma.sync kernel is gone from the library)
@pytest.mark.parametrize("B,heads,d,Nq,Nk", [(2, 8, 40, 4096, 4096), (1, 8, 80, 1024, 1024), (2, 8, 160, 256, 256), (1, 8, 160, 64, 64),
                                             (2, 8, 40, 4096, 77), (2, 8, 160, 64, 77), (1, 8, 80, 1024, 77)])
def test_attention(ops, cuda_device, B, heads, d, Nq, Nk, impl):
    g = torch.Generator(device="cuda").manual_seed(d + Nk)
    Cc = heads * d
    self_attn = Nq == Nk
    if self_attn:  # fused qkv buffer [B, N, 3C]
        qkv = bf(torch.randn(B, Nq, 3 * Cc, device=cuda_device, generator=g))
        q, k, v = qkv[..., :Cc], qkv[..., Cc:2 * Cc], qkv[..., 2 * Cc:]
        ldq = ldk = 3 * Cc
        q_bs, kv_bs = Nq * 3 * Cc, Nk * 3 * Cc
    else:  # q [B,N,C]; k,v inside a wide per-layer-stacked buffer [B,77,ldkv]
        ldkv = 2 * Cc + 256
        qb = bf(torch.randn(B, Nq, Cc, device=cuda_device, generator=g))
        kvb = bf(torch.randn(B, Nk, ldkv, device=cuda_device, generator=g))
        q, k, v = qb, kvb[..., 128:128 + Cc], kvb[..., 128 + Cc:128 + 2 * Cc]
        ldq, ldk = Cc, ldkv
        q_bs, kv_bs = Nq * Cc, Nk * ldkv
    o = torch.empty(B, Nq, Cc, dtype=DT, device=cuda_device)
    ops.attention(q, ldq, k, ldk, v, ldk, o, Cc, B, heads, d, Nq, Nk, q_bs, kv_bs, Nq * Cc, 1.0 / math.sqrt(d), impl=impl)
    split = lambda t: t.float().reshape(B, -1, heads, d).transpose(1, 2)  # noqa: E731
    ref = F.scaled_dot_product_attention(split(q), split(k), split(v)).transpose(1, 2).reshape(B, Nq, Cc)
    assert relerr(o, ref) < 2e-2
    # the warp-specialised pipeline (independent MMA issuers per query tile, shared K/V ring) must be race-free: bit-identical reruns
    for _ in range(3):
        o2 = torch.empty_like(o)
        ops.attention(q, ldq, k, ldk, v, ldk, o2, Cc, B, heads, d, Nq, Nk, q_bs, kv_bs, Nq * Cc, 1.0 / math.sqrt(d), impl=impl)
        assert torch.equal(o, o2)


# ---------------------------------------------------------------------------------------------- packing (LoRA fold)
def test_pack_linear_lora_fold(ops, cuda_device):
    g = torch.Generator(device="cuda").manual_seed(17)
    N, K, r = 320, 768, 16
    w = torch.randn(N, K, device=cuda_device, generator=g)
    A = torch.randn(r, K, device=cuda_device, generator=g) / r
    Bm = torch.randn(N, r, device=cuda_device, generator=g) * 0.02
    out = ops.pack_linear(w, A, Bm, scale=2.0, dtype=DT)
    ref = bf(w + 2.0 * (Bm @ A))
    # fp32 sum order may differ by an ulp before the bf16 rounding: allow 1 bf16 ulp on <0.1% of entries
    diff = (out.float() - ref.float()).abs()
    assert (diff > 0).float().mean().item() < 1e-3
    assert relerr(out, ref) < 1e-2
    assert torch.equal(ops.pack_linear(w, dtype=DT), bf(w))


# ---------------------------------------------------------------------------------------------- sliding-window merge
@pytest.mark.parametrize("H,W", [(512, 1024), (1024, 1024), (768, 1280)])
def test_slide_merge_matches_sequential_accumulate(ops, cuda_device, H, W):
    """feature_extractor.py:254-275: out[window] += crop; cnt[window] += 1; out /= cnt -- reproduced bit for bit by the gather kernel
    (same addition order per pixel)."""
    g = torch.Generator(device="cuda").manual_seed(H + W)
    s, n, Cc, crop, stride = 8, 2, 24, 512, 256
    wins = [(y, x) for y in range(0, H - crop + 1, stride) for x in range(0, W - crop + 1, stride)]
    hf = crop // s
    feats = torch.randn(len(wins) * n, Cc, hf, hf, device=cuda_device, generator=g)
    out = ops.slide_merge(feats, len(wins), [(y // s, x // s) for y, x in wins], H // s, W // s)
    ref = torch.zeros(n, Cc, H // s, W // s, device=cuda_device)
    cnt = torch.zeros(1, 1, H // s, W // s, device=cuda_device)
    for wi, (y, x) in enumerate(wins):
        ref[:, :, y // s:y // s + hf, x // s:x // s + hf] += feats[wi * n:(wi + 1) * n]
        cnt[..., y // s:y // s + hf, x // s:x // s + hf] += 1
    ref /= cnt
    assert torch.equal(out, ref)


@pytest.mark.parametrize("B,H,W,Cin,Cout,k", [(2, 32, 32, 128, 192, 3), (1, 64, 64, 320, 320, 3), (2, 16, 16, 640, 1280, 1), (1, 8, 128, 64, 128, 3), (3, 8, 8, 128, 320, 3)])
def test_conv_dgrad_is_the_same_implicit_gemm(ops, cuda_device, B, H, W, Cin, Cout, k):
    """First building block of SURVEY §8 row f-3: dX of a stride-1 conv = the forward implicit-GEMM kernel on dY with the weight's in / out
    roles swapped and the taps mirrored (madm_op_pack_conv_dgrad), against torch.autograd."""
    g = torch.Generator(device="cuda").manual_seed(Cin + H)
    x = torch.randn(B, Cin, H, W, device=cuda_device, generator=g, requires_grad=True)
    w = torch.randn(Cout, Cin, k, k, device=cuda_device, generator=g) / math.sqrt(k * k * Cin)
    dy = bf(torch.randn(B, Cout, H, W, device=cuda_device, generator=g))
    y = F.conv2d(x, bf(w).float(), padding=k // 2)
    (ref,) = torch.autograd.grad(y, x, dy.float())
    wp = ops.pack_conv_dgrad(w, dtype=DT)
    a = nhwc(dy)
    M = B * H * W
    out = torch.empty(M, Cin, device=cuda_device)
    seg = ops.make_seg(a, B, H, W, Cout, taps=ops.taps_3x3() if k == 3 else None)
    ops.gemm([seg], M, Cin, wp, out_f32=out, ldo32=Cin)
    assert relerr(out, nhwc(ref).reshape(M, Cin)) < 2e-3


def test_linear_dgrad_with_folded_lora(ops, cuda_device):
    """dX = dY (W + s B A): the transposed, LoRA-folded weight as the GEMM's B operand (madm_op_pack_linear_dgrad), against torch.autograd."""
    g = torch.Generator(device="cuda").manual_seed(9)
    M, K, N, r, sc = 4096, 320, 960, 16, 2.0
    x = torch.randn(M, K, device=cuda_device, generator=g, requires_grad=True)
    w = torch.randn(N, K, device=cuda_device, generator=g) / math.sqrt(K)
    la = torch.randn(r, K, device=cuda_device, generator=g) / math.sqrt(r)
    lb = torch.randn(N, r, device=cuda_device, generator=g) * 0.02
    dy = bf(torch.randn(M, N, device=cuda_device, generator=g))
    wp = ops.pack_linear_dgrad(w, la, lb, sc, dtype=DT)
    assert torch.equal(wp, ops.pack_linear(w, la, lb, sc, dtype=DT).t().contiguous())  # exactly the transpose of the forward operand
    (ref,) = torch.autograd.grad(F.linear(x, wp.float().t()), x, dy.float())
    out = torch.empty(M, K, device=cuda_device)
    ops.gemm([ops.make_seg(dy, 1, 1, M, N)], M, K, wp, out_f32=out, ldo32=K)
    assert relerr(out, ref) < 2e-3
