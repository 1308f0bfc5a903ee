"""Training path of the vae_decoder_loss / 's0' variant on the GPU (the configuration all shipped experiment files select,
config_files/SemSeg/MTMADISE/mtmadise_cityscapes_rgb_to_depth_11.py:47-55).

The VAE decoder runs under no_grad and its image is detached before it becomes the first feature (ldm_diffusers.py:191-201), so 's0'
back-propagates into feature_projections.0 only; 'before_vae.decoder' (return_unet_final_output=True, the UNet's final output that the
meta-arch's vae_decoder_loss differentiates) carries grad into the UNet through the frozen conv_out / conv_norm_out; 'after_vae.decoder'
carries none.  Product (autograd.Function around madm_extract(MADM_FLAG_TRAIN) / madm_backward) against torch.autograd through the fp32
oracle oracle.synthetic.build_backbone(variant='s0') (training_gradients_s0 below) with the gates S0_GATES below, plus the op-level check of
the K = 3 projection backward (madm_op_c3_gn_bwd) against torch.autograd.
"""
import ctypes as C

import pytest
import torch

from helpers import build_product_backbone, set_lora_adapter
from test_train_gpu import compare, make_trainable

pytestmark = pytest.mark.gpu

# (per-tensor, per-family / overall) cosine gates.  Below test_train_gpu.GATES because projection 0 differentiates the DECODED image: it carries the
# VAE decoder's operand rounding (decoder output 5.4e-3 max-rel at fp16, test_s0_gpu) into 512^2 maps whose ReLU masks then flip more often than the
# UNet taps'.  Measured on a B200 (2 images / 1 + 1 in flight): projection families at cosine 0.9964 - 0.9974 with fp16 (LoRA / conditioning
# 0.998), 0.972 - 0.979 with bf16 (LoRA 0.985 - 0.988; worst tensor 0.931); the UNet-output path alone (decoder-only loss) at 0.99999 / 0.9994.
# The K = 3 backward itself is checked exactly by test_c3_gn_bwd_matches_autograd.
S0_GATES = {"fp16": (0.99, 0.995), "bf16": (0.90, 0.965)}


def s0_functional(out, final, seed=99, feature_scale=1e-3, final_scale=1e-3):
    """The fixed linear functional of these tests: feature_scale * sum_k <feat_k, R_k> + final_scale * <before_vae.decoder, R> with seeded
    Gaussian R drawn on the CPU, the feature maps first (dict order), then the UNet's final output.  A scale of 0 drops the term."""
    g = torch.Generator().manual_seed(seed)
    loss = 0.0
    for v in out.values():
        r = torch.randn(v.shape, generator=g).to(v.device)
        if feature_scale:
            loss = loss + feature_scale * (v * r).sum()
    v = final["before_vae.decoder"]
    r = torch.randn(v.shape, generator=g).to(v.device)
    if final_scale:
        loss = loss + final_scale * (v * r).sum()
    return loss


def training_gradients_s0(bb, img, adapter="Depth", input_modal="others", seed=99, feature_scale=1e-3, final_scale=1e-3):
    """Reference gradients of the s0 variant, as oracle.synthetic.training_gradients computes them for the base one: the trainable set (active
    adapter's LoRA factors, feature projections, prompt / time parameters) of the fp32 oracle receives the gradient of s0_functional over
    {s0, s3, s4, s5} and 'before_vae.decoder' (return_unet_final_output=True).  The oracle's VAE decoder runs under no_grad and its image is
    detached (oracle/backbone.py), so s0 reaches feature_projections.0 only.  Returns (loss, {name: grad}), None where no gradient arrives."""
    from oracle.lora import set_adapter
    set_adapter(bb.feature_extractor.ldm_extractor.unet, [adapter])
    train = [(n, p) for n, p in bb.named_parameters()
             if ("lora_" in n and f".{adapter}." in n) or n.startswith("feature_projections.") or "clip_project_others" in n]
    for p in bb.parameters():
        p.requires_grad_(False)
        p.grad = None
    for _, p in train:
        p.requires_grad_(True)
    feats, final = bb(img, input_modal=input_modal, return_unet_final_output=True)
    loss = s0_functional(feats["output_features"], final, seed, feature_scale, final_scale)
    loss.backward()
    grads = {n: (None if p.grad is None else p.grad.detach().clone()) for n, p in train}
    for _, p in train:
        p.requires_grad_(False)
        p.grad = None
    return float(loss.detach()), grads


@pytest.fixture(scope="module", params=["bf16", "fp16"])
def pair(request, cuda_device):
    from oracle import synthetic
    ob = synthetic.build_backbone(variant="s0").to(cuda_device)
    pb = build_product_backbone(cuda_device, compute_dtype=request.param, variant="s0")
    missing, unexpected = pb.load_state_dict(ob.state_dict(), strict=False)
    assert not missing and not unexpected, (missing[:5], unexpected[:5])
    make_trainable(pb)
    yield ob, pb, request.param
    del pb, ob
    torch.cuda.empty_cache()


def _clear(params):
    for p in params.values():
        p.grad = None


def _loss_tol(mode, ref):  # the s0 map's 67 M values carry the decoder's rounding: 1.5e-2 measured with fp16 at 2 images
    return (8e-2 if mode == "bf16" else 3e-2) * max(1.0, abs(ref))


def test_s0_backward_matches_oracle_autograd(pair, cuda_device):
    """loss = functional(s0, s3, s4, s5) + functional(before_vae.decoder) at 2 images: every trainable gradient against oracle autograd;
    the same step again gives bit-identical gradients."""
    from oracle import synthetic
    ob, pb, mode = pair
    img = synthetic.synthetic_images(2, seed=7).to(cuda_device)
    loss_ref, grads_ref = training_gradients_s0(ob, img, adapter="Depth", input_modal="others")
    params = dict(pb.named_parameters())
    _clear(params)
    set_lora_adapter(pb.feature_extractor.ldm_extractor.unet, "Depth")
    feats, final = pb(img, input_modal="others", return_unet_final_output=True)
    out = feats["output_features"]
    assert list(out) == ["s0", "s3", "s4", "s5"] and all(v.requires_grad for v in out.values())
    assert final["before_vae.decoder"].requires_grad and not final["after_vae.decoder"].requires_grad
    loss = s0_functional(out, final)
    assert abs(float(loss.detach()) - loss_ref) <= _loss_tol(mode, loss_ref)
    loss.backward()
    compare(grads_ref, params, f"s0/others/Depth/{mode}", mode, S0_GATES[mode])
    assert all(p.grad is None for n, p in params.items() if ".default." in n)
    assert all(p.grad is None for n, p in params.items() if not p.requires_grad)
    first = {n: p.grad.clone() for n, p in params.items() if p.grad is not None}
    _clear(params)
    feats, final = pb(img, input_modal="others", return_unet_final_output=True)
    s0_functional(feats["output_features"], final).backward()
    for n, g in first.items():
        assert torch.equal(g, params[n].grad), n
    _clear(params)


def test_s0_detach_semantics(pair, cuda_device):
    """A loss on s0 alone reaches feature_projections.0 only; a loss on before_vae.decoder alone reaches the LoRA factors and the
    conditioning (against the oracle) and no projection."""
    from oracle import synthetic
    ob, pb, mode = pair
    img = synthetic.synthetic_images(1, seed=3).to(cuda_device)
    params = dict(pb.named_parameters())
    set_lora_adapter(pb.feature_extractor.ldm_extractor.unet, "Depth")
    # s0 alone
    _clear(params)
    feats, final = pb(img, input_modal="others", return_unet_final_output=True)
    g = torch.Generator().manual_seed(5)
    s0 = feats["output_features"]["s0"]
    (s0 * torch.randn(s0.shape, generator=g).to(cuda_device)).sum().backward()
    for n, p in params.items():
        if n.startswith("feature_projections.0."):
            assert p.grad is not None and float(p.grad.abs().max()) > 0.0, n
        else:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, n
    # before_vae.decoder alone
    _, grads_ref = training_gradients_s0(ob, img, adapter="Depth", input_modal="others", feature_scale=0.0)
    assert all(grads_ref[n] is None for n in grads_ref if n.startswith("feature_projections."))
    _clear(params)
    feats, final = pb(img, input_modal="others", return_unet_final_output=True)
    s0_functional(feats["output_features"], final, feature_scale=0.0).backward()
    assert any(p.grad is not None and float(p.grad.abs().max()) > 0.0 for n, p in params.items() if ".lora_A.Depth." in n)
    compare(grads_ref, params, f"s0/before_vae.decoder only/{mode}", mode, S0_GATES[mode])
    _clear(params)


def test_s0_two_passes_in_flight_source_and_mixed(pair, cuda_device):
    """The source pass ('rgb', adapter 'default', with the vae_decoder_loss term) and the mixed pass ('mixed', adapter 'Depth') in flight
    before ONE backward, as MTMADISE.forward runs them."""
    from oracle import synthetic
    from oracle.lora import set_adapter
    ob, pb, mode = pair
    src = synthetic.synthetic_images(1, seed=11).to(cuda_device)
    mix = synthetic.synthetic_images(1, seed=12).to(cuda_device)
    ounet = ob.feature_extractor.ldm_extractor.unet
    train = [(n, p) for n, p in ob.named_parameters() if "lora_" in n or n.startswith("feature_projections.") or
             n.startswith("feature_extractor.clip_project_")]
    for p in ob.parameters():
        p.requires_grad_(False); p.grad = None
    for _, p in train:
        p.requires_grad_(True)
    set_adapter(ounet, ["default"])
    f1, fin1 = ob(src, input_modal="rgb", return_unet_final_output=True)
    l1 = s0_functional(f1["output_features"], fin1, seed=5)
    set_adapter(ounet, ["Depth"])
    f2, fin2 = ob(mix, input_modal="mixed", return_unet_final_output=True)
    l2 = s0_functional(f2["output_features"], fin2, seed=6, final_scale=0.0)
    (l1 + l2).backward()
    grads_ref = {n: (None if p.grad is None else p.grad.detach().clone()) for n, p in train}
    for _, p in train:
        p.requires_grad_(False); p.grad = None
    params = dict(pb.named_parameters())
    _clear(params)
    punet = pb.feature_extractor.ldm_extractor.unet
    set_lora_adapter(punet, "default")
    p1f, p1fin = pb(src, input_modal="rgb", return_unet_final_output=True)
    p1 = s0_functional(p1f["output_features"], p1fin, seed=5)
    set_lora_adapter(punet, "Depth")
    p2f, p2fin = pb(mix, input_modal="mixed", return_unet_final_output=True)  # (no loss term on its final output: d_unet_sample = NULL)
    p2 = s0_functional(p2f["output_features"], p2fin, seed=6, final_scale=0.0)
    (p1 + p2).backward()
    ref = float((l1 + l2).detach())
    assert abs(float((p1 + p2).detach()) - ref) <= _loss_tol(mode, ref)
    compare(grads_ref, params, f"s0/rgb/default + mixed/Depth/{mode}", mode, S0_GATES[mode])
    _clear(params)


def test_s0_backward_launch_counts(cuda_device):
    """A training plan of the s0 variant has a backward pass at every supported batch size (B = 1, 2, 8)."""
    from oracle import synthetic
    pb = build_product_backbone(cuda_device, compute_dtype="fp16", variant="s0")
    make_trainable(pb)
    set_lora_adapter(pb.feature_extractor.ldm_extractor.unet, "Depth")
    eng = pb.feature_extractor.ldm_extractor.engine()
    counts = {}
    for B in (1, 2, 8):
        out = pb(synthetic.synthetic_images(B, seed=B).to(cuda_device), input_modal="others")["output_features"]
        out["s3"].sum().backward()
        counts[B] = int(eng.lib.madm_backward_launch_count(eng.ctx, B))
        del out
    print(f"[s0] backward launches per pass: {counts}")
    assert all(n > 0 for n in counts.values()), counts
    del pb
    torch.cuda.empty_cache()


@pytest.mark.parametrize("relu", [1, 0], ids=["conv1_relu", "shortcut"])
@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
def test_c3_gn_bwd_matches_autograd(cuda_device, relu, dtype):
    """madm_op_c3_gn_bwd (the s0 projection's K = 3 branches, conv1x1(3 -> 128) -> GroupNorm(32) [-> ReLU], backward from the image without
    the conv output) against torch.autograd in float64 on random 512^2 images: d weight, d gamma, d beta within 1e-4 relative.  The incoming
    gradient is zeroed where |z| < 1e-3, so the ReLU mask does not depend on the evaluation precision of z."""
    from madm_b200 import _lib
    lib = _lib.load()
    B, Ch, H = 2, 128, 512
    HW = H * H
    g = torch.Generator(device=cuda_device).manual_seed(17 + relu)
    x = torch.rand(B, 3, H, H, device=cuda_device, generator=g) * 2 - 1
    w = torch.randn(Ch, 3, 1, 1, device=cuda_device, generator=g) * 0.5
    gamma = 1.0 + 0.1 * torch.randn(Ch, device=cuda_device, generator=g)
    beta = 0.1 * torch.randn(Ch, device=cuda_device, generator=g)
    tdt = torch.float16 if dtype == "fp16" else torch.bfloat16
    dy = torch.randn(B, Ch, H, H, device=cuda_device, generator=g).to(tdt)
    xd, wd, gd, bd = (t.double().requires_grad_(t is not x) for t in (x, w, gamma, beta))
    z = torch.nn.functional.group_norm(torch.nn.functional.conv2d(xd, wd), 32, gd, bd, eps=1e-5)
    dyd = dy.double().masked_fill(z.detach().abs() < 1e-3, 0.0)
    dy = dyd.to(tdt)  # (exact: zeros and the 16-bit values themselves)
    (torch.relu(z) if relu else z).backward(dyd)
    img4 = torch.zeros(B, HW, 4, device=cuda_device)
    img4[..., :3] = x.permute(0, 2, 3, 1).reshape(B, HW, 3)
    dy16 = dy.permute(0, 2, 3, 1).contiguous()
    dw, dg, db = torch.empty(Ch, 3, device=cuda_device), torch.empty(Ch, device=cuda_device), torch.empty(Ch, device=cuda_device)
    scratch = torch.empty(int(lib.madm_op_c3_gn_bwd_scratch_floats(B, Ch)), device=cuda_device)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.madm_op_c3_gn_bwd(img4.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(), 1e-5, relu, B, HW, Ch, dy16.data_ptr(), 1.0,
                                     dw.data_ptr(), dg.data_ptr(), db.data_ptr(), scratch.data_ptr(),
                                     _lib.DTYPE_FP16 if dtype == "fp16" else _lib.DTYPE_BF16, st), None, "madm_op_c3_gn_bwd")
    torch.cuda.synchronize()
    for name, got, ref in (("weight", dw, wd.grad.reshape(Ch, 3)), ("norm.weight", dg, gd.grad), ("norm.bias", db, bd.grad)):
        err = ((got.double() - ref).abs().max() / ref.abs().max()).item()
        print(f"[c3_gn_bwd relu={relu} {dtype}] d {name}: max rel err {err:.2e}")
        assert err <= 1e-4, (name, err)
