"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol, the parameter holders expose the
reference's state_dict keys, LoRA adapter bookkeeping, loud failure without a GPU, and the batch-sharding helper under a
world_size-2 gloo group."""
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_all_declared_symbols():
    from madm_b200 import _lib
    lib = _lib.load()
    assert lib.madm_version() >= 100
    hdr = open(os.path.join(ROOT, "include", "madm_b200.h")).read()
    declared = set(re.findall(r"\b(madm_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"madm_ctx", "madm_stream"}
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(lib, name), f"libmadm_b200.so does not export {name}"
        assert name in _lib.SYMBOLS, f"{name} has no ctypes prototype"


def test_struct_layouts_match_header_sizes():
    """ctypes mirrors of the POD structs must have the C sizes (compiled check through a tiny C program is overkill:
    the fields are all 4/8-byte scalars and pointers, so sizes are deterministic)."""
    import ctypes as C
    from madm_b200 import _lib
    assert C.sizeof(_lib.MadmTensor) == 8 + 8 + 8 + 32  # name, data, ndim(+pad), shape[4]
    assert C.sizeof(_lib.MadmGemmSeg) == 8 + 6 * 4 + 9 + 9 + 2 + 9 * 4  # a, 6 ints, dx, dy, pad, b_off
    assert C.sizeof(_lib.MadmProfile) == 5 * (32 + 8 + 4 * 8)


def test_ctypes_structs_match_the_compiled_header(tmp_path):
    """sizeof / offsetof of the POD structs as gcc lays them out from include/madm_b200.h == the ctypes mirrors in madm_b200/_lib.py."""
    import ctypes as C
    import subprocess
    from madm_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('''#include <stdio.h>
#include <stddef.h>
#include "madm_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(madm_tensor), sizeof(madm_extract_args), sizeof(madm_gemm_seg), sizeof(madm_gemm_args),
         sizeof(madm_profile), offsetof(madm_extract_args, out), offsetof(madm_extract_args, packed), offsetof(madm_extract_args, logits),
         offsetof(madm_extract_args, decoded_raw));
  return 0;
}
''')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    A = _lib.MadmExtractArgs
    want = [C.sizeof(_lib.MadmTensor), C.sizeof(A), C.sizeof(_lib.MadmGemmSeg), C.sizeof(_lib.MadmGemmArgs), C.sizeof(_lib.MadmProfile),
            A.out.offset, A.packed.offset, A.logits.offset, A.decoded_raw.offset]
    assert got == want, (got, want)


def test_create_without_gpu_fails_loudly():
    """No CPU fallback: without a CUDA device madm_create must fail with a message, and the Engine must raise."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import ctypes as C
    from madm_b200 import _lib
    from madm_b200.engine import Engine
    lib = _lib.load()
    h = C.c_void_p()
    rc = lib.madm_create(C.byref(h), 0)
    assert rc != 0 and b"no CUDA device" in lib.madm_last_error(None)
    with pytest.raises(_lib.MadmError):
        Engine(torch.device("cpu"))


def test_state_dict_keys_match_oracle_and_reference_names():
    """Product holders expose exactly the oracle's (= diffusers / peft / detectron2) state_dict keys."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import build_product_backbone
    pb = build_product_backbone(torch.device("cpu"))
    keys = set(pb.state_dict().keys())
    pre = "feature_extractor.ldm_extractor."
    for k in [pre + "unet.conv_in.weight", pre + "unet.time_embedding.linear_1.weight",
              pre + "unet.down_blocks.0.attentions.0.transformer_blocks.0.attn1.to_q.base_layer.weight",
              pre + "unet.down_blocks.0.attentions.0.transformer_blocks.0.attn1.to_q.lora_A.Depth.weight",
              pre + "unet.up_blocks.3.attentions.2.transformer_blocks.0.attn2.to_out.0.lora_B.default.weight",
              pre + "unet.up_blocks.3.attentions.2.transformer_blocks.0.ff.net.0.proj.weight",
              pre + "vae.encoder.mid_block.attentions.0.to_q.bias", pre + "vae.quant_conv.weight",
              pre + "shared_noise", pre + "uncond_inputs",
              "feature_extractor.clip_project_rgb.prompt_embed", "feature_extractor.clip_project_others.alpha_cond_time",
              "feature_extractor.ema_clip_project_others.time_embed",
              "feature_projections.0.0.conv1.weight", "feature_projections.1.0.shortcut.norm.bias",
              "ema_feature_projections.3.0.conv3.norm.weight"]:
        assert k in keys, k
    assert "feature_projections.0.0.shortcut.weight" not in keys  # s2: 512 -> 512 has an identity shortcut
    unet = pb.feature_extractor.ldm_extractor.unet
    assert sum(p.numel() for n, p in unet.named_parameters() if "lora" not in n) == 859_520_964
    assert len(list(unet.lora_layers())) == 128
    shared = pb.feature_extractor.ldm_extractor.shared_noise
    assert torch.equal(shared.cpu(), torch.randn(1, 4, 64, 64, generator=torch.Generator().manual_seed(42)))


def test_s0_variant_state_dict_keys_match_oracle():
    """vae_decoder_loss / s0 variant (mtmadise_cityscapes_rgb_to_depth_11.py:47-55): the product holders expose exactly the
    oracle's (= diffusers) keys incl. vae.decoder.*, and the projection for 's0' is Bottleneck(3 -> 128 -> 128)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import build_product_backbone
    from oracle import synthetic
    pb = build_product_backbone(torch.device("cpu"), variant="s0")
    with torch.device("meta"):
        ob = synthetic.build_backbone(variant="s0", lora_configs=(), with_ema=False)
    pk = {k: tuple(v.shape) for k, v in pb.state_dict().items()}
    pre = "feature_extractor.ldm_extractor.vae."
    for k, v in ob.state_dict().items():
        if k.startswith(pre) or k.startswith("feature_projections."):
            assert pk.get(k) == tuple(v.shape), (k, pk.get(k), tuple(v.shape))
    assert pk[pre + "decoder.up_blocks.2.resnets.0.conv_shortcut.weight"] == (256, 512, 1, 1)
    assert pk["feature_projections.0.0.conv1.weight"] == (128, 3, 1, 1) and pk["feature_projections.0.0.shortcut.weight"] == (128, 3, 1, 1)
    assert pk["feature_projections.0.0.conv3.weight"] == (128, 128, 1, 1)
    assert sum(v.numel() for k, v in pb.state_dict().items() if k.startswith(pre + "decoder.")) == 49_490_179
    assert pb._out_features == ["s0", "s3", "s4", "s5"] and pb._out_feature_strides["s0"] == 1
    from madm_b200.backbone import AttentionFeatureExtractorBackbone
    with pytest.raises(NotImplementedError):  # s2 projection config on an s0 extractor
        AttentionFeatureExtractorBackbone(None, [512, 320, 640, 1280], None, feature_extractor=pb.feature_extractor,
                                          out_features=["s2", "s3", "s4", "s5"])


def test_adapter_selection_follows_reference_semantics():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import set_lora_adapter
    from madm_b200.sd14_params import UNetParams
    from types import SimpleNamespace
    with torch.device("meta"):
        unet = UNetParams(device="meta")
    cfg = SimpleNamespace(r=16, lora_alpha=32, init_lora_weights="gaussian", target_modules=["to_k", "to_q", "to_v", "to_out.0"])
    assert unet.active_adapter() is None  # no adapters: set_lora_adapter is a no-op in the reference (mtmadise.py:131-132)
    unet.add_adapter(cfg, "default")
    unet.add_adapter(cfg, "Depth")
    set_lora_adapter(unet, "Depth")
    assert unet.active_adapter() == "Depth" and unet.scaling_of("Depth") == 2.0
    set_lora_adapter(unet, ["default", "Depth"])
    with pytest.raises(NotImplementedError):
        unet.active_adapter()


def test_unsupported_configs_fail_loudly():
    from madm_b200.ldm import LdmDiffusers
    with pytest.raises(NotImplementedError):
        LdmDiffusers(None, [5], [5, 8, 11], (), input_range="-1+1", unet_block_indices_type="after", vae_decoder_loss=True, device="cpu")
    with pytest.raises(NotImplementedError):
        LdmDiffusers(None, [], [5, 8, 11], (), input_range="-1+1", unet_block_indices_type="after", device="cpu")


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from madm_b200.sharding import shard_items, gather_max
    items = list(range(21))  # e.g. the 21 crops of one 1024x2048 image
    mine = shard_items(items, rank, world)
    ms = gather_max(10.0 + rank)  # max-over-ranks timing reduction used by bench.py
    allv = [None] * world
    dist.all_gather_object(allv, mine)
    q.put((rank, mine, ms, allv))
    dist.destroy_process_group()


def test_batch_sharding_world_size_2_gloo():
    """The N>1 path: images / crops are split in contiguous blocks over ranks with no data-path collective; timing is the
    max over ranks.  Exercised with a real 2-process gloo group on CPU."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29000 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, m0, t0, all0), (r1, m1, t1, all1) = res
    assert m0 == list(range(0, 11)) and m1 == list(range(11, 21))
    assert sorted(m0 + m1) == list(range(21))
    assert t0 == t1 == 11.0
    assert all0 == all1 == [m0, m1]


# ---------------------------------------------------------------------------------------------- DAFormer head mirror (SURVEY §8 f-2)
_HEAD_KW = dict(in_channels=[512] * 4, in_keys=["s2", "s3", "s4", "s5"], channels=256, num_classes=19, in_index=[0, 1, 2, 3],
                norm_cfg=dict(type="BN", requires_grad=True), align_corners=False,
                decoder_params=dict(embed_dims=256, embed_cfg=dict(type="mlp", act_cfg=None, norm_cfg=None),
                                    embed_neck_cfg=dict(type="mlp", act_cfg=None, norm_cfg=None),
                                    fusion_cfg=dict(type="aspp", sep=True, dilations=(1, 6, 12, 18), pool=False, act_cfg=dict(type="ReLU"),
                                                    norm_cfg=dict(type="BN", requires_grad=True))))


def test_head_state_dict_keys_match_reference_layout():
    """Key names / shapes of the shipped DAFormerHead configuration (mmcv ConvModule = .conv/.bn, DepthwiseSeparableConvModule =
    .depthwise_conv/.pointwise_conv; daformer_head.py:341-479, 536-640) — checked against the oracle restatement."""
    from madm_b200.head import DAFormerHead
    from oracle.daformer_head import build_head
    ph, oh = DAFormerHead(**_HEAD_KW), build_head()
    so, sp = oh.state_dict(), ph.state_dict()
    assert set(so) == set(sp)
    assert all(tuple(so[k].shape) == tuple(sp[k].shape) for k in so)
    assert "fuse_layer.aspp_modules.2.depthwise_conv.conv.weight" in sp and sp["fuse_layer.aspp_modules.2.depthwise_conv.conv.weight"].shape == (1024, 1, 3, 3)
    ph.load_state_dict(so)


def test_head_rejects_unsupported_variants_and_has_no_cpu_path():
    import copy
    import pytest
    from madm_b200 import _lib
    from madm_b200.head import DAFormerHead
    for patch in (dict(final_fuse_vae_decoder_feat=True), dict(concat_attention_to_conv_seg=True), dict(align_corners=True)):
        with pytest.raises(NotImplementedError):
            DAFormerHead(**{**_HEAD_KW, **patch})
    kw = copy.deepcopy(_HEAD_KW)
    kw["decoder_params"]["fusion_cfg"]["dilations"] = (1, 2, 3, 4)
    with pytest.raises(NotImplementedError):
        DAFormerHead(**kw)
    head = DAFormerHead(**_HEAD_KW).eval()
    feats = {k: torch.zeros(1, 512, s, s) for k, s in zip(("s2", "s3", "s4", "s5"), (128, 64, 32, 16))}
    with pytest.raises(_lib.MadmError):  # CPU tensors: the product refuses instead of computing in PyTorch
        head({"output_features": feats})
    with pytest.raises(NotImplementedError):
        head.train()({"output_features": feats})


def test_teacher_ops_have_no_cpu_path():
    """SURVEY §8 f-4 helpers refuse CPU tensors instead of falling back to PyTorch; the oracle restatement runs on CPU."""
    import pytest
    from madm_b200 import _lib, teacher
    from oracle import teacher as ot
    logits = torch.randn(1, 19, 8, 8)
    with pytest.raises(_lib.MadmError):
        teacher.pseudo_labels(logits, (32, 32), 0.9)
    with pytest.raises(_lib.MadmError):
        teacher.generate_class_mask(torch.zeros(4, 4, dtype=torch.int64), torch.tensor([0]))
    lab, prob, w, val = ot.pseudo_labels(logits, (32, 32), 0.2, psweight_ignore_top=3)
    assert lab.shape == (1, 32, 32) and lab.dtype == torch.int64 and 0.0 <= val <= 1.0
    assert torch.count_nonzero(w[:, :3]) == 0 and torch.all(w[:, 3:] == val)
    m = ot.generate_class_mask(lab[0], torch.tensor([int(lab[0, 0, 0])]))
    assert m.shape == (1, 32, 32) and m[0, 0, 0] == 1


def _gloo_allreduce_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from madm_b200.optim import allreduce_grads
    torch.manual_seed(0)
    # two LoRA adapters' worth of parameters; each rank trained a different adapter this step (mtmadise.py:149-157)
    params = [torch.nn.Parameter(torch.zeros(16, 320)), torch.nn.Parameter(torch.zeros(320, 16)),     # adapter "default"
              torch.nn.Parameter(torch.zeros(16, 320)), torch.nn.Parameter(torch.zeros(320, 16)),     # adapter "Depth"
              torch.nn.Parameter(torch.zeros(7)), torch.nn.Parameter(torch.zeros(3), requires_grad=False)]
    mine = (0, 1) if rank == 0 else (2, 3)
    for i in mine:
        params[i].grad = torch.full_like(params[i], float(rank + 1))
    params[4].grad = torch.full_like(params[4], 10.0 * (rank + 1))
    flat = allreduce_grads(params)
    # plain python objects: tensors sent through an mp.Queue are shared by file descriptor and need the producer to stay alive
    q.put((rank, [None if p.grad is None else (tuple(p.grad.shape), sorted(set(p.grad.flatten().tolist()))) for p in params], flat.numel()))
    dist.destroy_process_group()


def test_lora_grad_allreduce_world_size_2_gloo():
    """Training configuration (SURVEY §8e, config 5): ONE all-reduce over the flat buffer of all trainable gradients, zeros
    materialised for the adapter a rank did not train, averaged over ranks; frozen parameters stay out of the buffer."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31000 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_allreduce_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=120) for _ in range(2)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
    for rank, grads, n in res:
        assert n == 2 * (16 * 320 + 320 * 16) + 7
        assert grads[0] == ((16, 320), [0.5]) and grads[1] == ((320, 16), [0.5])   # (1 + 0) / 2 everywhere
        assert grads[2] == ((16, 320), [1.0]) and grads[3] == ((320, 16), [1.0])   # (0 + 2) / 2 everywhere
        assert grads[4] == ((7,), [15.0])
        assert grads[5] is None


def test_allreduce_grads_single_process_views_and_zeros():
    """Without a process group the call still flattens: afterwards every trainable parameter's .grad is a VIEW of the returned flat buffer
    (zeros where there was no gradient, the reference's add_zero_grad_on_unused_lora, mtmadise.py:149-157), frozen parameters stay out."""
    import torch
    from madm_b200.optim import allreduce_grads
    a, b, c = torch.nn.Parameter(torch.zeros(4, 3)), torch.nn.Parameter(torch.zeros(5)), torch.nn.Parameter(torch.zeros(2), requires_grad=False)
    a.grad = torch.arange(12.0).reshape(4, 3)
    flat = allreduce_grads([a, b, c])
    assert flat.numel() == 17 and torch.equal(flat[:12], torch.arange(12.0)) and torch.count_nonzero(flat[12:]) == 0
    assert a.grad.data_ptr() == flat.data_ptr() and b.grad.data_ptr() == flat[12:].data_ptr() and c.grad is None
    flat.mul_(2.0)  # the views follow the buffer
    assert torch.equal(a.grad, 2.0 * torch.arange(12.0).reshape(4, 3))


def test_host_only_size_queries_of_the_training_ops():
    """Scratch-size entry points are plain host functions: they answer without a device, and the fused LoRA-gradient op reports the widths it
    does not support (-1) instead of guessing."""
    from madm_b200 import _lib
    lib = _lib.load()
    ctas = min((8192 + 63) // 64, 148)
    assert lib.madm_op_lora_grads_scratch_floats(8192, 320, 320) == ctas * 16 * (320 + 320)
    assert lib.madm_op_lora_grads_scratch_floats(154, 1280, 768) == 3 * 16 * (1280 + 768)
    assert lib.madm_op_lora_grads_scratch_floats(8192, 96, 320) == -1 and lib.madm_op_lora_grads_scratch_floats(8192, 320, 100) == -1
    assert lib.madm_op_attention_bwd_scratch_floats(2, 8, 40, 4096, 4096) >= 2 * 2 * 8 * 4096
    assert lib.madm_op_wgrad_scratch_floats(8192, 320, 16, 1) > 0


def test_optimizer_ops_have_no_cpu_path():
    from madm_b200 import _lib
    from madm_b200.optim import FusedAdamW, update_ema
    from madm_b200.teacher import gaussian_blur, image_mix
    p = torch.nn.Parameter(torch.ones(4))
    p.grad = torch.ones(4)
    opt = FusedAdamW([p], lr=1e-3)
    assert opt.param_groups[0]["weight_decay"] == 1e-2 and opt.param_groups[0]["betas"] == (0.9, 0.999)
    with pytest.raises(_lib.MadmError):
        opt.step()
    with pytest.raises(_lib.MadmError):
        update_ema([torch.nn.Parameter(torch.ones(4))], [p], 3)
    with pytest.raises(_lib.MadmError):
        image_mix(torch.ones(1, 4, 4, dtype=torch.long), torch.rand(2, 3, 4, 4))
    with pytest.raises(_lib.MadmError):
        gaussian_blur(0.9, torch.rand(1, 3, 64, 64), 0.5)
    x = torch.rand(1, 3, 64, 64)
    assert gaussian_blur(0.2, x, 0.5) is x  # not selected: untouched, like the reference
    from madm_b200.teacher import color_jitter, color_jitter_params
    with pytest.raises(_lib.MadmError):
        color_jitter(0.9, data=x)
    assert color_jitter(0.1, data=x, target=None)[0] is x
    prm = color_jitter_params(5, 0.25, torch.Generator().manual_seed(1))
    assert prm["order"].shape == (5, 4) and all(sorted(r) == [0, 1, 2, 3] for r in prm["order"].tolist())
    assert (prm["brightness_factor"] >= 0.75).all() and (prm["brightness_factor"] <= 1.25).all() and (prm["hue_factor"].abs() <= 0.25).all()


def test_training_plan_dry_runs_without_a_device(monkeypatch):
    """SURVEY §8 row f-3, host side: the planner's dry runs of the training path (input-gradient arena layout, training workspace size)
    on a device-less context (MADM_PLAN_ONLY test hook: nothing can be launched from it).  Checks that the layout / size / plan passes
    of the forward-with-saved-activations + backward traversal agree with each other and scale with the batch."""
    import ctypes as C
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import meta_training_params, tensor_table
    from madm_b200 import _lib
    monkeypatch.setenv("MADM_PLAN_ONLY", "1")
    lib = _lib.load()
    h = C.c_void_p()
    _lib.check(lib.madm_create(C.byref(h), 0), None, "madm_create")
    try:
        _lib.check(lib.madm_set_compute_dtype(h, _lib.DTYPE_BF16), h, "dtype")
        named = meta_training_params()
        arr, keep = tensor_table(named, 0x1000)
        _lib.check(lib.madm_set_tensors(h, arr, len(named)), h, "madm_set_tensors")
        fwd = lib.madm_packed_bytes(h)
        dg = lib.madm_dgrad_packed_bytes(h)
        assert fwd > 2 ** 30 and dg > 2 ** 30, (fwd, dg, lib.madm_last_error(h))
        grads = [(n, t) for n, t in named if ("lora_" in n and ".Depth." in n) or n.startswith("feature_projections.")]
        garr, gkeep = tensor_table(grads, 0x100000)
        _lib.check(lib.madm_set_grad_tensors(h, garr, len(grads)), h, "madm_set_grad_tensors")
        w1, w2, w4 = (lib.madm_train_workspace_bytes(h, b, b"Depth") for b in (1, 2, 4))
        assert 0 < w1 < w2 < w4 < 16 * 2 ** 30, (w1, w2, w4, lib.madm_last_error(h))
        assert lib.madm_train_workspace_bytes(h, 2, b"Depth") == w2
        assert lib.madm_train_workspace_bytes(h, 2, b"") <= w2  # no adapter: no LoRA gradient scratch
        # a gradient buffer for a name that is not a registered parameter is rejected
        bad, bkeep = tensor_table([("feature_projections.9.0.conv1.weight", dict(named)["feature_projections.0.0.conv1.weight"])], 0x200000)
        assert lib.madm_set_grad_tensors(h, bad, 1) == -2
        # nothing can be launched from a device-less context
        a = _lib.MadmExtractArgs()
        a.B, a.stages = 1, 7
        assert lib.madm_extract(h, C.byref(a), None) == -3
    finally:
        lib.madm_destroy(h)
