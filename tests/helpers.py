"""Shared helpers for the parity tests (oracle <-> product)."""
import copy
from types import SimpleNamespace

import torch.nn.functional as F

LORA_CONFIGS = ("default_r16_a16", "Depth_r16_a16")


def build_product_backbone(device, lora_configs=LORA_CONFIGS, with_ema=True, same_cond_params=False, compute_dtype="fp16", variant="base"):
    """Construct madm_b200's backbone exactly as the reference LazyCall config does
    (config_files/common/models/mtmadise_multi_lora.py:14-41) + MTMADISE.set_multi_lora (mtmadise.py:115-127)."""
    from madm_b200.backbone import AttentionFeatureExtractorBackbone
    from madm_b200.ldm import BasePromptTimeGenerator, LdmDiffusers
    s0 = variant == "s0"  # the overrides of config_files/SemSeg/MTMADISE/mtmadise_cityscapes_rgb_to_depth_11.py:47-55
    ldm = LdmDiffusers(stable_diffusion_name_or_path=None, encoder_block_indices=[] if s0 else [5], unet_block_indices=[5, 8, 11],
                       unet_block_indices_type="after", decoder_block_indices=(), input_range="-1+1", finetune_unet="all",
                       vae_decoder_loss=s0, device=device, compute_dtype=compute_dtype)
    gen = BasePromptTimeGenerator(learnable_cond_prompt=True, learnable_cond_time=True, clip_state="no", num_timesteps=1,
                                  clip_model_name="ViT-L-14-336", ldm_extractor=ldm, same_cond_params=same_cond_params)
    bb = AttentionFeatureExtractorBackbone(attention_features_res=None, feature_dims=[3 if s0 else 512, 320, 640, 1280],
                                           projection_dim=[128 if s0 else 512, 512, 512, 512], attention_features_location=None,
                                           feature_extractor=gen, num_res_blocks=1, out_features=["s0" if s0 else "s2", "s3", "s4", "s5"],
                                           use_checkpoint=False, slide_training=False)
    for cfg in lora_configs:
        name, rank, alpha = cfg.split("_")
        lc = SimpleNamespace(r=int(rank[1:]), lora_alpha=int(alpha[1:]), init_lora_weights="gaussian",
                             target_modules=["to_k", "to_q", "to_v", "to_out.0"])
        ldm.unet.add_adapter(adapter_config=lc, adapter_name=name)
    if lora_configs:
        ldm.unet.set_adapter([c.split("_")[0] for c in lora_configs])
        ldm._freeze()
    if with_ema:  # CMDISE._inti_ema_weights (cmdise.py:307-325)
        bb.ema_feature_projections = copy.deepcopy(bb.feature_projections)
        gen.ema_clip_project_others = copy.deepcopy(gen.clip_project_others)
    return bb


def set_lora_adapter(unet, state):
    """MTMADISE.set_lora_adapter (mtmadise.py:129-147): write ``_active_adapter`` on every tuner layer."""
    if isinstance(state, str):
        state = [state]
    for _, m in unet.named_modules():
        if hasattr(m, "lora_A") and hasattr(m, "_active_adapter"):
            m._active_adapter = state


def cosine(a, b):
    return F.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0).item()


def max_rel(a, b):
    """max|a-b| / max|b| per tensor (SURVEY §8d parity gates)."""
    return ((a.double() - b.double()).abs().max() / b.double().abs().max()).item()


def meta_training_params(proj_width=128):
    """(state_dict name, meta tensor) pairs of the host-only training dry runs: UNet with the LoRA adapters 'default' and 'Depth' (r = 16),
    VAE encoder, four GN-bottleneck projections (512 / 320 / 640 / 1280 -> 512, bottleneck width proj_width)."""
    from madm_b200.sd14_params import BottleneckParams, UNetParams, VAEParams, empty_init
    with empty_init():
        unet, vae = UNetParams(device="meta"), VAEParams(device="meta")
        for name in ("default", "Depth"):
            unet.add_adapter(SimpleNamespace(r=16, lora_alpha=16, init_lora_weights="gaussian",
                                             target_modules=["to_k", "to_q", "to_v", "to_out.0"]), name)
        projs = [BottleneckParams(c, 512, proj_width, device="meta") for c in (512, 320, 640, 1280)]
    named = [("feature_extractor.ldm_extractor.unet." + n, p) for n, p in unet.named_parameters()]
    named += [("feature_extractor.ldm_extractor.vae." + n, p) for n, p in vae.named_parameters()]
    for i, pr in enumerate(projs):
        named += [(f"feature_projections.{i}.0." + n, p) for n, p in pr.named_parameters()]
    return named


def tensor_table(items, base):
    """madm_tensor records of (name, tensor) pairs at fake device addresses base, base + 16, ... (dry runs never dereference them).
    Returns the array and the encoded names, which must outlive it."""
    from madm_b200 import _lib
    arr = (_lib.MadmTensor * len(items))()
    keep = [n.encode() for n, _ in items]
    for i, (n, t) in enumerate(items):
        arr[i].name, arr[i].data, arr[i].ndim = keep[i], base + 16 * i, t.dim()
        for k, s in enumerate(t.shape):
            arr[i].shape[k] = s
    return arr, keep
