"""Host-only checks of the s0 variant's training plans on a device-less context (MADM_PLAN_ONLY test hook): the training traversal of the
vae_decoder_loss / s0 configuration lays out its input-gradient arena and sizes its workspace."""
import ctypes as C
from types import SimpleNamespace

import pytest

from helpers import meta_training_params, tensor_table


def meta_s0_params():
    """(state_dict name, meta tensor) pairs of the s0 variant: UNet with the adapters 'default' and 'Depth' (r = 16), the VAE with its decoder,
    and the projections 3 -> 128 (bottleneck 128) and 320 / 640 / 1280 -> 512 (mtmadise_cityscapes_rgb_to_depth_11.py:47-55)."""
    from madm_b200.sd14_params import BottleneckParams, UNetParams, VAEParams, empty_init
    with empty_init():
        unet, vae = UNetParams(device="meta"), VAEParams(device="meta", with_decoder=True)
        for name in ("default", "Depth"):
            unet.add_adapter(SimpleNamespace(r=16, lora_alpha=16, init_lora_weights="gaussian",
                                             target_modules=["to_k", "to_q", "to_v", "to_out.0"]), name)
        projs = [BottleneckParams(3, 128, 128, device="meta")] + [BottleneckParams(c, 512, 128, device="meta") for c in (320, 640, 1280)]
    named = [("feature_extractor.ldm_extractor.unet." + n, p) for n, p in unet.named_parameters()]
    named += [("feature_extractor.ldm_extractor.vae." + n, p) for n, p in vae.named_parameters()]
    for i, pr in enumerate(projs):
        named += [(f"feature_projections.{i}.0." + n, p) for n, p in pr.named_parameters()]
    return named


def _context(lib, _lib, dtype, variant, named):
    h = C.c_void_p()
    _lib.check(lib.madm_create(C.byref(h), 0), None, "madm_create")
    _lib.check(lib.madm_set_compute_dtype(h, _lib.DTYPE_FP16 if dtype == "fp16" else _lib.DTYPE_BF16), h, "dtype")
    _lib.check(lib.madm_set_variant(h, variant), h, "variant")
    arr, keep = tensor_table(named, 0x1000)
    _lib.check(lib.madm_set_tensors(h, arr, len(named)), h, "madm_set_tensors")
    return h


@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
def test_s0_training_plan_sizes(monkeypatch, dtype):
    """The s0 context sizes a training workspace at B = 1, 2, 8 and an input-gradient arena.  The arena holds the base variant's UNet
    operands plus unet.conv_out's (the decoder body runs without gradient and needs none) and no input-gradient operands for projection 0,
    whose 3-channel input (the detached decoded image) takes no gradient."""
    from madm_b200 import _lib
    monkeypatch.setenv("MADM_PLAN_ONLY", "1")
    lib = _lib.load()
    h = _context(lib, _lib, dtype, _lib.VARIANT_S0, meta_s0_params())
    base = _context(lib, _lib, dtype, _lib.VARIANT_BASE, meta_training_params())
    try:
        fwd = lib.madm_packed_bytes(h)
        dgrad = lib.madm_dgrad_packed_bytes(h)
        assert fwd > 2 ** 30 and dgrad > 2 ** 30, (fwd, dgrad, lib.madm_last_error(h))
        # projection 0's conv1 / shortcut operands of the base variant ([512, 128] / [512, 512]) outweigh conv_out's [320, 64]
        assert dgrad < lib.madm_dgrad_packed_bytes(base)
        for B in (1, 2, 8):
            tws, ws = lib.madm_train_workspace_bytes(h, B, b"Depth"), lib.madm_workspace_bytes(h, B)
            assert tws > ws > 0, (B, tws, ws, lib.madm_last_error(h))
        assert lib.madm_packed_bytes(h) == fwd and lib.madm_dgrad_packed_bytes(h) == dgrad
    finally:
        lib.madm_destroy(h)
        lib.madm_destroy(base)
