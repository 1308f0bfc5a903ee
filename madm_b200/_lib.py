"""ctypes binding of ``libmadm_b200.so`` (C ABI declared in ``include/madm_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C madm_b200/csrc``.  There is no
fallback: if the shared object is missing, or no sm_100 device is present when a context is created,
the product path raises.
"""
import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# MADM_B200_LIB points at another build of the same C ABI (A/B runs of two kernel versions on one box)
LIB_PATH = os.environ.get("MADM_B200_LIB") or os.path.join(_HERE, "libmadm_b200.so")

MADM_OK = 0
STAGE_VAE, STAGE_UNET, STAGE_PROJ, STAGE_ALL = 1, 2, 4, 7
STAGE_HEAD = 8
STAGE_DEC, STAGE_ALL_S0 = 16, 23
VARIANT_BASE, VARIANT_S0 = 0, 1
FLAG_IMG_NORMALISED = 1
FLAG_TRAIN = 2
FLAG_OUT_FP16 = 4
ACT_NONE, ACT_SILU, ACT_GEGLU, ACT_RELU = 0, 1, 2, 3
DTYPE_BF16, DTYPE_FP16 = 0, 1

c_void_p, c_int, c_int32, c_int64, c_float, c_size_t, c_char_p = (
    C.c_void_p, C.c_int, C.c_int32, C.c_int64, C.c_float, C.c_size_t, C.c_char_p)


class MadmTensor(C.Structure):
    _fields_ = [("name", c_char_p), ("data", c_void_p), ("ndim", c_int32), ("shape", c_int64 * 4)]


class MadmExtractArgs(C.Structure):
    _fields_ = [
        ("B", c_int32), ("stages", c_int32), ("ema", c_int32), ("flags", c_int32),
        ("img", c_void_p), ("cond_inputs", c_void_p), ("cond_emb", c_void_p), ("timesteps", c_void_p),
        ("shared_noise", c_void_p), ("noisy_latents_in", c_void_p),
        ("out", c_void_p * 4),
        ("latents", c_void_p), ("noisy_latents", c_void_p), ("taps", c_void_p * 4),
        ("packed", c_void_p), ("workspace", c_void_p), ("workspace_bytes", c_size_t),
        ("range_flag", c_void_p), ("logits", c_void_p),
        ("unet_sample", c_void_p), ("decoded", c_void_p), ("decoded_raw", c_void_p),
        ("head_h", c_int32), ("head_w", c_int32),
        ("packed_dgrad", c_void_p), ("train_adapter", c_char_p), ("train_lora_scale", c_float), ("train_loss_scale", c_float),
    ]


class MadmBackwardArgs(C.Structure):
    _fields_ = [
        ("B", c_int32), ("reserved", c_int32),
        ("dout", c_void_p * 4), ("out", c_void_p * 4), ("cond_emb", c_void_p),
        ("d_cond_inputs", c_void_p), ("d_cond_emb", c_void_p),
        ("adapter", c_char_p), ("lora_alpha_over_r", c_float), ("loss_scale", c_float),
        ("packed", c_void_p), ("packed_dgrad", c_void_p), ("workspace", c_void_p), ("workspace_bytes", c_size_t),
        ("d_unet_sample", c_void_p),
    ]


class _MadmProfileKind(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("launches", c_int32), ("ms", C.c_double), ("flops", C.c_double), ("bytes", C.c_double),
                ("exec_flops", C.c_double)]


class MadmProfile(C.Structure):
    _fields_ = [("kind", _MadmProfileKind * 5)]


class MadmGemmSeg(C.Structure):
    _fields_ = [("a", c_void_p), ("Bt", c_int32), ("H", c_int32), ("W", c_int32), ("C", c_int32), ("ld", c_int32),
                ("ntaps", c_int32), ("dx", C.c_int8 * 9), ("dy", C.c_int8 * 9), ("b_off", c_int32 * 9)]


class MadmGemmArgs(C.Structure):
    _fields_ = [
        ("seg", MadmGemmSeg * 2), ("nseg", c_int32), ("M", c_int32), ("N", c_int32), ("Nw", c_int32), ("ldw", c_int32),
        ("w", c_void_p), ("bias", c_void_p), ("rowbias", c_void_p), ("rows_per_img", c_int32), ("ld_rowbias", c_int32),
        ("residual", c_void_p), ("ldr", c_int32), ("out_f32", c_void_p), ("ldo32", c_int32),
        ("out_bf16", c_void_p), ("ldo16", c_int32), ("act", c_int32), ("alpha", c_float), ("bn", c_int32), ("dtype", c_int32),
        ("colstats", c_void_p), ("stat_rows", c_int32), ("mt", c_int32), ("s2d_H", c_int32), ("s2d_W", c_int32), ("pair", c_int32), ("res16", c_int32),
    ]


# every symbol include/madm_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "madm_version": (c_int, []),
    "madm_last_error": (c_char_p, [c_void_p]),
    "madm_create": (c_int, [C.POINTER(c_void_p), c_int]),
    "madm_destroy": (c_int, [c_void_p]),
    "madm_set_compute_dtype": (c_int, [c_void_p, c_int32]),
    "madm_get_compute_dtype": (c_int, [c_void_p]),
    "madm_set_variant": (c_int, [c_void_p, c_int32]),
    "madm_get_variant": (c_int, [c_void_p]),
    "madm_set_tensors": (c_int, [c_void_p, C.POINTER(MadmTensor), c_int32]),
    "madm_packed_bytes": (c_size_t, [c_void_p]),
    "madm_pack_weights": (c_int, [c_void_p, c_void_p, c_char_p, c_float, c_int32, c_void_p]),
    "madm_workspace_bytes": (c_size_t, [c_void_p, c_int32]),
    "madm_workspace_bytes_head": (c_size_t, [c_void_p, c_int32, c_int32, c_int32]),
    "madm_extract": (c_int, [c_void_p, C.POINTER(MadmExtractArgs), c_void_p]),
    "madm_set_grad_tensors": (c_int, [c_void_p, C.POINTER(MadmTensor), c_int32]),
    "madm_dgrad_packed_bytes": (c_size_t, [c_void_p]),
    "madm_pack_dgrad_weights": (c_int, [c_void_p, c_void_p, c_char_p, c_float, c_int32, c_void_p]),
    "madm_train_workspace_bytes": (c_size_t, [c_void_p, c_int32, c_char_p]),
    "madm_backward": (c_int, [c_void_p, C.POINTER(MadmBackwardArgs), c_void_p]),
    "madm_backward_launch_count": (c_int, [c_void_p, c_int32]),
    "madm_launch_count": (c_int, [c_void_p, c_int32, c_int32]),
    "madm_set_profiling": (c_int, [c_void_p, c_int32]),
    "madm_get_profile": (c_int, [c_void_p, C.POINTER(MadmProfile)]),
    "madm_get_profile_stages": (c_int, [c_void_p, c_int32, C.POINTER(MadmProfile)]),
    "madm_op_gemm": (c_int, [C.POINTER(MadmGemmArgs), c_void_p]),
    "madm_op_groupnorm": (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_float,
                                  c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "madm_op_groupnorm_scratch_floats": (c_int, [c_int32, c_int32, c_int32]),
    "madm_op_groupnorm_from_colstats": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p,
                                                c_float, c_int32, c_void_p, c_void_p, c_int32, c_void_p]),
    "madm_op_layernorm": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_float, c_void_p, c_int32, c_void_p]),
    "madm_op_softmax_rows": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p]),
    "madm_op_attention": (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_int32,
                                  c_int32, c_int32, c_int32, c_int32, c_int64, c_int64, c_int64, c_float, c_int32, c_int32, c_void_p]),
    "madm_op_pack_linear": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_float, c_void_p, c_int32,
                                    c_int32, c_void_p]),
    "madm_op_pack_conv": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_int32, c_void_p]),
    "madm_op_pack_conv_dgrad": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_int32, c_void_p]),
    "madm_op_pack_linear_dgrad": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_float, c_void_p, c_int32, c_int32, c_void_p]),
    "madm_op_pack_geglu": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_void_p]),
    "madm_op_space_to_depth": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p]),
    "madm_op_nchw_to_nhwc16": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p]),
    "madm_op_bilinear_resize": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "madm_op_depthwise3x3": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "madm_op_pseudo_labels": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_float, c_int32, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p]),
    "madm_op_class_mask": (c_int, [c_void_p, c_int64, c_void_p, c_int32, c_void_p, c_void_p]),
    "madm_op_one_mix": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "madm_op_preprocess_image": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "madm_op_image_mix": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_void_p, c_void_p]),
    "madm_op_color_jitter": (c_int, [c_void_p, c_int32, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "madm_op_gaussian_blur": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_float, c_float, c_void_p, c_void_p, c_void_p]),
    "madm_op_ema_update": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_float, c_float, c_void_p]),
    "madm_op_grad_norm_scratch_floats": (c_int, [c_int32]),
    "madm_op_grad_norm": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "madm_op_adamw_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, C.c_double, C.c_double, C.c_double, C.c_double,
                                   C.c_double, c_int32, c_void_p, c_float, c_void_p]),
    "madm_op_slide_merge": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "madm_op_upsample2x": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p]),
    "madm_op_image_im2col": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_void_p]),
    "madm_op_groupnorm_bwd_scratch_floats": (c_int, [c_int32, c_int32, c_int32]),
    "madm_op_groupnorm_bwd": (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_float, c_int32,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_void_p]),
    "madm_op_c3_gn_bwd_scratch_floats": (c_int64, [c_int32, c_int32]),
    "madm_op_c3_gn_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int32, c_int32, c_int32, c_int32, c_void_p, c_float, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "madm_op_layernorm_bwd": (c_int, [c_void_p, c_int32, c_int32, c_void_p, c_float, c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "madm_op_geglu_fwd": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_int32, c_void_p]),
    "madm_op_geglu_bwd": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int32, c_void_p]),
    "madm_op_attention_bwd_scratch_floats": (c_int64, [c_int32, c_int32, c_int32, c_int32, c_int32]),
    "madm_op_attention_bwd": (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32,
                                      c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int64, c_int64, c_int64,
                                      c_int64, c_int64, c_int64, c_float, c_void_p, c_int32, c_void_p]),
    "madm_op_wgrad_scratch_floats": (c_int64, [c_int32, c_int32, c_int32, c_int32]),
    "madm_op_wgrad": (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_float, c_void_p,
                              c_int32, c_void_p, c_int32, c_void_p]),
    "madm_op_lora_grads_scratch_floats": (c_int64, [c_int32, c_int32, c_int32]),
    "madm_op_lora_grads": (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_float, c_void_p, c_void_p,
                                   c_void_p, c_int32, c_void_p]),
    "madm_op_colsum_per_image": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_int32, c_void_p]),
    "madm_op_zero_stuff2x": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "madm_op_sum2x2": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p]),
    "madm_op_relu_bwd_nchw": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_float, c_void_p, c_int32, c_void_p]),
    "madm_op_gn_add_relu_nchw": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_float,
                                         c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
}

_lib: Optional[C.CDLL] = None


class MadmError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the native library; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MadmError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). madm_b200 has no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, ctx=None, what: str = ""):
    if rc != MADM_OK:
        lib = load()
        msg = lib.madm_last_error(ctx)
        raise MadmError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
