/* madm_b200 — C ABI of the B200-native MADM diffusion feature-extraction hot path.
 *
 * The reference (XiaRho/MADM) has no FFI for this path: its boundary is the Python nn.Module
 *   AttentionFeatureExtractorBackbone.forward(img, input_modal, ema_forward, timestep, **kw)
 *       (reference modeling/backbone/feature_extractor.py:280-284, :156-170, :367-396)
 * which calls BasePromptTimeGenerator.forward (modeling/meta_arch/ldm_base.py:832-924) and
 * LdmDiffusers.forward (modeling/meta_arch/ldm_diffusers.py:143-217).  This library is what the drop-in
 * Python module (madm_b200/backbone.py) binds instead of diffusers/peft/detectron2: each entry point below
 * names the reference code it replaces.
 *
 * Conventions: extern "C", POD structs, raw device pointers, no torch types.  Every call returns 0 on success
 * or a negative MADM_E* code (never throws / aborts); madm_last_error() gives the message.  All device work is
 * enqueued asynchronously on the caller's stream (pass torch.cuda.current_stream().cuda_stream); there are no
 * hidden synchronisations.  The caller owns all memory: parameters (fp32, PyTorch layouts), the packed-weight
 * arena, the workspace and the outputs.  One madm_ctx per (process, device); not thread-safe.
 * Built for sm_100a only; there is no CPU fallback.
 */
#ifndef MADM_B200_H_
#define MADM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MADM_VERSION 100 /* 0.1.0 */

enum {
  MADM_OK = 0,
  MADM_EINVAL = -1,   /* bad argument / unsupported shape */
  MADM_ENOTFOUND = -2,/* a required parameter tensor was not registered */
  MADM_ECUDA = -3,    /* CUDA runtime / driver error */
  MADM_ESTATE = -4,   /* call order violation (e.g. extract before pack) */
  MADM_ENOMEM = -5    /* workspace or packed arena too small */
};

/* Compute dtype of the GEMM / attention operands (accumulation, norms, softmax and the residual stream are always fp32).
 * fp16 is the default: it is the reference's own AMP dtype (engine/train_loop.py:277, evaluation/evaluator.py:62-86) and it
 * meets the 2e-2 parity gate with margin; bf16 runs at the same tensor-core rate but its 8-bit mantissa puts the projected
 * maps at ~2.1e-2 on the synthetic model (DESIGN.md "Numerics"). */
#define MADM_DTYPE_BF16 0
#define MADM_DTYPE_FP16 1

typedef struct madm_ctx madm_ctx;
typedef void* madm_stream; /* cudaStream_t */

/* A named fp32 device tensor in its PyTorch layout (Conv2d [out,in,kh,kw], Linear [out,in], vectors [n]).
 * Names are the reference's state_dict keys relative to `backbone.` (SURVEY Appendix A.6), e.g.
 *   feature_extractor.ldm_extractor.unet.down_blocks.0.resnets.0.conv1.weight
 *   feature_extractor.ldm_extractor.unet....attn1.to_q.base_layer.weight / .lora_A.<adapter>.weight
 *   feature_extractor.ldm_extractor.vae.encoder.conv_in.weight
 *   feature_projections.0.0.conv1.weight, feature_projections.0.0.conv1.norm.weight
 *   ema_feature_projections.*  (EMA twins, reference modeling/meta_arch/cmdise.py:308) */
typedef struct madm_tensor {
  const char* name;
  const void* data;
  int32_t ndim;
  int64_t shape[4];
} madm_tensor;

int madm_version(void);
const char* madm_last_error(const madm_ctx* ctx); /* ctx may be NULL: error of the last failed madm_create */

int madm_create(madm_ctx** out, int device);
int madm_destroy(madm_ctx* ctx);

/* Select MADM_DTYPE_FP16 (default) or MADM_DTYPE_BF16.  Invalidates packed weights and plans: call before
 * madm_pack_weights. */
int madm_set_compute_dtype(madm_ctx* ctx, int32_t dtype);
int madm_get_compute_dtype(const madm_ctx* ctx);

/* Path variant (a property of the backbone's constructor config).
 * MADM_VARIANT_BASE: config_files/common/models/mtmadise_multi_lora.py:14-41 — encoder tap (encoder_block_indices=[5]) -> 's2'.
 * MADM_VARIANT_S0:   the configuration all shipped experiment files select
 *   (config_files/SemSeg/MTMADISE/mtmadise_cityscapes_rgb_to_depth_11.py:47-55: vae_decoder_loss=True, encoder_block_indices=[],
 *   feature_dims[0]=3, projection_dim[0]=128, out_features[0]='s0'): the UNet runs to its final output (conv_norm_out / conv_out,
 *   ldm_diffusers.py:608-611), the VAE decoder decodes it (vae_decoder, ldm_diffusers.py:314-346) and the decoded 3 x 512 x 512 image
 *   is the first feature, projected by Bottleneck(3 -> 128 -> 128) into 's0' [B,128,512,512] (SURVEY §8 row a-11 / f-1).
 * Needs the vae.decoder.* / vae.post_quant_conv.* / unet.conv_norm_out.* / unet.conv_out.* parameters registered.
 * Invalidates packed weights and plans: call before madm_pack_weights. */
#define MADM_VARIANT_BASE 0
#define MADM_VARIANT_S0 1
int madm_set_variant(madm_ctx* ctx, int32_t variant);
int madm_get_variant(const madm_ctx* ctx);

/* Register / refresh parameter pointers.  Replaces nn.Module parameter ownership: the library never copies or
 * owns model weights, it reads biases and norm affines in place and packs GEMM weights into the arena below. */
int madm_set_tensors(madm_ctx* ctx, const madm_tensor* named, int32_t n);

/* Bytes of the packed bf16 weight arena (K-major tiles for TMA) for the registered model. */
size_t madm_packed_bytes(madm_ctx* ctx);

/* fp32 -> bf16 K-major packing of every GEMM weight into `packed` (caller-allocated, madm_packed_bytes()).
 * `adapter` names the active LoRA adapter to fold (W' = W + alpha/r * B@A; replaces peft's LoRA Linear.forward and
 * MTMADISE.set_lora_adapter, reference modeling/meta_arch/mtmadise.py:115-147); NULL or "" = base weights.
 * lora_alpha_over_r: scaling for that adapter.  lora_only = 1 repacks just the 128 LoRA-targeted projections (adapter switch),
 * 2 those plus the feature_projections / ema_feature_projections convs (what a LoRA training step's optimizer / EMA update touches);
 * 0 repacks everything (after load_state_dict). */
int madm_pack_weights(madm_ctx* ctx, void* packed, const char* adapter, float lora_alpha_over_r, int32_t lora_only,
                      madm_stream stream);

#define MADM_STAGE_VAE 1   /* vae_encoder           (reference ldm_diffusers.py:283-311) */
#define MADM_STAGE_UNET 2  /* add_noise + diffusion_unet (ldm_diffusers.py:349-360, :454-616) */
#define MADM_STAGE_PROJ 4  /* forward_features      (reference feature_extractor.py:367-396) */
#define MADM_STAGE_ALL 7
/* SURVEY §8 row f-2 (next after the path): DAFormerHead.forward (modeling/sem_seg_head/daformer_head.py:702-749) on the feature
 * dict: reads args.out[0..3] (s2..s5, produced by MADM_STAGE_PROJ in the same call or supplied by the caller) and writes
 * args.logits.  Needs the head's parameters registered under "sem_seg_head." (a context may hold only those). */
#define MADM_STAGE_HEAD 8
/* MADM_VARIANT_S0 only: UNet conv_norm_out / conv_out (ldm_diffusers.py:608-611) + vae_decoder(output_final=True)
 * (ldm_diffusers.py:192, :314-346).  Runs between MADM_STAGE_UNET and MADM_STAGE_PROJ; MADM_STAGE_ALL_S0 is the whole variant path. */
#define MADM_STAGE_DEC 16
#define MADM_STAGE_ALL_S0 23

/* Workspace bytes needed by madm_extract for batch B (all stages). */
size_t madm_workspace_bytes(madm_ctx* ctx, int32_t B);
/* the same when the head stage runs on a head_h x head_w grid (madm_extract_args.head_h / head_w) */
size_t madm_workspace_bytes_head(madm_ctx* ctx, int32_t B, int32_t head_h, int32_t head_w);

#define MADM_FLAG_IMG_NORMALISED 1
/* out[0..3] are fp16 [B,C,H,W] tensors instead of fp32 (base variant, MADM_STAGE_PROJ; not with MADM_FLAG_TRAIN, whose madm_backward
 * reads the fp32 maps): an opt-in for host-bound consumers -- the
 * reference returns fp32 maps (GroupNorm runs in fp32 under autocast), so fp32 stays the default.  Halves the 357 MB per 8 images that
 * a caller who downloads the feature dict moves over PCIe. */
#define MADM_FLAG_OUT_FP16 4
typedef struct madm_extract_args {
  int32_t B;                   /* images (512x512 crops) in this call */
  int32_t stages;              /* MADM_STAGE_* mask; intermediate results live in the workspace between calls */
  int32_t ema;                 /* use ema_feature_projections (ema_forward=True) */
  int32_t flags;               /* MADM_FLAG_* */
  const float* img;            /* [B,3,512,512] fp32 NCHW in [0,1] (LdmDiffusers.forward input, input_range '-1+1'); with
                                  MADM_FLAG_IMG_NORMALISED already in [-1,1]: what the module-level vae_encoder() of the reference
                                  receives (ldm_diffusers.py:283-311, called from mtmadise.py:254,345,398,463 on colour targets) */
  const float* cond_inputs;    /* [B,77,768] fp32: batched_inputs['cond_inputs'] (ldm_base.py:915-917) */
  const float* cond_emb;       /* [B,1280] fp32: batched_inputs['cond_emb'][:,0] */
  const int64_t* timesteps;    /* [B] int64 device: torch.randint(lo,hi,(B,)) (ldm_diffusers.py:160) */
  const float* shared_noise;   /* [1,4,64,64] fp32: buffer shared_noise (ldm_diffusers.py:73-75) */
  const float* noisy_latents_in; /* optional [B,4,64,64] NCHW: overrides VAE+q-sample output for the UNet stage */
  float* out[4];               /* s2 [B,512,128,128] (MADM_VARIANT_S0: s0 [B,128,512,512]), s3 [B,512,64,64], s4 [B,512,32,32], s5 [B,512,16,16] fp32 NCHW */
  /* optional debug / parity taps (NULL to skip), fp32 NCHW */
  float* latents;              /* [B,4,64,64]  vae mean * 0.18215 */
  float* noisy_latents;        /* [B,4,64,64] */
  float* taps[4];              /* enc tap [B,512,128,128], unet taps [B,320,64,64], [B,640,32,32], [B,1280,16,16] */
  const void* packed;          /* arena filled by madm_pack_weights */
  void* workspace;
  size_t workspace_bytes;
  int32_t* range_flag;         /* optional device int: set to 1 if the normalised image leaves [-1,1]
                                  (the reference asserts this with a host sync, ldm_diffusers.py:147) */
  float* logits;               /* MADM_STAGE_HEAD: [B,num_classes,128,128] fp32 NCHW (DAFormerHead output, before any resize);
                                  MADM_VARIANT_S0: the head fuses on the s0 grid -> [B,num_classes,512,512] */
  /* MADM_VARIANT_S0 (MADM_STAGE_DEC); out[0] then is s0 [B,128,512,512].  Both optional (NULL to skip), fp32 NCHW: the dict
   * LdmDiffusers.forward returns under return_unet_final_output (ldm_diffusers.py:211-215) */
  float* unet_sample;          /* [B,4,64,64]   'before_vae.decoder': unet_final_output.sample */
  float* decoded;              /* [B,3,512,512] 'after_vae.decoder': clip(decoder_output, -1, 1) */
  float* decoded_raw;          /* [B,3,512,512] decoder_output itself: the first entry of the feature list (ldm_diffusers.py:199) */
  /* MADM_STAGE_HEAD alone: grid of the first feature map in out[0] (0, 0 = that of a 512 x 512 crop: 128 x 128, s0 variant 512 x 512).
   * Sliding-window inference merges the crops' features into full-image maps before the head runs (feature_extractor.py:270-275), e.g.
   * 256 x 512 for a 1024 x 2048 image; the other three maps are 1/2, 1/4, 1/8 of it (s0 variant: 1/8, 1/16, 1/32) and the logits
   * come out on this grid. */
  int32_t head_h, head_w;
  const void* packed_dgrad;    /* MADM_FLAG_TRAIN: the arena filled by madm_pack_dgrad_weights (holds the natural-order feed-forward weights
                                  of the training forward next to the input-gradient operands) */
  const char* train_adapter;   /* MADM_FLAG_TRAIN: the active LoRA adapter (names the lora_A / lora_B gradients); NULL / "" = none */
  float train_lora_scale;      /* its alpha / r */
  float train_loss_scale;      /* loss scale of the backward that will follow (> 0; 1.0 with bf16 operands) */
} madm_extract_args;

/* The whole path a-1..a-9 of SURVEY §8: VAE encode -> q-sample -> UNet forward with taps -> GN-bottleneck projections. */
int madm_extract(madm_ctx* ctx, const madm_extract_args* args, madm_stream stream);

/* Per-kernel-family device timing of the last madm_extract call (CUDA events recorded on the launch stream around every
 * launch while profiling is on), with the algorithmic FLOPs / HBM bytes of those launches: the inputs of the roofline
 * line bench.py prints.  madm_get_profile synchronises the device. */
#define MADM_KIND_GEMM 0        /* gemm_tc_kernel: all convs / linears (tensor-bound) */
#define MADM_KIND_ATTENTION 1   /* flash_attn_kernel */
#define MADM_KIND_GROUPNORM 2   /* gn_stats / gn_apply / gn_add_relu_nchw (HBM-bound) */
#define MADM_KIND_LAYERNORM 3
#define MADM_KIND_ELEMENTWISE 4 /* im2col, q-sample, space-to-depth, upsample, softmax rows, casts */
#define MADM_NUM_KINDS 5
typedef struct madm_profile {
  /* flops: ALGORITHMIC (2*MAC of the reference's convs / linears / attention products: no K padding, no identity-weight residual
   * segments) -- the numerator of the roofline line; exec_flops: what the launches execute (>= flops). */
  struct { char name[32]; int32_t launches; double ms; double flops; double bytes; double exec_flops; } kind[MADM_NUM_KINDS];
} madm_profile;
int madm_set_profiling(madm_ctx* ctx, int32_t on);
int madm_get_profile(madm_ctx* ctx, madm_profile* out);
/* the same, restricted to the launches of the stages in stage_mask (MADM_STAGE_*): e.g. MADM_STAGE_UNET for the UNet contractions */
int madm_get_profile_stages(madm_ctx* ctx, int32_t stage_mask, madm_profile* out);

/* Number of kernels one madm_extract call launches for batch B with the given stage mask (for bench accounting). */
int madm_launch_count(madm_ctx* ctx, int32_t B, int32_t stages);

/* ---------------------------------------------------------------------------------------------------------------
 * Operator-level entry points (the kernels the engine is built from), exposed so parity tests can check each one
 * against the oracle through the same C ABI.  All pointers are device pointers.  "*_bf16" parameters are 16-bit operand
 * tensors whose element type is given by `dtype` (MADM_DTYPE_*).
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct madm_gemm_seg {
  const void* a;     /* bf16 NHWC activations [Bt,H,W,ld] */
  int32_t Bt, H, W, C, ld, ntaps;
  int8_t dx[9], dy[9];
  int32_t b_off[9];
} madm_gemm_seg;

typedef struct madm_gemm_args {
  madm_gemm_seg seg[2];
  int32_t nseg, M, N, Nw, ldw;
  const void* w;          /* bf16 [Nw, ldw] K-major */
  const float* bias;      /* [N] or NULL */
  const float* rowbias;   /* [nimg, ld_rowbias] or NULL */
  int32_t rows_per_img, ld_rowbias;
  const float* residual;  /* fp32 [M, ldr] or NULL (16-bit if res16) */
  int32_t ldr;
  float* out_f32; int32_t ldo32;
  void* out_bf16; int32_t ldo16;
  int32_t act;            /* 0 none, 1 SiLU, 2 GEGLU (tile-interleaved weights), 3 ReLU */
  float alpha;
  int32_t bn;             /* N tile: 0 auto, else 16/32/64/128/160/192/256 */
  int32_t dtype;          /* MADM_DTYPE_* of a, w and out_bf16 */
  float* colstats;        /* optional [ceil(M/32)][N][2]: per-column (sum, sum of squares) of the stored outputs per 32-row block,
                             i.e. the GroupNorm statistics of the consumer fused into this epilogue (no atomics) */
  int32_t stat_rows;      /* 32 (0 = 32) */
  int32_t mt;             /* M sub-tiles per CTA tile when bn = 128: 0 auto, 1 (128-row tiles), 2 (256-row tiles) */
  int32_t s2d_H, s2d_W;   /* > 0: out_bf16 is written in space-to-depth layout [4][B][H/2][W/2][N] (operand of a stride-2 conv) */
  int32_t pair;           /* CTA pairs (tcgen05 cta_group::2, 256-row MMAs): 0 auto, 1 force, -1 never */
  int32_t res16;          /* residual points to a 16-bit [M, ldr] tensor of `dtype` (may alias out_bf16) instead of fp32 */
} madm_gemm_args;

int madm_op_gemm(const madm_gemm_args* a, madm_stream stream);
int madm_op_groupnorm(const void* x0, int32_t C0, const void* x1, int32_t C1, int32_t B, int32_t HW,
                      int32_t in16 /* inputs are 16-bit (dtype) instead of fp32 */, const float* gamma,
                      const float* beta, float eps, int32_t act, float* stats_scratch /* madm_op_groupnorm_scratch_floats() */,
                      void* y_bf16, void* raw_bf16, int32_t dtype, madm_stream stream);
/* GroupNorm whose statistics come from a producing GEMM's `colstats` instead of a statistics pass */
int madm_op_groupnorm_from_colstats(const void* x, int32_t C, int32_t B, int32_t HW, int32_t in16, const float* colstats,
                                    int32_t stat_rows, const float* gamma, const float* beta, float eps, int32_t act,
                                    float* scratch /*[B,32,32,2]*/, void* y_bf16, int32_t dtype, madm_stream stream);
int madm_op_groupnorm_scratch_floats(int32_t B, int32_t HW, int32_t C); /* scratch size (floats) for the two GN ops */
int madm_op_layernorm(const void* x, int32_t in16 /* x is 16-bit (dtype) instead of fp32 */, int32_t M, int32_t C, const float* gamma,
                      const float* beta, float eps, void* y_bf16, int32_t dtype, madm_stream stream);
int madm_op_softmax_rows(const float* s, int32_t R, int32_t L, void* p_bf16, int32_t dtype, madm_stream stream);
int madm_op_attention(const void* q, int32_t ldq, const void* k, int32_t ldk, const void* v, int32_t ldv, void* o, int32_t ldo,
                      int32_t B, int32_t heads, int32_t d, int32_t Nq, int32_t Nk, int64_t q_bstride, int64_t kv_bstride,
                      int64_t o_bstride, float scale, int32_t dtype, int32_t impl /* must be 0: the tcgen05/TMEM kernel */,
                      madm_stream stream);
int madm_op_pack_linear(const float* w, int32_t N, int32_t K, const float* lora_a, const float* lora_b, int32_t r, float scale,
                        void* out_bf16, int32_t ldo, int32_t dtype, madm_stream stream);
int madm_op_pack_conv(const float* w, int32_t N, int32_t C, int32_t taps, int32_t Cpad, void* out_bf16, int32_t ldo,
                      int32_t dtype, madm_stream stream);
/* dgrad operands (first building block of SURVEY §8 row f-3, the backward pass): the input gradient of a stride-1 conv / a linear is
 * madm_op_gemm on the output gradient with these packed weights — conv [Cout,Cin,kh,kw] -> [Cin, taps*CoPad] with mirrored taps (the
 * forward tap offsets apply as is), linear [N,K] (+ LoRA: W + s B A) -> its transpose [K, ldo >= N]. */
int madm_op_pack_conv_dgrad(const float* w, int32_t Cout, int32_t Cin, int32_t taps, int32_t CoPad, void* out_bf16, int32_t ldo, int32_t dtype,
                            madm_stream stream);
int madm_op_pack_linear_dgrad(const float* w, int32_t N, int32_t K, const float* lora_a, const float* lora_b, int32_t r, float scale,
                              void* out_bf16, int32_t ldo, int32_t dtype, madm_stream stream);
int madm_op_pack_geglu(const float* w, const float* bias, int32_t C4, int32_t K, void* out_bf16, float* out_bias,
                       int32_t dtype, madm_stream stream);
int madm_op_space_to_depth(const float* x, int32_t B, int32_t H, int32_t W, int32_t C, void* out_bf16, int32_t dtype,
                           madm_stream stream);
/* head stage kernels (SURVEY §8 f-2; reference daformer_head.py:702-749, mmseg resize, mmcv DepthwiseSeparableConvModule) */
int madm_op_nchw_to_nhwc16(const float* x, int32_t B, int32_t C, int32_t HW, void* out16, int32_t dtype, madm_stream stream);
int madm_op_bilinear_resize(const void* src16, int32_t B, int32_t Hs, int32_t Ws, int32_t C, void* dst16, int32_t Hd, int32_t Wd,
                            int32_t dst_pitch, int32_t dtype, madm_stream stream); /* F.interpolate(bilinear, align_corners=False), NHWC */
int madm_op_depthwise3x3(const void* src16, int32_t B, int32_t H, int32_t W, int32_t C, int32_t dilation, const float* w9 /*[9][C]*/,
                         const float* shift /*[C]*/, void* dst16, int32_t dtype, madm_stream stream); /* + shift + ReLU */
/* teacher post-processing + DACS mixing (SURVEY §8 f-4; reference mtmadise.py:337-352, utils/dacs_transforms.py:87-112) */
int madm_op_pseudo_labels(const float* logits /*[B,C,h,w]*/, int32_t B, int32_t C, int32_t h, int32_t w, int32_t H, int32_t W, float threshold,
                          int32_t ignore_top, int64_t* label /*[B,H,W]*/, float* prob /*[B,H,W]*/, float* weight /*[B,H,W] or NULL*/,
                          int32_t* count /*device scalar: pixels with prob >= threshold*/, madm_stream stream);
int madm_op_class_mask(const int64_t* label, int64_t n, const int64_t* classes, int32_t k, int64_t* mask, madm_stream stream);
int madm_op_one_mix(const int64_t* mask, int64_t n, const int64_t* label_a, const int64_t* label_b, int64_t* label_out /*or NULL*/,
                    const float* weight_a, const float* weight_b, float* weight_out /*or NULL*/, madm_stream stream);
/* FeatureExtractorBackbone.preprocess_image (reference modeling/backbone/feature_extractor.py:140-146, :77-79): T.Resize(backbone_in_size,
 * BILINEAR) — on tensors with the reference's pinned torchvision 0.16.1 that is F.interpolate(bilinear, align_corners=False) WITHOUT
 * antialiasing — to Hr x Wr, then the zero padding of ImageList.from_tensors up to Hd x Wd; fp32 planes (B*3 of them). */
int madm_op_preprocess_image(const float* src /*[planes,Hs,Ws]*/, int32_t planes, int32_t Hs, int32_t Ws, int32_t Hr, int32_t Wr, int32_t Hd,
                             int32_t Wd, float* dst /*[planes,Hd,Wd]*/, madm_stream stream);
/* image side of the DACS mixing (SURVEY §8 f-4; reference utils/dacs_transforms.py:98-112 one_mix on `data`, :62-84 gaussian_blur =
 * kornia.filters.GaussianBlur2d(kernel_size, (sigma, sigma)), separable, border 'reflect') */
int madm_op_image_mix(const int64_t* mask /*[HW] 0/1*/, const float* a /*[C,HW]*/, const float* b, int32_t C, int64_t HW, float* out,
                      madm_stream stream);
/* dacs_transforms.color_jitter (:41-59) = kornia.augmentation.ColorJitter.apply_transform (classic 0.6.x - 0.7.0 arithmetic: additive
 * brightness, multiplicative contrast, saturation / hue through HSV; the reference does not pin a kornia release) between denorm_ / renorm_.
 * in / out [B,3,HW] fp32; order [B][4] device int32 = permutation of (0 brightness, 1 contrast, 2 saturation, 3 hue); factors [B][4] device =
 * (brightness_factor - 1, contrast_factor, saturation_factor, hue_factor * 2 pi); mean / std: device [3] or both NULL. */
int madm_op_color_jitter(const float* in, int32_t B, int64_t HW, const int32_t* order, const float* factors, const float* mean, const float* stdv,
                         float* out, madm_stream stream);
int madm_op_gaussian_blur(const float* src /*[planes,H,W]*/, int32_t planes, int32_t H, int32_t W, int32_t ky, int32_t kx, float sigma_y,
                          float sigma_x, float* tmp /*scratch, same size*/, float* dst, madm_stream stream);
/* optimizer side of the training step (SURVEY §8 f-3).  Pointer tables are HOST arrays of n DEVICE pointers (fp32 tensors of numel[i]
 * elements); everything is enqueued on `stream`, nothing returns to the host.
 *   madm_op_ema_update : CMDISE._update_ema (modeling/meta_arch/cmdise.py:337-349): ema = alpha * ema + one_minus_alpha * param
 *   madm_op_grad_norm  : the global L2 norm torch.nn.utils.clip_grad_norm_ computes (engine/train_loop.py:123-124, :201-210) -> device scalar
 *   madm_op_adamw_step : one torch.optim.AdamW step (config_files/common/optim.py:9-18), step counted from 1; with grad_norm (device
 *                        scalar) and max_norm > 0 the gradients are scaled by min(max_norm / (norm + 1e-6), 1) first.
 *                        Hyper-parameters are doubles: torch derives 1 - beta, lr / (1 - beta1^t), ... in Python floats before casting */
int madm_op_ema_update(float* const* ema, const float* const* param, const int64_t* numel, int32_t n, float alpha, float one_minus_alpha,
                       madm_stream stream);
int madm_op_grad_norm_scratch_floats(int32_t n);
int madm_op_grad_norm(const float* const* grad, const int64_t* numel, int32_t n, float* scratch, float* out_norm, madm_stream stream);
int madm_op_adamw_step(float* const* param, const float* const* grad, float* const* exp_avg, float* const* exp_avg_sq, const int64_t* numel,
                       int32_t n, double lr, double beta1, double beta2, double eps, double weight_decay, int32_t step, const float* grad_norm,
                       float max_norm, madm_stream stream);
/* sliding-window merge of per-crop feature maps (reference feature_extractor.py:254-275: accumulate, divide by the count matrix):
 * feats [nwin*n, C, hf, wf] window-major, wins [nwin][2] = window origin (y1, x1) in feature pixels -> out [n, C, Hf, Wf] */
int madm_op_slide_merge(const float* feats, int32_t nwin, int32_t n, int32_t C, int32_t hf, int32_t wf, const int32_t* wins, int32_t Hf,
                        int32_t Wf, float* out, madm_stream stream);
int madm_op_upsample2x(const float* x, int32_t B, int32_t H, int32_t W, int32_t C, void* out_bf16, int32_t dtype,
                       madm_stream stream);
int madm_op_image_im2col(const float* img, int32_t B, int32_t H, int32_t W, void* out_bf16, int32_t* range_flag,
                         int32_t dtype, madm_stream stream);
int madm_op_gn_add_relu_nchw(const float* a, const float* ga, const float* ba, const float* s, const float* gs, const float* bs,
                             int32_t has_shortcut_norm, float eps, int32_t B, int32_t HW, int32_t C, float* stats_scratch,
                             float* out_nchw, madm_stream stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Training path (SURVEY §8 row f-3 / BASELINE config 5): the backward pass of madm_extract for the LoRA training step's trainable set
 *   - the active adapter's lora_A / lora_B factors on to_q / to_k / to_v / to_out.0 of all 32 attentions (mtmadise.py:115-147),
 *   - feature_projections.* (conv weights and GroupNorm affines of the four GN bottlenecks, feature_extractor.py:347-359),
 *   - the learned prompt / time conditioning, through d(cond_inputs) and d(cond_emb) (ldm_base.py:632-717: tiny tanh(alpha) * embed
 *     arithmetic that stays with the caller),
 * i.e. what `loss.backward()` produces in the reference's AMPTrainer.run_step (engine/train_loop.py:277-302) once the base UNet weights
 * are frozen, as BASELINE.json narrows config 5.  The VAE encoder runs without gradient (ldm_diffusers.py:282).
 * MADM_VARIANT_S0 (stages MADM_STAGE_ALL_S0): the VAE decoder runs without gradient too and its image is detached before it becomes the first
 * feature (ldm_diffusers.py:191-201), so d(s0) reaches feature_projections.0.* only; madm_backward_args.d_unet_sample, the gradient of
 * 'before_vae.decoder' (the UNet's final output, which the meta-arch's vae_decoder_loss differentiates), enters the UNet through the frozen
 * conv_out / conv_norm_out and joins the gradient of up layer 11's output.
 *
 * Protocol: madm_pack_dgrad_weights (after every parameter update / adapter switch, next to madm_pack_weights) -> madm_extract with
 * MADM_FLAG_TRAIN (keeps every activation the backward needs in the training workspace; B <= 8) -> madm_backward with the gradients of
 * the four feature maps.  Gradients are WRITTEN (not accumulated) into the buffers registered with madm_set_grad_tensors under the
 * parameters' names; parameters without a registered buffer get no gradient.  16-bit gradient tensors have the context's operand dtype;
 * with fp16 operands pass a loss_scale (the incoming gradients are multiplied by it, every output is divided by it again), with bf16 1.0.
 * ------------------------------------------------------------------------------------------------------------- */
#define MADM_FLAG_TRAIN 2
int madm_set_grad_tensors(madm_ctx* ctx, const madm_tensor* named, int32_t n); /* fp32 device buffers shaped like the parameters */
size_t madm_dgrad_packed_bytes(madm_ctx* ctx);
/* trainable_only != 0 repacks just what an optimizer step or an adapter switch can change (LoRA-folded linears, LoRA factors,
 * feature_projections convs) in an arena that was fully packed before */
int madm_pack_dgrad_weights(madm_ctx* ctx, void* packed_dgrad, const char* adapter, float lora_alpha_over_r, int32_t trainable_only,
                            madm_stream stream);
/* workspace of a MADM_FLAG_TRAIN forward + madm_backward at batch B with this adapter active (call after madm_set_grad_tensors) */
size_t madm_train_workspace_bytes(madm_ctx* ctx, int32_t B, const char* adapter);
typedef struct madm_backward_args {
  int32_t B;
  int32_t reserved;
  const float* dout[4];        /* gradients of out[0..3] (s2..s5), fp32 NCHW */
  const float* out[4];         /* the forward's outputs themselves (ReLU mask of the projections' last pass) */
  const float* cond_emb;       /* [B,1280]: the forward's cond_emb (time path SiLU backward) */
  float* d_cond_inputs;        /* [B,77,768] or NULL */
  float* d_cond_emb;           /* [B,1280] or NULL */
  const char* adapter;         /* active LoRA adapter of the forward ("" / NULL: none, no LoRA gradients) */
  float lora_alpha_over_r;
  float loss_scale;            /* > 0; 1.0 for bf16 operands */
  const void* packed;          /* forward arena (madm_pack_weights) */
  const void* packed_dgrad;    /* madm_pack_dgrad_weights arena */
  void* workspace;             /* the training workspace the MADM_FLAG_TRAIN forward ran in */
  size_t workspace_bytes;
  const float* d_unet_sample;  /* MADM_VARIANT_S0: gradient of madm_extract_args.unet_sample ('before_vae.decoder'), fp32 NCHW [B,4,64,64];
                                  NULL = no loss term on it (the UNet-output backward does no work) */
} madm_backward_args;
int madm_backward(madm_ctx* ctx, const madm_backward_args* args, madm_stream stream);
/* number of kernels one madm_backward call launches (after a MADM_FLAG_TRAIN forward at this B) */
int madm_backward_launch_count(madm_ctx* ctx, int32_t B);

/* ---- backward pass of the LoRA training step (SURVEY §8 row f-3), operator level.  "16" tensors have the operand dtype `dtype`. ---- */
/* GroupNorm(32)(+act) backward.  x = channel concat of x0 / x1 (fp32, or 16-bit if in16); stats = group sums [B,32,2] (sum, sum of squares)
 * of x; dy16 [B,HW,C] = gradient of act(GN(x)); scratch = madm_op_groupnorm_bwd_scratch_floats(B,HW,C) floats.  Any subset of outputs:
 * out16 [B,HW,C]; fp32 dx0 [B,HW,C0] / dx1 [B,HW,C1] (acc != 0: accumulated); `extra` fp32 [B,HW,C] is added to dx; dgamma / dbeta [C]. */
int madm_op_groupnorm_bwd_scratch_floats(int32_t B, int32_t HW, int32_t C);
int madm_op_groupnorm_bwd(const void* x0, int32_t C0, const void* x1, int32_t C1, int32_t B, int32_t HW, int32_t in16, const float* stats,
                          const float* gamma, const float* beta, float eps, int32_t act, const void* dy16, const float* extra, float* scratch,
                          void* out16, float* dx0, int32_t acc0, float* dx1, int32_t acc1, float* dgamma, float* dbeta, int32_t dtype,
                          madm_stream stream);
/* backward of z = GroupNorm(32)(conv1x1(x; w [C,3], no bias)) (-> ReLU if relu) on a 3-channel image, the K = 3 branches of the s0 projection
 * (feature_projections.0 conv1 with its ReLU, shortcut without), without materialising z or the conv output: img4 fp32 [B*HW][4] (3 used);
 * dy16 [B,HW,C] = gradient of the branch output.  Writes dw [C,3], dgamma [C], dbeta [C] (any may be NULL), multiplied by `scale`.  C % 32 == 0,
 * C <= 1024, C/8 divides 256; scratch = madm_op_c3_gn_bwd_scratch_floats(B, C) floats */
int64_t madm_op_c3_gn_bwd_scratch_floats(int32_t B, int32_t C);
int madm_op_c3_gn_bwd(const float* img4, const float* w, const float* gamma, const float* beta, float eps, int32_t relu, int32_t B, int32_t HW,
                      int32_t C, const void* dy16, float scale, float* dw, float* dgamma, float* dbeta, float* scratch, int32_t dtype, madm_stream stream);
int madm_op_layernorm_bwd(const float* x, int32_t M, int32_t C, const float* gamma, float eps, const void* dy16, float* dx, int32_t accumulate,
                          int32_t dtype, madm_stream stream);
/* GEGLU, natural column order: raw16 [M,2H] = (hidden | gate) -> out16 [M,H]; backward: draw16 [M,2H] */
int madm_op_geglu_fwd(const void* raw16, int64_t M, int32_t H, void* out16, int32_t dtype, madm_stream stream);
int madm_op_geglu_bwd(const void* raw16, const void* dout16, int64_t M, int32_t H, void* draw16, int32_t dtype, madm_stream stream);
/* softmax(Q K^T scale) V backward per (image, head): same addressing as madm_op_attention; scratch = madm_op_attention_bwd_scratch_floats(..) floats */
int64_t madm_op_attention_bwd_scratch_floats(int32_t B, int32_t heads, int32_t d, int32_t Nq, int32_t Nk);
int madm_op_attention_bwd(const void* q, int32_t ldq, const void* k, int32_t ldk, const void* v, int32_t ldv, const void* o, int32_t ldo,
                          const void* dout, int32_t lddo, void* dq, int32_t lddq, void* dk, int32_t lddk, void* dv, int32_t lddv, int32_t B,
                          int32_t heads, int32_t d, int32_t Nq, int32_t Nk, int64_t q_bs, int64_t kv_bs, int64_t o_bs, int64_t do_bs, int64_t dq_bs,
                          int64_t dkv_bs, float scale, float* scratch, int32_t dtype, madm_stream stream);
/* weight gradient dW[n,k] = alpha * sum_m dY[m,n] X[m,k]; taps = 9: implicit im2col of X [Bimg,H,W,K] -> PyTorch conv layout [N,K,3,3];
 * transpose_out != 0 (taps = 1): out[k,n].  scratch = madm_op_wgrad_scratch_floats(M,N,K,taps) floats */
int64_t madm_op_wgrad_scratch_floats(int32_t M, int32_t N, int32_t K, int32_t taps);
int madm_op_wgrad(const void* dy16, int32_t lda, const void* x16, int32_t ldb, int32_t M, int32_t N, int32_t K, int32_t taps, int32_t Bimg, int32_t H,
                  int32_t W, float alpha, float* out, int32_t transpose_out, float* scratch, int32_t dtype, madm_stream stream);
/* fused LoRA factor gradients of one rank-16 wrapped linear y = (W + s B A) x (the reference trains them through peft's Linear under autograd,
 * modeling/meta_arch/mtmadise.py:115-147): gB [N,16] = alpha dY^T (X A^T), gA [16,K] = alpha (dY B)^T X; a16 = A [16,K], bt16 = B^T [16,N] in the
 * operand dtype; N in {320,640,1280}, K in {320,640,768,1280}; scratch = madm_op_lora_grads_scratch_floats(M,N,K) floats; gA / gB may be null */
int64_t madm_op_lora_grads_scratch_floats(int32_t M, int32_t N, int32_t K);
int madm_op_lora_grads(const void* x16, int32_t ldx, const void* dy16, int32_t ldy, const void* a16, const void* bt16, int32_t M, int32_t N, int32_t K,
                       float alpha, float* gA, float* gB, float* scratch, int32_t dtype, madm_stream stream);
int madm_op_colsum_per_image(const void* x16, int32_t B, int32_t HW, int32_t C, float* out, int32_t ldo, int32_t dtype, madm_stream stream);
int madm_op_zero_stuff2x(const void* x16, int32_t B, int32_t h, int32_t w, int32_t C, void* out16, madm_stream stream);
int madm_op_sum2x2(const float* x, int32_t B, int32_t h, int32_t w, int32_t C, float* out, int32_t accumulate, madm_stream stream);
int madm_op_relu_bwd_nchw(const float* dout, const float* out, int32_t B, int32_t C, int32_t HW, float scale, void* dz16, int32_t dtype,
                          madm_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* MADM_B200_H_ */
