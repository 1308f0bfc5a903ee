// Host-side launchers of the non-GEMM kernels.  "_bf16" in a parameter name means "16-bit operand tensor": its element
// type is bf16 or fp16 according to the `fp16` flag (the compute dtype is a per-context runtime choice).
//  Every function enqueues on `st`, never synchronises, and returns
// nullptr on success or a static error string.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "gemm_tc.h"

namespace madm {

// ---- norm.cu
// GroupNorm(32) statistics are per-slab partial sums [B, slabs, 32, 2] (no atomics: deterministic, batch-size invariant);
// groupnorm_apply reduces them in fixed order, groupnorm_finalize produces [B,32,2] for gn_add_relu_nchw.
int groupnorm_slabs(int HW, int C);
// x0 / x1: fp32 NHWC, or 16-bit (dtype per `fp16`) when in16 != 0
const char* groupnorm_stats(const void* x0, int C0, const void* x1, int C1, int B, int HW, int in16, int fp16, float* partial,
                            cudaStream_t st);
const char* groupnorm_finalize(const float* partial, int B, int HW, int C, float* stats, cudaStream_t st);
// per-column statistics from a GEMM epilogue (GemmDesc::colstats, 32-row blocks) -> slab partials [B, S, 32, 2] with
// S = groupnorm_colstats_chunks(nblocks); feed groupnorm_apply(stats_slabs = S) or groupnorm_finalize_slabs
int groupnorm_colstats_chunks(int nblocks);
const char* groupnorm_finalize_slabs(const float* partial, int B, int slabs, float* stats, cudaStream_t st);
const char* groupnorm_colstats_reduce(const float* cs0, int C0, const float* cs1, int C1, int B, int nblocks, float* out, cudaStream_t st);
// stats_slabs: number of slabs behind `partial` (0 = the geometry of groupnorm_stats for this shape)
const char* groupnorm_apply(const void* x0, int C0, const void* x1, int C1, int B, int HW, int in16, const float* partial, int stats_slabs,
                            const float* gamma, const float* beta, float eps, int act, void* y_bf16, void* raw_bf16,
                            int fp16, cudaStream_t st);
const char* layernorm(const void* x, int in16 /* x is 16-bit (operand dtype) instead of fp32 */, int M, int C, const float* gamma, const float* beta,
                      float eps, void* y_bf16, int fp16, cudaStream_t st);
const char* softmax_rows(const float* s, int R, int L, void* p_bf16, int fp16, cudaStream_t st);
// out_fp16 != 0: out_nchw is an fp16 [B,C,HW] tensor (MADM_FLAG_OUT_FP16: halves the feature dict's bytes for host-bound consumers)
const char* gn_add_relu_nchw(const float* a, const float* stats_a, const float* ga, const float* ba, const float* s,
                             const float* stats_s, const float* gs, const float* bs, float eps, int B, int HW, int C,
                             float* out_nchw, cudaStream_t st, int out_fp16 = 0);

// 3-channel input of the s0 projection (SURVEY §8 a-11): image moments -> analytic GroupNorm statistics of its K = 3 1x1 convs
int image_moments_floats(int B);
const char* image_moments(const float* img4 /*[B*HW][4]*/, int B, int HW, float* partial /*image_moments_floats(B)*/, cudaStream_t st);
// coef[B][C][4] = (a0, a1, a2, d) with GN32(conv1x1(x; w [C][3]))_c = a . x + d
const char* c3_gn_coeffs(const float* mom, const float* w, const float* gamma, const float* beta, float eps, int B, int HW, int C, float* coef,
                         cudaStream_t st);
// out16[B*HW, C] = relu(a_c . x + d_c) in one pass
const char* c3_conv_gn_relu(const float* img4, const float* coef, int B, int HW, int C, void* out16, int fp16, cudaStream_t st);
// out NCHW = relu(GN(a; stats_a) + as_c . x + ds_c): the shortcut branch recomputed from the image
const char* gn_add_relu_nchw_c3(const float* a, const float* stats_a, const float* ga, const float* ba, const float* img4, const float* coef_s, float eps,
                                int B, int HW, int C, float* out_nchw, cudaStream_t st);
// backward of one such branch z = GN32(conv1x1(x; w [C][3])) (-> ReLU if relu) from the image, its moments `mom` and the forward's `coef` (ReLU
// mask): dy16 [B*HW, C] = gradient of the branch output -> dw [C][3], dgamma / dbeta [C] (each may be null), written, times `scale`.
// Scratch: partial = c3_gn_bwd_scratch_floats(B, C) floats.
size_t c3_gn_bwd_scratch_floats(int B, int C);
const char* c3_gn_bwd(const float* img4, const float* mom, const float* coef, const float* w, const float* gamma, float eps, int relu, int B, int HW,
                      int C, const void* dy16, int fp16, float scale, float* dw, float* dgamma, float* dbeta, float* partial, cudaStream_t st);

// ---- attention_tc.cu : O[b, i, h*d:(h+1)*d] = softmax(Q K^T * scale) V per (image, head); 16-bit in/out, fp32 softmax, on tcgen05 / TMEM
// (prepared launch: TMA tensor maps encoded once)
struct FaLaunch {
  alignas(64) unsigned char params[512];
  int d = 0;
  int nqt = 1;  // query tiles (128 rows) per CTA
  dim3 grid;
};
const char* flash_attention_tc_prepare(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o, int ldo, int B,
                                       int heads, int d, int Nq, int Nk, long q_bstride, long kv_bstride, long o_bstride, float scale,
                                       int fp16, FaLaunch* out, float* lse = nullptr /* optional [B,heads,Nq] log-sum-exp output */);
const char* flash_attention_tc_launch(const FaLaunch& l, cudaStream_t st);
// tensor map of the [d, heads, tokens, batch] view of a 16-bit [batch, tokens, ld] buffer whose head h occupies columns [h*d, (h+1)*d):
// box = 64 columns (zero-filled past d) x box_rows tokens; errors start with `op`
const char* attention_head_map(CUtensorMap* tm, const char* op, const void* ptr, int d, int heads, int ntok, int B, int ld, long bstride, int box_rows);

// ---- elementwise.cu
// img NCHW fp32 in [0,1] -> (img-0.5)/0.5 -> 3x3 im2col rows [B*H*W, 64] bf16 (27 real columns, tap-major (ky,kx,c))
// normalised != 0: img already is in [-1,1] (no (img-0.5)/0.5)
const char* image_im2col(const float* img, int B, int H, int W, void* out_bf16, int* range_flag, int fp16, cudaStream_t st, int normalised = 0);
// noisy[b,p,:] = sqrt(ac[t_b])*lat[b,p,:] + sqrt(1-ac[t_b])*noise[:,p]  (latents NHWC fp32 [B*HW,4], noise NCHW [4,HW])
const char* qsample(const float* lat, const float* noise_nchw, const int64_t* t, const float* alphas_cumprod, int B, int HW,
                    float* noisy_nhwc, float* noisy_nchw_or_null, cudaStream_t st);
// noisy NHWC fp32 [B,H,W,4] -> 3x3 im2col rows [B*H*W, 64] bf16 (36 real columns, tap-major)
const char* latent_im2col(const float* noisy_nhwc, int B, int H, int W, void* out_bf16, int fp16, cudaStream_t st);
// t[B] -> [B,320] bf16 sinusoid (cos | sin), diffusers Timesteps(320, flip_sin_to_cos=True, shift 0)
const char* timestep_sinusoid(const int64_t* t, int B, void* out_bf16, int fp16, cudaStream_t st);
// generic fp32 -> bf16 with optional SiLU and per-row add (emb + cond_emb)
const char* f32_to_bf16(const float* x, const float* add_or_null, long n, int act, void* y_bf16, float* y_f32_or_null,
                        int fp16, cudaStream_t st);
// fp32 NHWC [B,H,W,C] -> 4 stride-2 phase images bf16 [4][B][H/2][W/2][C]; phase = (y&1)*2 + (x&1)
const char* space_to_depth(const float* x, int B, int H, int W, int C, void* out_bf16, int fp16, cudaStream_t st);
// fp32 NHWC [B,H,W,C] -> nearest 2x bf16 [B,2H,2W,C]
const char* upsample_nearest2x(const float* x, int B, int H, int W, int C, void* out_bf16, int fp16, cudaStream_t st);
// fp32 planes [planes,Hs,Ws] -> bilinear (align_corners=False, no antialias) to Hr x Wr, written into the top-left corner of zero-filled
// [planes,Hd,Wd] planes (Hd >= Hr, Wd >= Wr): T.Resize + ImageList.from_tensors padding of FeatureExtractorBackbone.preprocess_image
const char* resize_bilinear_nchw(const float* src, int planes, int Hs, int Ws, int Hr, int Wr, int Hd, int Wd, float* dst, cudaStream_t st);
// 16-bit NHWC [B,H,W,C] -> nearest 2x 16-bit [B,2H,2W,C] (the VAE decoder's 16-bit stream)
const char* upsample_nearest2x_16(const void* x16, int B, int H, int W, int C, void* out16, cudaStream_t st);
// VAE decoder entry: z = post_quant_conv(sample * inv_scale), a 1x1 conv 4 -> 4 in fp32 (ldm_diffusers.py:319-320); NHWC [M,4]
const char* post_quant_conv(const float* sample, const float* w /*[4,4]*/, const float* bias /*[4]*/, float inv_scale, long M, float* z,
                            cudaStream_t st);
// decoder image fp32 NHWC [B*HW, 4] (3 real channels) -> 16-bit operand rows [B*HW, 64] (zero padded) for the s0 projection's 1x1
// convs, and optionally clip(x, -1, 1) ('after_vae.decoder') and x itself as fp32 NCHW [B,3,HW]
const char* decoder_image_pack(const float* img4, int B, int HW, void* rows16, float* clipped_nchw_or_null, float* raw_nchw_or_null, int fp16,
                               cudaStream_t st);
// split-K: out = act(sum_s partial[s] + bias + rowbias + residual), partial[s] = part + s*split_stride, each [M,N] fp32
const char* splitk_reduce(const float* part, int splits, long split_stride, int M, int N, const float* bias, const float* rowbias,
                          int rows_per_img, int ld_rowbias, const float* residual, int ldr, float* out32, int ldo32, void* out16, int ldo16,
                          int act, int fp16, cudaStream_t st, int res16 = 0);
// fp32 NHWC [B,HW,C] -> NCHW fp32 [B,C,HW]
const char* nhwc_to_nchw(const float* x, int B, int HW, int C, float* out, cudaStream_t st);
const char* nhwc_to_nchw_strided(const float* x, int B, int HW, int C, int ld, float* out, cudaStream_t st);

// ---- head.cu (DAFormer head stage, SURVEY §8 f-2)
// fp32 NCHW [B,C,HW] -> 16-bit NHWC [B,HW,C]
const char* nchw_to_nhwc16(const float* x, int B, int C, int HW, void* out16, int fp16, cudaStream_t st);
// bilinear resize (align_corners=False) of 16-bit NHWC [B,Hs,Ws,C] -> [B,Hd,Wd,C] written with channel pitch ldd
const char* bilinear_resize_nhwc16(const void* src, int B, int Hs, int Ws, int C, void* dst, int Hd, int Wd, int ldd, int fp16, cudaStream_t st);
// depthwise 3x3 conv, dilation = padding = dil, + shift + ReLU; w9 fp32 [9][C] (BatchNorm scale folded), shift fp32 [C]
const char* depthwise3x3_nhwc16(const void* src, int B, int H, int W, int C, int dil, const float* w9, const float* shift, void* dst, int fp16,
                                cudaStream_t st);
// eval-mode BatchNorm -> out[0..N) = scale, out[N..2N) = shift (conv_bias optional)
const char* bn_fold(const float* gamma, const float* beta, const float* mean, const float* var, const float* conv_bias, float eps, int N,
                    float* out, cudaStream_t st);
// depthwise weight [C,1,3,3] * scale[c] -> fp32 [9][C]
const char* pack_depthwise(const float* w, const float* scale, int C, float* out, cudaStream_t st);

// ---- teacher.cu (teacher post-processing + DACS mixing, SURVEY §8 f-4)
// logits [B,C,h,w] fp32 NCHW -> bilinear (align_corners=False) to HxW -> softmax max / argmax -> label int64, prob fp32 [B,H,W];
// count (device int scratch) = #pixels with prob >= threshold; weight (optional) = count/pixels, 0 in the top ignore_top rows
const char* pseudo_labels(const float* logits, int B, int C, int h, int w, int H, int W, float threshold, int ignore_top, int64_t* label,
                          float* prob, float* weight, int* count, cudaStream_t st);
const char* class_mask(const int64_t* label, long n, const int64_t* classes, int k, int64_t* mask, cudaStream_t st);
const char* one_mix(const int64_t* mask, long n, const int64_t* la, const int64_t* lb, int64_t* lout, const float* wa, const float* wb,
                    float* wout, cudaStream_t st);

// sliding-window merge: feats [nwin*n,C,hf,wf] (window-major), wins [nwin][2] = (y1,x1) in feature pixels -> out [n,C,Hf,Wf] = mean over covering windows
const char* slide_merge(const float* feats, int nwin, int n, int C, int hf, int wf, const int* wins, int Hf, int Wf, float* out, cudaStream_t st);

// ---- optim.cu (optimizer side of the training step, SURVEY §8 f-3; image side of the DACS mixing, f-4)
// Pointer tables are HOST arrays of n device pointers.  ema = wa * ema + wb * param   (wa = alpha, wb = 1 - alpha)
const char* ema_update(float* const* ema, const float* const* param, const long* numel, int n, float wa, float wb, cudaStream_t st);
int grad_norm_scratch_floats(int n);
// out_norm (device scalar) = sqrt(sum over all tensors of g^2); partial: device scratch of grad_norm_scratch_floats(n) floats
const char* grad_norm(const float* const* grad, const long* numel, int n, float* partial, float* out_norm, cudaStream_t st);
// torch.optim.AdamW step `step` (>= 1) on n tensors; grad_norm_dev (device scalar or null) + max_norm > 0: clip_grad_norm_ folded in
const char* adamw_step(float* const* param, const float* const* grad, float* const* exp_avg, float* const* exp_avg_sq, const long* numel, int n,
                       double lr, double beta1, double beta2, double eps, double weight_decay, int step, const float* grad_norm_dev, float max_norm,
                       cudaStream_t st);
// out[c, i] = mask[i] * a[c, i] + (1 - mask[i]) * b[c, i]
const char* image_mix(const int64_t* mask, const float* a, const float* b, int C, long HW, float* out, cudaStream_t st);
// kornia ColorJitter.apply_transform on [B,3,HW] fp32: order [B][4] = permutation of (0 brightness, 1 contrast, 2 saturation, 3 hue),
// factors [B][4] = (brightness_factor - 1, contrast_factor, saturation_factor, hue_factor * 2 pi); mean / std [3] or null (denorm_ / renorm_)
const char* color_jitter(const float* in, int B, long HW, const int* order, const float* factors, const float* mean, const float* stdv, float* out,
                         cudaStream_t st);
// separable Gaussian blur of `planes` HxW fp32 planes, reflect border; tmp: scratch of the same size (may not alias src / dst)
const char* gaussian_blur(const float* src, int planes, int H, int W, int ky, int kx, float sigma_y, float sigma_x, float* tmp, float* dst,
                          cudaStream_t st);

// ---- backward.cu (SURVEY §8 row f-3: backward of the HBM-bound layers; 16-bit gradients have the context's operand dtype)
// GroupNorm(32)(+act) backward.  x = channel concat of x0 / x1 (fp32, or 16-bit if in16); stats = the forward's finalised group sums
// [B,32,2] (sum, sum of squares); dy16 [B,HW,C] = gradient of act(GN(x)).  Scratch: partial [B][groupnorm_bwd_slabs(HW)][C][2], coef
// [B][32][2], chan [B][C][2] (only for affine gradients).  Outputs (any subset): out16 [B,HW,C]; fp32 dx0 [B,HW,C0] / dx1 [B,HW,C1], each
// stored or accumulated; `extra` (fp32 [B,HW,C]) is added to dx; dgamma / dbeta [C] = affine_scale * sums over (B, HW).
int groupnorm_bwd_slabs(int HW);
const char* groupnorm_bwd(const void* x0, int C0, const void* x1, int C1, int B, int HW, int in16, const float* stats, const float* gamma,
                          const float* beta, float eps, int act, const void* dy16, int fp16, float* partial, float* coef, float* chan,
                          const float* extra, void* out16, float* dx0, int acc0, float* dx1, int acc1, float* dgamma, float* dbeta,
                          float affine_scale, cudaStream_t st);
// LayerNorm backward over rows of x fp32 [M,C] (statistics recomputed): dx stored or accumulated (fp32)
const char* layernorm_bwd(const float* x, int M, int C, const float* gamma, float eps, const void* dy16, int fp16, float* dx, int accumulate,
                          cudaStream_t st, void* dx16 = nullptr /* optional 16-bit copy of the updated dx */);
// GEGLU in natural column order: raw16 [M, 2H] = (hidden | gate) -> out16 [M,H] = hidden * gelu(gate); backward -> draw16 [M, 2H]
const char* geglu_fwd(const void* raw16, long M, int H, void* out16, int fp16, cudaStream_t st);
const char* geglu_bwd(const void* raw16, const void* dout16, long M, int H, void* draw16, int fp16, cudaStream_t st);
// out[b * ldo + c] = sum over the pixels of image b of x16[b, :, c]   (gradient of a per-image row bias: time_emb_proj)
const char* colsum_per_image(const void* x16, int B, int HW, int C, int fp16, float* out, int ldo, cudaStream_t st);
// 16-bit [B,h,w,C] -> [B,2h,2w,C], values at even positions, zeros elsewhere (operand of a stride-2 conv's input gradient)
const char* zero_stuff2x(const void* x16, int B, int h, int w, int C, void* out16, cudaStream_t st);
// fp32 [B,2h,2w,C] -> [B,h,w,C]: 2x2 block sums (backward of nearest-2x upsampling), stored or accumulated
const char* sum2x2(const float* x, int B, int h, int w, int C, float* out, int accumulate, cudaStream_t st);
// dz16 [B,HW,C] = scale * dout[b,c,p] * (out[b,c,p] > 0): ReLU backward of the projections' last pass + NCHW -> NHWC
const char* relu_bwd_nchw_to_nhwc16(const float* dout, const float* out, int B, int C, int HW, float scale, void* dz16, int fp16, cudaStream_t st);
const char* scale_copy_f32(const float* src, long n, float scale, float* dst, cudaStream_t st);
const char* temb_silu_bwd(const float* d_act, const float* emb, const float* cond_emb, long n, float scale, float* d_cond_emb, cudaStream_t st);

// ---- attention_bwd.cu: gradients of softmax(Q K^T scale) V per (image, head); scratch = attention_bwd_scratch_floats(B, heads, d, Nq, Nk) floats
// (prepared launch: shapes checked, parameter blocks filled and tensor maps encoded once)
struct AttnBwdLaunch {
  alignas(64) unsigned char tc[2][640];   // tcgen05 roles (dK / dV, then dQ) when attention_bwd_tc_supported: parameter blocks, tensor maps encoded
  alignas(64) unsigned char params[256];  // parameter block of the warp-level kernels, query split included
  dim3 gq, gk, gtc[2];                    // grids: query blocks, key blocks x query split, the two tcgen05 roles
  int B = 0;
  int fp16 = 0, dp = 0;                   // dispatch: operand dtype, head dim padded to a multiple of 16
  bool have_lse = false;                  // the forward's log-sum-exp is given: the L / D pass only computes D
};
size_t attention_bwd_scratch_floats(int B, int heads, int d, int Nq, int Nk);
const char* attention_bwd_prepare(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, const void* o, int ldo, const void* dout,
                                  int lddo, void* dq, int lddq, void* dk, int lddk, void* dv, int lddv, int B, int heads, int d, int Nq, int Nk, long q_bs,
                                  long k_bs, long v_bs, long o_bs, long do_bs, long dq_bs, long dk_bs, long dv_bs, float scale, float* scratch, int fp16,
                                  AttnBwdLaunch* out,
                                  const float* lse = nullptr /* [B,heads,Nq] from the forward kernel: skips the backward's own Q K^T pass */);
const char* attention_bwd_launch(const AttnBwdLaunch& l, cudaStream_t st);

// fused LoRA factor gradients of one rank-16 wrapped linear (wgrad.cu): gB [N,16] = alpha dY^T (X A^T), gA [16,K] = alpha (dY B)^T X;
// a16 = lora_A [16,K], bt16 = lora_B^T [16,N] in the operand dtype; scratch = lora_grads_scratch_floats(M, N, K) floats
bool lora_grads_supported(int N, int K);
size_t lora_grads_scratch_floats(int M, int N, int K);
const char* lora_grads(const void* x16, int ldx, const void* dy16, int ldy, const void* a16, const void* bt16, int M, int N, int K, float alpha, float* gA,
                       float* gB, float* scratch, int fp16, cudaStream_t st);

// ---- attention_bwd_tc.cu: the same gradients on tcgen05 / TMEM for d = 40 / 80 and token counts that are multiples of 128 (the UNet's 64x64 and
// 32x32 self-attention); attention_bwd_launch hands over to it after its L / D pass.  L2 = log-sum-exp * log2(e), D = rowsum(dO * O), both
// [B, heads, Nq].  The prepare fills AttnBwdLaunch::tc and ::gtc.
bool attention_bwd_tc_supported(int d, int Nq, int Nk);
const char* attention_bwd_tc_prepare(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, const void* dout, int lddo, void* dq,
                                     int lddq, void* dk, int lddk, void* dv, int lddv, int B, int heads, int d, int Nq, int Nk, long q_bs, long k_bs,
                                     long v_bs, long do_bs, long dq_bs, long dk_bs, long dv_bs, float scale, const float* L2, const float* D,
                                     AttnBwdLaunch* out);
const char* attention_bwd_tc_launch(const AttnBwdLaunch& l, cudaStream_t st);

// ---- wgrad.cu: dW[n,k] = alpha * sum_m dY[m,n] X[m,k] (taps = 9: implicit im2col of X [Bimg,H,W,K]) -> out[n*so_n + k*so_k + tap*so_tap]
int wgrad_splits(int M, int N, int K, int taps);
size_t wgrad_scratch_floats(int M, int N, int K, int taps);
const char* wgrad(const void* dy16, int lda, const void* x16, int ldb, int M, int N, int K, int taps, int Bimg, int H, int W, float alpha,
                  float* out, long so_n, long so_k, long so_tap, float* scratch, int fp16, cudaStream_t st);

// ---- pack.cu (weight packing; fp32 PyTorch layouts -> bf16 K-major GEMM operands)
// conv weight [N, C, kh, kw] fp32 -> [N, kh*kw*Cpad] bf16 with K index = tap*Cpad + c (zero fill for c >= C)
const char* pack_conv_weight(const float* w, int N, int C, int taps, int Cpad, int Kpad, int ldo, void* out_bf16, int fp16,
                             cudaStream_t st, const float* row_scale = nullptr);
// linear weight [N, K] (+ LoRA: + scale * B[N,r] @ A[r,K]) -> bf16 [N, K] written at row offset / interleave
const char* pack_linear_weight(const float* w, int N, int K, const float* lora_a, const float* lora_b, int r, float scale,
                               int ldo, void* out_bf16, int fp16, cudaStream_t st);
// dgrad operands (SURVEY §8 f-3): conv weight [Cout, Cin, kh, kw] -> [Cin, taps*CoPad] with mirrored taps; linear (+ LoRA) -> its transpose [K, N]
const char* pack_conv_dgrad_weight(const float* w, int Cout, int Cin, int taps, int CoPad, int Kpad, int ldo, void* out_bf16, int fp16,
                                   cudaStream_t st);
const char* pack_linear_dgrad_weight(const float* w, int N, int K, const float* lora_a, const float* lora_b, int r, float scale, int ldo,
                                     void* out_bf16, int fp16, cudaStream_t st);
// many linears in one launch: out = 16-bit(w + scale * lb la) as [N, ldo] rows (transpose = 0) or transposed [K, ldo] rows (transpose = 1);
// la = null: plain conversion.  r <= 16.
struct LoraPackEntry { const float* w; const float* la; const float* lb; void* out; int N, K, r, ldo; };
constexpr int kLoraPackMax = 48;
struct LoraPackTable { LoraPackEntry e[kLoraPackMax]; int n; float scale; int transpose; int fp16; };
const char* pack_lora_multi(const LoraPackEntry* entries, int n, float scale, int transpose, int fp16, cudaStream_t st);
// GEGLU: rows of W[8C, C] reordered so each 128-row tile holds 64 value rows then their 64 gate rows (bias likewise)
const char* pack_geglu_weight(const float* w, const float* bias, int C4 /* = 4C */, int K, void* out_bf16, float* out_bias,
                              int fp16, cudaStream_t st);
// fold quant_conv(8->8, 1x1) and the 0.18215 scale into conv_out(512->8, 3x3): rows 0..3 of the product, N padded to 16
const char* pack_vae_latent_head(const float* w_out /*[8,512,3,3]*/, const float* b_out, const float* w_q /*[8,8]*/,
                                 const float* b_q, float scale, int C, void* out_bf16 /*[16, 9*C]*/, float* out_bias /*[16]*/,
                                 int fp16, cudaStream_t st);

}  // namespace madm
