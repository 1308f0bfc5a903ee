// C-ABI operator-level entry points (include/madm_b200.h, "Operator-level entry points"): thin adapters from the POD
// argument structs to the kernel launchers, used by the parity tests and by nothing else in the product path.
#include "../../include/madm_b200.h"
#include "api_internal.h"
#include "kernels.h"

#include <string.h>

using namespace madm;

namespace madm {
static thread_local char g_err[512] = "";
void set_global_error(const char* msg) {
  strncpy(g_err, msg ? msg : "", sizeof(g_err) - 1);
  g_err[sizeof(g_err) - 1] = 0;
}
const char* global_error() { return g_err; }
}  // namespace madm

static int fail(const char* e) {
  set_global_error(e);
  return MADM_EINVAL;
}
#define RUN(expr)                      \
  do {                                 \
    const char* _e = (expr);           \
    if (_e) return fail(_e);           \
    return MADM_OK;                    \
  } while (0)

extern "C" {

int madm_op_gemm(const madm_gemm_args* a, madm_stream stream) {
  if (!a) return fail("madm_op_gemm: null args");
  GemmDesc d;
  d.nseg = a->nseg;
  for (int s = 0; s < 2; ++s) {
    const madm_gemm_seg& g = a->seg[s];
    GemmASeg& t = d.seg[s];
    t.ptr = g.a; t.Bt = g.Bt; t.H = g.H; t.W = g.W; t.C = g.C; t.ld = g.ld; t.ntaps = g.ntaps;
    for (int i = 0; i < 9; ++i) { t.dx[i] = g.dx[i]; t.dy[i] = g.dy[i]; t.b_off[i] = g.b_off[i]; }
  }
  d.M = a->M; d.N = a->N; d.w = a->w; d.Nw = a->Nw; d.ldw = a->ldw;
  d.bias = a->bias; d.rowbias = a->rowbias; d.rows_per_img = a->rows_per_img; d.ld_rowbias = a->ld_rowbias;
  d.residual = a->residual; d.ldr = a->ldr;
  d.out_f32 = a->out_f32; d.ldo32 = a->ldo32; d.out_bf16 = a->out_bf16; d.ldo16 = a->ldo16;
  d.act = a->act; d.alpha = a->alpha; d.bn = a->bn; d.fp16 = a->dtype == MADM_DTYPE_FP16;
  if (a->colstats && a->stat_rows != 0 && a->stat_rows != 32) return fail("gemm: stat_rows must be 32");
  d.colstats = a->colstats; d.mt = a->mt; d.s2d_H = a->s2d_H; d.s2d_W = a->s2d_W; d.pair = a->pair; d.res16 = a->res16;
  GemmLaunch L;
  if (const char* e = gemm_prepare(d, &L)) return fail(e);
  RUN(gemm_launch(L, static_cast<cudaStream_t>(stream)));
}

int madm_op_groupnorm(const void* x0, int32_t C0, const void* x1, int32_t C1, int32_t B, int32_t HW, int32_t in16, const float* gamma,
                      const float* beta, float eps, int32_t act, float* stats, void* y, void* raw, int32_t dtype, madm_stream stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int f16 = dtype == MADM_DTYPE_FP16;
  if (const char* e = groupnorm_stats(x0, C0, x1, C1, B, HW, in16, f16, stats, st)) return fail(e);
  RUN(groupnorm_apply(x0, C0, x1, C1, B, HW, in16, stats, 0, gamma, beta, eps, act, y, raw, f16, st));
}

int madm_op_layernorm(const void* x, int32_t in16, int32_t M, int32_t C, const float* gamma, const float* beta, float eps, void* y,
                      int32_t dtype, madm_stream stream) {
  RUN(layernorm(x, in16, M, C, gamma, beta, eps, y, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_softmax_rows(const float* s, int32_t R, int32_t L, void* p, int32_t dtype, madm_stream stream) {
  RUN(softmax_rows(s, R, L, p, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_attention(const void* q, int32_t ldq, const void* k, int32_t ldk, const void* v, int32_t ldv, void* o, int32_t ldo,
                      int32_t B, int32_t heads, int32_t d, int32_t Nq, int32_t Nk, int64_t q_bs, int64_t kv_bs, int64_t o_bs,
                      float scale, int32_t dtype, int32_t impl, madm_stream stream) {
  if (impl != 0) return fail("madm_op_attention: impl must be 0 (the mma.sync kernel of round 1 was removed from the library)");
  FaLaunch L;
  if (const char* e = flash_attention_tc_prepare(q, ldq, k, ldk, v, ldv, o, ldo, B, heads, d, Nq, Nk, q_bs, kv_bs, o_bs, scale,
                                                 dtype == MADM_DTYPE_FP16, &L))
    return fail(e);
  RUN(flash_attention_tc_launch(L, static_cast<cudaStream_t>(stream)));
}

int madm_op_pack_linear(const float* w, int32_t N, int32_t K, const float* la, const float* lb, int32_t r, float scale, void* out,
                        int32_t ldo, int32_t dtype, madm_stream stream) {
  RUN(pack_linear_weight(w, N, K, la, lb, r, scale, ldo ? ldo : K, out, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_pack_conv(const float* w, int32_t N, int32_t C, int32_t taps, int32_t Cpad, void* out, int32_t ldo, int32_t dtype,
                      madm_stream stream) {
  const int Kpad = taps * Cpad;
  RUN(pack_conv_weight(w, N, C, taps, Cpad, Kpad, ldo ? ldo : Kpad, out, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_pack_conv_dgrad(const float* w, int32_t Cout, int32_t Cin, int32_t taps, int32_t CoPad, void* out, int32_t ldo, int32_t dtype,
                            madm_stream stream) {
  const int Kpad = taps * CoPad;
  RUN(pack_conv_dgrad_weight(w, Cout, Cin, taps, CoPad, Kpad, ldo ? ldo : Kpad, out, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_pack_linear_dgrad(const float* w, int32_t N, int32_t K, const float* lora_a, const float* lora_b, int32_t r, float scale, void* out,
                              int32_t ldo, int32_t dtype, madm_stream stream) {
  RUN(pack_linear_dgrad_weight(w, N, K, lora_a, lora_b, r, scale, ldo ? ldo : N, out, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_pack_geglu(const float* w, const float* bias, int32_t C4, int32_t K, void* out, float* out_bias, int32_t dtype,
                       madm_stream stream) {
  RUN(pack_geglu_weight(w, bias, C4, K, out, out_bias, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_space_to_depth(const float* x, int32_t B, int32_t H, int32_t W, int32_t C, void* out, int32_t dtype, madm_stream stream) {
  RUN(space_to_depth(x, B, H, W, C, out, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_upsample2x(const float* x, int32_t B, int32_t H, int32_t W, int32_t C, void* out, int32_t dtype, madm_stream stream) {
  RUN(upsample_nearest2x(x, B, H, W, C, out, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_nchw_to_nhwc16(const float* x, int32_t B, int32_t C, int32_t HW, void* out, int32_t dtype, madm_stream stream) {
  RUN(nchw_to_nhwc16(x, B, C, HW, out, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_bilinear_resize(const void* src, int32_t B, int32_t Hs, int32_t Ws, int32_t C, void* dst, int32_t Hd, int32_t Wd, int32_t ldd,
                            int32_t dtype, madm_stream stream) {
  RUN(bilinear_resize_nhwc16(src, B, Hs, Ws, C, dst, Hd, Wd, ldd, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_depthwise3x3(const void* src, int32_t B, int32_t H, int32_t W, int32_t C, int32_t dilation, const float* w9, const float* shift,
                         void* dst, int32_t dtype, madm_stream stream) {
  RUN(depthwise3x3_nhwc16(src, B, H, W, C, dilation, w9, shift, dst, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_pseudo_labels(const float* logits, int32_t B, int32_t C, int32_t h, int32_t w, int32_t H, int32_t W, float threshold,
                          int32_t ignore_top, int64_t* label, float* prob, float* weight, int32_t* count, madm_stream stream) {
  RUN(pseudo_labels(logits, B, C, h, w, H, W, threshold, ignore_top, label, prob, weight, count, static_cast<cudaStream_t>(stream)));
}

int madm_op_class_mask(const int64_t* label, int64_t n, const int64_t* classes, int32_t k, int64_t* mask, madm_stream stream) {
  RUN(class_mask(label, long(n), classes, k, mask, static_cast<cudaStream_t>(stream)));
}

int madm_op_one_mix(const int64_t* mask, int64_t n, const int64_t* label_a, const int64_t* label_b, int64_t* label_out, const float* weight_a,
                    const float* weight_b, float* weight_out, madm_stream stream) {
  RUN(one_mix(mask, long(n), label_a, label_b, label_out, weight_a, weight_b, weight_out, static_cast<cudaStream_t>(stream)));
}

int madm_op_ema_update(float* const* ema, const float* const* param, const int64_t* numel, int32_t n, float alpha, float one_minus_alpha,
                       madm_stream stream) {
  if (!ema || !param || !numel || n < 1) return fail("madm_op_ema_update: null argument");
  RUN(ema_update(ema, param, reinterpret_cast<const long*>(numel), n, alpha, one_minus_alpha, static_cast<cudaStream_t>(stream)));
}

int madm_op_grad_norm_scratch_floats(int32_t n) { return grad_norm_scratch_floats(n); }

int madm_op_grad_norm(const float* const* grad, const int64_t* numel, int32_t n, float* scratch, float* out_norm, madm_stream stream) {
  if (!grad || !numel || !scratch || !out_norm || n < 1) return fail("madm_op_grad_norm: null argument");
  RUN(grad_norm(grad, reinterpret_cast<const long*>(numel), n, scratch, out_norm, static_cast<cudaStream_t>(stream)));
}

int madm_op_adamw_step(float* const* param, const float* const* grad, float* const* exp_avg, float* const* exp_avg_sq, const int64_t* numel,
                       int32_t n, double lr, double beta1, double beta2, double eps, double weight_decay, int32_t step, const float* grad_norm,
                       float max_norm, madm_stream stream) {
  if (!param || !grad || !exp_avg || !exp_avg_sq || !numel || n < 1) return fail("madm_op_adamw_step: null argument");
  RUN(adamw_step(param, grad, exp_avg, exp_avg_sq, reinterpret_cast<const long*>(numel), n, lr, beta1, beta2, eps, weight_decay, step, grad_norm,
                 max_norm, static_cast<cudaStream_t>(stream)));
}

int madm_op_preprocess_image(const float* src, int32_t planes, int32_t Hs, int32_t Ws, int32_t Hr, int32_t Wr, int32_t Hd, int32_t Wd, float* dst,
                             madm_stream stream) {
  if (!src || !dst) return fail("madm_op_preprocess_image: null argument");
  RUN(resize_bilinear_nchw(src, planes, Hs, Ws, Hr, Wr, Hd, Wd, dst, static_cast<cudaStream_t>(stream)));
}

int madm_op_image_mix(const int64_t* mask, const float* a, const float* b, int32_t C, int64_t HW, float* out, madm_stream stream) {
  if (!mask || !a || !b || !out) return fail("madm_op_image_mix: null argument");
  RUN(image_mix(mask, a, b, C, long(HW), out, static_cast<cudaStream_t>(stream)));
}

int madm_op_color_jitter(const float* in, int32_t B, int64_t HW, const int32_t* order, const float* factors, const float* mean, const float* stdv,
                         float* out, madm_stream stream) {
  if (!in || !order || !factors || !out) return fail("madm_op_color_jitter: null argument");
  RUN(color_jitter(in, B, long(HW), order, factors, mean, stdv, out, static_cast<cudaStream_t>(stream)));
}

int madm_op_gaussian_blur(const float* src, int32_t planes, int32_t H, int32_t W, int32_t ky, int32_t kx, float sigma_y, float sigma_x, float* tmp,
                          float* dst, madm_stream stream) {
  if (!src || !tmp || !dst) return fail("madm_op_gaussian_blur: null argument");
  RUN(gaussian_blur(src, planes, H, W, ky, kx, sigma_y, sigma_x, tmp, dst, static_cast<cudaStream_t>(stream)));
}

int madm_op_slide_merge(const float* feats, int32_t nwin, int32_t n, int32_t C, int32_t hf, int32_t wf, const int32_t* wins, int32_t Hf, int32_t Wf,
                        float* out, madm_stream stream) {
  RUN(slide_merge(feats, nwin, n, C, hf, wf, wins, Hf, Wf, out, static_cast<cudaStream_t>(stream)));
}

int madm_op_image_im2col(const float* img, int32_t B, int32_t H, int32_t W, void* out, int32_t* range_flag, int32_t dtype,
                         madm_stream stream) {
  RUN(image_im2col(img, B, H, W, out, range_flag, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

int madm_op_groupnorm_from_colstats(const void* x, int32_t C, int32_t B, int32_t HW, int32_t in16, const float* colstats, int32_t stat_rows,
                                    const float* gamma, const float* beta, float eps, int32_t act, float* scratch /*[B,32 chunks,32,2]*/, void* y,
                                    int32_t dtype, madm_stream stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int f16 = dtype == MADM_DTYPE_FP16;
  if (HW % stat_rows != 0) return fail("groupnorm_from_colstats: HW must be a multiple of stat_rows");
  if (stat_rows != 32) return fail("groupnorm_from_colstats: stat_rows must be 32");
  const int nb = HW / stat_rows;
  if (const char* e = groupnorm_colstats_reduce(colstats, C, nullptr, 0, B, nb, scratch, st)) return fail(e);
  RUN(groupnorm_apply(x, C, nullptr, 0, B, HW, in16, scratch, groupnorm_colstats_chunks(nb), gamma, beta, eps, act, y, nullptr, f16, st));
}

int madm_op_groupnorm_scratch_floats(int32_t B, int32_t HW, int32_t C) {
  return int(size_t(2) * B * groupnorm_slabs(HW, C) * 64 + size_t(2) * B * 64);
}

int madm_op_gn_add_relu_nchw(const float* a, const float* ga, const float* ba, const float* s, const float* gs, const float* bs,
                             int32_t has_shortcut_norm, float eps, int32_t B, int32_t HW, int32_t C, float* stats, float* out,
                             madm_stream stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t per = size_t(B) * groupnorm_slabs(HW, C) * 64;  // scratch: partials(a), partials(s), final(a), final(s)
  float* pa = stats;
  float* ps = stats + per;
  float* st_a = stats + 2 * per;
  float* st_s = st_a + size_t(B) * 64;
  if (const char* e = groupnorm_stats(a, C, nullptr, 0, B, HW, 0, 0, pa, st)) return fail(e);
  if (const char* e = groupnorm_finalize(pa, B, HW, C, st_a, st)) return fail(e);
  if (has_shortcut_norm) {
    if (const char* e = groupnorm_stats(s, C, nullptr, 0, B, HW, 0, 0, ps, st)) return fail(e);
    if (const char* e = groupnorm_finalize(ps, B, HW, C, st_s, st)) return fail(e);
  }
  RUN(gn_add_relu_nchw(a, st_a, ga, ba, s, has_shortcut_norm ? st_s : nullptr, gs, bs, eps, B, HW, C, out, st));
}

// ---- backward pass (SURVEY §8 row f-3)
int madm_op_groupnorm_bwd_scratch_floats(int32_t B, int32_t HW, int32_t C) {
  return int(size_t(B) * groupnorm_bwd_slabs(HW) * C * 2 + size_t(B) * 64 + size_t(B) * C * 2);
}
int madm_op_groupnorm_bwd(const void* x0, int32_t C0, const void* x1, int32_t C1, int32_t B, int32_t HW, int32_t in16, const float* stats,
                          const float* gamma, const float* beta, float eps, int32_t act, const void* dy16, const float* extra, float* scratch,
                          void* out16, float* dx0, int32_t acc0, float* dx1, int32_t acc1, float* dgamma, float* dbeta, int32_t dtype,
                          madm_stream stream) {
  const int C = C0 + C1;
  float* partial = scratch;
  float* coef = partial + size_t(B) * groupnorm_bwd_slabs(HW) * C * 2;
  float* chan = coef + size_t(B) * 64;
  RUN(groupnorm_bwd(x0, C0, x1, C1, B, HW, in16, stats, gamma, beta, eps, act, dy16, dtype == MADM_DTYPE_FP16, partial, coef, chan, extra, out16, dx0,
                    acc0, dx1, acc1, dgamma, dbeta, 1.0f, static_cast<cudaStream_t>(stream)));
}
int64_t madm_op_c3_gn_bwd_scratch_floats(int32_t B, int32_t C) {
  return int64_t(image_moments_floats(B)) + int64_t(B) * C * 4 + int64_t(c3_gn_bwd_scratch_floats(B, C));
}
int madm_op_c3_gn_bwd(const float* img4, const float* w, const float* gamma, const float* beta, float eps, int32_t relu, int32_t B, int32_t HW,
                      int32_t C, const void* dy16, float scale, float* dw, float* dgamma, float* dbeta, float* scratch, int32_t dtype, madm_stream stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* mom = scratch;  // the forward's quantities the backward reads: image moments, folded conv + GroupNorm coefficients (ReLU mask)
  float* coef = mom + image_moments_floats(B);
  float* partial = coef + size_t(B) * C * 4;
  if (const char* e = image_moments(img4, B, HW, mom, st)) return fail(e);
  if (const char* e = c3_gn_coeffs(mom, w, gamma, beta, eps, B, HW, C, coef, st)) return fail(e);
  RUN(c3_gn_bwd(img4, mom, coef, w, gamma, eps, relu, B, HW, C, dy16, dtype == MADM_DTYPE_FP16, scale, dw, dgamma, dbeta, partial, st));
}
int madm_op_layernorm_bwd(const float* x, int32_t M, int32_t C, const float* gamma, float eps, const void* dy16, float* dx, int32_t accumulate,
                          int32_t dtype, madm_stream stream) {
  RUN(layernorm_bwd(x, M, C, gamma, eps, dy16, dtype == MADM_DTYPE_FP16, dx, accumulate, static_cast<cudaStream_t>(stream)));
}
int madm_op_geglu_fwd(const void* raw16, int64_t M, int32_t H, void* out16, int32_t dtype, madm_stream stream) {
  RUN(geglu_fwd(raw16, long(M), H, out16, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}
int madm_op_geglu_bwd(const void* raw16, const void* dout16, int64_t M, int32_t H, void* draw16, int32_t dtype, madm_stream stream) {
  RUN(geglu_bwd(raw16, dout16, long(M), H, draw16, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}
int64_t madm_op_attention_bwd_scratch_floats(int32_t B, int32_t heads, int32_t d, int32_t Nq, int32_t Nk) {
  return int64_t(attention_bwd_scratch_floats(B, heads, d, Nq, Nk));
}
int madm_op_attention_bwd(const void* q, int32_t ldq, const void* k, int32_t ldk, const void* v, int32_t ldv, const void* o, int32_t ldo,
                          const void* dout, int32_t lddo, void* dq, int32_t lddq, void* dk, int32_t lddk, void* dv, int32_t lddv, int32_t B,
                          int32_t heads, int32_t d, int32_t Nq, int32_t Nk, int64_t q_bs, int64_t kv_bs, int64_t o_bs, int64_t do_bs, int64_t dq_bs,
                          int64_t dkv_bs, float scale, float* scratch, int32_t dtype, madm_stream stream) {
  AttnBwdLaunch L;
  if (const char* e = attention_bwd_prepare(q, ldq, k, ldk, v, ldv, o, ldo, dout, lddo, dq, lddq, dk, lddk, dv, lddv, B, heads, d, Nq, Nk, long(q_bs),
                                            long(kv_bs), long(kv_bs), long(o_bs), long(do_bs), long(dq_bs), long(dkv_bs), long(dkv_bs), scale, scratch,
                                            dtype == MADM_DTYPE_FP16, &L))
    return fail(e);
  RUN(attention_bwd_launch(L, static_cast<cudaStream_t>(stream)));
}
int64_t madm_op_wgrad_scratch_floats(int32_t M, int32_t N, int32_t K, int32_t taps) { return int64_t(wgrad_scratch_floats(M, N, K, taps)); }
int madm_op_wgrad(const void* dy16, int32_t lda, const void* x16, int32_t ldb, int32_t M, int32_t N, int32_t K, int32_t taps, int32_t Bimg, int32_t H,
                  int32_t W, float alpha, float* out, int32_t transpose_out, float* scratch, int32_t dtype, madm_stream stream) {
  long so_n = K, so_k = 1, so_tap = 0;
  if (taps == 9) { so_n = long(K) * 9; so_k = 9; so_tap = 1; }
  else if (transpose_out) { so_n = 1; so_k = N; }
  RUN(wgrad(dy16, lda, x16, ldb, M, N, K, taps, Bimg, H, W, alpha, out, so_n, so_k, so_tap, scratch, dtype == MADM_DTYPE_FP16,
            static_cast<cudaStream_t>(stream)));
}
int64_t madm_op_lora_grads_scratch_floats(int32_t M, int32_t N, int32_t K) { return lora_grads_supported(N, K) ? int64_t(lora_grads_scratch_floats(M, N, K)) : -1; }
int madm_op_lora_grads(const void* x16, int32_t ldx, const void* dy16, int32_t ldy, const void* a16, const void* bt16, int32_t M, int32_t N, int32_t K,
                       float alpha, float* gA, float* gB, float* scratch, int32_t dtype, madm_stream stream) {
  RUN(lora_grads(x16, ldx, dy16, ldy, a16, bt16, M, N, K, alpha, gA, gB, scratch, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}
int madm_op_colsum_per_image(const void* x16, int32_t B, int32_t HW, int32_t C, float* out, int32_t ldo, int32_t dtype, madm_stream stream) {
  RUN(colsum_per_image(x16, B, HW, C, dtype == MADM_DTYPE_FP16, out, ldo, static_cast<cudaStream_t>(stream)));
}
int madm_op_zero_stuff2x(const void* x16, int32_t B, int32_t h, int32_t w, int32_t C, void* out16, madm_stream stream) {
  RUN(zero_stuff2x(x16, B, h, w, C, out16, static_cast<cudaStream_t>(stream)));
}
int madm_op_sum2x2(const float* x, int32_t B, int32_t h, int32_t w, int32_t C, float* out, int32_t accumulate, madm_stream stream) {
  RUN(sum2x2(x, B, h, w, C, out, accumulate, static_cast<cudaStream_t>(stream)));
}
int madm_op_relu_bwd_nchw(const float* dout, const float* out, int32_t B, int32_t C, int32_t HW, float scale, void* dz16, int32_t dtype,
                          madm_stream stream) {
  RUN(relu_bwd_nchw_to_nhwc16(dout, out, B, C, HW, scale, dz16, dtype == MADM_DTYPE_FP16, static_cast<cudaStream_t>(stream)));
}

}  // extern "C"
