// Host-side engine: owns no model memory.  It (1) keeps a registry of the caller's fp32 parameter pointers under their
// reference state_dict names, (2) defines the packed bf16 weight arena layout and the pack pass (with LoRA folding),
// (3) builds, per batch size, a static plan of kernel launches over a caller-provided workspace (TMA tensor maps are
// encoded once at plan time), and (4) replays the plan on the caller's stream.
//
// The SD-1.4 topology below restates the control flow of the reference's own forward re-implementations:
//   vae_encoder      modeling/meta_arch/ldm_diffusers.py:283-311
//   add_noise        modeling/meta_arch/ldm_diffusers.py:349-360
//   diffusion_unet   modeling/meta_arch/ldm_diffusers.py:454-616 (+ :363-451 up blocks, taps 'after' resnet+attn)
//   forward_features modeling/backbone/feature_extractor.py:367-396 (+ detectron2 BottleneckBlock, norm="GN")
#include "../../include/madm_b200.h"
#include "api_internal.h"
#include "kernels.h"
#include "launch.cuh"

#include <algorithm>
#include <cuda_bf16.h>
#include <functional>
#include <map>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <memory>
#include <string>
#include <tuple>
#include <unordered_map>
#include <vector>

using namespace madm;

namespace {

typedef __nv_bfloat16 bf16;
using Op = std::function<const char*(cudaStream_t)>;

struct ParamRef {
  const float* p = nullptr;
  int ndim = 0;
  int64_t shape[4] = {0, 0, 0, 0};
  int64_t numel() const {
    int64_t n = 1;
    for (int i = 0; i < ndim; ++i) n *= shape[i];
    return n;
  }
};

// ---- packed arena entries.  Two arenas use them: the forward arena (madm_pack_weights) and the training path's input-gradient
// ("dgrad") arena (madm_pack_dgrad_weights): transposed / tap-mirrored 16-bit copies of the frozen weights (LoRA folded), the skinny
// LoRA factor operands, and the natural-order feed-forward weight of the training forward.
enum PackKind { PK_CONV,       // conv [N,C,k,k] -> [N, taps*Cpad] inside rows of pitch ldo
                PK_CONV_DGRAD, // conv [Cout=N,Cin=C,k,k] -> [Cin, taps*Cpad], mirrored taps (Cpad = Cout)
                PK_LINEAR,     // linear [N,K=C] (+ LoRA) in natural row order, rows of pitch ldo
                PK_LINEAR_T,   // linear [N,K=C] (+ LoRA) -> its transpose, written at a column offset of a [K, ldo] region
                PK_LORA_A,     // lora_A [r,in] -> [r,in]       (operand of U = X A^T)
                PK_LORA_BT,    // lora_B [out,r] -> [r,out]     (operand of V = dY B)
                PK_GEGLU, PK_VAE_HEAD, PK_F32_COPY, PK_F32_SUM2,
                PK_BN_FOLD,    // eval-mode BatchNorm -> fp32 [scale | shift] (bias_off = N floats each)
                PK_CONV_BN,    // conv weight with the BatchNorm scale (at bias_off) folded into its rows
                PK_DW_BN,      // depthwise 3x3 weight * BatchNorm scale -> fp32 [9][C]
                PK_IDENTITY,   // N x N identity block (16-bit) inside a wider packed row: the residual add as an extra K segment
                PK_REGION };   // bytes reserved for entries registered into it
struct PackEntry {
  PackKind kind;
  std::string src, src2, src3, src4;  // parameter names (linear / LoRA factor: the module path)
  size_t off = 0;                     // byte offset in arena
  int N = 0, C = 0, taps = 1, Cpad = 0, Kpad = 0, ldo = 0;
  bool lora = false;                  // LoRA-targeted linear
  bool trainable = false;             // an optimizer or EMA step can change it: the subset a partial repack rewrites
  size_t bias_off = 0;                // for GEGLU / VAE head: fp32 bias region
};

// An arena's layout: its entries by key, laid out by a LAYOUT pass of the traversal and looked up by the other passes
struct Arena {
  std::vector<PackEntry> entries;
  std::map<std::string, size_t> index;  // key -> index in entries
  size_t bytes = 0;
  bool done = false;                    // laid out for the current parameter shapes, operand dtype and variant
  size_t reserve(size_t n) {
    const size_t off = bytes;
    bytes += (n + 1023) & ~size_t(1023);
    return off;
  }
};

struct IoBind {  // per-call pointers read by the plan's first/last ops
  madm_extract_args a;
  madm_backward_args b;  // training plans: the arguments of the madm_backward call being replayed
};

struct F32T { float* p = nullptr; size_t off = 0; size_t bytes = 0; };
struct B16T { bf16* p = nullptr; size_t off = 0; size_t bytes = 0; };

// gradient of an fp32-stream activation in a training plan: allocated by its first contributor; later contributors accumulate
struct GradBuf {
  F32T f;
  bool written = false;  // at least one contribution has been emitted
  bool stop = false;     // nothing trainable lies upstream: contributions are skipped
};

constexpr int kStatRows = 32;  // rows per block of a GEMM epilogue's column statistics (GemmDesc::colstats: one block per epilogue warp)

// fp32 residual-stream activation, NHWC, optionally with a bf16 copy for consumers that take it as a GEMM operand
struct Act {
  F32T f; B16T h;
  std::shared_ptr<struct GradBuf> gr;  // training plans: gradient of this activation (fp32 [M,C]), shared by all copies of the handle
  float* cs = nullptr;  // per-column statistics written by the producing GEMM's epilogue ([M/kStatRows][C][2]), if any
  bool has_cs = false;  // valid in every builder mode (cs itself is null outside PLAN mode)
  bool h_s2d = false;   // the 16-bit copy `h` is stored in space-to-depth layout [4][B][H/2][W/2][C] (input of a stride-2 conv)
  int B = 0, H = 0, W = 0, C = 0;
  int HW() const { return H * W; }
  long M() const { return long(B) * H * W; }
};

// One kernel launch of a plan and what the profile accounts to it
struct Launch {
  Op run;
  int stage;          // MADM_STAGE_* bit
  int branch;         // 0 = the caller's stream; 1..4 = independent projection branches (run on side streams, forked / joined by events)
  int kind;           // MADM_KIND_*
  bool optional;      // debug/taps launch that does work only when the caller asks for the extra output
  double flops;       // algorithmic FLOPs (2*MAC of the reference's convs / linears: no K padding, no identity segments)
  double exec_flops;  // FLOPs the launch executes (padded K, identity-weight residual segments, GEGLU both halves)
  double bytes;       // algorithmic HBM bytes (HBM-bound kernels)
};

// Heap-allocated and never moved: its launches point into `io`.
struct Plan {
  const void* packed = nullptr;
  void* ws = nullptr;
  size_t ws_bytes = 0;
  std::vector<Launch> ops;
  std::vector<Launch> bops;   // training plans: the backward pass (replayed by madm_backward)
  bool train = false;
  const void* dpacked = nullptr;
  float loss_scale = 1.0f, lora_scale = 0.f;
  std::string adapter;
  std::vector<cudaEvent_t> ev;  // 2 per op, created on demand when profiling
  Plan() = default;
  Plan(const Plan&) = delete;
  ~Plan() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
  IoBind io;
  size_t stats_bytes = 0;
};

}  // namespace

struct madm_ctx {
  int device = 0;
  int fp16 = 1;  // compute dtype of GEMM operands (MADM_DTYPE_FP16 default)
  int variant = MADM_VARIANT_BASE;
  std::string err;
  std::unordered_map<std::string, ParamRef> params;
  Arena fwd;    // forward arena (madm_pack_weights)
  Arena dgrad;  // input-gradient arena of the training path (madm_pack_dgrad_weights)
  float* alphas_cumprod = nullptr;  // [1000] device
  bool profiling = false;
  cudaStream_t side[4] = {nullptr, nullptr, nullptr, nullptr};  // projection branches (created on first use)
  cudaEvent_t ev_fork[4] = {nullptr, nullptr, nullptr, nullptr}, ev_join[4] = {nullptr, nullptr, nullptr, nullptr};
  Plan* last_plan = nullptr;
  int last_stages = 0;
  std::map<std::tuple<int, int, int, int>, std::unique_ptr<Plan>> plans;  // (B, ema, head_h, head_w)
  std::map<std::tuple<int, int, int>, size_t> ws_bytes_cache;             // (B, head_h, head_w)
  // training path
  std::unordered_map<std::string, float*> grads;     // gradient output buffers by parameter name (madm_set_grad_tensors)
  std::map<std::pair<int, uintptr_t>, std::unique_ptr<Plan>> train_plans;  // (B, training workspace) -> forward (activations kept) + backward
};

namespace {

const std::string kUnet = "feature_extractor.ldm_extractor.unet.";
const std::string kVae = "feature_extractor.ldm_extractor.vae.";

struct BuildError {
  std::string msg;
  int code;
};

// ------------------------------------------------------------------------------------------------ builder
// One traversal of the model serves three purposes, selected by `mode`:
//   LAYOUT: register packed-arena entries (B-independent)      SIZE: compute workspace bytes for B
//   PLAN:   emit launches with real pointers
enum Mode { LAYOUT, SIZE, PLAN };

IoBind dry_io;  // what the launches of a dry pass would read: they are not kept, so nothing reads it

struct Builder {
  madm_ctx* ctx;
  Mode mode;
  int B;
  bool ema;
  Plan* plan = nullptr;
  IoBind* io = &dry_io;  // per-call pointers the launches read (the plan's in PLAN mode)
  uint8_t* ws = nullptr;
  const uint8_t* packed = nullptr;
  int cur_stage = MADM_STAGE_VAE;
  int cur_branch = 0;            // branch tag of the ops being emitted (build_proj)
  bool defer_free = false;       // concurrent branches must not recycle each other's buffers: frees are collected and released at the join
  std::vector<std::pair<size_t, size_t>> deferred;
  int head_h = 0, head_w = 0;  // grid of the head's first feature map (0 = the 512 x 512 crop's: 128 x 128, s0 variant 512 x 512)
  // ---- training plans (SURVEY §8 row f-3): the forward keeps what the backward needs; every builder function records its backward on
  // the tape, which build_all() replays in reverse into plan->bops
  bool train = false;
  bool bwd = false;            // currently emitting the backward pass
  const uint8_t* dpacked = nullptr;
  float loss_scale = 1.0f;
  std::string adapter;         // active LoRA adapter of this training plan ("" = none)
  float lora_scale = 0.f;
  std::vector<std::pair<int, std::function<void()>>> tape;  // (stage of the forward that recorded it, its backward)
  bool frozen = false;         // emitting a part of a differentiated stage that runs without gradient (the s0 variant's VAE decoder body)
  // forward of a stage the training plan differentiates (not the VAE encoder): its tensors stay allocated and each block records its backward
  bool recording() const { return train && !bwd && !frozen && cur_stage != MADM_STAGE_VAE; }

  // ---- workspace allocator (first-fit free list, 1 KB granularity); identical sequence in SIZE and PLAN modes
  struct Blk { size_t off, bytes; };
  std::vector<Blk> free_list;
  size_t top = 0, peak = 0;
  size_t alloc(size_t bytes) {
    bytes = (bytes + 1023) & ~size_t(1023);
    for (size_t i = 0; i < free_list.size(); ++i) {
      if (free_list[i].bytes >= bytes) {
        size_t off = free_list[i].off;
        if (free_list[i].bytes == bytes) free_list.erase(free_list.begin() + i);
        else { free_list[i].off += bytes; free_list[i].bytes -= bytes; }
        return off;
      }
    }
    size_t off = top;
    top += bytes;
    if (top > peak) peak = top;
    return off;
  }
  void release(size_t off, size_t bytes) {
    if (bytes == 0) return;
    bytes = (bytes + 1023) & ~size_t(1023);
    if (off + bytes == top) {  // shrink the top, merging trailing free blocks
      top = off;
      bool merged = true;
      while (merged) {
        merged = false;
        for (size_t i = 0; i < free_list.size(); ++i)
          if (free_list[i].off + free_list[i].bytes == top) {
            top = free_list[i].off;
            free_list.erase(free_list.begin() + i);
            merged = true;
            break;
          }
      }
      return;
    }
    // insert + coalesce neighbours
    Blk nb{off, bytes};
    for (size_t i = 0; i < free_list.size();) {
      if (free_list[i].off + free_list[i].bytes == nb.off) { nb.off = free_list[i].off; nb.bytes += free_list[i].bytes; free_list.erase(free_list.begin() + i); }
      else if (nb.off + nb.bytes == free_list[i].off) { nb.bytes += free_list[i].bytes; free_list.erase(free_list.begin() + i); }
      else ++i;
    }
    free_list.push_back(nb);
  }
  F32T f32(size_t n) { F32T t; t.bytes = n * 4; t.off = alloc(t.bytes); t.p = reinterpret_cast<float*>(ws + t.off); return t; }
  B16T b16(size_t n) { B16T t; t.bytes = n * 2; t.off = alloc(t.bytes); t.p = reinterpret_cast<bf16*>(ws + t.off); return t; }
  // pinned buffers (feature taps) survive free(): they are consumed by the projection stage
  std::vector<size_t> pinned;
  bool is_pinned(size_t off, size_t bytes) const {
    if (bytes == 0) return false;
    for (size_t o : pinned) if (o == off) return true;
    return false;
  }
  void pin(const Act& a) {
    if (a.f.bytes) pinned.push_back(a.f.off);
    if (a.h.bytes) pinned.push_back(a.h.off);
  }
  void release_or_defer(size_t off, size_t bytes) { if (defer_free) deferred.push_back({off, bytes}); else release(off, bytes); }
  void flush_deferred() { for (auto& d : deferred) release(d.first, d.second); deferred.clear(); }
  void free(F32T& t) { if (recording()) return; if (!is_pinned(t.off, t.bytes)) release_or_defer(t.off, t.bytes); t.bytes = 0; t.p = nullptr; }
  void free(B16T& t) { if (recording()) return; if (!is_pinned(t.off, t.bytes)) release_or_defer(t.off, t.bytes); t.bytes = 0; t.p = nullptr; }
  void free(Act& a) { free(a.f); free(a.h); }
  Act act(int B_, int H, int W, int C, bool with_f32, bool with_b16) {
    Act a; a.B = B_; a.H = H; a.W = W; a.C = C;
    if (with_f32) a.f = f32(size_t(a.M()) * C);
    if (with_b16) a.h = b16(size_t(a.M()) * C);
    if (train) a.gr = std::make_shared<GradBuf>();
    return a;
  }
  // gradient buffer of an activation: allocated by the first contributor.  Returns the pointer and whether to accumulate.
  float* grad(const Act& a, int* accumulate) {
    GradBuf& g = *a.gr;
    if (g.f.bytes == 0) g.f = f32(size_t(a.M()) * a.C);
    *accumulate = g.written ? 1 : 0;
    g.written = true;
    return g.f.p;
  }
  static bool wants_grad(const Act& a) { return a.gr && !a.gr->stop; }
  float* grad_buf(const std::string& name) {  // registered gradient output buffer of a parameter, or null
    auto it = ctx->grads.find(name);
    return it == ctx->grads.end() ? nullptr : it->second;
  }

  // ---- per-GroupNorm statistics slots: per-slab partial sums [B, slabs, 32, 2] fp32 (each slot written by exactly one CTA
  // per call, so no zeroing and no atomics) or finalised [B,32,2] (slabs = 1)
  size_t stats_used = 0;
  float* stats_base = nullptr;
  float* new_stats(int slabs) {
    float* p = stats_base ? stats_base + stats_used : nullptr;
    stats_used += size_t(B) * slabs * 64;
    return p;
  }

  // per-column statistics buffer for a GEMM whose output feeds a GroupNorm; lives in the statistics arena
  void attach_colstats(Act& a, GemmDesc& d) {
    if (a.HW() % kStatRows != 0 || a.C % 32 != 0) return;  // shape not eligible: the consumer falls back to a statistics pass
    // The fused statistics add ~25 % to the epilogue's instruction count (separate kernel variant, gemm_tc_kernel<BN,true>):
    // measured +0.25 ms on the GEMM family against -1.0 ms of statistics passes, at every K.
    if (choose_splits(d) > 1) return;  // split-K launches leave the statistics to a separate pass
    const size_t n = size_t((a.M() + kStatRows - 1) / kStatRows) * a.C * 2;
    a.cs = stats_base ? stats_base + stats_used : nullptr;
    stats_used += n;
    a.has_cs = true;
    d.colstats = a.cs;
  }

  // ---- parameters
  [[noreturn]] void fail(int code, const std::string& m) { throw BuildError{m, code}; }
  const ParamRef* find(const std::string& name) {
    auto it = ctx->params.find(name);
    return it == ctx->params.end() ? nullptr : &it->second;
  }
  const float* param(const std::string& name, int64_t numel = -1) {
    const ParamRef* r = find(name);
    if (!r) fail(MADM_ENOTFOUND, "parameter not registered: " + name);
    if (numel >= 0 && r->numel() != numel) fail(MADM_EINVAL, "parameter has unexpected size: " + name);
    return r->p;
  }

  // ---- packed arenas
  // returns an arena's entry, registering it in a LAYOUT pass.  The training traversal's LAYOUT pass only adds to the dgrad arena: the
  // caller has sized the forward arena already (madm_packed_bytes).
  const PackEntry& entry(Arena& a, const std::string& key, const std::function<PackEntry()>& make) {
    auto it = a.index.find(key);
    if (it != a.index.end()) return a.entries[it->second];
    if (mode != LAYOUT) fail(MADM_ESTATE, "packed entry missing from layout: " + key);
    if (train && &a == &ctx->fwd) fail(MADM_ESTATE, "training layout reached a forward-arena entry the forward layout lacks: " + key);
    PackEntry e = make();
    e.trainable = e.lora || e.kind == PK_LORA_A || e.kind == PK_LORA_BT || cur_stage == MADM_STAGE_PROJ;
    a.index[key] = a.entries.size();
    a.entries.push_back(e);
    return a.entries.back();
  }
  const bf16* pw(size_t off) const { return reinterpret_cast<const bf16*>(packed + off); }
  const float* pf(size_t off) const { return reinterpret_cast<const float*>(packed + off); }

  // conv weight [N,C,k,k] -> [N, taps*Cpad] (optionally inside a wider row of pitch ldo at column col_off)
  size_t conv_w(const std::string& name, int N, int C, int taps, int Cpad = 0) {
    if (Cpad == 0) Cpad = (C + 63) / 64 * 64;
    const int Kpad = (taps * Cpad + 63) / 64 * 64;
    return entry(ctx->fwd, "conv:" + name, [&] {
      PackEntry e; e.kind = PK_CONV; e.src = name + ".weight"; e.N = N; e.C = C; e.taps = taps; e.Cpad = Cpad; e.Kpad = Kpad; e.ldo = Kpad;
      e.off = ctx->fwd.reserve(size_t(N) * Kpad * 2);
      return e;
    }).off;
  }
  // conv3x3 (Cout -> Cout) and 1x1 shortcut (Cin -> Cout) packed side by side: [Cout, 9*Cout + Cin]; bias = b_conv + b_sc
  struct Fused { size_t w_off, b_off; };
  Fused conv_plus_shortcut(const std::string& conv, const std::string& sc, int Cout, int Cin) {
    const int K0 = 9 * Cout, K = K0 + Cin;
    const PackEntry& e0 = entry(ctx->fwd, "convsc:" + conv, [&] {
      PackEntry e; e.kind = PK_CONV; e.src = conv + ".weight"; e.N = Cout; e.C = Cout; e.taps = 9; e.Cpad = Cout; e.Kpad = K0; e.ldo = K;
      e.off = ctx->fwd.reserve(size_t(Cout) * K * 2);
      return e;
    });
    const size_t w_off = e0.off;
    entry(ctx->fwd, "convsc_sc:" + conv, [&] {
      PackEntry e; e.kind = PK_CONV; e.src = sc + ".weight"; e.N = Cout; e.C = Cin; e.taps = 1; e.Cpad = Cin; e.Kpad = Cin; e.ldo = K;
      e.off = w_off + size_t(K0) * 2;
      return e;
    });
    const size_t b_off = entry(ctx->fwd, "convsc_b:" + conv, [&] {
      PackEntry e; e.kind = PK_F32_SUM2; e.src = conv + ".bias"; e.src2 = sc + ".bias"; e.N = Cout;
      e.off = ctx->fwd.reserve(size_t(Cout) * 4);
      return e;
    }).off;
    return Fused{w_off, b_off};
  }
  // conv3x3 (C -> C) with the residual add folded in as a second K segment with identity weights: [C, 9*C + C].  The residual
  // operand then is the 16-bit stream itself, read by TMA like any A tile (exact: 1.0 * x accumulated in fp32), so the epilogue
  // needs no fp32 residual tensor.
  size_t conv_plus_identity(const std::string& conv, int C) {
    const int K0 = 9 * C, K = K0 + C;
    const size_t w_off = entry(ctx->fwd, "convid:" + conv, [&] {
      PackEntry e; e.kind = PK_CONV; e.src = conv + ".weight"; e.N = C; e.C = C; e.taps = 9; e.Cpad = C; e.Kpad = K0; e.ldo = K;
      e.off = ctx->fwd.reserve(size_t(C) * K * 2);
      return e;
    }).off;
    entry(ctx->fwd, "convid_i:" + conv, [&] {
      PackEntry e; e.kind = PK_IDENTITY; e.N = C; e.ldo = K; e.off = w_off + size_t(K0) * 2;
      return e;
    });
    return w_off;
  }
  // a region holding several linears stacked along N (fused QKV, all cross-attn K/V, all time_emb_proj)
  size_t region(const std::string& key, size_t bytes) {
    return entry(ctx->fwd, "region:" + key, [&] { PackEntry e; e.kind = PK_REGION; e.off = ctx->fwd.reserve(bytes); return e; }).off;
  }
  void linear_part(const std::string& module, size_t region_off, int row_off, int N, int K, bool lora) {
    entry(ctx->fwd, "lin:" + module, [&] {
      PackEntry e; e.kind = PK_LINEAR; e.src = module; e.N = N; e.C = K; e.ldo = K; e.lora = lora;
      e.off = region_off + size_t(row_off) * K * 2;
      return e;
    });
  }
  size_t linear_w(const std::string& module, int N, int K, bool lora) {
    return entry(ctx->fwd, "lin:" + module, [&] {
      PackEntry e; e.kind = PK_LINEAR; e.src = module; e.N = N; e.C = K; e.ldo = K; e.lora = lora;
      e.off = ctx->fwd.reserve(size_t(N) * K * 2);
      return e;
    }).off;
  }
  // mmcv ConvModule (conv without bias -> BatchNorm(eval) -> ReLU): BN scale folded into the packed weight rows, shift = epilogue bias
  struct ConvBn { size_t w_off, shift_off; };
  ConvBn conv_bn(const std::string& mod, int N, int C, int taps) {
    const size_t fold = entry(ctx->fwd, "bnfold:" + mod, [&] {
      PackEntry e; e.kind = PK_BN_FOLD; e.src = mod + ".bn"; e.N = N; e.off = ctx->fwd.reserve(size_t(2) * N * 4);
      return e;
    }).off;
    const int Kpad = taps * C;
    const size_t w = entry(ctx->fwd, "convbn:" + mod, [&] {
      PackEntry e; e.kind = PK_CONV_BN; e.src = mod + ".conv.weight"; e.N = N; e.C = C; e.taps = taps; e.Cpad = C; e.Kpad = Kpad; e.ldo = Kpad;
      e.bias_off = fold; e.off = ctx->fwd.reserve(size_t(N) * Kpad * 2);
      return e;
    }).off;
    return ConvBn{w, fold + size_t(N) * 4};
  }
  // depthwise ConvModule: fp32 [9][C] weights (scale folded) + shift
  ConvBn depthwise_bn(const std::string& mod, int C) {
    const size_t fold = entry(ctx->fwd, "bnfold:" + mod, [&] {
      PackEntry e; e.kind = PK_BN_FOLD; e.src = mod + ".bn"; e.N = C; e.off = ctx->fwd.reserve(size_t(2) * C * 4);
      return e;
    }).off;
    const size_t w = entry(ctx->fwd, "dwbn:" + mod, [&] {
      PackEntry e; e.kind = PK_DW_BN; e.src = mod + ".conv.weight"; e.C = C; e.bias_off = fold; e.off = ctx->fwd.reserve(size_t(9) * C * 4);
      return e;
    }).off;
    return ConvBn{w, fold + size_t(C) * 4};
  }
  void f32_part(const std::string& name, size_t region_off, int elem_off, int n) {
    entry(ctx->fwd, "f32:" + name, [&] {
      PackEntry e; e.kind = PK_F32_COPY; e.src = name; e.N = n; e.off = region_off + size_t(elem_off) * 4;
      return e;
    });
  }

  // ---- op emission
  void emit(Op op, bool optional = false, int kind = MADM_KIND_ELEMENTWISE, double flops = 0.0, double bytes = 0.0, double exec_flops = -1.0) {
    if (mode != PLAN) return;
    (bwd ? plan->bops : plan->ops)
        .push_back(Launch{std::move(op), cur_stage, cur_branch, kind, optional, flops, exec_flops < 0 ? flops : exec_flops, bytes});
  }
  // launches emitted so far into the pass being built (PLAN mode; 0 otherwise)
  size_t emitted() const { return mode == PLAN ? (bwd ? plan->bops : plan->ops).size() : 0; }
  // makes the launches emitted since `from` do nothing in a call whose optional input *arg is null
  void only_if_set(size_t from, const float* const* arg) {
    if (mode != PLAN) return;
    std::vector<Launch>& ops = bwd ? plan->bops : plan->ops;
    for (size_t k = from; k < ops.size(); ++k) {
      Op run = std::move(ops[k].run);
      ops[k].run = [arg, run](cudaStream_t st) -> const char* { return *arg ? run(st) : nullptr; };
    }
  }
  // algo_flops < 0: 2*M*N*K from the descriptor (K counts real channels only when k_real is given)
  // split-K factor for a GEMM whose M x N tiling cannot fill the 148 SMs (8x8-resolution convs, small batches): the K range
  // is divided over `splits` CTAs per output tile; raw fp32 partials are reduced in fixed order by splitk_reduce, which
  // also applies the fused epilogue.  Deterministic (no atomics).  MADM_NO_SPLITK=1 turns it off: the reference summation order.
  static int choose_splits(const GemmDesc& d) {
    if (getenv("MADM_NO_SPLITK")) return 1;
    if (d.act == ACT_GEGLU || d.N % 4 != 0 || d.N < 128) return 1;
    const int tiles = ((d.M + 127) / 128) * ((d.N + 127) / 128);  // the split launch uses 128-wide N tiles
    int chunks = 0;
    for (int sgi = 0; sgi < d.nseg; ++sgi) chunks += d.seg[sgi].ntaps * d.seg[sgi].C / 64;
    if (tiles > 74 || chunks < 32) return 1;
    int s = 148 / tiles;
    if (s > chunks / 16) s = chunks / 16;
    if (s > 8) s = 8;
    return s < 2 ? 1 : s;
  }

  // algorithmic HBM bytes of one GEMM: every operand / result element crosses HBM once (A is read once, not once per filter tap)
  static double gemm_algo_bytes(const GemmDesc& d) {
    double by = 0;
    for (int sgi = 0; sgi < d.nseg; ++sgi) by += double(d.M) * d.seg[sgi].C * 2 + double(d.N) * d.seg[sgi].ntaps * d.seg[sgi].C * 2;
    const double mn = double(d.M) * ((d.act == ACT_GEGLU) ? d.N : d.N);
    if (d.act == ACT_GEGLU) by += double(d.N) * (d.seg[0].ntaps * d.seg[0].C) * 2;  // the gate half of the weight
    if (d.out_f32) by += mn * 4;
    if (d.out_bf16) by += mn * 2;
    if (d.residual) by += mn * (d.res16 ? 2 : 4);
    if (d.colstats) by += mn / 32 * 8;
    return by;
  }
  void gemm(const GemmDesc& d0, double algo_flops = -1.0) {
    const int splits = choose_splits(d0);
    F32T part;
    if (splits > 1) part = f32(size_t(splits) * d0.M * d0.N);  // identical allocation sequence in every builder mode
    if (mode == PLAN) {
      GemmDesc d = d0;
      d.fp16 = ctx->fp16;
      if (splits > 1) {  // raw fp32 partials; splitk_reduce applies the epilogue
        d.bias = nullptr; d.rowbias = nullptr; d.residual = nullptr; d.res16 = 0; d.out_bf16 = nullptr; d.act = ACT_NONE; d.colstats = nullptr; d.alpha = 1.0f;
        d.out_f32 = part.p; d.ldo32 = d0.N; d.splits = splits; d.split_stride = long(d0.M) * d0.N; d.bn = 128;
      }
      GemmLaunch L;
      if (const char* e = gemm_prepare(d, &L)) fail(MADM_EINVAL, std::string(e));
      double K = 0;
      for (int sgi = 0; sgi < d.nseg; ++sgi) K += double(d.seg[sgi].ntaps) * d.seg[sgi].C;
      const double exec = 2.0 * double(d.M) * ((d.act == ACT_GEGLU) ? 2.0 * d.N : double(d.N)) * K;
      if (algo_flops < 0) algo_flops = exec;
      if (getenv("MADM_DUMP_PLAN")) {  // tools/layer_report.py parses these lines
        char tail[48];
        if (splits > 1) snprintf(tail, sizeof(tail), "splits=%d tma=%d stats=0", splits, L.p.tma_epi);
        else snprintf(tail, sizeof(tail), "tma=%d stats=%d", L.p.tma_epi, (d.colstats ? 1 : 0) | (d.s2d_W > 0 ? 2 : 0));
        fprintf(stderr, "MADM_PLAN gemm M=%d N=%d K=%d bn=%d tiles=%d taps=%d nseg=%d act=%d res=%d f32=%d h16=%d gflop=%.3f %s\n", d.M, d.N, int(K), L.bn,
                L.p.num_tiles, d.seg[0].ntaps, d.nseg, d0.act, d0.residual ? 1 : 0, d0.out_f32 ? 1 : 0, d0.out_bf16 ? 1 : 0, algo_flops / 1e9, tail);
      }
      emit([L](cudaStream_t st) { return gemm_launch(L, st); }, false, MADM_KIND_GEMM, algo_flops, gemm_algo_bytes(d), exec);
      if (splits > 1) {
        const GemmDesc e0 = d0; const float* pp = part.p; const int f16 = ctx->fp16; const long ss = d.split_stride;
        if (e0.alpha != 1.0f) fail(MADM_EINVAL, "split-K with alpha != 1 is not supported");
        emit([=](cudaStream_t st) {
          return splitk_reduce(pp, splits, ss, e0.M, e0.N, e0.bias, e0.rowbias, e0.rows_per_img, e0.ld_rowbias, e0.residual, e0.ldr, e0.out_f32,
                               e0.ldo32, e0.out_bf16, e0.ldo16, e0.act, f16, st, e0.res16);
        }, false, MADM_KIND_ELEMENTWISE, 0.0, double(splits + 2) * e0.M * e0.N * 4);
      }
    }
    if (splits > 1) free(part);
  }

  // fused attention: tcgen05/TMEM kernel (tensor maps encoded at plan time)
  void attention(const bf16* q, int ldq, const bf16* k, int ldk, const bf16* v, int ldv, bf16* o, int ldo, int Bn, int heads, int d, int Nq,
                 int Nk, long q_bs, long kv_bs, long o_bs, float scale, float* lse = nullptr) {
    const double flops = 4.0 * double(Bn) * Nq * Nk * heads * d;
    if (mode != PLAN) return;
    const int h16 = ctx->fp16;
    FaLaunch L;
    if (const char* e = flash_attention_tc_prepare(q, ldq, k, ldk, v, ldv, o, ldo, Bn, heads, d, Nq, Nk, q_bs, kv_bs, o_bs, scale, h16, &L, lse))
      fail(MADM_EINVAL, std::string(e));
    emit([L](cudaStream_t st) { return flash_attention_tc_launch(L, st); }, false, MADM_KIND_ATTENTION, flops, 0.0);
  }
  // its backward (training plans): prepared like the forward, with the gradient kernels' scratch
  void attention_bwd(const bf16* q, int ldq, const bf16* k, int ldk, const bf16* v, int ldv, const bf16* o, int ldo, const bf16* dout, int lddo, bf16* dq,
                     int lddq, bf16* dk, int lddk, bf16* dv, int lddv, int Bn, int heads, int d, int Nq, int Nk, long q_bs, long k_bs, long v_bs, long o_bs,
                     long do_bs, long dq_bs, long dk_bs, long dv_bs, float scale, float* scratch, const float* lse) {
    if (mode != PLAN) return;
    AttnBwdLaunch L;
    if (const char* e = attention_bwd_prepare(q, ldq, k, ldk, v, ldv, o, ldo, dout, lddo, dq, lddq, dk, lddk, dv, lddv, Bn, heads, d, Nq, Nk, q_bs, k_bs,
                                              v_bs, o_bs, do_bs, dq_bs, dk_bs, dv_bs, scale, scratch, ctx->fp16, &L, lse))
      fail(MADM_EINVAL, std::string(e));
    emit([L](cudaStream_t st) { return attention_bwd_launch(L, st); });
  }

  static GemmASeg seg_1x1(const bf16* p, int Bn, int H, int W, int C, int ld = 0) {
    GemmASeg s; s.ptr = p; s.Bt = Bn; s.H = H; s.W = W; s.C = C; s.ld = ld; s.ntaps = 1;
    return s;
  }
  static GemmASeg seg_3x3(const bf16* p, int Bn, int H, int W, int C) {
    GemmASeg s; s.ptr = p; s.Bt = Bn; s.H = H; s.W = W; s.C = C; s.ntaps = 9;
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) { s.dy[ky * 3 + kx] = int8_t(ky - 1); s.dx[ky * 3 + kx] = int8_t(kx - 1); }
    return s;
  }
  static GemmASeg seg_plain(const bf16* p, long M, int K, int ld = 0) {
    GemmASeg s; s.ptr = p; s.Bt = 1; s.H = 1; s.W = int(M); s.C = K; s.ld = ld; s.ntaps = 1;
    return s;
  }
  // stride-2 3x3 conv over the space-to-depth tensor [4][B][Ho][Wo][C]; pad1: PyTorch padding=1; else F.pad(0,1,0,1)+padding 0
  static GemmASeg seg_s2(const bf16* p, int Bn, int Ho, int Wo, int C, bool pad1) {
    GemmASeg s; s.ptr = p; s.Bt = 4 * Bn; s.H = Ho; s.W = Wo; s.C = C; s.ntaps = 9;
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        int py, dy, px, dx;
        if (pad1) { py = (ky == 1) ? 0 : 1; dy = (ky == 0) ? -1 : 0; px = (kx == 1) ? 0 : 1; dx = (kx == 0) ? -1 : 0; }
        else      { py = (ky == 1) ? 1 : 0; dy = (ky == 2) ? 1 : 0;  px = (kx == 1) ? 1 : 0; dx = (kx == 2) ? 1 : 0; }
        s.dy[ky * 3 + kx] = int8_t(dy); s.dx[ky * 3 + kx] = int8_t(dx); s.b_off[ky * 3 + kx] = (py * 2 + px) * Bn;
      }
    return s;
  }

  // GroupNorm(32) over an NHWC tensor (fp32 stream, or a 16-bit intermediate when in16; optionally the channel concat of
  // two fp32 sources) -> 16-bit operand tensor (+ raw 16-bit copy of the input)
  struct GnSaved { float* stats = nullptr; int slabs = 0; };  // per-slab partial sums [B, slabs, 32, 2] the backward finalises again
  GnSaved groupnorm(const Act& x0, const Act* x1, const std::string& norm, float eps, int actfn, bf16* y, bf16* raw, bool in16 = false) {
    const int C0 = x0.C, C1 = x1 ? x1->C : 0;
    const float* g = (mode == LAYOUT) ? nullptr : param(norm + ".weight", C0 + C1);
    const float* b = (mode == LAYOUT) ? nullptr : param(norm + ".bias", C0 + C1);
    const void* p0 = in16 ? static_cast<const void*>(x0.h.p) : static_cast<const void*>(x0.f.p);
    const void* p1 = x1 ? static_cast<const void*>(x1->f.p) : nullptr;
    const int Bn = x0.B, HW = x0.HW();
    const double elems = double(Bn) * HW * (C0 + C1);
    const int f16 = ctx->fp16, i16 = in16 ? 1 : 0;
    const double in_b = in16 ? 2 : 4;
    const bool fused = x0.has_cs && (!x1 || x1->has_cs);
    float* stats;
    int slabs;
    if (fused) {  // statistics came out of the producing GEMM epilogues: one small fixed-order reduction, no pass over x
      const int nb = HW / kStatRows;
      slabs = groupnorm_colstats_chunks(nb);
      stats = new_stats(slabs);
      const float* c0 = x0.cs; const float* c1 = x1 ? x1->cs : nullptr;
      emit([=](cudaStream_t st) { return groupnorm_colstats_reduce(c0, C0, c1, C1, Bn, nb, stats, st); }, false, MADM_KIND_GROUPNORM, 0.0,
           double(Bn) * nb * (C0 + C1) * 8);
    } else {
      slabs = groupnorm_slabs(HW, C0 + C1);
      stats = new_stats(slabs);
      emit([=](cudaStream_t st) { return groupnorm_stats(p0, C0, p1, C1, Bn, HW, i16, f16, stats, st); }, false, MADM_KIND_GROUPNORM, 0.0,
           elems * in_b);
    }
    emit([=](cudaStream_t st) { return groupnorm_apply(p0, C0, p1, C1, Bn, HW, i16, stats, slabs, g, b, eps, actfn, y, raw, f16, st); }, false,
         MADM_KIND_GROUPNORM, 0.0, elems * (in_b + 2 + (raw ? 2 : 0)));
    GnSaved sv; sv.stats = stats; sv.slabs = slabs;
    return sv;
  }

  // ---- backward of groupnorm() (training plans): dy16 = gradient of act(GN(x)); any subset of the outputs of kernels.h groupnorm_bwd.
  // fin = already finalised group sums [B,32,2] (projection tails), else the forward's slab partials in `sv` are finalised first.
  void groupnorm_bwd(const Act& x0, const Act* x1, bool in16, const GnSaved& sv, const float* fin, const std::string& norm, float eps, int actfn,
                     const bf16* dy, const float* extra, bf16* out16, float* dx0, int acc0, float* dx1, int acc1, float* dgamma, float* dbeta) {
    const int C0 = x0.C, C1 = x1 ? x1->C : 0, C = C0 + C1, Bn = x0.B, HW = x0.HW();
    const float* g = (mode == LAYOUT) ? nullptr : param(norm + ".weight", C);
    const float* be = (mode == LAYOUT) ? nullptr : param(norm + ".bias", C);
    const void* p0 = in16 ? static_cast<const void*>(x0.h.p) : static_cast<const void*>(x0.f.p);
    const void* p1 = x1 ? static_cast<const void*>(x1->f.p) : nullptr;
    F32T part = f32(size_t(Bn) * groupnorm_bwd_slabs(HW) * C * 2), coef = f32(size_t(Bn) * 64), chan = f32(size_t(Bn) * C * 2), fsum = f32(size_t(Bn) * 64);
    float* pp = part.p; float* cp = coef.p; float* chp = chan.p; float* fp = fsum.p;
    const float* stats = sv.stats; const int slabs = sv.slabs;
    const int f16 = ctx->fp16, i16 = in16 ? 1 : 0;
    const float inv_scale = 1.0f / loss_scale;
    emit([=](cudaStream_t st) -> const char* {
      const float* sums = fin;
      if (!sums) {
        if (const char* e = groupnorm_finalize_slabs(stats, Bn, slabs, fp, st)) return e;
        sums = fp;
      }
      return madm::groupnorm_bwd(p0, C0, p1, C1, Bn, HW, i16, sums, g, be, eps, actfn, dy, f16, pp, cp, chp, extra, out16, dx0, acc0, dx1, acc1, dgamma,
                                 dbeta, inv_scale, st);
    });
    free(part); free(coef); free(chan); free(fsum);
  }

  // ---- dgrad arena (training plans)
  const bf16* dpw(size_t off) const { return dpacked ? reinterpret_cast<const bf16*>(dpacked + off) : nullptr; }
  // conv [Cout,Cin,k,k] -> [Cin, taps*Cout] (Cout % 64 == 0), the B operand of dX = dY (*) W^T.  CoPad > 0: a few output channels, each tap
  // padded to CoPad, K to a multiple of 64 (the layout latent_im2col gives the output gradient: taps x 4 channels, zero-padded to 64)
  size_t dconv_w(const std::string& name, int Cout, int Cin, int taps, int CoPad = 0) {
    const int Cp = CoPad > 0 ? CoPad : Cout, Kpad = CoPad > 0 ? (taps * CoPad + 63) / 64 * 64 : taps * Cout;
    return entry(ctx->dgrad, "dconv:" + name, [&] {
      PackEntry e; e.kind = PK_CONV_DGRAD; e.src = name + ".weight"; e.N = Cout; e.C = Cin; e.taps = taps; e.Cpad = Cp; e.Kpad = Kpad;
      e.ldo = Kpad; e.off = ctx->dgrad.reserve(size_t(Cin) * Kpad * 2);
      return e;
    }).off;
  }
  size_t dregion(const std::string& key, size_t bytes) {
    return entry(ctx->dgrad, "dregion:" + key, [&] { PackEntry e; e.kind = PK_REGION; e.off = ctx->dgrad.reserve(bytes); return e; }).off;
  }
  // linear [N,K] (+LoRA) transposed into columns [col_off, col_off+N) of a [K, ldo] region
  void dlinear_part(const std::string& module, size_t region_off, int col_off, int N, int K, int ldo, bool lora) {
    entry(ctx->dgrad, "dlin:" + module, [&] {
      PackEntry e; e.kind = PK_LINEAR_T; e.src = module; e.N = N; e.C = K; e.ldo = ldo; e.lora = lora; e.off = region_off + size_t(col_off) * 2;
      return e;
    });
  }
  size_t dlinear_w(const std::string& module, int N, int K, bool lora) {
    return entry(ctx->dgrad, "dlin:" + module, [&] {
      PackEntry e; e.kind = PK_LINEAR_T; e.src = module; e.N = N; e.C = K; e.ldo = N; e.lora = lora; e.off = ctx->dgrad.reserve(size_t(N) * K * 2);
      return e;
    }).off;
  }
  // linear [N,K] in natural row order: the forward operand of ff.net.0.proj in the training forward
  size_t dlinear_fwd(const std::string& module, int N, int K) {
    return entry(ctx->dgrad, "dlinfwd:" + module, [&] {
      PackEntry e; e.kind = PK_LINEAR; e.src = module; e.N = N; e.C = K; e.ldo = K; e.off = ctx->dgrad.reserve(size_t(N) * K * 2);
      return e;
    }).off;
  }
  size_t dlora_a(const std::string& module, int K) {
    return entry(ctx->dgrad, "dloraA:" + module, [&] {
      PackEntry e; e.kind = PK_LORA_A; e.src = module; e.N = 16; e.C = K; e.ldo = K; e.off = ctx->dgrad.reserve(size_t(16) * K * 2);
      return e;
    }).off;
  }
  size_t dlora_bt(const std::string& module, int N) {
    return entry(ctx->dgrad, "dloraB:" + module, [&] {
      PackEntry e; e.kind = PK_LORA_BT; e.src = module; e.N = N; e.C = 16; e.ldo = N; e.off = ctx->dgrad.reserve(size_t(16) * N * 2);
      return e;
    }).off;
  }
};

// ------------------------------------------------------------------------------------------------ model pieces
struct Model {
  Builder& b;
  explicit Model(Builder& bb) : b(bb) {}
  int f16() const { return b.ctx->fp16; }
  const float* P(const std::string& n, int64_t numel = -1) { return b.mode == LAYOUT ? nullptr : b.param(n, numel); }

  // ---- time embedding projections of all 22 UNet ResBlocks, stacked along N
  std::vector<std::pair<std::string, int>> temb_layers;  // (resnet prefix, Cout)
  std::map<std::string, int> temb_off;
  int temb_total = 0;
  F32T temb_all;  // [B, temb_total]
  // ---- cross-attention K/V of all 16 transformer blocks, stacked along N
  std::vector<std::pair<std::string, int>> xattn_layers;  // (attn2 prefix, C)
  std::map<std::string, int> kv_off;
  int kv_total = 0;
  B16T kv_all;  // [B*77, kv_total]

  void enumerate_unet() {
    auto res = [&](const std::string& p, int cout) { temb_layers.push_back({p, cout}); temb_off[p] = temb_total; temb_total += cout; };
    auto att = [&](const std::string& p, int c) { xattn_layers.push_back({p + ".transformer_blocks.0.attn2", c}); kv_off[p + ".transformer_blocks.0.attn2"] = kv_total; kv_total += 2 * c; };
    const int ch[4] = {320, 640, 1280, 1280};
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 2; ++j) {
        res(kUnet + "down_blocks." + std::to_string(i) + ".resnets." + std::to_string(j), ch[i]);
        if (i < 3) att(kUnet + "down_blocks." + std::to_string(i) + ".attentions." + std::to_string(j), ch[i]);
      }
    res(kUnet + "mid_block.resnets.0", 1280);
    att(kUnet + "mid_block.attentions.0", 1280);
    res(kUnet + "mid_block.resnets.1", 1280);
    const int rev[4] = {1280, 1280, 640, 320};
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 3; ++j) {
        res(kUnet + "up_blocks." + std::to_string(i) + ".resnets." + std::to_string(j), rev[i]);
        if (i > 0) att(kUnet + "up_blocks." + std::to_string(i) + ".attentions." + std::to_string(j), rev[i]);
      }
  }

  // ---- ResnetBlock2D.  x = channel concat of x0 (and x1).  Returns fp32 (+bf16 copy if want_b16) output.
  // A 16-bit-only input (x0.f null: the VAE's high-resolution stages with fp16 operands, where the reference itself runs the
  // whole VAE in fp16) is read as is by norm1 and enters conv2 as a second K segment (conv_shortcut weights, or identity weights
  // for the plain residual); out16_only then also drops the fp32 copy of the output.
  Act resblock(const std::string& p, const Act& x0, const Act* x1, int Cout, float eps, bool has_temb, bool want_b16, bool want_s2d = false,
               bool out16_only = false) {
    const int Bn = x0.B, H = x0.H, W = x0.W, Cin = x0.C + (x1 ? x1->C : 0);
    const bool shortcut = Cin != Cout;
    const bool in16 = x0.f.bytes == 0 && x0.h.bytes != 0;  // (valid in every builder mode: sizes, not pointers)
    if (x1 && !shortcut) b.fail(MADM_EINVAL, "resblock: concat input without shortcut");
    if (in16 && (x1 || x0.h_s2d)) b.fail(MADM_EINVAL, "resblock: a 16-bit stream input must be a single linear tensor");
    B16T n1 = b.b16(size_t(x0.M()) * Cin);
    B16T raw; if (shortcut && !in16) raw = b.b16(size_t(x0.M()) * Cin);
    const Builder::GnSaved s1 = b.groupnorm(x0, x1, p + ".norm1", eps, ACT_SILU, n1.p, (shortcut && !in16) ? raw.p : nullptr, in16);
    // conv1 (+ bias + time embedding row bias) -> 16-bit intermediate (it only feeds norm2)
    Act h1 = b.act(Bn, H, W, Cout, false, true);
    {
      GemmDesc d; d.seg[0] = Builder::seg_3x3(n1.p, Bn, H, W, Cin); d.M = int(x0.M()); d.N = Cout;
      d.w = b.pw(b.conv_w(p + ".conv1", Cout, Cin, 9)); d.Nw = Cout;
      d.bias = P(p + ".conv1.bias", Cout);
      if (has_temb) { d.rowbias = temb_all.p ? temb_all.p + temb_off[p] : nullptr; d.ld_rowbias = temb_total; d.rows_per_img = H * W; }
      d.out_bf16 = h1.h.p; d.ldo16 = Cout;
      b.attach_colstats(h1, d);  // norm2 statistics come out of this epilogue
      b.gemm(d);
    }
    b.free(n1);
    B16T n2 = b.b16(size_t(x0.M()) * Cout);
    const Builder::GnSaved s2 = b.groupnorm(h1, nullptr, p + ".norm2", eps, ACT_SILU, n2.p, nullptr, /*in16=*/true);
    b.free(h1);
    Act out = b.act(Bn, H, W, Cout, !out16_only, want_b16 || want_s2d || out16_only);
    out.h_s2d = want_s2d;
    {
      GemmDesc d; d.seg[0] = Builder::seg_3x3(n2.p, Bn, H, W, Cout); d.M = int(x0.M()); d.N = Cout; d.Nw = Cout;
      if (want_s2d) { d.s2d_H = H; d.s2d_W = W; }
      if (shortcut) {  // out = conv2(n2) + conv_shortcut(x): one GEMM, K = 9*Cout + Cin
        Builder::Fused f = b.conv_plus_shortcut(p + ".conv2", p + ".conv_shortcut", Cout, Cin);
        d.nseg = 2; d.seg[1] = Builder::seg_1x1(in16 ? x0.h.p : raw.p, Bn, H, W, Cin);
        d.w = b.pw(f.w_off); d.bias = b.pf(f.b_off);
      } else if (in16) {  // out = conv2(n2) + I x: the residual is the 16-bit stream, added on the tensor core
        d.nseg = 2; d.seg[1] = Builder::seg_1x1(x0.h.p, Bn, H, W, Cout);
        d.w = b.pw(b.conv_plus_identity(p + ".conv2", Cout)); d.bias = P(p + ".conv2.bias", Cout);
      } else {
        d.w = b.pw(b.conv_w(p + ".conv2", Cout, Cout, 9)); d.bias = P(p + ".conv2.bias", Cout);
        d.residual = x0.f.p; d.ldr = Cout;
      }
      d.out_f32 = out.f.p; d.ldo32 = Cout; d.out_bf16 = out.h.p; d.ldo16 = Cout;
      b.attach_colstats(out, d);  // statistics for whichever GroupNorm consumes this block's output
      // the identity-weight segment is the reference's residual ADD: executed on the tensor core, but not algorithmic work
      b.gemm(d, (!shortcut && in16) ? 2.0 * double(d.M) * Cout * (9.0 * Cout) : -1.0);
    }
    b.free(n2);
    if (shortcut && !in16) b.free(raw);
    if (!b.recording()) return out;
    // ---- backward
    const Act xa = x0, xb = x1 ? *x1 : Act();
    const bool has_b = x1 != nullptr;
    b.tape.push_back({b.cur_stage, [=]() {
      // dgrad operands are registered whether or not this block ends up on the gradient path (the layout must not depend on it)
      const size_t w2 = b.dconv_w(p + ".conv2", Cout, Cout, 9), w1 = b.dconv_w(p + ".conv1", Cout, Cin, 9);
      const size_t wsc = shortcut ? b.dconv_w(p + ".conv_shortcut", Cout, Cin, 1) : 0;
      if (!out.gr->written) return;
      const long M = xa.M();
      B16T g16 = b.b16(size_t(M) * Cout);
      to16(out.gr->f.p, M * Cout, g16.p);
      B16T dn2 = b.b16(size_t(M) * Cout);
      { GemmDesc d; d.seg[0] = Builder::seg_3x3(g16.p, Bn, H, W, Cout); d.M = int(M); d.N = Cout; d.Nw = Cout; d.w = b.dpw(w2);
        d.out_bf16 = dn2.p; d.ldo16 = Cout; b.gemm(d); }
      B16T dh1 = b.b16(size_t(M) * Cout);
      b.groupnorm_bwd(h1, nullptr, true, s2, nullptr, p + ".norm2", eps, ACT_SILU, dn2.p, nullptr, dh1.p, nullptr, 0, nullptr, 0, nullptr, nullptr);
      b.free(dn2);
      { const bf16* src = dh1.p; float* dst = d_temb_all.p ? d_temb_all.p + temb_off.at(p) : nullptr; const int tt = temb_total, h16 = f16(), HWi = H * W;
        b.emit([=](cudaStream_t st) { return colsum_per_image(src, Bn, HWi, Cout, h16, dst, tt, st); }); }
      const bool need_a = Builder::wants_grad(xa), need_b = has_b && Builder::wants_grad(xb);
      if (need_a || need_b) {
        B16T dn1 = b.b16(size_t(M) * Cin);
        { GemmDesc d; d.seg[0] = Builder::seg_3x3(dh1.p, Bn, H, W, Cout); d.M = int(M); d.N = Cin; d.Nw = Cin; d.w = b.dpw(w1);
          d.out_bf16 = dn1.p; d.ldo16 = Cin; b.gemm(d); }
        F32T T;
        const float* extra = out.gr->f.p;  // identity residual: d(x) += d(out)
        if (shortcut) {
          T = b.f32(size_t(M) * Cin);
          GemmDesc d; d.seg[0] = Builder::seg_1x1(g16.p, Bn, H, W, Cout); d.M = int(M); d.N = Cin; d.Nw = Cin; d.w = b.dpw(wsc);
          d.out_f32 = T.p; d.ldo32 = Cin; b.gemm(d);
          extra = T.p;
        }
        int acc_a = 0, acc_b = 0;
        float* da = need_a ? b.grad(xa, &acc_a) : nullptr;
        float* db = need_b ? b.grad(xb, &acc_b) : nullptr;
        b.groupnorm_bwd(xa, has_b ? &xb : nullptr, false, s1, nullptr, p + ".norm1", eps, ACT_SILU, dn1.p, extra, nullptr, da, acc_a, db, acc_b, nullptr, nullptr);
        if (shortcut) b.free(T);
        b.free(dn1);
      }
      b.free(dh1); b.free(g16);
    }});
    return out;
  }

  // ---- Transformer2DModel (one BasicTransformerBlock): returns fp32 (+bf16) output; x is NOT freed
  Act transformer(const std::string& p, const Act& x, bool want_b16, bool want_s2d = false) {
    const bool train = b.recording();
    const int Bn = x.B, H = x.H, W = x.W, C = x.C;
    const long M = x.M();
    const int heads = 8, d_head = C / heads, n_tok = H * W;
    const float sc = 1.0f / sqrtf(float(d_head));
    const std::string tb = p + ".transformer_blocks.0";
    const int h16 = f16(), Mi = int(M);
    B16T n = b.b16(size_t(M) * C);
    const Builder::GnSaved sn = b.groupnorm(x, nullptr, p + ".norm", 1e-6f, ACT_NONE, n.p, nullptr);
    // The block's fp32 hidden state in its three versions: proj_in's output and the results of the two attention out-projections.
    // Inference updates one buffer in place (hs += GEMM); a training plan keeps every version for the LayerNorm backward.
    F32T hs0 = b.f32(size_t(M) * C), hs1 = train ? b.f32(size_t(M) * C) : hs0, hs2 = train ? b.f32(size_t(M) * C) : hs0;
    { GemmDesc d; d.seg[0] = Builder::seg_1x1(n.p, Bn, H, W, C); d.M = Mi; d.N = C; d.Nw = C;
      d.w = b.pw(b.conv_w(p + ".proj_in", C, C, 1)); d.bias = P(p + ".proj_in.bias", C); d.out_f32 = hs0.p; d.ldo32 = C; b.gemm(d); }
    b.free(n);
    auto ln = [&](const std::string& name, const float* src, bf16* y) {
      const float* g = P(name + ".weight", C); const float* be = P(name + ".bias", C);
      b.emit([=](cudaStream_t st) { return layernorm(src, 0, Mi, C, g, be, 1e-5f, y, h16, st); }, false, MADM_KIND_LAYERNORM, 0.0, double(Mi) * C * 6);
    };
    // --- self attention
    B16T l1 = b.b16(size_t(M) * C);
    ln(tb + ".norm1", hs0.p, l1.p);
    B16T qkv = b.b16(size_t(M) * 3 * C);
    { const size_t reg = b.region("qkv:" + tb, size_t(3) * C * C * 2);
      b.linear_part(tb + ".attn1.to_q", reg, 0, C, C, true);
      b.linear_part(tb + ".attn1.to_k", reg, C, C, C, true);
      b.linear_part(tb + ".attn1.to_v", reg, 2 * C, C, C, true);
      GemmDesc d; d.seg[0] = Builder::seg_plain(l1.p, M, C); d.M = Mi; d.N = 3 * C; d.Nw = 3 * C; d.w = b.pw(reg);
      d.out_bf16 = qkv.p; d.ldo16 = 3 * C; b.gemm(d); }
    b.free(l1);
    B16T att = b.b16(size_t(M) * C);
    F32T lse1, lse2;  // training: log-sum-exp rows of both attentions (for the backward)
    if (train) { lse1 = b.f32(size_t(Bn) * heads * n_tok); lse2 = b.f32(size_t(Bn) * heads * n_tok); }
    { const bf16* q = qkv.p;
      b.attention(q, 3 * C, q + C, 3 * C, q + 2 * C, 3 * C, att.p, C, Bn, heads, d_head, n_tok, n_tok, long(n_tok) * 3 * C, long(n_tok) * 3 * C,
                  long(n_tok) * C, sc, lse1.p); }
    b.free(qkv);
    { GemmDesc d; d.seg[0] = Builder::seg_plain(att.p, M, C); d.M = Mi; d.N = C; d.Nw = C;
      d.w = b.pw(b.linear_w(tb + ".attn1.to_out.0", C, C, true)); d.bias = lora_bias(tb + ".attn1.to_out.0", C);
      d.residual = hs0.p; d.ldr = C; d.out_f32 = hs1.p; d.ldo32 = C; b.gemm(d); }
    // --- cross attention (K/V precomputed for all layers in kv_all)
    B16T l2 = b.b16(size_t(M) * C);
    ln(tb + ".norm2", hs1.p, l2.p);
    B16T q2 = b.b16(size_t(M) * C);
    { GemmDesc d; d.seg[0] = Builder::seg_plain(l2.p, M, C); d.M = Mi; d.N = C; d.Nw = C;
      d.w = b.pw(b.linear_w(tb + ".attn2.to_q", C, C, true)); d.out_bf16 = q2.p; d.ldo16 = C; b.gemm(d); }
    b.free(l2);
    const B16T att2 = train ? b.b16(size_t(M) * C) : att;  // inference reuses the self-attention's output buffer (freed once, as att)
    const int kvo = kv_off[tb + ".attn2"], ldkv = kv_total;
    { const bf16* kv = kv_all.p;
      b.attention(q2.p, C, kv ? kv + kvo : nullptr, ldkv, kv ? kv + kvo + C : nullptr, ldkv, att2.p, C, Bn, heads, d_head, n_tok, 77, long(n_tok) * C,
                  long(77) * ldkv, long(n_tok) * C, sc, lse2.p); }
    b.free(q2);
    { GemmDesc d; d.seg[0] = Builder::seg_plain(att2.p, M, C); d.M = Mi; d.N = C; d.Nw = C;
      d.w = b.pw(b.linear_w(tb + ".attn2.to_out.0", C, C, true)); d.bias = lora_bias(tb + ".attn2.to_out.0", C);
      d.residual = hs1.p; d.ldr = C; d.out_f32 = hs2.p; d.ldo32 = C; b.gemm(d); }
    b.free(att);
    // --- feed-forward.  Inference: GEGLU fused in the first GEMM's epilogue.  Training keeps the pre-activation: raw = l3 W1^T + b1 in
    // natural column order (hidden | gate; weight from the dgrad arena), then the GEGLU pass.
    B16T l3 = b.b16(size_t(M) * C);
    ln(tb + ".norm3", hs2.p, l3.p);
    B16T rawff; if (train) rawff = b.b16(size_t(M) * 8 * C);
    B16T ff = b.b16(size_t(M) * 4 * C);
    if (train) {
      { GemmDesc d; d.seg[0] = Builder::seg_plain(l3.p, M, C); d.M = Mi; d.N = 8 * C; d.Nw = 8 * C;
        d.w = b.dpw(b.dlinear_fwd(tb + ".ff.net.0.proj", 8 * C, C)); d.bias = P(tb + ".ff.net.0.proj.bias", 8 * C);
        d.out_bf16 = rawff.p; d.ldo16 = 8 * C; b.gemm(d); }
      const bf16* src = rawff.p; bf16* dst = ff.p; const int Hh = 4 * C;
      b.emit([=](cudaStream_t st) { return geglu_fwd(src, M, Hh, dst, h16, st); }, false, MADM_KIND_ELEMENTWISE, 0.0, double(M) * C * 24);
    } else {
      const PackEntry& e = b.entry(b.ctx->fwd, "geglu:" + tb, [&] {
        PackEntry pe; pe.kind = PK_GEGLU; pe.src = tb + ".ff.net.0.proj.weight"; pe.src2 = tb + ".ff.net.0.proj.bias"; pe.N = 4 * C; pe.C = C;
        pe.off = b.ctx->fwd.reserve(size_t(8) * C * C * 2); pe.bias_off = b.ctx->fwd.reserve(size_t(8) * C * 4);
        return pe; });
      GemmDesc d; d.seg[0] = Builder::seg_plain(l3.p, M, C); d.M = Mi; d.N = 4 * C; d.Nw = 8 * C; d.w = b.pw(e.off);
      d.bias = b.pf(e.bias_off); d.act = ACT_GEGLU; d.out_bf16 = ff.p; d.ldo16 = 4 * C; b.gemm(d);
    }
    b.free(l3);
    B16T hsb = b.b16(size_t(M) * C);
    { GemmDesc d; d.seg[0] = Builder::seg_plain(ff.p, M, 4 * C); d.M = Mi; d.N = C; d.Nw = C;
      d.w = b.pw(b.linear_w(tb + ".ff.net.2", C, 4 * C, false)); d.bias = P(tb + ".ff.net.2.bias", C);
      d.residual = hs2.p; d.ldr = C; d.out_bf16 = hsb.p; d.ldo16 = C; b.gemm(d); }
    b.free(ff);
    b.free(hs0);
    Act out = b.act(Bn, H, W, C, true, want_b16 || want_s2d);
    out.h_s2d = want_s2d;
    { GemmDesc d; d.seg[0] = Builder::seg_1x1(hsb.p, Bn, H, W, C); d.M = Mi; d.N = C; d.Nw = C;
      if (want_s2d) { d.s2d_H = H; d.s2d_W = W; }
      d.w = b.pw(b.conv_w(p + ".proj_out", C, C, 1)); d.bias = P(p + ".proj_out.bias", C);
      d.residual = x.f.p; d.ldr = C; d.out_f32 = out.f.p; d.ldo32 = C; d.out_bf16 = out.h.p; d.ldo16 = C;
      b.attach_colstats(out, d); b.gemm(d); }
    b.free(hsb);
    if (!train) return out;
    // ---- backward
    const Act xin = x;
    b.tape.push_back({b.cur_stage, [=]() {
      const size_t w_po = b.dconv_w(p + ".proj_out", C, C, 1), w_pi = b.dconv_w(p + ".proj_in", C, C, 1);
      const size_t w_ff2 = b.dlinear_w(tb + ".ff.net.2", C, 4 * C, false), w_ff1 = b.dlinear_w(tb + ".ff.net.0.proj", 8 * C, C, false);
      const size_t w_o2 = b.dlinear_w(tb + ".attn2.to_out.0", C, C, true), w_q2 = b.dlinear_w(tb + ".attn2.to_q", C, C, true);
      const size_t w_o1 = b.dlinear_w(tb + ".attn1.to_out.0", C, C, true);
      const size_t w_qkv = b.dregion("qkv:" + tb, size_t(3) * C * C * 2);
      b.dlinear_part(tb + ".attn1.to_q", w_qkv, 0, C, C, 3 * C, true);
      b.dlinear_part(tb + ".attn1.to_k", w_qkv, C, C, C, 3 * C, true);
      b.dlinear_part(tb + ".attn1.to_v", w_qkv, 2 * C, C, C, 3 * C, true);
      if (b.mode == LAYOUT) {  // the LoRA factor operands of this block
        for (const char* m : {".attn1.to_q", ".attn1.to_k", ".attn1.to_v", ".attn1.to_out.0", ".attn2.to_q", ".attn2.to_out.0"}) { b.dlora_a(tb + m, C); b.dlora_bt(tb + m, C); }
        b.dlora_a(tb + ".attn2.to_k", 768); b.dlora_bt(tb + ".attn2.to_k", C);
        b.dlora_a(tb + ".attn2.to_v", 768); b.dlora_bt(tb + ".attn2.to_v", C);
      }
      if (!out.gr->written) return;
      // dh = gradient of the block's hidden state (fp32), carried backwards through the three residual branches
      B16T g16 = b.b16(size_t(M) * C);
      to16(out.gr->f.p, M * C, g16.p);
      F32T dh = b.f32(size_t(M) * C);
      B16T dh16 = b.b16(size_t(M) * C);
      { GemmDesc d; d.seg[0] = Builder::seg_1x1(g16.p, Bn, H, W, C); d.M = Mi; d.N = C; d.Nw = C; d.w = b.dpw(w_po);
        d.out_f32 = dh.p; d.ldo32 = C; d.out_bf16 = dh16.p; d.ldo16 = C; b.gemm(d); }
      b.free(g16);
      // --- feed-forward
      B16T dff = b.b16(size_t(M) * 4 * C);
      { GemmDesc d; d.seg[0] = Builder::seg_plain(dh16.p, M, C); d.M = Mi; d.N = 4 * C; d.Nw = 4 * C; d.w = b.dpw(w_ff2); d.out_bf16 = dff.p; d.ldo16 = 4 * C; b.gemm(d); }
      B16T draw = b.b16(size_t(M) * 8 * C);
      { const bf16* r = rawff.p; const bf16* dy = dff.p; bf16* dst = draw.p; const int Hh = 4 * C;
        b.emit([=](cudaStream_t st) { return geglu_bwd(r, dy, M, Hh, dst, h16, st); }); }
      b.free(dff);
      B16T dl = b.b16(size_t(M) * C);
      { GemmDesc d; d.seg[0] = Builder::seg_plain(draw.p, M, 8 * C); d.M = Mi; d.N = C; d.Nw = C; d.w = b.dpw(w_ff1); d.out_bf16 = dl.p; d.ldo16 = C; b.gemm(d); }
      b.free(draw);
      auto ln_bwd = [&](const std::string& name, const float* xs) {  // dh += LayerNorm'(xs) dl ; dh16 = 16-bit(dh)
        const float* g = P(name + ".weight", C); const bf16* dy = dl.p; float* dst = dh.p; bf16* d16 = dh16.p;
        b.emit([=](cudaStream_t st) -> const char* {
          return layernorm_bwd(xs, Mi, C, g, 1e-5f, dy, h16, dst, 1, st, d16);  // (writes the 16-bit copy of dh as well)
        });
      };
      ln_bwd(tb + ".norm3", hs2.p);
      F32T ascr = b.f32(attention_bwd_scratch_floats(Bn, heads, d_head, n_tok, n_tok > 77 ? n_tok : 77) + attention_bwd_scratch_floats(Bn, heads, d_head, n_tok, 77));
      // --- cross attention
      B16T datt = b.b16(size_t(M) * C);
      { GemmDesc d; d.seg[0] = Builder::seg_plain(dh16.p, M, C); d.M = Mi; d.N = C; d.Nw = C; d.w = b.dpw(w_o2); d.out_bf16 = datt.p; d.ldo16 = C; b.gemm(d); }
      lora_wgrad(tb + ".attn2.to_out.0", att2.p, C, dh16.p, C, M, C, C);
      B16T dq2 = b.b16(size_t(M) * C);
      { const bf16* kv = kv_all.p; bf16* dkv = dkv_all.p;
        b.attention_bwd(q2.p, C, kv ? kv + kvo : nullptr, ldkv, kv ? kv + kvo + C : nullptr, ldkv, att2.p, C, datt.p, C, dq2.p, C, dkv ? dkv + kvo : nullptr,
                        ldkv, dkv ? dkv + kvo + C : nullptr, ldkv, Bn, heads, d_head, n_tok, 77, long(n_tok) * C, long(77) * ldkv, long(77) * ldkv,
                        long(n_tok) * C, long(n_tok) * C, long(n_tok) * C, long(77) * ldkv, long(77) * ldkv, sc, ascr.p, lse2.p); }
      lora_wgrad(tb + ".attn2.to_q", l2.p, C, dq2.p, C, M, C, C);
      lora_wgrad(tb + ".attn2.to_k", ctx16_saved.p, 768, dkv_all.p ? dkv_all.p + kvo : nullptr, ldkv, long(Bn) * 77, C, 768);
      lora_wgrad(tb + ".attn2.to_v", ctx16_saved.p, 768, dkv_all.p ? dkv_all.p + kvo + C : nullptr, ldkv, long(Bn) * 77, C, 768);
      { GemmDesc d; d.seg[0] = Builder::seg_plain(dq2.p, M, C); d.M = Mi; d.N = C; d.Nw = C; d.w = b.dpw(w_q2); d.out_bf16 = dl.p; d.ldo16 = C; b.gemm(d); }
      b.free(dq2);
      ln_bwd(tb + ".norm2", hs1.p);
      // --- self attention
      { GemmDesc d; d.seg[0] = Builder::seg_plain(dh16.p, M, C); d.M = Mi; d.N = C; d.Nw = C; d.w = b.dpw(w_o1); d.out_bf16 = datt.p; d.ldo16 = C; b.gemm(d); }
      lora_wgrad(tb + ".attn1.to_out.0", att.p, C, dh16.p, C, M, C, C);
      B16T dqkv = b.b16(size_t(M) * 3 * C);
      { const bf16* q = qkv.p; bf16* dq = dqkv.p;
        b.attention_bwd(q, 3 * C, q + C, 3 * C, q + 2 * C, 3 * C, att.p, C, datt.p, C, dq, 3 * C, dq + C, 3 * C, dq + 2 * C, 3 * C, Bn, heads, d_head, n_tok,
                        n_tok, long(n_tok) * 3 * C, long(n_tok) * 3 * C, long(n_tok) * 3 * C, long(n_tok) * C, long(n_tok) * C, long(n_tok) * 3 * C,
                        long(n_tok) * 3 * C, long(n_tok) * 3 * C, sc, ascr.p, lse1.p); }
      b.free(datt);
      lora_wgrad(tb + ".attn1.to_q", l1.p, C, dqkv.p, 3 * C, M, C, C);
      lora_wgrad(tb + ".attn1.to_k", l1.p, C, dqkv.p ? dqkv.p + C : nullptr, 3 * C, M, C, C);
      lora_wgrad(tb + ".attn1.to_v", l1.p, C, dqkv.p ? dqkv.p + 2 * C : nullptr, 3 * C, M, C, C);
      { GemmDesc d; d.seg[0] = Builder::seg_plain(dqkv.p, M, 3 * C); d.M = Mi; d.N = C; d.Nw = C; d.w = b.dpw(w_qkv); d.out_bf16 = dl.p; d.ldo16 = C; b.gemm(d); }
      b.free(dqkv); b.free(ascr);
      ln_bwd(tb + ".norm1", hs0.p);
      // --- proj_in, GroupNorm; the block's residual adds d(out) to d(x)
      if (Builder::wants_grad(xin)) {
        B16T dn = b.b16(size_t(M) * C);
        { GemmDesc d; d.seg[0] = Builder::seg_1x1(dh16.p, Bn, H, W, C); d.M = Mi; d.N = C; d.Nw = C; d.w = b.dpw(w_pi); d.out_bf16 = dn.p; d.ldo16 = C; b.gemm(d); }
        int acc = 0;
        float* dx = b.grad(xin, &acc);
        b.groupnorm_bwd(xin, nullptr, false, sn, nullptr, p + ".norm", 1e-6f, ACT_NONE, dn.p, out.gr->f.p, nullptr, dx, acc, nullptr, 0, nullptr, nullptr);
        b.free(dn);
      }
      b.free(dl); b.free(dh16); b.free(dh);
    }});
    return out;
  }

  // bias of a (possibly LoRA-wrapped) Linear: "<m>.base_layer.bias" if wrapped else "<m>.bias"
  const float* lora_bias(const std::string& module, int n) {
    if (b.mode == LAYOUT) return nullptr;
    if (b.find(module + ".base_layer.bias")) return b.param(module + ".base_layer.bias", n);
    return b.param(module + ".bias", n);
  }

  Act downsample(const std::string& p, const Act& x, bool pad1, bool out16_only = false) {
    const int Bn = x.B, H = x.H, W = x.W, C = x.C;
    // the producer's epilogue writes the stride-2 conv's space-to-depth operand (resblock / transformer with want_s2d)
    if (!x.h_s2d) b.fail(MADM_EINVAL, "downsample: the input has no space-to-depth operand");
    Act out = b.act(Bn, H / 2, W / 2, C, !out16_only, out16_only);
    { GemmDesc d; d.seg[0] = Builder::seg_s2(x.h.p, Bn, H / 2, W / 2, C, pad1); d.M = int(out.M()); d.N = C; d.Nw = C;
      d.w = b.pw(b.conv_w(p + ".conv", C, C, 9)); d.bias = P(p + ".conv.bias", C);
      if (out16_only) { d.out_bf16 = out.h.p; d.ldo16 = C; } else { d.out_f32 = out.f.p; d.ldo32 = C; }
      b.attach_colstats(out, d); b.gemm(d); }
    if (!b.recording()) return out;
    const Act xin = x;
    b.tape.push_back({b.cur_stage, [=]() {
      const size_t w = b.dconv_w(p + ".conv", C, C, 9);
      if (!out.gr->written || !Builder::wants_grad(xin)) return;
      // input gradient of the stride-2 conv: zero-stuff d(out) onto the input grid, then the stride-1 dgrad GEMM with mirrored taps
      const long Mo = out.M(), Mx = xin.M();
      B16T g16 = b.b16(size_t(Mo) * C);
      to16(out.gr->f.p, Mo * C, g16.p);
      B16T z = b.b16(size_t(Mx) * C);
      { const bf16* src = g16.p; bf16* dst = z.p; b.emit([=](cudaStream_t st) { return zero_stuff2x(src, Bn, H / 2, W / 2, C, dst, st); }); }
      int acc = 0;
      float* dx = b.grad(xin, &acc);
      { GemmDesc d; d.seg[0] = Builder::seg_3x3(z.p, Bn, H, W, C); d.M = int(Mx); d.N = C; d.Nw = C; d.w = b.dpw(w);
        if (acc) { d.residual = dx; d.ldr = C; }
        d.out_f32 = dx; d.ldo32 = C; b.gemm(d); }
      b.free(z); b.free(g16);
    }});
    return out;
  }

  // Upsample2D: nearest 2x (materialised as a 16-bit operand) + conv3x3.  A 16-bit-only input (x.f empty: the VAE decoder's
  // high-resolution stream) is replicated as is; out16_only keeps the result on the 16-bit stream.
  Act upsample(const std::string& p, const Act& x, bool out16_only = false) {
    const int Bn = x.B, H = x.H, W = x.W, C = x.C;
    const bool in16 = x.f.bytes == 0 && x.h.bytes != 0;
    B16T up = b.b16(size_t(x.M()) * 4 * C);
    { const float* src = x.f.p; const bf16* src16 = x.h.p; bf16* dst = up.p;
      const int h16 = f16();
      if (in16) b.emit([=](cudaStream_t st) { return upsample_nearest2x_16(src16, Bn, H, W, C, dst, st); }, false, MADM_KIND_ELEMENTWISE, 0.0,
                       double(x.M()) * C * 10);
      else b.emit([=](cudaStream_t st) { return upsample_nearest2x(src, Bn, H, W, C, dst, h16, st); }, false, MADM_KIND_ELEMENTWISE, 0.0,
                  double(x.M()) * C * 12); }
    Act out = b.act(Bn, 2 * H, 2 * W, C, !out16_only, out16_only);
    { GemmDesc d; d.seg[0] = Builder::seg_3x3(up.p, Bn, 2 * H, 2 * W, C); d.M = int(out.M()); d.N = C; d.Nw = C;
      d.w = b.pw(b.conv_w(p + ".conv", C, C, 9)); d.bias = P(p + ".conv.bias", C);
      if (out16_only) { d.out_bf16 = out.h.p; d.ldo16 = C; } else { d.out_f32 = out.f.p; d.ldo32 = C; }
      b.attach_colstats(out, d); b.gemm(d); }
    b.free(up);
    if (!b.recording()) return out;
    const Act xin = x;
    b.tape.push_back({b.cur_stage, [=]() {
      const size_t w = b.dconv_w(p + ".conv", C, C, 9);
      if (!out.gr->written || !Builder::wants_grad(xin)) return;
      const long Mo = out.M();
      B16T g16 = b.b16(size_t(Mo) * C);
      to16(out.gr->f.p, Mo * C, g16.p);
      F32T dup = b.f32(size_t(Mo) * C);
      { GemmDesc d; d.seg[0] = Builder::seg_3x3(g16.p, Bn, 2 * H, 2 * W, C); d.M = int(Mo); d.N = C; d.Nw = C; d.w = b.dpw(w);
        d.out_f32 = dup.p; d.ldo32 = C; b.gemm(d); }
      int acc = 0;
      float* dx = b.grad(xin, &acc);
      { const float* src = dup.p; b.emit([=](cudaStream_t st) { return sum2x2(src, Bn, H, W, C, dx, acc, st); }); }
      b.free(dup); b.free(g16);
    }});
    return out;
  }

  // ---- VAE mid-block attention (1 head, d = 512, 4096 tokens): QK^T / softmax / PV as three GEMM passes per image
  Act vae_attention(const std::string& p, const Act& x) {
    const int Bn = x.B, H = x.H, W = x.W, C = x.C, T = H * W;
    const long M = x.M();
    B16T n = b.b16(size_t(M) * C);
    b.groupnorm(x, nullptr, p + ".group_norm", 1e-6f, ACT_NONE, n.p, nullptr);
    B16T qk = b.b16(size_t(M) * 2 * C);
    { const size_t reg = b.region("vae_qk:" + p, size_t(2) * C * C * 2);
      b.linear_part(p + ".to_q", reg, 0, C, C, false);
      b.linear_part(p + ".to_k", reg, C, C, C, false);
      const size_t breg = b.region("vae_qk_bias:" + p, size_t(2) * C * 4);
      b.f32_part(p + ".to_q.bias", breg, 0, C);
      b.f32_part(p + ".to_k.bias", breg, C, C);
      GemmDesc d; d.seg[0] = Builder::seg_plain(n.p, M, C); d.M = int(M); d.N = 2 * C; d.Nw = 2 * C; d.w = b.pw(reg); d.bias = b.pf(breg);
      d.out_bf16 = qk.p; d.ldo16 = 2 * C; b.gemm(d); }
    const size_t wv = b.linear_w(p + ".to_v", C, C, false);
    B16T o = b.b16(size_t(M) * C);
    B16T vt = b.b16(size_t(C) * T);
    F32T S = b.f32(size_t(T) * T);
    B16T Pm = b.b16(size_t(T) * T);
    for (int i = 0; i < Bn; ++i) {
      const bf16* ni = n.p ? n.p + size_t(i) * T * C : nullptr;
      const bf16* qi = qk.p ? qk.p + size_t(i) * T * 2 * C : nullptr;
      { // V^T[c, t] = sum_k Wv[c,k] * n[t,k]   (bias added after PV: softmax rows sum to 1)
        GemmDesc d; d.seg[0] = Builder::seg_plain(b.pw(wv), C, C); d.M = C; d.N = T; d.Nw = T; d.w = ni; d.ldw = C;
        d.out_bf16 = vt.p; d.ldo16 = T; b.gemm(d); }
      { GemmDesc d; d.seg[0] = Builder::seg_plain(qi, T, C, 2 * C); d.M = T; d.N = T; d.Nw = T; d.w = qi ? qi + C : nullptr; d.ldw = 2 * C;
        d.alpha = 1.0f / sqrtf(float(C)); d.out_f32 = S.p; d.ldo32 = T; b.gemm(d); }
      { const float* s = S.p; bf16* pm = Pm.p;
        const int h16 = f16();
        b.emit([=](cudaStream_t st) { return softmax_rows(s, T, T, pm, h16, st); }, false, MADM_KIND_ELEMENTWISE, 0.0, double(T) * T * 6); }
      { GemmDesc d; d.seg[0] = Builder::seg_plain(Pm.p, T, T); d.M = T; d.N = C; d.Nw = C; d.w = vt.p; d.ldw = T;
        d.bias = P(p + ".to_v.bias", C); d.out_bf16 = o.p ? o.p + size_t(i) * T * C : nullptr; d.ldo16 = C; b.gemm(d); }
    }
    b.free(Pm); b.free(S); b.free(vt); b.free(qk); b.free(n);
    Act out = b.act(Bn, H, W, C, true, false);
    { GemmDesc d; d.seg[0] = Builder::seg_plain(o.p, M, C); d.M = int(M); d.N = C; d.Nw = C;
      d.w = b.pw(b.linear_w(p + ".to_out.0", C, C, false)); d.bias = P(p + ".to_out.0.bias", C);
      d.residual = x.f.p; d.ldr = C; d.out_f32 = out.f.p; d.ldo32 = C; b.attach_colstats(out, d); b.gemm(d); }
    b.free(o);
    return out;
  }

  // persistent cross-stage buffers
  bool s0() const { return b.ctx->variant == MADM_VARIANT_S0; }

  Act enc_tap;           // [B,128,128,512] fp32 + bf16; MADM_VARIANT_S0: the decoded image, C = 3, `h` = zero-padded rows [B*512*512, 64]
  F32T unet_sample;      // MADM_VARIANT_S0: [B*4096, 4] UNet final output (NHWC)
  F32T latents;          // [B*4096, 4]
  Act unet_tap[3];       // 64x64x320, 32x32x640, 16x16x1280 (fp32 + bf16)

  void nchw_debug(const Act& a, int which) {  // taps[which] if requested
    IoBind* io = b.io;
    const float* src = a.f.p; const int Bn = a.B, HW = a.HW(), C = a.C;
    b.emit([=](cudaStream_t st) -> const char* {
      float* dst = io->a.taps[which];
      return dst ? nhwc_to_nchw(src, Bn, HW, C, dst, st) : nullptr;
    }, true);
  }


  // ============================================================================================== training path (SURVEY §8 row f-3)
  // A block's forward is the same builder function for inference and training; in a training plan (Builder::recording()) it also records
  // its backward on the tape.  The training forward differs in three data choices: nothing is freed in the differentiated stages, the
  // transformer's hidden state is not updated in place (LayerNorm backward needs every version), and GEGLU keeps its pre-activation
  // (natural-order feed-forward weight from the dgrad arena + one elementwise pass).
  F32T d_temb_all;   // [B, temb_total] gradient of all 22 time_emb_proj outputs
  B16T dkv_all;      // [B*77, kv_total] gradient of all cross-attention K / V
  F32T emb_saved;    // [B,1280] time_embedding output before (+ cond_emb, SiLU)
  B16T ctx16_saved;  // [B*77,768] 16-bit cond_inputs

  void to16(const float* src, long n, bf16* dst) {
    const int h16 = f16();
    b.emit([=](cudaStream_t st) { return f32_to_bf16(src, nullptr, n, ACT_NONE, dst, nullptr, h16, st); });
  }
  void check_lora_rank(const std::string& module) {
    if (b.mode == LAYOUT || b.adapter.empty()) return;
    const ParamRef* A = b.find(module + ".lora_A." + b.adapter + ".weight");
    if (A && A->shape[0] != 16) b.fail(MADM_EINVAL, "training path: LoRA rank must be 16 (" + module + ")");
  }
  // gradients of one LoRA-wrapped linear y = (W + s B A) x: dB = s dY^T (X A^T), dA = s (dY B)^T X.  X [M,K] pitch ldx, dY [M,N] pitch ldy.
  void lora_wgrad(const std::string& module, const bf16* X, int ldx, const bf16* dY, int ldy, long M, int N, int K) {
    const size_t oa = b.dlora_a(module, K), ob = b.dlora_bt(module, N);  // (registered in the layout pass whatever the adapter)
    if (b.mode == LAYOUT) return;
    if (b.adapter.empty()) return;
    float* gA = b.grad_buf(module + ".lora_A." + b.adapter + ".weight");
    float* gB = b.grad_buf(module + ".lora_B." + b.adapter + ".weight");
    if (!gA && !gB) return;
    check_lora_rank(module);
    const float alpha = b.lora_scale / b.loss_scale;
    const int h16 = f16(), Mi = int(M);
    if (!lora_grads_supported(N, K))
      b.fail(MADM_EINVAL, "training path: no LoRA gradient kernel for N = " + std::to_string(N) + ", K = " + std::to_string(K) + " (" + module + ")");
    // both factor gradients in one kernel + one reduce (wgrad.cu)
    F32T scr = b.f32(lora_grads_scratch_floats(Mi, N, K));
    const bf16* a16 = b.dpw(oa); const bf16* bt16 = b.dpw(ob); float* sp = scr.p;
    b.emit([=](cudaStream_t st) { return lora_grads(X, ldx, dY, ldy, a16, bt16, Mi, N, K, alpha, gA, gB, sp, h16, st); });
    b.free(scr);
  }

  // =========================================================================== VAE encoder
  void build_vae() {
    b.cur_stage = MADM_STAGE_VAE;
    const int Bn = b.B, R = 512;
    const std::string e = kVae + "encoder.";
    IoBind* io = b.io;
    B16T col = b.b16(size_t(Bn) * R * R * 64);
    { bf16* dst = col.p; const int h16 = f16();
      b.emit([=](cudaStream_t st) { return image_im2col(io->a.img, Bn, R, R, dst, io->a.range_flag, h16, st, io->a.flags & MADM_FLAG_IMG_NORMALISED); }); }
    // fp16 operands: the residual stream of the 512^2 and 256^2 stages (3/4 of the VAE's bytes) is kept in fp16 like the
    // reference's VAE (AutoencoderKL loaded with torch_dtype=float16, ldm_diffusers.py:246-249); bf16 keeps the fp32 stream.
    const bool s16 = f16();
    Act x = b.act(Bn, R, R, 128, !s16, s16);
    { GemmDesc d; d.seg[0] = Builder::seg_plain(col.p, long(Bn) * R * R, 64); d.M = Bn * R * R; d.N = 128; d.Nw = 128;
      d.w = b.pw(b.conv_w(e + "conv_in", 128, 3, 9, /*Cpad=*/3)); d.bias = P(e + "conv_in.bias", 128);
      if (s16) { d.out_bf16 = x.h.p; d.ldo16 = 128; } else { d.out_f32 = x.f.p; d.ldo32 = 128; }
      b.attach_colstats(x, d);
      b.gemm(d, 2.0 * double(d.M) * 128 * 27); }
    b.free(col);
    const int ch[4] = {128, 256, 512, 512};
    int index = 0;
    for (int i = 0; i < 4; ++i) {
      for (int j = 0; j < 2; ++j) {
        const std::string p = e + "down_blocks." + std::to_string(i) + ".resnets." + std::to_string(j);
        ++index;
        const bool is_tap = index == 5 && !s0();  // encoder_block_indices=[5] (counter increments before the check, :289-293); [] in the s0 variant
        const bool feeds_down = (j == 1 && i < 3);  // its output is the input of this stage's stride-2 conv
        const bool o16 = s16 && i < 2;  // this block's output stays on the 16-bit stream
        Act y = resblock(p, x, nullptr, ch[i], 1e-6f, false, is_tap, feeds_down && !is_tap, o16);
        b.free(x);
        x = y;
        if (is_tap) {  // keep the tap alive for the projection stage
          enc_tap = x;
          b.pin(enc_tap);
          nchw_debug(enc_tap, 0);
        }
      }
      if (i < 3) {
        Act y = downsample(e + "down_blocks." + std::to_string(i) + ".downsamplers.0", x, /*pad1=*/false, /*out16_only=*/s16 && i < 2);
        b.free(x);
        x = y;
      }
    }
    {
      Act y = resblock(e + "mid_block.resnets.0", x, nullptr, 512, 1e-6f, false, false); b.free(x); x = y;
      y = vae_attention(e + "mid_block.attentions.0", x); b.free(x); x = y;
      y = resblock(e + "mid_block.resnets.1", x, nullptr, 512, 1e-6f, false, false); b.free(x); x = y;
    }
    B16T n = b.b16(size_t(x.M()) * 512);
    b.groupnorm(x, nullptr, e + "conv_norm_out", 1e-6f, ACT_SILU, n.p, nullptr);
    latents = b.f32(size_t(x.M()) * 4);
    { const PackEntry& pe = b.entry(b.ctx->fwd, "vae_head", [&] {
        PackEntry q; q.kind = PK_VAE_HEAD; q.src = e + "conv_out.weight"; q.src2 = e + "conv_out.bias"; q.src3 = kVae + "quant_conv.weight";
        q.src4 = kVae + "quant_conv.bias"; q.C = 512; q.off = b.ctx->fwd.reserve(size_t(16) * 9 * 512 * 2); q.bias_off = b.ctx->fwd.reserve(64);
        return q; });
      GemmDesc d; d.seg[0] = Builder::seg_3x3(n.p, Bn, x.H, x.W, 512); d.M = int(x.M()); d.N = 4; d.Nw = 16; d.w = b.pw(pe.off);
      d.bias = b.pf(pe.bias_off); d.out_f32 = latents.p; d.ldo32 = 4; d.bn = 16;
      b.gemm(d, 2.0 * double(d.M) * 8 * (9 * 512 + 8)); }  // algorithmic: conv_out 512->8 (3x3) + quant_conv 8->8
    b.free(n);
    b.free(x);
    { const float* src = latents.p;
      b.emit([=](cudaStream_t st) -> const char* {
        return io->a.latents ? nhwc_to_nchw(src, Bn, 64 * 64, 4, io->a.latents, st) : nullptr; }, true); }
  }

  // =========================================================================== UNet
  void build_unet() {
    b.cur_stage = MADM_STAGE_UNET;
    const int Bn = b.B;
    IoBind* io = b.io;
    // ---- q-sample (or external noisy latents) + conv_in im2col
    F32T noisy = b.f32(size_t(Bn) * 4096 * 4);
    B16T col = b.b16(size_t(Bn) * 4096 * 64);
    {
      const float* lat = latents.p; float* nz = noisy.p; bf16* cdst = col.p; const float* ac = b.ctx->alphas_cumprod;
      b.emit([=](cudaStream_t st) -> const char* {
        if (io->a.noisy_latents_in) return nchw_to_nhwc4(io->a.noisy_latents_in, Bn, 4096, nz, st);
        return qsample(lat, io->a.shared_noise, io->a.timesteps, ac, Bn, 4096, nz, io->a.noisy_latents, st);
      });
      const int h16 = f16();
      b.emit([=](cudaStream_t st) { return latent_im2col(nz, Bn, 64, 64, cdst, h16, st); });
    }
    // ---- time embedding: sinusoid -> linear_1 -> SiLU -> linear_2 (+ cond_emb) -> SiLU -> all 22 time_emb_proj at once
    B16T sinus = b.b16(size_t(Bn) * 320);
    { bf16* dst = sinus.p; const int h16 = f16(); b.emit([=](cudaStream_t st) { return timestep_sinusoid(io->a.timesteps, Bn, dst, h16, st); }); }
    B16T e1 = b.b16(size_t(Bn) * 1280);
    { GemmDesc d; d.seg[0] = Builder::seg_plain(sinus.p, Bn, 320); d.M = Bn; d.N = 1280; d.Nw = 1280;
      d.w = b.pw(b.linear_w(kUnet + "time_embedding.linear_1", 1280, 320, false)); d.bias = P(kUnet + "time_embedding.linear_1.bias", 1280);
      d.act = ACT_SILU; d.out_bf16 = e1.p; d.ldo16 = 1280; b.gemm(d); }
    emb_saved = b.f32(size_t(Bn) * 1280);
    { GemmDesc d; d.seg[0] = Builder::seg_plain(e1.p, Bn, 1280); d.M = Bn; d.N = 1280; d.Nw = 1280;
      d.w = b.pw(b.linear_w(kUnet + "time_embedding.linear_2", 1280, 1280, false)); d.bias = P(kUnet + "time_embedding.linear_2.bias", 1280);
      d.out_f32 = emb_saved.p; d.ldo32 = 1280; b.gemm(d); }
    B16T emb_act = b.b16(size_t(Bn) * 1280);
    { const float* src = emb_saved.p; bf16* dst = emb_act.p; const int h16 = f16();
      b.emit([=](cudaStream_t st) { return f32_to_bf16(src, io->a.cond_emb, long(Bn) * 1280, ACT_SILU, dst, nullptr, h16, st); }); }
    temb_all = b.f32(size_t(Bn) * temb_total);
    { const size_t reg = b.region("temb_w", size_t(temb_total) * 1280 * 2);
      const size_t breg = b.region("temb_b", size_t(temb_total) * 4);
      for (auto& l : temb_layers) {
        b.linear_part(l.first + ".time_emb_proj", reg, temb_off[l.first], l.second, 1280, false);
        b.f32_part(l.first + ".time_emb_proj.bias", breg, temb_off[l.first], l.second);
      }
      GemmDesc d; d.seg[0] = Builder::seg_plain(emb_act.p, Bn, 1280); d.M = Bn; d.N = temb_total; d.Nw = temb_total; d.w = b.pw(reg);
      d.bias = b.pf(breg); d.out_f32 = temb_all.p; d.ldo32 = temb_total; b.gemm(d); }
    b.free(sinus); b.free(e1); b.free(emb_saved); b.free(emb_act);
    // ---- cross-attention K/V of every transformer block in one GEMM
    ctx16_saved = b.b16(size_t(Bn) * 77 * 768);
    { bf16* dst = ctx16_saved.p; const int h16 = f16();
      b.emit([=](cudaStream_t st) { return f32_to_bf16(io->a.cond_inputs, nullptr, long(Bn) * 77 * 768, ACT_NONE, dst, nullptr, h16, st); }); }
    kv_all = b.b16(size_t(Bn) * 77 * kv_total);
    { const size_t reg = b.region("xattn_kv", size_t(kv_total) * 768 * 2);
      for (auto& l : xattn_layers) {
        b.linear_part(l.first + ".to_k", reg, kv_off[l.first], l.second, 768, true);
        b.linear_part(l.first + ".to_v", reg, kv_off[l.first] + l.second, l.second, 768, true);
      }
      GemmDesc d; d.seg[0] = Builder::seg_plain(ctx16_saved.p, long(Bn) * 77, 768); d.M = Bn * 77; d.N = kv_total; d.Nw = kv_total; d.w = b.pw(reg);
      d.out_bf16 = kv_all.p; d.ldo16 = kv_total; b.gemm(d); }
    b.free(ctx16_saved);
    if (b.recording()) {
      d_temb_all = b.f32(size_t(Bn) * temb_total);
      dkv_all = b.b16(size_t(Bn) * 77 * kv_total);
      // ---- backward of the prologue (runs last): time path -> d(cond_emb), stacked K/V projections -> d(cond_inputs)
      b.tape.push_back({b.cur_stage, [=]() {
        const size_t wt = b.dregion("temb_w", size_t(temb_total) * 1280 * 2);
        for (auto& l : temb_layers) b.dlinear_part(l.first + ".time_emb_proj", wt, temb_off[l.first], l.second, 1280, temb_total, false);
        const size_t wk = b.dregion("xattn_kv", size_t(kv_total) * 768 * 2);
        for (auto& l : xattn_layers) {
          b.dlinear_part(l.first + ".to_k", wk, kv_off[l.first], l.second, 768, kv_total, true);
          b.dlinear_part(l.first + ".to_v", wk, kv_off[l.first] + l.second, l.second, 768, kv_total, true);
        }
        const float inv = 1.0f / b.loss_scale;
        {  // d(emb + cond_emb) = (d_temb_all W_temb) * silu'(emb + cond_emb)
          B16T dt16 = b.b16(size_t(Bn) * temb_total);
          to16(d_temb_all.p, long(Bn) * temb_total, dt16.p);
          F32T dact = b.f32(size_t(Bn) * 1280);
          { GemmDesc d; d.seg[0] = Builder::seg_plain(dt16.p, Bn, temb_total); d.M = Bn; d.N = 1280; d.Nw = 1280; d.w = b.dpw(wt);
            d.out_f32 = dact.p; d.ldo32 = 1280; b.gemm(d); }
          { const float* da = dact.p; const float* em = emb_saved.p;
            b.emit([=](cudaStream_t st) -> const char* {
              if (!io->b.d_cond_emb) return nullptr;
              if (!io->b.cond_emb) return "madm_backward: cond_emb is required for d_cond_emb";
              return temb_silu_bwd(da, em, io->b.cond_emb, long(Bn) * 1280, inv, io->b.d_cond_emb, st); }); }
          b.free(dact); b.free(dt16);
        }
        {  // d(cond_inputs) = dkv_all W_kv : fp32 [B*77, 768] into a scratch, copied out if the caller asked for it
          F32T dc = b.f32(size_t(Bn) * 77 * 768);
          { GemmDesc d; d.seg[0] = Builder::seg_plain(dkv_all.p, long(Bn) * 77, kv_total); d.M = Bn * 77; d.N = 768; d.Nw = 768; d.w = b.dpw(wk);
            d.out_f32 = dc.p; d.ldo32 = 768; b.gemm(d); }
          { const float* src = dc.p; const long n = long(Bn) * 77 * 768;
            b.emit([=](cudaStream_t st) -> const char* {
              if (!io->b.d_cond_inputs) return nullptr;
              return scale_copy_f32(src, n, inv, io->b.d_cond_inputs, st); }); }
          b.free(dc);
        }
      }});
    }
    // ---- conv_in (nothing trainable upstream: its output stops the gradient)
    Act x = b.act(Bn, 64, 64, 320, true, false);
    if (b.recording()) x.gr->stop = true;
    { GemmDesc d; d.seg[0] = Builder::seg_plain(col.p, long(Bn) * 4096, 64); d.M = Bn * 4096; d.N = 320; d.Nw = 320;
      d.w = b.pw(b.conv_w(kUnet + "conv_in", 320, 4, 9, /*Cpad=*/4)); d.bias = P(kUnet + "conv_in.bias", 320); d.out_f32 = x.f.p; d.ldo32 = 320;
      b.attach_colstats(x, d);
      b.gemm(d, 2.0 * double(d.M) * 320 * 36); }
    b.free(col); b.free(noisy);
    // ---- down path
    std::vector<Act> skips;
    skips.push_back(x);
    const int ch[4] = {320, 640, 1280, 1280};
    for (int i = 0; i < 4; ++i) {
      const std::string blk = kUnet + "down_blocks." + std::to_string(i);
      for (int j = 0; j < 2; ++j) {
        Act y = resblock(blk + ".resnets." + std::to_string(j), x, nullptr, ch[i], 1e-5f, true, false);
        if (i < 3) { Act z = transformer(blk + ".attentions." + std::to_string(j), y, false, /*want_s2d=*/j == 1); b.free(y); y = z; }
        x = y;
        skips.push_back(x);
      }
      if (i < 3) { x = downsample(blk + ".downsamplers.0", x, /*pad1=*/true); skips.push_back(x); }
    }
    // ---- mid
    {
      Act y = resblock(kUnet + "mid_block.resnets.0", x, nullptr, 1280, 1e-5f, true, false);
      Act z = transformer(kUnet + "mid_block.attentions.0", y, false); b.free(y);
      x = resblock(kUnet + "mid_block.resnets.1", z, nullptr, 1280, 1e-5f, true, false); b.free(z);
      // (the mid input is skips.back(); it is freed when popped below)
    }
    // ---- up path; taps after layers 5, 8, 11 (unet_block_indices=[5,8,11], type 'after')
    const int rev[4] = {1280, 1280, 640, 320};
    int idx = 0;
    for (int i = 0; i < 4; ++i) {
      const std::string blk = kUnet + "up_blocks." + std::to_string(i);
      for (int j = 0; j < 3; ++j) {
        Act skip = skips.back(); skips.pop_back();
        const bool is_tap = (idx == 5 || idx == 8 || idx == 11);
        Act y = resblock(blk + ".resnets." + std::to_string(j), x, &skip, rev[i], 1e-5f, true, is_tap && i == 0);
        b.free(x); b.free(skip);
        if (i > 0) { Act z = transformer(blk + ".attentions." + std::to_string(j), y, is_tap); b.free(y); y = z; }
        x = y;
        if (is_tap) {
          const int t = (idx == 5) ? 2 : (idx == 8 ? 1 : 0);
          unet_tap[t] = x;
          b.pin(x);
          nchw_debug(x, 1 + t);
          build_proj_early(1 + t);  // this tap's projection can run beside the rest of the UNet
        }
        ++idx;
      }
      if (i < 3) {
        Act y = upsample(blk + ".upsamplers.0", x);
        b.free(x);  // (pinned taps stay alive for the projection stage)
        x = y;
      }
    }
    b.free(temb_all);
    b.free(kv_all);
  }

  // =========================================================================== UNet tail + VAE decoder (MADM_VARIANT_S0)
  // unet.conv_norm_out / conv_act / conv_out (reference ldm_diffusers.py:608-611) -> sample [B,4,64,64] ('before_vae.decoder'), then
  // vae_decoder(latents=sample, output_final=True) (ldm_diffusers.py:192, :314-346): 1/0.18215 scale, post_quant_conv, conv_in,
  // mid block, 4 up blocks x 3 ResBlocks (512, 512, 256, 128 channels) with nearest-2x + conv between, GN + SiLU + conv 128 -> 3.
  // The decoded image (not clipped, ldm_diffusers.py:199) becomes the first feature of forward_features.
  // Training plans: the UNet tail carries grad (the meta-arch's vae_decoder_loss differentiates 'before_vae.decoder') and records its backward;
  // the decoder body runs without gradient and its image is detached (ldm_diffusers.py:191-201), so it records nothing.
  void build_dec() {
    b.cur_stage = MADM_STAGE_DEC;
    const int Bn = b.B;
    IoBind* io = b.io;
    const int h16 = f16();
    {
      const Act& x = unet_tap[0];  // output of up layer 11 (64x64x320), the UNet's last hidden state
      B16T n = b.b16(size_t(x.M()) * 320);
      const Builder::GnSaved sv = b.groupnorm(x, nullptr, kUnet + "conv_norm_out", 1e-5f, ACT_SILU, n.p, nullptr);
      unet_sample = b.f32(size_t(x.M()) * 4);
      GemmDesc d; d.seg[0] = Builder::seg_3x3(n.p, Bn, 64, 64, 320); d.M = int(x.M()); d.N = 4; d.Nw = 4; d.bn = 16;
      d.w = b.pw(b.conv_w(kUnet + "conv_out", 4, 320, 9)); d.bias = P(kUnet + "conv_out.bias", 4); d.out_f32 = unet_sample.p; d.ldo32 = 4;
      b.gemm(d);
      b.free(n);
      { const float* src = unet_sample.p;
        b.emit([=](cudaStream_t st) -> const char* {
          return io->a.unet_sample ? nhwc_to_nchw(src, Bn, 64 * 64, 4, io->a.unet_sample, st) : nullptr; }, true); }
      if (b.recording()) {
        // ---- backward: d(unet_sample) -> conv_out input gradient -> conv_norm_out (GN + SiLU) backward, added to d(up layer 11 output)
        const Act xin = x;
        b.tape.push_back({b.cur_stage, [=]() {
          const size_t w = b.dconv_w(kUnet + "conv_out", 4, 320, 9, /*CoPad=*/4);
          const long M = xin.M();
          const size_t from = b.emitted();
          F32T g = b.f32(size_t(M) * 4);
          B16T col = b.b16(size_t(M) * 64);
          { float* gp = g.p; bf16* cp = col.p; const float S = b.loss_scale;
            b.emit([=](cudaStream_t st) { return nchw_to_nhwc4(io->b.d_unet_sample, Bn, 4096, gp, st, S); });
            b.emit([=](cudaStream_t st) { return latent_im2col(gp, Bn, 64, 64, cp, h16, st); }); }
          B16T dn = b.b16(size_t(M) * 320);
          { GemmDesc d; d.seg[0] = Builder::seg_plain(col.p, M, 64); d.M = int(M); d.N = 320; d.Nw = 320; d.w = b.dpw(w);
            d.out_bf16 = dn.p; d.ldo16 = 320; b.gemm(d); }
          int acc = 0;
          float* dx = b.grad(xin, &acc);
          // projection 1 has written this gradient already (its backward replays first), so a call without d_unet_sample may skip the term
          if (!acc) b.fail(MADM_ESTATE, "training plan: the UNet-output backward must accumulate onto projection 1's input gradient");
          b.groupnorm_bwd(xin, nullptr, false, sv, nullptr, kUnet + "conv_norm_out", 1e-5f, ACT_SILU, dn.p, nullptr, nullptr, dx, acc, nullptr, 0, nullptr,
                          nullptr);
          b.only_if_set(from, &io->b.d_unet_sample);
          b.free(dn); b.free(col); b.free(g);
        }});
      }
    }
    b.frozen = b.train;  // the decoder body: no gradient in a training plan
    const std::string dc = kVae + "decoder.";
    const long M0 = long(Bn) * 4096;
    F32T z = b.f32(size_t(M0) * 4);
    { const float* src = unet_sample.p; float* dst = z.p;
      const float* w = P(kVae + "post_quant_conv.weight", 16); const float* bi = P(kVae + "post_quant_conv.bias", 4);
      b.emit([=](cudaStream_t st) { return post_quant_conv(src, w, bi, 1.0f / 0.18215f, M0, dst, st); }); }
    b.free(unet_sample);
    B16T col = b.b16(size_t(M0) * 64);
    { const float* src = z.p; bf16* dst = col.p;
      b.emit([=](cudaStream_t st) { return latent_im2col(src, Bn, 64, 64, dst, h16, st); }); }
    Act x = b.act(Bn, 64, 64, 512, true, false);
    { GemmDesc d; d.seg[0] = Builder::seg_plain(col.p, M0, 64); d.M = int(M0); d.N = 512; d.Nw = 512;
      d.w = b.pw(b.conv_w(dc + "conv_in", 512, 4, 9, /*Cpad=*/4)); d.bias = P(dc + "conv_in.bias", 512); d.out_f32 = x.f.p; d.ldo32 = 512;
      b.attach_colstats(x, d);
      b.gemm(d, 2.0 * double(d.M) * 512 * 36 + 2.0 * double(d.M) * 16); }  // + post_quant_conv
    b.free(col); b.free(z);
    {
      Act y = resblock(dc + "mid_block.resnets.0", x, nullptr, 512, 1e-6f, false, false); b.free(x); x = y;
      y = vae_attention(dc + "mid_block.attentions.0", x); b.free(x); x = y;
      y = resblock(dc + "mid_block.resnets.1", x, nullptr, 512, 1e-6f, false, false); b.free(x); x = y;
    }
    // fp16 operands: the 256^2 and 512^2 stages keep their residual stream in fp16, like the encoder's (and the reference's fp16 VAE)
    const bool s16 = f16();
    const int ch[4] = {512, 512, 256, 128};
    for (int i = 0; i < 4; ++i) {
      const bool o16 = s16 && i >= 2;
      for (int j = 0; j < 3; ++j) {
        Act y = resblock(dc + "up_blocks." + std::to_string(i) + ".resnets." + std::to_string(j), x, nullptr, ch[i], 1e-6f, false, false, false, o16);
        b.free(x);
        x = y;
      }
      if (i < 3) {
        Act y = upsample(dc + "up_blocks." + std::to_string(i) + ".upsamplers.0", x, /*out16_only=*/s16 && i + 1 >= 2);
        b.free(x);
        x = y;
      }
    }
    const long M = x.M();
    B16T n = b.b16(size_t(M) * 128);
    b.groupnorm(x, nullptr, dc + "conv_norm_out", 1e-6f, ACT_SILU, n.p, nullptr, /*in16=*/x.f.bytes == 0);
    b.free(x);
    F32T img = b.f32(size_t(M) * 4);
    { GemmDesc d; d.seg[0] = Builder::seg_3x3(n.p, Bn, 512, 512, 128); d.M = int(M); d.N = 3; d.Nw = 3; d.bn = 16;
      d.w = b.pw(b.conv_w(dc + "conv_out", 3, 128, 9)); d.bias = P(dc + "conv_out.bias", 3); d.out_f32 = img.p; d.ldo32 = 4;
      b.gemm(d); }
    b.free(n);
    // the decoded image stays as fp32 [B*512*512][4] (3 used): the s0 projection consumes it directly (build_proj, 3-channel input)
    enc_tap = Act(); enc_tap.B = Bn; enc_tap.H = 512; enc_tap.W = 512; enc_tap.C = 3;
    enc_tap.f = img;
    { const float* src = img.p;
      b.emit([=](cudaStream_t st) -> const char* {
        if (!io->a.decoded && !io->a.decoded_raw) return nullptr;
        return decoder_image_pack(src, Bn, 512 * 512, nullptr, io->a.decoded, io->a.decoded_raw, h16, st); }, true); }
    b.pin(enc_tap);
    b.frozen = false;
  }

  static const char* nchw_to_nhwc4(const float* src, int Bn, int HW, float* dst, cudaStream_t st, float scale = 1.0f);

  // =========================================================================== feature projections
  // The four bottleneck projections are independent chains of small launches (1.0 ms of latency-bound kernels at B = 8).  Each is tagged as a
  // branch (1..4) and emitted as soon as its tap exists -- the encoder tap's right after the VAE stage, the UNet taps' after up layers 5 / 8 / 11 --
  // so madm_extract can run it on a side stream that forks there and joins at the end of the plan (inside a CUDA-graph capture: parallel graph
  // branches): the projections fill the SMs the under-filled 16x16 / 8x8 UNet levels leave idle.  A branch's buffers are not recycled before the
  // end of the plan.
  bool proj_built[4] = {false, false, false, false};
  void build_proj_early(int i) {  // called where tap i has just been produced
    if (!s0() && !b.train) build_proj_one(i);
  }
  void build_proj() {
    for (int i = 0; i < 4; ++i) build_proj_one(i);
    b.flush_deferred();
  }
  void build_proj_one(int i) {
    if (proj_built[i]) return;
    proj_built[i] = true;
    const int saved_stage = b.cur_stage;
    b.cur_stage = MADM_STAGE_PROJ;
    IoBind* io = b.io;
    const std::string root = b.ema ? "ema_feature_projections." : "feature_projections.";
    const Act* taps[4] = {&enc_tap, &unet_tap[0], &unet_tap[1], &unet_tap[2]};
    b.defer_free = true;
    {
      b.cur_branch = 1 + i;
      const Act& x = *taps[i];
      const std::string p = root + std::to_string(i) + ".0.";
      const int h16 = f16();
      const ParamRef* w1 = b.find(p + "conv1.weight"); const ParamRef* w3 = b.find(p + "conv3.weight");
      if (!w1 || !w3) b.fail(MADM_ENOTFOUND, "parameter not registered: " + p + "conv1.weight / conv3.weight");
      const int Bn = x.B, H = x.H, W = x.W, Cin = x.C, Cb = int(w1->shape[0]), Cout = int(w3->shape[0]);
      if (int(w1->shape[1]) != Cin || Cb % 64 != 0 || Cout % 64 != 0) b.fail(MADM_EINVAL, "feature projection " + std::to_string(i) + ": unsupported channels");
      const long M = x.M();
      const bool shortcut = Cin != Cout;
      // The 3-channel decoded image of the s0 variant: its K = 3 1x1 convs are not GEMMs.  conv1 -> GN -> ReLU is one elementwise pass with
      // GroupNorm statistics derived from the image's moments, and the shortcut branch is recomputed inside the final pass (norm.cu).
      const bool rgb3 = Cin == 3;
      if (Cin % 64 != 0 && !rgb3) b.fail(MADM_EINVAL, "feature projection " + std::to_string(i) + ": input channels must be 3 or a multiple of 64");
      F32T mom, coef1, coefs;
      const float* img4 = x.f.p;
      if (rgb3) {
        if (!shortcut) b.fail(MADM_EINVAL, "feature projection: a 3-channel input needs a shortcut conv");
        mom = b.f32(size_t(image_moments_floats(Bn)));
        coef1 = b.f32(size_t(Bn) * Cb * 4);
        coefs = b.f32(size_t(Bn) * Cout * 4);
        const int HWi = H * W;
        float* mp = mom.p; float* c1p = coef1.p; float* csp = coefs.p;
        const float* w1p = P(p + "conv1.weight", int64_t(Cb) * 3); const float* g1 = P(p + "conv1.norm.weight", Cb); const float* b1 = P(p + "conv1.norm.bias", Cb);
        const float* wsp = P(p + "shortcut.weight", int64_t(Cout) * 3); const float* gsp = P(p + "shortcut.norm.weight", Cout);
        const float* bsp = P(p + "shortcut.norm.bias", Cout);
        b.emit([=](cudaStream_t st) { return image_moments(img4, Bn, HWi, mp, st); }, false, MADM_KIND_GROUPNORM, 0.0, double(M) * 16);
        b.emit([=](cudaStream_t st) { return c3_gn_coeffs(mp, w1p, g1, b1, 1e-5f, Bn, HWi, Cb, c1p, st); }, false, MADM_KIND_GROUPNORM, 0.0, 0.0);
        b.emit([=](cudaStream_t st) { return c3_gn_coeffs(mp, wsp, gsp, bsp, 1e-5f, Bn, HWi, Cout, csp, st); }, false, MADM_KIND_GROUPNORM, 0.0, 0.0);
      }
      // every GroupNorm of the bottleneck takes its statistics from the producing GEMM's epilogue
      B16T a1 = b.b16(size_t(M) * Cb);
      Act c1;
      Builder::GnSaved s1;
      if (rgb3) {
        bf16* a1p = a1.p; const float* c1p = coef1.p; const int HWi = H * W;
        b.emit([=](cudaStream_t st) { return c3_conv_gn_relu(img4, c1p, Bn, HWi, Cb, a1p, h16, st); }, false, MADM_KIND_GROUPNORM, 0.0, double(M) * (16 + 2.0 * Cb));
      } else {
        c1 = b.act(Bn, H, W, Cb, false, true);
        { GemmDesc d; d.seg[0] = Builder::seg_1x1(x.h.p, Bn, H, W, Cin); d.M = int(M); d.N = Cb; d.Nw = Cb;
          d.w = b.pw(b.conv_w(p + "conv1", Cb, Cin, 1)); d.out_bf16 = c1.h.p; d.ldo16 = Cb; b.attach_colstats(c1, d); b.gemm(d); }
        s1 = b.groupnorm(c1, nullptr, p + "conv1.norm", 1e-5f, ACT_RELU, a1.p, nullptr, /*in16=*/true);
        b.free(c1);
      }
      Act c2 = b.act(Bn, H, W, Cb, false, true);
      { GemmDesc d; d.seg[0] = Builder::seg_3x3(a1.p, Bn, H, W, Cb); d.M = int(M); d.N = Cb; d.Nw = Cb;
        d.w = b.pw(b.conv_w(p + "conv2", Cb, Cb, 9)); d.out_bf16 = c2.h.p; d.ldo16 = Cb; b.attach_colstats(c2, d); b.gemm(d); }
      b.free(a1);
      B16T a2 = b.b16(size_t(M) * Cb);
      const Builder::GnSaved s2 = b.groupnorm(c2, nullptr, p + "conv2.norm", 1e-5f, ACT_RELU, a2.p, nullptr, /*in16=*/true);
      b.free(c2);
      Act c3 = b.act(Bn, H, W, Cout, true, false);
      { GemmDesc d; d.seg[0] = Builder::seg_1x1(a2.p, Bn, H, W, Cb); d.M = int(M); d.N = Cout; d.Nw = Cout;
        d.w = b.pw(b.conv_w(p + "conv3", Cout, Cb, 1)); d.out_f32 = c3.f.p; d.ldo32 = Cout; b.attach_colstats(c3, d); b.gemm(d); }
      b.free(a2);
      Act sc;
      if (shortcut && !rgb3) {
        sc = b.act(Bn, H, W, Cout, true, false);
        GemmDesc d; d.seg[0] = Builder::seg_1x1(x.h.p, Bn, H, W, Cin); d.M = int(M); d.N = Cout; d.Nw = Cout;
        d.w = b.pw(b.conv_w(p + "shortcut", Cout, Cin, 1)); d.out_f32 = sc.f.p; d.ldo32 = Cout; b.attach_colstats(sc, d); b.gemm(d);
      }
      const int HW = H * W;
      float* st3 = b.new_stats(1);
      float* sts = (shortcut && !rgb3) ? b.new_stats(1) : nullptr;
      const float* c3p = c3.f.p; const float* scp = rgb3 ? nullptr : (shortcut ? sc.f.p : x.f.p);
      const double pel = double(Bn) * HW * Cout;
      auto tail_stats = [&](const Act& t, const float* src, float* dst) {  // [B,32,2] group sums of a fp32 [M,Cout] tensor
        if (t.has_cs) {
          const float* cst = t.cs; const int nb = HW / kStatRows; const int S = groupnorm_colstats_chunks(nb);
          float* part = b.new_stats(S);
          b.emit([=](cudaStream_t st) { return groupnorm_colstats_reduce(cst, Cout, nullptr, 0, Bn, nb, part, st); }, false, MADM_KIND_GROUPNORM,
                 0.0, double(Bn) * nb * Cout * 8);
          b.emit([=](cudaStream_t st) { return groupnorm_finalize_slabs(part, Bn, S, dst, st); }, false, MADM_KIND_GROUPNORM, 0.0, 0.0);
        } else {
          float* part = b.new_stats(groupnorm_slabs(HW, Cout));
          b.emit([=](cudaStream_t st) { return groupnorm_stats(src, Cout, nullptr, 0, Bn, HW, 0, 0, part, st); }, false, MADM_KIND_GROUPNORM, 0.0,
                 pel * 4);
          b.emit([=](cudaStream_t st) { return groupnorm_finalize(part, Bn, HW, Cout, dst, st); }, false, MADM_KIND_GROUPNORM, 0.0, 0.0);
        }
      };
      tail_stats(c3, c3p, st3);
      if (shortcut && !rgb3) tail_stats(sc, scp, sts);
      const float* g3 = P(p + "conv3.norm.weight", Cout); const float* b3 = P(p + "conv3.norm.bias", Cout);
      const float* gs = shortcut ? P(p + "shortcut.norm.weight", Cout) : nullptr;
      const float* bs = shortcut ? P(p + "shortcut.norm.bias", Cout) : nullptr;
      if (rgb3) {
        const float* csp = coefs.p;
        b.emit([=](cudaStream_t st) -> const char* {
          float* dst = io->a.out[i];
          if (!dst) return "madm_extract: output pointer is null";
          return gn_add_relu_nchw_c3(c3p, st3, g3, b3, img4, csp, 1e-5f, Bn, HW, Cout, dst, st);
        }, false, MADM_KIND_GROUPNORM, 0.0, pel * 8);
      } else b.emit([=](cudaStream_t st) -> const char* {
        float* dst = io->a.out[i];
        if (!dst) return "madm_extract: output pointer is null";
        return gn_add_relu_nchw(c3p, st3, g3, b3, scp, sts, gs, bs, 1e-5f, Bn, HW, Cout, dst, st, (io->a.flags & MADM_FLAG_OUT_FP16) ? 1 : 0);
      }, false, MADM_KIND_GROUPNORM, 0.0, pel * 12);
      b.free(c3);
      if (shortcut && !rgb3) b.free(sc);
      if (rgb3) { b.free(mom); b.free(coef1); b.free(coefs); }
      if (b.recording()) {
        // ---- backward
        b.tape.push_back({b.cur_stage, [=]() {
          const size_t wd3 = b.dconv_w(p + "conv3", Cout, Cb, 1), wd2 = b.dconv_w(p + "conv2", Cb, Cb, 9);
          // (a 3-channel input is the detached decoded image: no input gradient, so no operands for it)
          const size_t wd1 = rgb3 ? 0 : b.dconv_w(p + "conv1", Cb, Cin, 1), wds = shortcut && !rgb3 ? b.dconv_w(p + "shortcut", Cout, Cin, 1) : 0;
          const float S = b.loss_scale, inv = 1.0f / b.loss_scale;
          const int Mi = int(M);
          // d(z) = d(out) * (out > 0), NCHW -> NHWC, scaled by the loss scale
          B16T dz = b.b16(size_t(M) * Cout);
          { bf16* dst = dz.p;
            b.emit([=](cudaStream_t st) -> const char* {
              if (!io->b.dout[i] || !io->b.out[i]) return "madm_backward: dout / out pointer is null";
              return relu_bwd_nchw_to_nhwc16(io->b.dout[i], io->b.out[i], Bn, Cout, HW, S, dst, h16, st); }); }
          auto wg = [&](const std::string& name, const bf16* dy, int N, const bf16* xx, int K, int taps) {  // weight gradient of one conv
            float* g = b.grad_buf(p + name + ".weight");
            if (!g) return;
            F32T scr = b.f32(wgrad_scratch_floats(Mi, N, K, taps));
            float* sp = scr.p;
            const long so_n = taps == 9 ? long(K) * 9 : K, so_k = taps == 9 ? 9 : 1, so_t = taps == 9 ? 1 : 0;
            b.emit([=](cudaStream_t st) { return wgrad(dy, N, xx, K, Mi, N, K, taps, Bn, H, W, inv, g, so_n, so_k, so_t, sp, h16, st); });
            b.free(scr);
          };
          int acc = 0;
          float* dtap = Builder::wants_grad(x) ? b.grad(x, &acc) : nullptr;
          // conv3 branch
          B16T dc3 = b.b16(size_t(M) * Cout);
          b.groupnorm_bwd(c3, nullptr, false, Builder::GnSaved(), st3, p + "conv3.norm", 1e-5f, ACT_NONE, dz.p, nullptr, dc3.p, nullptr, 0, nullptr, 0,
                          b.grad_buf(p + "conv3.norm.weight"), b.grad_buf(p + "conv3.norm.bias"));
          wg("conv3", dc3.p, Cout, a2.p, Cb, 1);
          B16T da2 = b.b16(size_t(M) * Cb);
          { GemmDesc d; d.seg[0] = Builder::seg_1x1(dc3.p, Bn, H, W, Cout); d.M = Mi; d.N = Cb; d.Nw = Cb; d.w = b.dpw(wd3); d.out_bf16 = da2.p; d.ldo16 = Cb; b.gemm(d); }
          b.free(dc3);
          B16T dc2 = b.b16(size_t(M) * Cb);
          b.groupnorm_bwd(c2, nullptr, true, s2, nullptr, p + "conv2.norm", 1e-5f, ACT_RELU, da2.p, nullptr, dc2.p, nullptr, 0, nullptr, 0,
                          b.grad_buf(p + "conv2.norm.weight"), b.grad_buf(p + "conv2.norm.bias"));
          b.free(da2);
          wg("conv2", dc2.p, Cb, a1.p, Cb, 9);
          B16T da1 = b.b16(size_t(M) * Cb);
          { GemmDesc d; d.seg[0] = Builder::seg_3x3(dc2.p, Bn, H, W, Cb); d.M = Mi; d.N = Cb; d.Nw = Cb; d.w = b.dpw(wd2); d.out_bf16 = da1.p; d.ldo16 = Cb; b.gemm(d); }
          b.free(dc2);
          if (rgb3) {
            // the two K = 3 branches: their conv / GroupNorm gradients from the image, its moments and the forward's folded coefficients
            // (norm.cu c3_gn_bwd), without the conv outputs the forward never stored
            auto c3_bwd = [&](const std::string& name, int C, const float* coef, const bf16* dy, int relu) {
              F32T part = b.f32(c3_gn_bwd_scratch_floats(Bn, C));
              const float* mp = mom.p; const float* wp = P(p + name + ".weight", int64_t(C) * 3); const float* gp = P(p + name + ".norm.weight", C);
              float* dw = b.grad_buf(p + name + ".weight"); float* dg = b.grad_buf(p + name + ".norm.weight"); float* db = b.grad_buf(p + name + ".norm.bias");
              float* pp = part.p;
              b.emit([=](cudaStream_t st) { return c3_gn_bwd(img4, mp, coef, wp, gp, 1e-5f, relu, Bn, HW, C, dy, h16, inv, dw, dg, db, pp, st); }, false,
                     MADM_KIND_GROUPNORM, 0.0, double(M) * (16 + 2.0 * C));
              b.free(part);
            };
            c3_bwd("conv1", Cb, coef1.p, da1.p, 1);
            b.free(da1);
            c3_bwd("shortcut", Cout, coefs.p, dz.p, 0);
            b.free(dz);
            return;
          }
          B16T dc1 = b.b16(size_t(M) * Cb);
          b.groupnorm_bwd(c1, nullptr, true, s1, nullptr, p + "conv1.norm", 1e-5f, ACT_RELU, da1.p, nullptr, dc1.p, nullptr, 0, nullptr, 0,
                          b.grad_buf(p + "conv1.norm.weight"), b.grad_buf(p + "conv1.norm.bias"));
          b.free(da1);
          wg("conv1", dc1.p, Cb, x.h.p, Cin, 1);
          if (dtap) {
            GemmDesc d; d.seg[0] = Builder::seg_1x1(dc1.p, Bn, H, W, Cb); d.M = Mi; d.N = Cin; d.Nw = Cin; d.w = b.dpw(wd1);
            if (acc) { d.residual = dtap; d.ldr = Cin; }
            d.out_f32 = dtap; d.ldo32 = Cin; b.gemm(d);
            acc = 1;
          }
          b.free(dc1);
          if (shortcut) {
            B16T dsc = b.b16(size_t(M) * Cout);
            b.groupnorm_bwd(sc, nullptr, false, Builder::GnSaved(), sts, p + "shortcut.norm", 1e-5f, ACT_NONE, dz.p, nullptr, dsc.p, nullptr, 0, nullptr, 0,
                            b.grad_buf(p + "shortcut.norm.weight"), b.grad_buf(p + "shortcut.norm.bias"));
            wg("shortcut", dsc.p, Cout, x.h.p, Cin, 1);
            if (dtap) {
              GemmDesc d; d.seg[0] = Builder::seg_1x1(dsc.p, Bn, H, W, Cout); d.M = Mi; d.N = Cin; d.Nw = Cin; d.w = b.dpw(wds);
              if (acc) { d.residual = dtap; d.ldr = Cin; }
              d.out_f32 = dtap; d.ldo32 = Cin; b.gemm(d);
            }
            b.free(dsc);
          }
          b.free(dz);
        }});
      }
    }
    b.cur_branch = 0;
    b.defer_free = false;
    b.cur_stage = saved_stage;
  }

  // ---- DAFormerHead.forward (reference modeling/sem_seg_head/daformer_head.py:702-749; SURVEY §8 f-2) on the feature dict
  // s2..s5 (fp32 NCHW, args.out[0..3]): MLP embeds 512 -> E at native resolution, bilinear resize (align_corners=False) to the s2
  // grid, concat, depthwise-separable ASPP (1x1 + 3 dilated branches) with eval-mode BatchNorm folded + ReLU, 3x3 bottleneck,
  // 1x1 classifier -> args.logits [B, classes, 128, 128].
  bool has_head() const { return b.ctx->params.count("sem_seg_head.conv_seg.weight") != 0; }
  void build_head() {
    b.cur_stage = MADM_STAGE_HEAD;
    IoBind* io = b.io;
    const std::string h = "sem_seg_head.";
    const ParamRef* cs = b.find(h + "conv_seg.weight");
    const ParamRef* e0 = b.find(h + "embed_layers.0.proj.weight");
    if (!cs || !e0) b.fail(MADM_ENOTFOUND, "sem_seg_head parameters are not registered");
    const int ncls = int(cs->shape[0]), CH = int(cs->shape[1]), E = int(e0->shape[0]), Cin0 = int(e0->shape[1]);
    // base: s2..s5, four 512-channel maps, fused on the 128^2 grid.  s0 variant (in_keys[0]='s0', in_channels[0]=128,
    // mtmadise_cityscapes_rgb_to_depth_11.py:51-55): the first map is 128 x 512^2, so the head fuses on the 512^2 grid.
    // grid of the first map: the 512^2 crop's by default; sliding-window inference hands the head full-image maps (feature_extractor.py:
    // 270-275 merges the crops before the head runs), so the grid is a call argument (madm_extract_args.head_h / head_w)
    const int H = b.head_h > 0 ? b.head_h : (s0() ? 512 : 128), W = b.head_w > 0 ? b.head_w : (s0() ? 512 : 128);
    if (Cin0 != (s0() ? 128 : 512) || E % 64 != 0 || CH % 64 != 0 || ncls > 32) b.fail(MADM_EINVAL, "sem_seg_head: unsupported channel configuration");
    const int ratio[4] = {1, s0() ? 8 : 2, s0() ? 16 : 4, s0() ? 32 : 8};
    if (H % ratio[3] != 0 || W % ratio[3] != 0 || !(W % 128 == 0 || 128 % W == 0)) b.fail(MADM_EINVAL, "sem_seg_head: unsupported feature grid");
    const int Bn = b.B, CAT = 4 * E;
    const long M = long(Bn) * H * W;
    const int f16v = f16();
    B16T cat = b.b16(size_t(M) * CAT);
    for (int i = 0; i < 4; ++i) {
      const int Hi = H / ratio[i], Wi = W / ratio[i], HWi = Hi * Wi, Cin = i == 0 ? Cin0 : 512;
      const long Mi = long(Bn) * HWi;
      B16T x = b.b16(size_t(Mi) * Cin);
      {
        bf16* xp = x.p;
        b.emit([=](cudaStream_t st) -> const char* {
          const float* src = io->a.out[i];
          if (!src) return "madm_extract: the head stage needs the feature maps in args.out[0..3]";
          return nchw_to_nhwc16(src, Bn, Cin, HWi, xp, f16v, st);
        }, false, MADM_KIND_ELEMENTWISE, 0.0, double(Mi) * Cin * 6);
      }
      const std::string lin = h + "embed_layers." + std::to_string(i) + ".proj";
      GemmDesc d; d.seg[0] = Builder::seg_plain(x.p, Mi, Cin); d.M = int(Mi); d.N = E; d.Nw = E;
      d.w = b.pw(b.linear_w(lin, E, Cin, false)); d.bias = P(lin + ".bias", E);
      if (i == 0) {  // already on the s2 grid: straight into its slice of the concat buffer
        d.out_bf16 = cat.p; d.ldo16 = CAT;
        b.gemm(d);
      } else {
        B16T e = b.b16(size_t(Mi) * E);
        d.out_bf16 = e.p; d.ldo16 = E;
        b.gemm(d);
        bf16* ep = e.p; bf16* dst = cat.p + size_t(i) * E;
        b.emit([=](cudaStream_t st) { return bilinear_resize_nhwc16(ep, Bn, Hi, Wi, E, dst, H, W, CAT, f16v, st); }, false, MADM_KIND_ELEMENTWISE,
               0.0, double(M) * E * 2 + double(Mi) * E * 2);
        b.free(e);
      }
      b.free(x);
    }
    // ASPP: branch 0 = 1x1 ConvModule, branches 1..3 = depthwise 3x3 (dilation 6/12/18) -> pointwise 1x1; outputs concatenated
    const std::string as = h + "fuse_layer.aspp_modules.";
    B16T aspp = b.b16(size_t(M) * 4 * CH);
    {
      const Builder::ConvBn c = b.conv_bn(as + "0", CH, CAT, 1);
      GemmDesc d; d.seg[0] = Builder::seg_1x1(cat.p, Bn, H, W, CAT); d.M = int(M); d.N = CH; d.Nw = CH;
      d.w = b.pw(c.w_off); d.bias = b.pf(c.shift_off); d.act = ACT_RELU; d.out_bf16 = aspp.p; d.ldo16 = 4 * CH;
      b.gemm(d);
    }
    const int dil[3] = {6, 12, 18};
    for (int j = 1; j <= 3; ++j) {
      const std::string m = as + std::to_string(j);
      const Builder::ConvBn dw = b.depthwise_bn(m + ".depthwise_conv", CAT);
      B16T t = b.b16(size_t(M) * CAT);
      { const bf16* src = cat.p; bf16* dst = t.p; const float* w9 = b.pf(dw.w_off); const float* sh = b.pf(dw.shift_off); const int dl = dil[j - 1];
        b.emit([=](cudaStream_t st) { return depthwise3x3_nhwc16(src, Bn, H, W, CAT, dl, w9, sh, dst, f16v, st); }, false, MADM_KIND_ELEMENTWISE, 0.0,
               double(M) * CAT * 4); }
      const Builder::ConvBn pwc = b.conv_bn(m + ".pointwise_conv", CH, CAT, 1);
      GemmDesc d; d.seg[0] = Builder::seg_1x1(t.p, Bn, H, W, CAT); d.M = int(M); d.N = CH; d.Nw = CH;
      d.w = b.pw(pwc.w_off); d.bias = b.pf(pwc.shift_off); d.act = ACT_RELU; d.out_bf16 = aspp.p + size_t(j) * CH; d.ldo16 = 4 * CH;
      b.gemm(d);
      b.free(t);
    }
    b.free(cat);
    B16T bott = b.b16(size_t(M) * CH);
    {
      const Builder::ConvBn c = b.conv_bn(h + "fuse_layer.bottleneck", CH, 4 * CH, 9);
      GemmDesc d; d.seg[0] = Builder::seg_3x3(aspp.p, Bn, H, W, 4 * CH); d.M = int(M); d.N = CH; d.Nw = CH;
      d.w = b.pw(c.w_off); d.bias = b.pf(c.shift_off); d.act = ACT_RELU; d.out_bf16 = bott.p; d.ldo16 = CH;
      b.gemm(d);
    }
    b.free(aspp);
    // classifier: 1x1 conv CH -> classes (+bias); N padded to 32 columns in the fp32 NHWC scratch, then NCHW into args.logits
    F32T lg = b.f32(size_t(M) * 32);
    {
      GemmDesc d; d.seg[0] = Builder::seg_1x1(bott.p, Bn, H, W, CH); d.M = int(M); d.N = ncls; d.Nw = ncls;
      d.w = b.pw(b.conv_w(h + "conv_seg", ncls, CH, 1)); d.bias = P(h + "conv_seg.bias", ncls); d.out_f32 = lg.p; d.ldo32 = 32; d.bn = 32;
      b.gemm(d);
    }
    b.free(bott);
    {
      const float* lp = lg.p;
      b.emit([=](cudaStream_t st) -> const char* {
        float* dst = io->a.logits;
        if (!dst) return "madm_extract: logits pointer is null";
        return nhwc_to_nchw_strided(lp, Bn, H * W, ncls, 32, dst, st);
      }, false, MADM_KIND_ELEMENTWISE, 0.0, double(M) * ncls * 8);
    }
    b.free(lg);
  }

  bool has_path() const { return b.ctx->params.count(kUnet + "conv_in.weight") != 0; }
  void build_all() {
    if (b.train) {  // forward that keeps its activations + the backward pass (SURVEY §8 row f-3)
      if (!has_path()) b.fail(MADM_ESTATE, "training path: UNet / VAE parameters are not registered");
    }
    if (has_path() || !has_head()) {  // a context that holds only sem_seg_head.* runs the head alone
      enumerate_unet();
      build_vae();
      if (enc_tap.gr) enc_tap.gr->stop = true;  // training: the VAE encoder runs without gradient (ldm_diffusers.py:282)
      build_proj_early(0);  // the encoder tap's projection overlaps the whole UNet
      build_unet();
      if (s0()) build_dec();
      build_proj();
    }
    if (!b.train) {
      if (has_head()) build_head();
      return;
    }
    b.bwd = true;
    { float* dt = d_temb_all.p; bf16* dk = dkv_all.p; const size_t nt = size_t(b.B) * temb_total * 4, nk = size_t(b.B) * 77 * kv_total * 2;
      b.emit([=](cudaStream_t st) -> const char* {
        if (cudaMemsetAsync(dt, 0, nt, st) != cudaSuccess || cudaMemsetAsync(dk, 0, nk, st) != cudaSuccess) return "cudaMemsetAsync failed";
        return nullptr; }); }
    for (auto it = b.tape.rbegin(); it != b.tape.rend(); ++it) {
      b.cur_stage = it->first;  // the dgrad entries a backward registers belong to its forward's stage
      it->second();
    }
    b.bwd = false;
  }
};

__global__ void nchw_to_nhwc4_kernel(const float* __restrict__ src, int Bn, int HW, float scale, float* __restrict__ dst) {
  const long i = long(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= long(Bn) * HW) return;
  const int p = int(i % HW), bb = int(i / HW);
  const float* s = src + size_t(bb) * 4 * HW + p;
  *reinterpret_cast<float4*>(dst + i * 4) = make_float4(s[0] * scale, s[HW] * scale, s[2 * HW] * scale, s[3 * HW] * scale);
}
const char* Model::nchw_to_nhwc4(const float* src, int Bn, int HW, float* dst, cudaStream_t st, float scale) {
  const long total = long(Bn) * HW;
  nchw_to_nhwc4_kernel<<<unsigned((total + 255) / 256), 256, 0, st>>>(src, Bn, HW, scale, dst);
  return cudaGetLastError() == cudaSuccess ? nullptr : "nchw_to_nhwc4 launch failed";
}

int extract_train(madm_ctx* ctx, const madm_extract_args* a, cudaStream_t st);

int set_err(madm_ctx* ctx, int code, const std::string& m) {
  if (ctx) ctx->err = m;
  set_global_error(m.c_str());
  return code;
}

// Runs the model traversal in the builder's mode.
int traverse(madm_ctx* ctx, Builder& bld) {
  Model m(bld);
  try {
    m.build_all();
  } catch (const BuildError& e) {
    return set_err(ctx, e.code, e.msg);
  }
  return MADM_OK;
}

// Bytes of the GroupNorm statistics slots a traversal used; they sit at the start of the workspace, the activations after them.
size_t stats_region(const Builder& bld) { return (bld.stats_used * 4 + 1023) & ~size_t(1023); }

// Runs the traversal in a dry mode; in SIZE mode returns the workspace bytes (stats region + peak).
int dry_run(madm_ctx* ctx, Mode mode, int B, size_t* ws_bytes, int head_h = 0, int head_w = 0, bool train = false, const std::string& adapter = "") {
  Builder bld{ctx, mode, B, false};
  bld.head_h = head_h; bld.head_w = head_w;
  bld.train = train; bld.adapter = adapter; bld.lora_scale = 1.0f;
  const int rc = traverse(ctx, bld);
  if (rc == MADM_OK && ws_bytes) *ws_bytes = stats_region(bld) + bld.peak + 1024;
  return rc;
}

// Emits `plan` (its pointers and workspace already set) with the settings of `cfg`: a SIZE pass of the same traversal sizes the
// statistics region, then the PLAN pass lays the launches out over the workspace.
int build_plan(madm_ctx* ctx, const Builder& cfg, Plan* plan) {
  Builder probe = cfg;
  probe.mode = SIZE;
  int rc = traverse(ctx, probe);
  if (rc != MADM_OK) return rc;
  plan->stats_bytes = stats_region(probe);
  Builder bld = cfg;
  bld.mode = PLAN;
  bld.plan = plan;
  bld.io = &plan->io;
  bld.packed = static_cast<const uint8_t*>(plan->packed);
  bld.dpacked = static_cast<const uint8_t*>(plan->dpacked);
  bld.stats_base = reinterpret_cast<float*>(plan->ws);
  bld.ws = static_cast<uint8_t*>(plan->ws) + plan->stats_bytes;
  rc = traverse(ctx, bld);
  if (rc != MADM_OK) return rc;
  if (plan->stats_bytes + bld.peak > plan->ws_bytes)
    return set_err(ctx, MADM_ENOMEM, plan->train ? "madm_extract: training workspace too small for plan" : "madm_extract: workspace too small for plan");
  return MADM_OK;
}

// Runs the launches of `ops` whose stage is in `stages` on `st`.  With `side`, branch launches run on the context's side streams: each
// branch forks from `st` before its first launch and joins back before the first head launch (the head consumes the projections'
// outputs) and at the end.  With `ev` (2 per launch), each launch is bracketed by its events.  A failing launch i is reported as
// "<its message> (<what> i)".
int replay(madm_ctx* ctx, const std::vector<Launch>& ops, int stages, cudaStream_t st, bool side, const cudaEvent_t* ev, const char* what) {
  unsigned forked = 0;  // bit k: side stream k has work of this call
  auto join = [&]() {
    for (int k = 0; k < 4; ++k)
      if (forked & (1u << k)) { cudaEventRecord(ctx->ev_join[k], ctx->side[k]); cudaStreamWaitEvent(st, ctx->ev_join[k], 0); }
    forked = 0;
  };
  for (size_t i = 0; i < ops.size(); ++i) {
    const Launch& l = ops[i];
    if (!(l.stage & stages)) continue;
    const int br = side ? l.branch : 0;
    cudaStream_t s = st;
    if (br > 0) {
      if (!(forked & (1u << (br - 1)))) {  // fork here: everything this branch reads (its tap) has been enqueued on the caller's stream
        cudaEventRecord(ctx->ev_fork[br - 1], st);
        cudaStreamWaitEvent(ctx->side[br - 1], ctx->ev_fork[br - 1], 0);
        forked |= 1u << (br - 1);
      }
      s = ctx->side[br - 1];
    } else if (forked && (l.stage & MADM_STAGE_HEAD)) {
      join();
    }
    if (ev) cudaEventRecord(ev[2 * i], s);
    if (const char* e = l.run(s)) { join(); return set_err(ctx, MADM_ECUDA, std::string(e) + " (" + what + " " + std::to_string(i) + ")"); }
    if (ev) cudaEventRecord(ev[2 * i + 1], s);
  }
  join();
  return MADM_OK;
}

int ensure_layout(madm_ctx* ctx) {
  if (ctx->fwd.done) return MADM_OK;
  ctx->fwd = Arena();
  int rc = dry_run(ctx, LAYOUT, 1, nullptr);
  if (rc != MADM_OK) return rc;
  // EMA projection twins share the layout pass (registered only if the caller provided them)
  if (ctx->params.count("ema_feature_projections.0.0.conv1.weight")) {
    Builder bld{ctx, LAYOUT, 1, true};
    Model m(bld);
    try {
      m.enumerate_unet();
      // projections need tap shapes only
      m.enc_tap.B = 1; m.enc_tap.H = 128; m.enc_tap.W = 128; m.enc_tap.C = 512;
      if (m.s0()) { m.enc_tap.H = 512; m.enc_tap.W = 512; m.enc_tap.C = 3; }
      const int hw[3] = {64, 32, 16}, cc[3] = {320, 640, 1280};
      for (int i = 0; i < 3; ++i) { m.unet_tap[i].B = 1; m.unet_tap[i].H = hw[i]; m.unet_tap[i].W = hw[i]; m.unet_tap[i].C = cc[i]; }
      m.build_proj();
    } catch (const BuildError& e) {
      return set_err(ctx, e.code, e.msg);
    }
  }
  ctx->fwd.done = true;
  return MADM_OK;
}

// The dgrad arena is laid out by a LAYOUT pass of the training traversal, which reads the forward arena's entries.
int ensure_dlayout(madm_ctx* ctx) {
  int rc = ensure_layout(ctx);
  if (rc != MADM_OK) return rc;
  if (ctx->dgrad.done) return MADM_OK;
  ctx->dgrad = Arena();
  rc = dry_run(ctx, LAYOUT, 1, nullptr, 0, 0, /*train=*/true);
  if (rc != MADM_OK) return rc;
  ctx->dgrad.done = true;
  return MADM_OK;
}

// What a setter changed.  Each level drops everything the levels before it drop.
enum Change {
  GRAD_BUFFERS,    // training plans capture the gradient buffers
  PARAM_POINTERS,  // every plan captures parameter pointers
  LAYOUT_INPUTS,   // parameter shapes, operand dtype or variant: the arena layouts and the workspace sizes follow from them
};
void invalidate(madm_ctx* ctx, Change what) {
  ctx->train_plans.clear();
  if (what >= PARAM_POINTERS) {
    ctx->plans.clear();
    ctx->last_plan = nullptr;
  }
  if (what >= LAYOUT_INPUTS) {
    ctx->fwd.done = false;
    ctx->dgrad.done = false;
    ctx->ws_bytes_cache.clear();
  }
}

__global__ void identity16_kernel(uint16_t* out, int N, int ldo, uint16_t one) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N * N) out[size_t(i / N) * ldo + (i % N)] = (i / N == i % N) ? one : uint16_t(0);
}

__global__ void f32_sum2_kernel(const float* a, const float* b2, int n, float* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] + b2[i];
}

// Which entries of an arena a pack rewrites: all, the LoRA-targeted linears (adapter switch), or what an optimizer or EMA step can
// change (PackEntry::trainable), in an arena that was fully packed before.
enum Subset { PACK_ALL, PACK_LORA, PACK_TRAINABLE };

// Packs the `subset` of `arena` into `base`, folding the LoRA adapter `ad` ("" = base weights) scaled by `scale`.
int pack_arena(madm_ctx* ctx, const Arena& arena, uint8_t* base, const std::string& ad, float scale, Subset subset, cudaStream_t st) {
  auto get = [&](const std::string& name) -> const ParamRef* {
    auto it = ctx->params.find(name);
    return it == ctx->params.end() ? nullptr : &it->second;
  };
  // a linear's weight: "<m>.base_layer.weight" if a LoRA adapter wraps it, else "<m>.weight"; folded with the active adapter's factors
  // when wrapped (le.la = null and le.r = 0 otherwise)
  auto linear = [&](const PackEntry& e, LoraPackEntry* le) -> int {
    const ParamRef* w = get(e.src + ".base_layer.weight");
    const bool wrapped = w != nullptr;
    if (!w) w = get(e.src + ".weight");
    if (!w) return set_err(ctx, MADM_ENOTFOUND, "parameter not registered: " + e.src + ".weight");
    if (w->numel() != int64_t(e.N) * e.C) return set_err(ctx, MADM_EINVAL, "unexpected shape: " + e.src);
    *le = LoraPackEntry{w->p, nullptr, nullptr, base + e.off, e.N, e.C, 0, e.ldo};
    if (wrapped && !ad.empty()) {
      const ParamRef* A = get(e.src + ".lora_A." + ad + ".weight");
      const ParamRef* Bm = get(e.src + ".lora_B." + ad + ".weight");
      if (!A || !Bm) return set_err(ctx, MADM_ENOTFOUND, "LoRA adapter '" + ad + "' not registered for " + e.src);
      le->r = int(A->shape[0]);
      if (A->shape[1] != e.C || Bm->shape[0] != e.N || Bm->shape[1] != le->r) return set_err(ctx, MADM_EINVAL, "LoRA shape mismatch: " + e.src);
      le->la = A->p; le->lb = Bm->p;
    }
    return MADM_OK;
  };
  std::vector<LoraPackEntry> multi[2];  // natural-order [0] / transposed [1] outputs of the multi-tensor pack kernel
  for (const PackEntry& e : arena.entries) {
    if ((subset == PACK_LORA && !e.lora) || (subset == PACK_TRAINABLE && !e.trainable)) continue;
    const char* err = nullptr;
    switch (e.kind) {
      case PK_CONV: case PK_CONV_BN: case PK_CONV_DGRAD: {
        const ParamRef* w = get(e.src);
        if (!w) return set_err(ctx, MADM_ENOTFOUND, "parameter not registered: " + e.src);
        if (w->numel() != int64_t(e.N) * e.C * e.taps) return set_err(ctx, MADM_EINVAL, "unexpected shape: " + e.src);
        if (e.kind == PK_CONV_DGRAD) err = pack_conv_dgrad_weight(w->p, e.N, e.C, e.taps, e.Cpad, e.Kpad, e.ldo, base + e.off, ctx->fp16, st);
        else err = pack_conv_weight(w->p, e.N, e.C, e.taps, e.Cpad, e.Kpad, e.ldo, base + e.off, ctx->fp16, st,
                                    e.kind == PK_CONV_BN ? reinterpret_cast<const float*>(base + e.bias_off) : nullptr);
        break;
      }
      case PK_LINEAR: case PK_LINEAR_T: {
        LoraPackEntry le;
        if (const int rc = linear(e, &le)) return rc;
        const bool t = e.kind == PK_LINEAR_T;
        if (e.lora && le.r <= 16) {  // the 128 LoRA-targeted projections: folded by the multi-tensor kernel after the loop
          multi[t].push_back(le);
          break;
        }
        err = (t ? pack_linear_dgrad_weight : pack_linear_weight)(le.w, e.N, e.C, le.la, le.lb, le.r, scale, e.ldo, base + e.off, ctx->fp16, st);
        break;
      }
      case PK_LORA_A: case PK_LORA_BT: {
        if (ad.empty()) break;
        const ParamRef* f = get(e.src + (e.kind == PK_LORA_A ? ".lora_A." : ".lora_B.") + ad + ".weight");
        if (!f) break;  // module not wrapped (zero-adapter configuration)
        LoraPackEntry le{f->p, nullptr, nullptr, base + e.off, 0, 0, 0, e.ldo};
        if (e.kind == PK_LORA_A) {
          if (f->shape[0] != 16 || f->shape[1] != e.C) return set_err(ctx, MADM_EINVAL, "training path: lora_A must be [16, in]: " + e.src);
          le.N = 16; le.K = e.C;
          multi[0].push_back(le);  // [16, in] as is
        } else {
          if (f->shape[0] != e.N || f->shape[1] != 16) return set_err(ctx, MADM_EINVAL, "training path: lora_B must be [out, 16]: " + e.src);
          le.N = e.N; le.K = 16;
          multi[1].push_back(le);  // [out, 16] -> [16, out]
        }
        break;
      }
      case PK_GEGLU: {
        const ParamRef* w = get(e.src); const ParamRef* bb = get(e.src2);
        if (!w || !bb) return set_err(ctx, MADM_ENOTFOUND, "parameter not registered: " + e.src);
        err = pack_geglu_weight(w->p, bb->p, e.N, e.C, base + e.off, reinterpret_cast<float*>(base + e.bias_off), ctx->fp16, st);
        break;
      }
      case PK_VAE_HEAD: {
        const ParamRef *w = get(e.src), *b1 = get(e.src2), *wq = get(e.src3), *bq = get(e.src4);
        if (!w || !b1 || !wq || !bq) return set_err(ctx, MADM_ENOTFOUND, "parameter not registered: " + e.src);
        err = pack_vae_latent_head(w->p, b1->p, wq->p, bq->p, 0.18215f, e.C, base + e.off, reinterpret_cast<float*>(base + e.bias_off),
                                   ctx->fp16, st);
        break;
      }
      case PK_F32_COPY: {
        const ParamRef* s = get(e.src);
        if (!s) return set_err(ctx, MADM_ENOTFOUND, "parameter not registered: " + e.src);
        if (cudaMemcpyAsync(base + e.off, s->p, size_t(e.N) * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess) err = "cudaMemcpyAsync failed";
        break;
      }
      case PK_BN_FOLD: {
        const ParamRef *g = get(e.src + ".weight"), *bt = get(e.src + ".bias"), *mu = get(e.src + ".running_mean"), *var = get(e.src + ".running_var");
        if (!g || !bt || !mu || !var) return set_err(ctx, MADM_ENOTFOUND, "BatchNorm parameters / running statistics not registered: " + e.src);
        if (g->numel() != e.N || bt->numel() != e.N || mu->numel() != e.N || var->numel() != e.N)
          return set_err(ctx, MADM_EINVAL, "unexpected shape: " + e.src);
        err = bn_fold(g->p, bt->p, mu->p, var->p, nullptr, 1e-5f, e.N, reinterpret_cast<float*>(base + e.off), st);
        break;
      }
      case PK_DW_BN: {
        const ParamRef* w = get(e.src);
        if (!w) return set_err(ctx, MADM_ENOTFOUND, "parameter not registered: " + e.src);
        if (w->numel() != int64_t(e.C) * 9) return set_err(ctx, MADM_EINVAL, "unexpected shape: " + e.src);
        err = pack_depthwise(w->p, reinterpret_cast<const float*>(base + e.bias_off), e.C, reinterpret_cast<float*>(base + e.off), st);
        break;
      }
      case PK_IDENTITY: {
        identity16_kernel<<<(e.N * e.N + 255) / 256, 256, 0, st>>>(reinterpret_cast<uint16_t*>(base + e.off), e.N, e.ldo,
                                                                  ctx->fp16 ? uint16_t(0x3C00) : uint16_t(0x3F80));
        if (cudaGetLastError() != cudaSuccess) err = "identity16 launch failed";
        break;
      }
      case PK_F32_SUM2: {
        const ParamRef *a = get(e.src), *b2 = get(e.src2);
        if (!a || !b2) return set_err(ctx, MADM_ENOTFOUND, "parameter not registered: " + e.src);
        f32_sum2_kernel<<<(e.N + 255) / 256, 256, 0, st>>>(a->p, b2->p, e.N, reinterpret_cast<float*>(base + e.off));
        if (cudaGetLastError() != cudaSuccess) err = "f32_sum2 launch failed";
        break;
      }
      case PK_REGION: break;
    }
    if (err) return set_err(ctx, MADM_ECUDA, err);
  }
  for (int t = 0; t < 2; ++t)
    if (!multi[t].empty())
      if (const char* err = pack_lora_multi(multi[t].data(), int(multi[t].size()), scale, t, ctx->fp16, st)) return set_err(ctx, MADM_ECUDA, err);
  return MADM_OK;
}

}  // namespace

// ================================================================================================ C ABI
extern "C" {

int madm_version(void) { return MADM_VERSION; }

const char* madm_last_error(const madm_ctx* ctx) { return ctx ? ctx->err.c_str() : global_error(); }

int madm_create(madm_ctx** out, int device) {
  if (!out) return set_err(nullptr, MADM_EINVAL, "madm_create: null out");
  int ndev = 0;
  if (getenv("MADM_PLAN_ONLY")) {
    // host-side test hook: a context without a device, good for the planner's dry runs only (packed-arena layouts, workspace sizes,
    // launch counts); nothing can be launched from it -- there is no CPU compute path
    std::unique_ptr<madm_ctx> c(new madm_ctx());
    c->device = -1;
    *out = c.release();
    return MADM_OK;
  }
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_err(nullptr, MADM_ECUDA, "madm_create: no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return set_err(nullptr, MADM_EINVAL, "madm_create: bad device index");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return set_err(nullptr, MADM_ECUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10) return set_err(nullptr, MADM_ECUDA, "madm_create: device is not sm_100 (B200); kernels are built for sm_100a only");
  if (cudaSetDevice(device) != cudaSuccess) return set_err(nullptr, MADM_ECUDA, "cudaSetDevice failed");
  std::unique_ptr<madm_ctx> c(new madm_ctx());
  c->device = device;
  // DDPM alphas_cumprod (scaled_linear 0.00085..0.012, 1000 steps; fp32 like DDPMScheduler) — SURVEY Appendix A.3
  std::vector<float> ac(1000);
  {
    const float s0 = sqrtf(0.00085f), s1 = sqrtf(0.012f);
    float prod = 1.0f;
    for (int i = 0; i < 1000; ++i) {
      const float step = (s1 - s0) / 999.0f;
      // torch.linspace computes the upper half from the end point for symmetry
      const float v = (i < 500) ? s0 + step * float(i) : s1 - step * float(999 - i);
      const float beta = v * v;
      prod *= (1.0f - beta);
      ac[i] = prod;
    }
  }
  if (cudaMalloc(&c->alphas_cumprod, 1000 * sizeof(float)) != cudaSuccess) return set_err(nullptr, MADM_ECUDA, "cudaMalloc failed");
  if (cudaMemcpy(c->alphas_cumprod, ac.data(), 1000 * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess)
    return set_err(nullptr, MADM_ECUDA, "cudaMemcpy failed");
  *out = c.release();
  return MADM_OK;
}

int madm_destroy(madm_ctx* ctx) {
  if (!ctx) return MADM_OK;
  if (ctx->alphas_cumprod) cudaFree(ctx->alphas_cumprod);
  for (int k = 0; k < 4; ++k) {
    if (ctx->ev_fork[k]) cudaEventDestroy(ctx->ev_fork[k]);
    if (ctx->ev_join[k]) cudaEventDestroy(ctx->ev_join[k]);
    if (ctx->side[k]) cudaStreamDestroy(ctx->side[k]);
  }
  delete ctx;
  return MADM_OK;
}

int madm_set_compute_dtype(madm_ctx* ctx, int32_t dtype) {
  if (!ctx || (dtype != MADM_DTYPE_BF16 && dtype != MADM_DTYPE_FP16)) return set_err(ctx, MADM_EINVAL, "madm_set_compute_dtype: bad argument");
  const int f = dtype == MADM_DTYPE_FP16 ? 1 : 0;
  if (f != ctx->fp16) {
    ctx->fp16 = f;
    invalidate(ctx, LAYOUT_INPUTS);  // the packed layout depends on the operand dtype (16-bit VAE stream: identity segments)
  }
  return MADM_OK;
}

int madm_get_compute_dtype(const madm_ctx* ctx) { return ctx && !ctx->fp16 ? MADM_DTYPE_BF16 : MADM_DTYPE_FP16; }

int madm_set_variant(madm_ctx* ctx, int32_t variant) {
  if (!ctx || (variant != MADM_VARIANT_BASE && variant != MADM_VARIANT_S0)) return set_err(ctx, MADM_EINVAL, "madm_set_variant: bad argument");
  if (variant != ctx->variant) {
    ctx->variant = variant;
    invalidate(ctx, LAYOUT_INPUTS);
  }
  return MADM_OK;
}

int madm_get_variant(const madm_ctx* ctx) { return ctx ? ctx->variant : MADM_VARIANT_BASE; }

int madm_set_tensors(madm_ctx* ctx, const madm_tensor* named, int32_t n) {
  if (!ctx || (!named && n > 0)) return set_err(ctx, MADM_EINVAL, "madm_set_tensors: null argument");
  for (int i = 0; i < n; ++i) {
    const madm_tensor& t = named[i];
    if (!t.name || !t.data || t.ndim < 0 || t.ndim > 4) return set_err(ctx, MADM_EINVAL, "madm_set_tensors: bad tensor record");
    ParamRef r;
    r.p = static_cast<const float*>(t.data);
    r.ndim = t.ndim;
    for (int k = 0; k < t.ndim; ++k) r.shape[k] = t.shape[k];
    auto it = ctx->params.find(t.name);
    // a new name (adapters / EMA twins added) or a new shape under a known one: the model changed shape
    if (it == ctx->params.end() || it->second.ndim != r.ndim || !std::equal(r.shape, r.shape + r.ndim, it->second.shape))
      invalidate(ctx, LAYOUT_INPUTS);
    ctx->params[t.name] = r;
  }
  invalidate(ctx, PARAM_POINTERS);
  return MADM_OK;
}

size_t madm_packed_bytes(madm_ctx* ctx) {
  if (!ctx) return 0;
  if (ensure_layout(ctx) != MADM_OK) return 0;
  return ctx->fwd.bytes;
}

int madm_pack_weights(madm_ctx* ctx, void* packed, const char* adapter, float scale, int32_t lora_only, madm_stream stream) {
  if (!ctx || !packed) return set_err(ctx, MADM_EINVAL, "madm_pack_weights: null argument");
  if (ctx->device < 0) return set_err(ctx, MADM_ECUDA, "madm_pack_weights: this context was created without a device (MADM_PLAN_ONLY)");
  const int rc = ensure_layout(ctx);
  if (rc != MADM_OK) return rc;
  const Subset subset = lora_only == 1 ? PACK_LORA : lora_only == 2 ? PACK_TRAINABLE : PACK_ALL;
  return pack_arena(ctx, ctx->fwd, static_cast<uint8_t*>(packed), adapter ? adapter : "", scale, subset, static_cast<cudaStream_t>(stream));
}

size_t madm_workspace_bytes(madm_ctx* ctx, int32_t B) { return madm_workspace_bytes_head(ctx, B, 0, 0); }

size_t madm_workspace_bytes_head(madm_ctx* ctx, int32_t B, int32_t head_h, int32_t head_w) {
  if (!ctx || B < 1 || head_h < 0 || head_w < 0) return 0;
  if (ensure_layout(ctx) != MADM_OK) return 0;
  const std::tuple<int, int, int> key{B, head_h, head_w};
  auto it = ctx->ws_bytes_cache.find(key);
  if (it != ctx->ws_bytes_cache.end()) return it->second;
  size_t bytes = 0;
  if (dry_run(ctx, SIZE, B, &bytes, head_h, head_w) != MADM_OK) return 0;
  ctx->ws_bytes_cache[key] = bytes;
  return bytes;
}

int madm_set_profiling(madm_ctx* ctx, int32_t on) {
  if (!ctx) return MADM_EINVAL;
  ctx->profiling = on != 0;
  return MADM_OK;
}

int madm_get_profile(madm_ctx* ctx, madm_profile* out) { return madm_get_profile_stages(ctx, ~0, out); }

int madm_get_profile_stages(madm_ctx* ctx, int32_t stage_mask, madm_profile* out) {
  if (!ctx || !out) return set_err(ctx, MADM_EINVAL, "madm_get_profile: null argument");
  Plan* plan = ctx->last_plan;
  if (!plan || plan->ev.size() != 2 * plan->ops.size()) return set_err(ctx, MADM_ESTATE, "madm_get_profile: no profiled madm_extract call");
  static const char* names[MADM_NUM_KINDS] = {"gemm_tc", "flash_attention", "groupnorm", "layernorm", "elementwise"};
  for (int k = 0; k < MADM_NUM_KINDS; ++k) {
    snprintf(out->kind[k].name, sizeof(out->kind[k].name), "%s", names[k]);
    out->kind[k].launches = 0; out->kind[k].ms = 0; out->kind[k].flops = 0; out->kind[k].bytes = 0; out->kind[k].exec_flops = 0;
  }
  if (cudaDeviceSynchronize() != cudaSuccess) return set_err(ctx, MADM_ECUDA, "cudaDeviceSynchronize failed");
  for (size_t i = 0; i < plan->ops.size(); ++i) {
    const Launch& l = plan->ops[i];
    if (!(l.stage & ctx->last_stages) || !(l.stage & stage_mask) || l.optional) continue;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, plan->ev[2 * i], plan->ev[2 * i + 1]) != cudaSuccess) continue;
    out->kind[l.kind].launches += 1; out->kind[l.kind].ms += ms; out->kind[l.kind].flops += l.flops; out->kind[l.kind].bytes += l.bytes;
    out->kind[l.kind].exec_flops += l.exec_flops;
  }
  return MADM_OK;
}

int madm_launch_count(madm_ctx* ctx, int32_t B, int32_t stages) {
  if (!ctx || B < 1) return -1;
  auto it = ctx->plans.end();
  for (auto p = ctx->plans.begin(); p != ctx->plans.end(); ++p)
    if (std::get<0>(p->first) == B) { it = p; break; }
  if (it == ctx->plans.end()) return -1;
  int n = 0;
  for (const Launch& l : it->second->ops)
    if ((l.stage & stages) && !l.optional) ++n;
  return n;
}

int madm_extract(madm_ctx* ctx, const madm_extract_args* a, madm_stream stream) {
  if (!ctx || !a) return set_err(ctx, MADM_EINVAL, "madm_extract: null argument");
  if (ctx->device < 0) return set_err(ctx, MADM_ECUDA, "madm_extract: this context was created without a device (MADM_PLAN_ONLY)");
  if (a->B < 1) return set_err(ctx, MADM_EINVAL, "madm_extract: B must be >= 1");
  if (!a->packed || !a->workspace) return set_err(ctx, MADM_ESTATE, "madm_extract: packed arena and workspace are required");
  if ((a->stages & MADM_STAGE_VAE) && !a->img) return set_err(ctx, MADM_EINVAL, "madm_extract: img is null");
  if ((a->stages & MADM_STAGE_DEC) && ctx->variant != MADM_VARIANT_S0)
    return set_err(ctx, MADM_EINVAL, "madm_extract: MADM_STAGE_DEC needs madm_set_variant(MADM_VARIANT_S0)");
  if ((a->unet_sample || a->decoded || a->decoded_raw) && !(a->stages & MADM_STAGE_DEC))
    return set_err(ctx, MADM_EINVAL, "madm_extract: unet_sample / decoded / decoded_raw are outputs of MADM_STAGE_DEC");
  if ((a->stages & MADM_STAGE_UNET) && (!a->cond_inputs || !a->cond_emb || !a->timesteps || (!a->shared_noise && !a->noisy_latents_in)))
    return set_err(ctx, MADM_EINVAL, "madm_extract: conditioning / timesteps / shared_noise are required for the UNet stage");
  int rc = ensure_layout(ctx);
  if (rc != MADM_OK) return rc;
  if (a->flags & MADM_FLAG_TRAIN) return extract_train(ctx, a, static_cast<cudaStream_t>(stream));
  if (a->head_h < 0 || a->head_w < 0 || ((a->head_h > 0) != (a->head_w > 0))) return set_err(ctx, MADM_EINVAL, "madm_extract: bad head_h / head_w");
  if ((a->flags & MADM_FLAG_OUT_FP16) && (ctx->variant != MADM_VARIANT_BASE || (a->stages & MADM_STAGE_HEAD)))
    return set_err(ctx, MADM_EINVAL, "madm_extract: MADM_FLAG_OUT_FP16 is for the base variant's feature maps (not with MADM_STAGE_HEAD in the same call)");
  const size_t need = madm_workspace_bytes_head(ctx, a->B, a->head_h, a->head_w);
  if (need == 0) return MADM_EINVAL;
  if (a->workspace_bytes < need) return set_err(ctx, MADM_ENOMEM, "madm_extract: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  const std::tuple<int, int, int, int> key{a->B, a->ema ? 1 : 0, a->head_h, a->head_w};
  Plan* plan = nullptr;
  auto it = ctx->plans.find(key);
  if (it != ctx->plans.end() && it->second->packed == a->packed && it->second->ws == a->workspace) plan = it->second.get();
  if (!plan) {
    std::unique_ptr<Plan> np(new Plan());
    np->packed = a->packed; np->ws = a->workspace; np->ws_bytes = a->workspace_bytes;
    Builder cfg{ctx, PLAN, a->B, a->ema != 0};
    cfg.head_h = a->head_h; cfg.head_w = a->head_w;
    rc = build_plan(ctx, cfg, np.get());
    if (rc != MADM_OK) return rc;
    plan = np.get();
    ctx->plans[key] = std::move(np);
  }
  plan->io.a = *a;
  const bool prof = ctx->profiling;
  if (prof && plan->ev.size() != 2 * plan->ops.size()) {
    plan->ev.resize(2 * plan->ops.size());
    for (cudaEvent_t& e : plan->ev)
      if (cudaEventCreate(&e) != cudaSuccess) return set_err(ctx, MADM_ECUDA, "cudaEventCreate failed");
  }
  // Branch ops (the four projections) run on side streams between a fork and a join event unless per-launch profiling is on
  // (its per-family accounting assumes one stream).
  bool use_side = !prof;
  if (use_side) {
    bool any = false;
    for (size_t i = 0; i < plan->ops.size() && !any; ++i) any = plan->ops[i].branch != 0 && (plan->ops[i].stage & a->stages);
    use_side = any;
  }
  if (use_side && !ctx->ev_fork[0]) {
    bool ok = true;
    for (int k = 0; k < 4 && ok; ++k)
      ok = cudaStreamCreateWithFlags(&ctx->side[k], cudaStreamNonBlocking) == cudaSuccess &&
           cudaEventCreateWithFlags(&ctx->ev_fork[k], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&ctx->ev_join[k], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) return set_err(ctx, MADM_ECUDA, "madm_extract: could not create the projection streams");
  }
  rc = replay(ctx, plan->ops, a->stages, st, use_side, prof ? plan->ev.data() : nullptr, "op");
  if (rc != MADM_OK) return rc;
  ctx->last_plan = plan;
  ctx->last_stages = a->stages;
  return MADM_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ training path (SURVEY §8 row f-3)
extern "C" size_t madm_train_workspace_bytes(madm_ctx* ctx, int32_t B, const char* adapter);
namespace {
// madm_extract with MADM_FLAG_TRAIN: the forward of a training plan (activations kept for madm_backward)
int extract_train(madm_ctx* ctx, const madm_extract_args* a, cudaStream_t st) {
  if (a->stages != (ctx->variant == MADM_VARIANT_S0 ? MADM_STAGE_ALL_S0 : MADM_STAGE_ALL))
    return set_err(ctx, MADM_EINVAL, "madm_extract: MADM_FLAG_TRAIN runs all stages (MADM_STAGE_ALL; MADM_STAGE_ALL_S0 in the s0 variant)");
  if (a->ema) return set_err(ctx, MADM_EINVAL, "madm_extract: MADM_FLAG_TRAIN with the EMA projections (the teacher runs without gradient)");
  if (a->flags & MADM_FLAG_OUT_FP16) return set_err(ctx, MADM_EINVAL, "madm_extract: MADM_FLAG_OUT_FP16 with MADM_FLAG_TRAIN (madm_backward reads the fp32 outputs)");
  if (!a->packed_dgrad) return set_err(ctx, MADM_ESTATE, "madm_extract: MADM_FLAG_TRAIN needs packed_dgrad (madm_pack_dgrad_weights)");
  if (!(a->train_loss_scale > 0.f)) return set_err(ctx, MADM_EINVAL, "madm_extract: train_loss_scale must be > 0");
  if (a->B > 8) return set_err(ctx, MADM_EINVAL, "madm_extract: MADM_FLAG_TRAIN supports B <= 8");
  int rc = ensure_dlayout(ctx);
  if (rc != MADM_OK) return rc;
  const std::string ad = a->train_adapter ? a->train_adapter : "";
  Plan* plan = nullptr;
  const std::pair<int, uintptr_t> tkey{a->B, reinterpret_cast<uintptr_t>(a->workspace)};
  auto it = ctx->train_plans.find(tkey);
  if (it != ctx->train_plans.end()) {
    Plan* q = it->second.get();
    if (q->packed == a->packed && q->dpacked == a->packed_dgrad && q->ws == a->workspace && q->adapter == ad && q->loss_scale == a->train_loss_scale &&
        q->lora_scale == a->train_lora_scale)
      plan = q;
  }
  if (!plan) {
    const size_t need = madm_train_workspace_bytes(ctx, a->B, ad.c_str());
    if (need == 0) return MADM_EINVAL;
    if (a->workspace_bytes < need) return set_err(ctx, MADM_ENOMEM, "madm_extract: training workspace too small (madm_train_workspace_bytes)");
    std::unique_ptr<Plan> np(new Plan());
    np->packed = a->packed; np->dpacked = a->packed_dgrad; np->ws = a->workspace; np->ws_bytes = a->workspace_bytes;
    np->train = true; np->adapter = ad; np->loss_scale = a->train_loss_scale; np->lora_scale = a->train_lora_scale;
    Builder cfg{ctx, PLAN, a->B, false};
    cfg.train = true; cfg.adapter = ad; cfg.lora_scale = a->train_lora_scale; cfg.loss_scale = a->train_loss_scale;
    rc = build_plan(ctx, cfg, np.get());
    if (rc != MADM_OK) return rc;
    plan = np.get();
    ctx->train_plans[tkey] = std::move(np);
  }
  plan->io.a = *a;
  PdlTrainScope pdl;  // programmatic dependent launch for the training forward's ~550 small launches (launch.cuh)
  return replay(ctx, plan->ops, ~0, st, false, nullptr, "training forward op");
}
}  // namespace

extern "C" {

int madm_set_grad_tensors(madm_ctx* ctx, const madm_tensor* named, int32_t n) {
  if (!ctx || (!named && n > 0)) return set_err(ctx, MADM_EINVAL, "madm_set_grad_tensors: null argument");
  ctx->grads.clear();
  for (int i = 0; i < n; ++i) {
    if (!named[i].name || !named[i].data) return set_err(ctx, MADM_EINVAL, "madm_set_grad_tensors: bad tensor record");
    auto it = ctx->params.find(named[i].name);
    if (it == ctx->params.end()) return set_err(ctx, MADM_ENOTFOUND, std::string("madm_set_grad_tensors: no such parameter: ") + named[i].name);
    int64_t numel = 1;
    for (int k = 0; k < named[i].ndim; ++k) numel *= named[i].shape[k];
    if (numel != it->second.numel()) return set_err(ctx, MADM_EINVAL, std::string("madm_set_grad_tensors: shape mismatch: ") + named[i].name);
    ctx->grads[named[i].name] = static_cast<float*>(const_cast<void*>(named[i].data));
  }
  invalidate(ctx, GRAD_BUFFERS);
  return MADM_OK;
}

size_t madm_dgrad_packed_bytes(madm_ctx* ctx) {
  if (!ctx || ensure_dlayout(ctx) != MADM_OK) return 0;
  return ctx->dgrad.bytes;
}

int madm_pack_dgrad_weights(madm_ctx* ctx, void* packed, const char* adapter, float scale, int32_t trainable_only, madm_stream stream) {
  if (!ctx || !packed) return set_err(ctx, MADM_EINVAL, "madm_pack_dgrad_weights: null argument");
  if (ctx->device < 0) return set_err(ctx, MADM_ECUDA, "madm_pack_dgrad_weights: this context was created without a device (MADM_PLAN_ONLY)");
  const int rc = ensure_dlayout(ctx);
  if (rc != MADM_OK) return rc;
  return pack_arena(ctx, ctx->dgrad, static_cast<uint8_t*>(packed), adapter ? adapter : "", scale, trainable_only ? PACK_TRAINABLE : PACK_ALL,
                    static_cast<cudaStream_t>(stream));
}

size_t madm_train_workspace_bytes(madm_ctx* ctx, int32_t B, const char* adapter) {
  if (!ctx || B < 1) return 0;
  if (ensure_dlayout(ctx) != MADM_OK) return 0;
  size_t bytes = 0;
  if (dry_run(ctx, SIZE, B, &bytes, 0, 0, /*train=*/true, adapter ? adapter : "") != MADM_OK) return 0;
  return bytes;
}

int madm_backward_launch_count(madm_ctx* ctx, int32_t B) {
  if (!ctx) return -1;
  for (auto& kv : ctx->train_plans)
    if (kv.first.first == B) return int(kv.second->bops.size());
  return -1;
}

int madm_backward(madm_ctx* ctx, const madm_backward_args* a, madm_stream stream) {
  if (!ctx || !a) return set_err(ctx, MADM_EINVAL, "madm_backward: null argument");
  if (ctx->device < 0) return set_err(ctx, MADM_ECUDA, "madm_backward: this context was created without a device (MADM_PLAN_ONLY)");
  auto it = ctx->train_plans.find({a->B, reinterpret_cast<uintptr_t>(a->workspace)});
  if (it == ctx->train_plans.end()) return set_err(ctx, MADM_ESTATE, "madm_backward: no MADM_FLAG_TRAIN forward at this batch size in this workspace");
  Plan* plan = it->second.get();
  const std::string ad = a->adapter ? a->adapter : "";
  if (plan->ws != a->workspace || plan->packed != a->packed || plan->dpacked != a->packed_dgrad || plan->adapter != ad ||
      plan->loss_scale != a->loss_scale || plan->lora_scale != a->lora_alpha_over_r)
    return set_err(ctx, MADM_ESTATE, "madm_backward: arguments differ from the MADM_FLAG_TRAIN forward this plan was built for");
  plan->io.b = *a;
  PdlTrainScope pdl;  // programmatic dependent launch for the backward's ~640 small launches (launch.cuh)
  return replay(ctx, plan->bops, ~0, static_cast<cudaStream_t>(stream), false, nullptr, "backward op");
}

}  // extern "C"
