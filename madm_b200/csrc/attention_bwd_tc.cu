// tcgen05 / TMEM backward of softmax(Q K^T * scale) V for the UNet's large self-attention layers (d <= 64: the 64x64-token level, d = 40,
// n = 4096 -- 5 of the 16 transformer blocks and ~60 % of the training step's attention FLOPs).  SURVEY §8 row f-3; the reference
// back-propagates through diffusers' Attention processors (modeling/meta_arch/mtmadise.py:240-302 under engine/train_loop.py:277-302).
//
// Flash-style, no stored probabilities, deterministic (no atomics): one kernel template, two roles.
//   MODE 0 (dK, dV)  CTA = 128 keys of one (image, head), resident K_j, V_j; streams the query tiles (Q_i, dO_i, L_i, D_i):
//                      X = K_j Q_i^T = S^T        Y = V_j dO_i^T = dP^T                (128 x 128 x d, both operands K-major in smem)
//                      P^T = 2^(X c - L2[col])    dS^T = P^T (Y - D[col])              (thread = key row; L2 / D per column from smem)
//                      dV_j += P^T dO_i           dK_j += dS^T Q_i                     (A = 16-bit tile in TENSOR MEMORY, B = the streamed
//                                                                                       tile read MN-major: no transposes anywhere)
//   MODE 1 (dQ)      CTA = 128 queries, resident Q_i, dO_i; streams the key tiles (K_j, V_j):
//                      X = Q_i K_j^T = S          Y = dO_i V_j^T = dP                  P = 2^(X c - L2[row]), dS = P (Y - D[row])
//                      dQ_i += dS K_j
// L2 = log-sum-exp of the scaled scores times log2(e) (the forward kernel writes the log-sum-exp), D = rowsum(dO * O).
// TMEM (512 columns): X 128 | Y 128 | P 64 | dS 64 | acc(P product) 64 | acc(dS product) 64 -- every fp32 accumulator of the two
// running products stays in tensor memory for the whole loop.  Warp roles: warp 0 TMA producer (2-stage ring), warp 1 TMEM allocator +
// MMA issuer, warps 4-11 softmax (two warps per TMEM lane quarter: each thread owns one row and 64 of its 128 columns).
// The 16-bit P / dS tiles are pre-scaled by powers of two (fp16 subnormals: dS ~ 1e-8..1e-5) exactly like the warp-level kernels in
// attention_bwd.cu, which remain the path for d = 160, ragged token counts and the 77-key cross-attention.
// Template axes: KC = 64-column chunks per operand row (1: d <= 64, 2: d = 80) and TN = rows of a streamed tile (128, or 64 for KC = 2 so
// that two 80-column accumulators fit: X 64 | Y 64 | P 32 | dS 32 | acc 96 | acc 96 = 384 columns).
#include "cvt.cuh"
#include "kernels.h"
#include "launch.cuh"
#include "ptx.cuh"

#include <mutex>
#include <stdio.h>

namespace madm {

namespace {

constexpr int BT_TILE = 128 * 128;   // bytes of one [128 rows][64 x 16-bit] swizzled operand chunk
constexpr int BT_STAGES = 4;     // streamed-tile ring: the refill of a slot starts when its products retire, two to three tiles before it is needed
constexpr int BT_THREADS = 384;
constexpr float kPScale = 256.0f;      // P <= 1
constexpr float kDsScale = 16384.0f;   // same constants as attention_bwd.cu
template <int KC, int TN>
struct BtCfg {
  static constexpr int RES = KC * BT_TILE;        // bytes of a resident operand tile (128 rows)
  static constexpr int STR = KC * TN * 128;       // bytes of a streamed operand tile (TN rows)
  static constexpr int SLOT = 2 * STR;            // ring slot: T1 | T2
  static constexpr int ACC = KC == 1 ? 64 : 96;   // TMEM columns per accumulator
  static constexpr int CPT = TN / 2;              // columns of X / Y per softmax thread
  static constexpr int NCH = CPT / 32;            // 32-column chunks per thread
  static constexpr size_t SMEM = size_t(2) * RES + size_t(BT_STAGES) * (SLOT + 1024) + 256 + 1024;
  static_assert(3 * TN + 2 * ACC <= 512, "TMEM budget");
  static_assert(SMEM <= 227 * 1024, "smem budget");
};

struct BwdTcParams {
  CUtensorMap tmR1, tmR2, tmT1, tmT2;  // resident / streamed operand maps: MODE 0: K, V, Q, dO; MODE 1: Q, dO, K, V
  const float* L2;                     // [B, heads, Nq] log2-domain log-sum-exp
  const float* D;                      // [B, heads, Nq]
  uint16_t* out_s; int ld_s; long bs_s;  // dS product: dK (MODE 0) / dQ (MODE 1)
  uint16_t* out_p; int ld_p; long bs_p;  // P product: dV (MODE 0)
  int Nq, n_stream;                    // streamed tiles per CTA
  int d, ksteps, dv;                   // head dim, 16-wide k-steps carrying data, output columns (UMMA N)
  float scale_log2, out_scale_s, out_scale_p;
};

__device__ __forceinline__ float bt_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

template <int MODE, bool FP16, int KC, int TN>
__global__ void __launch_bounds__(BT_THREADS, 1) attn_bwd_tc_kernel(const __grid_constant__ BwdTcParams p) {
  using Cf = BtCfg<KC, TN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sR1 = base, sR2 = base + Cf::RES;
  auto sT1 = [&](int st) { return base + 2 * Cf::RES + uint32_t(st) * Cf::SLOT; };
  auto sT2 = [&](int st) { return sT1(st) + Cf::STR; };
  const uint32_t sVec = base + 2 * Cf::RES + BT_STAGES * Cf::SLOT;  // per stage: L2[TN] | (at +512 B) D[TN] floats
  const uint32_t sBar = sVec + BT_STAGES * 1024;
  const uint32_t r_full = sBar;
  auto t_full = [&](int s) { return sBar + 8u * (1 + s); };
  auto t_empty = [&](int s) { return sBar + 8u * (1 + BT_STAGES + s); };
  // x_full: X / Y complete -> softmax; xy_free: the softmax warps hold all of X / Y in registers -> the next tile's X / Y MMAs may overwrite them
  // (they then run under the second half of this tile's softmax arithmetic); p_ready: the 16-bit P / dS tiles are in tensor memory
  constexpr uint32_t kB0 = 1 + 2 * BT_STAGES;
  const uint32_t x_full = sBar + 8u * kB0, xy_free = sBar + 8u * (kB0 + 1), o_done = sBar + 8u * (kB0 + 2), p_ready = sBar + 8u * (kB0 + 3);
  const uint32_t tmem_slot = sBar + 8u * (kB0 + 4);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = blockIdx.x * 128, h = blockIdx.y, b = blockIdx.z;
  const int n = p.n_stream;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tmR1); prefetch_tmap(&p.tmR2); prefetch_tmap(&p.tmT1); prefetch_tmap(&p.tmT2);
    mbar_init(r_full, 1);
    for (int s = 0; s < BT_STAGES; ++s) { mbar_init(t_full(s), 1); mbar_init(t_empty(s), 1); }
    mbar_init(x_full, 1); mbar_init(xy_free, 8); mbar_init(o_done, 1); mbar_init(p_ready, 8);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  const uint32_t tX = tmem, tY = tmem + TN, tP = tmem + 2 * TN, tdS = tmem + 2 * TN + TN / 2, tAccP = tmem + 3 * TN, tAccS = tmem + 3 * TN + Cf::ACC;
  pdl_trigger();
  pdl_wait();

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      mbar_arrive_expect_tx(r_full, 2 * Cf::RES);
#pragma unroll
      for (int kc = 0; kc < KC; ++kc) {
        tma_load_4d(sR1 + kc * BT_TILE, &p.tmR1, r_full, kc * 64, h, r0, b);
        tma_load_4d(sR2 + kc * BT_TILE, &p.tmR2, r_full, kc * 64, h, r0, b);
      }
      const float* l2g = p.L2 + (size_t(b) * gridDim.y + h) * p.Nq;
      const float* dg = p.D + (size_t(b) * gridDim.y + h) * p.Nq;
      for (int it = 0; it < n; ++it) {
        const int st = it % BT_STAGES;
        mbar_wait(t_empty(st), ((it / BT_STAGES) & 1) ^ 1u);
        mbar_arrive_expect_tx(t_full(st), 2 * Cf::STR + (MODE == 0 ? 2 * TN * 4 : 0));
#pragma unroll
        for (int kc = 0; kc < KC; ++kc) {
          tma_load_4d(sT1(st) + kc * (TN * 128), &p.tmT1, t_full(st), kc * 64, h, it * TN, b);
          tma_load_4d(sT2(st) + kc * (TN * 128), &p.tmT2, t_full(st), kc * 64, h, it * TN, b);
        }
        if constexpr (MODE == 0) {  // the streamed query tile's L2 / D vectors
          bulk_load_1d(sVec + st * 1024, l2g + it * TN, TN * 4, t_full(st));
          bulk_load_1d(sVec + st * 1024 + 512, dg + it * TN, TN * 4, t_full(st));
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      const uint32_t idesc_x = make_idesc_16(128, TN, FP16 ? 1 : 0);
      const uint32_t idesc_o = make_idesc_16(128, p.dv, FP16 ? 1 : 0) | (1u << 16);  // B operand MN-major
      const int ksteps = p.ksteps;
      const uint64_t r1d = make_smem_desc_sw128(sR1), r2d = make_smem_desc_sw128(sR2);
      // descriptors of ring slot 0; slot s is the same descriptor + s * (slot bytes >> 4) in the start-address field (no carry: smem < 256 KB)
      const uint64_t t1d0 = make_smem_desc_sw128(sT1(0)), t2d0 = make_smem_desc_sw128(sT2(0));
      const uint64_t t1mn0 = make_smem_desc_sw128_mn(sT1(0), TN * 128), t2mn0 = make_smem_desc_sw128_mn(sT2(0), TN * 128);
      constexpr uint64_t kSlot = Cf::SLOT >> 4;
      constexpr uint64_t kResChunk = BT_TILE >> 4, kStrChunk = (TN * 128) >> 4;  // 64-column chunk strides of the K-major operands
      auto issue_xy = [&](int it) {  // X = R1 T1^T, Y = R2 T2^T
        const int st = it % BT_STAGES;
        mbar_wait(t_full(st), (it / BT_STAGES) & 1);
        tc_fence_after();
        const uint64_t a1 = t1d0 + uint64_t(st) * kSlot, a2 = t2d0 + uint64_t(st) * kSlot;
#pragma unroll
        for (int ks = 0; ks < 4 * KC; ++ks)
          if (ks < ksteps)
            umma_bf16_ss(tX, r1d + uint64_t(ks >> 2) * kResChunk + uint64_t(2 * (ks & 3)), a1 + uint64_t(ks >> 2) * kStrChunk + uint64_t(2 * (ks & 3)), idesc_x, ks != 0);
#pragma unroll
        for (int ks = 0; ks < 4 * KC; ++ks)
          if (ks < ksteps)
            umma_bf16_ss(tY, r2d + uint64_t(ks >> 2) * kResChunk + uint64_t(2 * (ks & 3)), a2 + uint64_t(ks >> 2) * kStrChunk + uint64_t(2 * (ks & 3)), idesc_x, ks != 0);
        umma_commit(x_full);
      };
      mbar_wait(r_full, 0);
      issue_xy(0);
      for (int it = 0; it < n; ++it) {
        if (it + 1 < n) {
          mbar_wait(xy_free, it & 1);  // X / Y of this tile are in the softmax warps' registers
          tc_fence_after();
          issue_xy(it + 1);            // first: the next tile's softmax waits for nothing but these
        }
        mbar_wait(p_ready, it & 1);    // the 16-bit P / dS tiles of this tile are posted
        tc_fence_after();
        const int st = it % BT_STAGES;
        const uint64_t b1 = t1mn0 + uint64_t(st) * kSlot, b2 = t2mn0 + uint64_t(st) * kSlot;
#pragma unroll
        for (int kk = 0; kk < TN / 16; ++kk) umma_f16_ts(tAccS, tdS + kk * 8, b1 + uint64_t(kk * (2048 >> 4)), idesc_o, (it > 0 || kk > 0) ? 1u : 0u);
        if constexpr (MODE == 0) {
#pragma unroll
          for (int kk = 0; kk < TN / 16; ++kk) umma_f16_ts(tAccP, tP + kk * 8, b2 + uint64_t(kk * (2048 >> 4)), idesc_o, (it > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(o_done);
        umma_commit(t_empty(st));
      }
    }
  } else if (warp >= 4) {
    // ===================== softmax-gradient warps: thread = row, TN / 2 of its TN columns =====================
    const int q = warp & 3, hf = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const uint32_t lane_base = uint32_t(q * 32) << 16;
    const float sl = p.scale_log2;
    float l2r = 0.f, dr = 0.f;
    if constexpr (MODE == 1) {
      const size_t o = (size_t(b) * gridDim.y + h) * p.Nq + r0 + row;
      l2r = p.L2[o];
      dr = p.D[o];
    }
    for (int it = 0; it < n; ++it) {
      const int st = it % BT_STAGES;
      mbar_wait(x_full, it & 1);
      tc_fence_after();
      uint32_t pkS[Cf::NCH * 16], pkP[MODE == 0 ? Cf::NCH * 16 : 1];
#pragma unroll
      for (int ch = 0; ch < Cf::NCH; ++ch) {
        const int c0 = hf * Cf::CPT + ch * 32;
        uint32_t xr[32], yr[32];
        __syncwarp();
        tmem_ld32(tX + lane_base + c0, xr);
        tmem_ld32(tY + lane_base + c0, yr);
        tmem_ld_wait();
        if (ch == Cf::NCH - 1) {  // every column of X / Y this warp owns is in registers
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(xy_free);
        }
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          float4 l4, d4;
          if constexpr (MODE == 0) {
            l4 = lds_f4(sVec + st * 1024 + uint32_t(c0 + i) * 4);
            d4 = lds_f4(sVec + st * 1024 + 512 + uint32_t(c0 + i) * 4);
          } else {
            l4 = make_float4(l2r, l2r, l2r, l2r);
            d4 = make_float4(dr, dr, dr, dr);
          }
          const float p0 = bt_ex2(fmaf(__uint_as_float(xr[i]), sl, -l4.x)), p1 = bt_ex2(fmaf(__uint_as_float(xr[i + 1]), sl, -l4.y));
          const float p2 = bt_ex2(fmaf(__uint_as_float(xr[i + 2]), sl, -l4.z)), p3 = bt_ex2(fmaf(__uint_as_float(xr[i + 3]), sl, -l4.w));
          const float s0 = p0 * (__uint_as_float(yr[i]) - d4.x) * kDsScale, s1 = p1 * (__uint_as_float(yr[i + 1]) - d4.y) * kDsScale;
          const float s2 = p2 * (__uint_as_float(yr[i + 2]) - d4.z) * kDsScale, s3 = p3 * (__uint_as_float(yr[i + 3]) - d4.w) * kDsScale;
          pkS[ch * 16 + (i >> 1)] = pack2_16(s0, s1, FP16 ? 1 : 0);
          pkS[ch * 16 + (i >> 1) + 1] = pack2_16(s2, s3, FP16 ? 1 : 0);
          if constexpr (MODE == 0) {
            pkP[ch * 16 + (i >> 1)] = pack2_16(p0 * kPScale, p1 * kPScale, FP16 ? 1 : 0);
            pkP[ch * 16 + (i >> 1) + 1] = pack2_16(p2 * kPScale, p3 * kPScale, FP16 ? 1 : 0);
          }
        }
      }
      // the previous tile's products have consumed the P / dS tiles (their MMAs ran behind this tile's X / Y while the loop above computed)
      if (it > 0) mbar_wait(o_done, (it - 1) & 1);
      tc_fence_after();
      __syncwarp();
      {
        uint32_t t16[16];
#pragma unroll
        for (int ch = 0; ch < Cf::NCH; ++ch) {
          const uint32_t col = uint32_t(hf * (Cf::CPT / 2) + ch * 16);  // 32 16-bit columns = 16 packed 32-bit TMEM columns
#pragma unroll
          for (int i = 0; i < 16; ++i) t16[i] = pkS[ch * 16 + i];
          tmem_st16(tdS + lane_base + col, t16);
          if constexpr (MODE == 0) {
#pragma unroll
            for (int i = 0; i < 16; ++i) t16[i] = pkP[ch * 16 + i];
            tmem_st16(tP + lane_base + col, t16);
          }
        }
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_ready);
    }
    // ---- accumulators -> 16-bit gradients (dS product: half 0; P product: half 1)
    mbar_wait(o_done, (n - 1) & 1);
    tc_fence_after();
    if (hf == 0 || MODE == 0) {
      const uint32_t tacc = (hf == 0 ? tAccS : tAccP) + lane_base;
      const float osc = hf == 0 ? p.out_scale_s : p.out_scale_p;
      uint16_t* op = (hf == 0 ? p.out_s + size_t(b) * p.bs_s + size_t(r0 + row) * p.ld_s : p.out_p + size_t(b) * p.bs_p + size_t(r0 + row) * p.ld_p) + h * p.d;
      uint32_t ro[Cf::ACC >= 80 ? 80 : 64];
      __syncwarp();
      tmem_ld16_at<0>(tacc, ro);
      tmem_ld16_at<16>(tacc + 16, ro);
      tmem_ld16_at<32>(tacc + 32, ro);
      if (p.dv > 48) tmem_ld16_at<48>(tacc + 48, ro);
      if constexpr (Cf::ACC >= 80) { if (p.dv > 64) tmem_ld16_at<64>(tacc + 64, ro); }
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < (Cf::ACC >= 80 ? 80 : 64); c += 8) {
        if (c < p.d) {
          uint4 v;
          v.x = pack2_16(__uint_as_float(ro[c]) * osc, __uint_as_float(ro[c + 1]) * osc, FP16 ? 1 : 0);
          v.y = pack2_16(__uint_as_float(ro[c + 2]) * osc, __uint_as_float(ro[c + 3]) * osc, FP16 ? 1 : 0);
          v.z = pack2_16(__uint_as_float(ro[c + 4]) * osc, __uint_as_float(ro[c + 5]) * osc, FP16 ? 1 : 0);
          v.w = pack2_16(__uint_as_float(ro[c + 6]) * osc, __uint_as_float(ro[c + 7]) * osc, FP16 ? 1 : 0);
          *reinterpret_cast<uint4*>(op + c) = v;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn bt_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* q = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(q);
  });
  return fn;
}
// [d, heads, tokens, batch] view of a [batch, tokens, ld] buffer whose head h occupies columns [h*d, (h+1)*d); box = 64 columns (zero-filled
// past d) x 128 tokens
const char* bt_map(CUtensorMap* tm, const void* ptr, int d, int heads, int ntok, int B, int ld, long bstride, int box_rows) {
  EncodeTiledFn fn = bt_encode_fn();
  if (!fn) return "attention_bwd: cuTensorMapEncodeTiled unavailable";
  cuuint64_t dims[4] = {cuuint64_t(d), cuuint64_t(heads), cuuint64_t(ntok), cuuint64_t(B)};
  cuuint64_t strides[3] = {cuuint64_t(d) * 2, cuuint64_t(ld) * 2, cuuint64_t(bstride) * 2};
  if (B == 1) strides[2] = cuuint64_t(ntok) * ld * 2;
  cuuint32_t box[4] = {64, 1, cuuint32_t(box_rows), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? nullptr : "attention_bwd: cuTensorMapEncodeTiled failed";
}

template <int MODE, bool FP16, int KC, int TN>
const char* bt_launch(const BwdTcParams& p, dim3 grid, cudaStream_t st) {
  static bool attr = false;
  if (!attr) {
    if (cudaFuncSetAttribute(attn_bwd_tc_kernel<MODE, FP16, KC, TN>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(BtCfg<KC, TN>::SMEM)) != cudaSuccess)
      return "attention_bwd: cudaFuncSetAttribute failed";
    attr = true;
  }
  if (launch_k(attn_bwd_tc_kernel<MODE, FP16, KC, TN>, grid, dim3(BT_THREADS), BtCfg<KC, TN>::SMEM, st, p) != cudaSuccess)
    return "attention_bwd: tcgen05 kernel launch failed";
  return nullptr;
}
template <int MODE>
const char* bt_dispatch(const BwdTcParams& p, dim3 grid, int fp16, cudaStream_t st) {
  if (p.d <= 64) return fp16 ? bt_launch<MODE, true, 1, 128>(p, grid, st) : bt_launch<MODE, false, 1, 128>(p, grid, st);
  return fp16 ? bt_launch<MODE, true, 2, 64>(p, grid, st) : bt_launch<MODE, false, 2, 64>(p, grid, st);
}

}  // namespace

bool attention_bwd_tc_supported(int d, int Nq, int Nk) {
  return (d == 40 || d == 80) && Nq % 128 == 0 && Nk % 128 == 0 && Nq >= 128 && Nk >= 128;
}

// dK / dV and dQ of one attention layer on the tcgen05 kernels.  L2 = log2-domain log-sum-exp, D = rowsum(dO * O), both [B, heads, Nq].
const char* attention_bwd_tc(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, const void* dout, int lddo, void* dq, int lddq,
                             void* dk, int lddk, void* dv, int lddv, int B, int heads, int d, int Nq, int Nk, long q_bs, long k_bs, long v_bs, long do_bs,
                             long dq_bs, long dk_bs, long dv_bs, float scale, const float* L2, const float* D, int fp16, cudaStream_t st) {
  if (!attention_bwd_tc_supported(d, Nq, Nk)) return "attention_bwd_tc: unsupported shape";
  BwdTcParams p;
  p.L2 = L2; p.D = D; p.Nq = Nq; p.d = d;
  p.ksteps = (d + 15) / 16;
  p.dv = (d + 15) / 16 * 16;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.out_scale_s = scale / kDsScale;
  p.out_scale_p = 1.0f / kPScale;
  const int TN = d <= 64 ? 128 : 64;  // rows of a streamed tile (BtCfg)
  CUtensorMap tq, tk, tv, tdo, tqs, tks, tvs, tdos;  // resident-role maps (128-row boxes) and streamed-role maps (TN-row boxes)
  if (const char* e = bt_map(&tq, q, d, heads, Nq, B, ldq, q_bs, 128)) return e;
  if (const char* e = bt_map(&tk, k, d, heads, Nk, B, ldk, k_bs, 128)) return e;
  if (const char* e = bt_map(&tv, v, d, heads, Nk, B, ldv, v_bs, 128)) return e;
  if (const char* e = bt_map(&tdo, dout, d, heads, Nq, B, lddo, do_bs, 128)) return e;
  if (const char* e = bt_map(&tqs, q, d, heads, Nq, B, ldq, q_bs, TN)) return e;
  if (const char* e = bt_map(&tks, k, d, heads, Nk, B, ldk, k_bs, TN)) return e;
  if (const char* e = bt_map(&tvs, v, d, heads, Nk, B, ldv, v_bs, TN)) return e;
  if (const char* e = bt_map(&tdos, dout, d, heads, Nq, B, lddo, do_bs, TN)) return e;
  {  // dK, dV
    p.tmR1 = tk; p.tmR2 = tv; p.tmT1 = tqs; p.tmT2 = tdos;
    p.out_s = static_cast<uint16_t*>(dk); p.ld_s = lddk; p.bs_s = dk_bs;
    p.out_p = static_cast<uint16_t*>(dv); p.ld_p = lddv; p.bs_p = dv_bs;
    p.n_stream = Nq / TN;
    const dim3 grid(Nk / 128, heads, B);
    if (const char* e = bt_dispatch<0>(p, grid, fp16, st)) return e;
  }
  {  // dQ
    p.tmR1 = tq; p.tmR2 = tdo; p.tmT1 = tks; p.tmT2 = tvs;
    p.out_s = static_cast<uint16_t*>(dq); p.ld_s = lddq; p.bs_s = dq_bs;
    p.out_p = nullptr; p.ld_p = 0; p.bs_p = 0;
    p.n_stream = Nk / TN;
    const dim3 grid(Nq / 128, heads, B);
    if (const char* e = bt_dispatch<1>(p, grid, fp16, st)) return e;
  }
  return cudaGetLastError() == cudaSuccess ? nullptr : "attention_bwd_tc launch failed";
}

}  // namespace madm
