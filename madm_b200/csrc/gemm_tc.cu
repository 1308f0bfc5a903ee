// tcgen05/TMEM implicit-GEMM for sm_100a: every dense contraction of the MADM feature-extraction path
// (ResBlock conv3x3/1x1, up/down-sample convs, attention q/k/v/out projections with the LoRA update already
// folded into the packed weight, GEGLU feed-forward, VAE convs, feature projections) runs through this kernel.
//
//   D[M,N] = act( alpha * sum_seg sum_tap A_seg(tap)[M,C] * W[N, k-slice]^T + bias[N] + rowbias[img(m),N] + residual[M,N] )
//
// A is never materialised as an im2col matrix: each 64-channel K chunk of each filter tap is one 4-D TMA box over the
// NHWC bf16 activation tensor, shifted by (dx,dy); out-of-bounds rows/columns are zero-filled by TMA, which is exactly
// the convolution's zero padding.  W tiles are 2-D TMA boxes over the packed K-major weight matrix.  Both land in
// 128B-swizzled shared memory and are consumed directly by tcgen05.mma (UMMA 128xBNx16, fp32 accumulators in TMEM).
// Persistent, warp-specialised: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (behind elect.sync), warps 2-9 = epilogue
// (tcgen05.ld -> per-warp smem transpose -> fused bias / time-embedding row bias / fp32 or 16-bit residual / SiLU / ReLU / GEGLU ->
// fp32 and/or 16-bit stores, optionally in space-to-depth layout, optionally with the consumer GroupNorm's column statistics).
// One CTA per SM (~200 KB of smem stages, two TMEM accumulator stages so the MMAs of tile i+1 overlap the epilogue of tile i);
// tiles >= 128 wide run as cta_group::2 pairs (256-row MMAs, each CTA stages half of W).  See DESIGN.md section 5.
#include "gemm_tc.h"
#include "cvt.cuh"
#include "launch.cuh"
#include "ptx.cuh"

#include <mutex>
#include <stdio.h>
#include <string.h>

namespace madm {

static constexpr int BM = 128;
static constexpr int BK = 64;
static constexpr int kEpiWarps = 8;                 // two warps per TMEM lane quarter, interleaved over 32-column chunks
static constexpr int kThreads = 64 + 32 * kEpiWarps;
static constexpr int A_STAGE_BYTES = BM * BK * 2;  // 16 KB
static constexpr int STG_LD = 36;                   // floats per staging row (32 + 4 pad: conflict-free 128-bit access)
// Per-epilogue-warp staging: the transpose buffer of the coalesced epilogue (32 x 36 floats) or, on the TMA-store path, EPI_NBUF
// swizzled 32 x 32 tiles (4 KB each, 1024-byte aligned: the TMA swizzle pattern is a function of the shared-memory address bits).
#ifndef EPI_NBUF
#define EPI_NBUF 2
#endif
static constexpr int TMA_TILE_BYTES = 4096;
static constexpr int STG_WARP_BYTES = EPI_NBUF * TMA_TILE_BYTES > 5120 ? EPI_NBUF * TMA_TILE_BYTES : 5120;
static_assert(STG_WARP_BYTES >= 32 * STG_LD * 4 && STG_WARP_BYTES % 1024 == 0, "staging");
enum { TMA_EPI_NONE = 0, TMA_EPI_F32 = 1, TMA_EPI_RED = 2, TMA_EPI_H16 = 3, TMA_EPI_RES_H16 = 4 };
#ifndef EPI_BATCH
#define EPI_BATCH 4
#endif

struct GemmParams {
  CUtensorMap tmA[2];
  CUtensorMap tmB;
  CUtensorMap tmR;   // TMA_EPI_RES_H16: the out-of-place fp32 residual (box 32 x 32, 128B swizzle), loaded per chunk into the warp's staging
  CUtensorMap tmO;   // output tensor map of the TMA-store epilogue (box 32 columns x 32 rows; fp32 with 128B swizzle or 16-bit with 64B swizzle)
  int tma_epi;       // TMA_EPI_*: 0 = coalesced-store epilogue, else the epilogue hands 32x32 tiles to cp(.reduce).async.bulk.tensor
  int nseg;
  int kchunks[2];
  int cpt[2];
  int8_t dx[2][9];
  int8_t dy[2][9];
  int boff[2][9];
  int M, N;
  int W, pix;  // output grid width and pixels per image
  int box_w, box_h, box_b;
  const float* bias;
  const float* rowbias;
  int rows_per_img;
  int ld_rowbias;
  const float* residual;
  int ldr;
  int res16;  // the residual is a 16-bit tensor (operand dtype) instead of fp32
  float* out_f32;
  int ldo32;
  __nv_bfloat16* out_bf16;
  int ldo16;
  int act;
  float alpha;
  int vec_ok;
  int n_tiles;
  int fp16;
  int num_tiles;
  int s2d_H, s2d_W;  // if s2d_W > 0 the 16-bit output is written in space-to-depth layout [4 phases][B][H/2][W/2][N] of an HxW image grid
  int s2d_B;
  int splits;        // split-K factor: tile t covers K range (t % splits) of output tile (t / splits) and writes raw partials
  long split_stride; // elements between the partial outputs of consecutive splits (out_f32 + split * split_stride)
  float* colstats;   // [ceil(M/32)][N][2] per-column (sum, sum of squares) of the stored outputs per 32-row block, or null
  int stat_rows;     // always 32 (one block per epilogue warp)
};

// MT = M sub-tiles (128 rows each) per CTA tile.  MT = 2 loads one W box per K chunk for two A boxes (tile 256 x BN): the
// L2->SM operand traffic per FLOP drops from (128+BN) to (256+BN)/2 bytes-equivalents, which is what bounds the BN = 128
// layers (measured 12.7 TB/s of L2->SM reads at 42 % tensor-pipe activity on the VAE 512^2 convs).
enum { EPI_PLAIN = 0, EPI_STATS = 1, EPI_S2D = 2, EPI_TMA = 4 };  // epilogue variants (bit mask; EPI_TMA never with EPI_S2D) compiled as separate kernels

// PAIR: the CTA is one half of a cta_group::2 pair (cluster of 2): the pair's tile is 2*MT*128 rows x BN, each CTA stages its own
// A rows and HALF of the W tile (BN/2 rows), and the leader's tcgen05.mma.cta_group::2 (M = 256) reads both halves.  Per CTA the
// TMA fill per tensor-clock drops from (128*MT + BN) to (128*MT + BN/2) rows, which is what bounds these tiles.
template <int BN, int MT, bool PAIR = false>
struct Cfg {
  static constexpr int A_BYTES = MT * A_STAGE_BYTES;
  static constexpr int B_ROWS = PAIR ? BN / 2 : BN;  // W rows staged by this CTA
  static constexpr int B_STAGE_BYTES = B_ROWS * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_STAGE_BYTES;
  static constexpr int EPI_BYTES = kEpiWarps * STG_WARP_BYTES;  // per-epilogue-warp transpose staging
  static constexpr int BUDGET = 227 * 1024 - 1024 /*align*/ - 256 /*barriers*/ - EPI_BYTES;
  static constexpr int STAGES = (BUDGET / STAGE_BYTES) > 8 ? 8 : (BUDGET / STAGE_BYTES);
  static constexpr int ACC_STRIDE = BN <= 16 ? 16 : (BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256)));
  static constexpr int NACC = 2;  // accumulator stages: the MMAs of tile i+1 overlap the epilogue of tile i
  static constexpr int TMEM_COLS = NACC * MT * ACC_STRIDE < 32 ? 32 : NACC * MT * ACC_STRIDE;
  static constexpr size_t SMEM = size_t(STAGES) * STAGE_BYTES + EPI_BYTES + 1024 + 256;
  static_assert(TMEM_COLS <= 512, "two accumulator stages must fit the 512 TMEM columns");
};

__device__ __forceinline__ float silu_f(float v) { return v / (1.0f + __expf(-v)); }
// exact (erf) GELU with erf from Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7, i.e. fp32-exact for a 16-bit output):
// 5 FMAs + one MUFU.RCP + one MUFU.EX2 instead of libdevice erff's branchy ~25-instruction polynomial.
__device__ __forceinline__ float gelu_erf_f(float v) {
  const float x = fabsf(v) * 0.70710678118654752f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, x, 1.0f)));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  poly *= t;
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-x * x * 1.4426950408889634f));
  const float erf_abs = fmaf(-poly, e, 1.0f);
  return 0.5f * v * (1.0f + copysignf(erf_abs, v));
}
__device__ __forceinline__ float4 ld_shared_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void st_shared_f4(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Fused epilogue of one 32x32 fp32 block that sits transposed in this warp's staging buffer: lane = (row sub-index, 4
// columns), 8 iterations of 4 rows -> every global access is a full 128-byte row segment.  `bb` already holds
// bias (+ the per-image time-embedding row bias).  Compile-time flags keep the loop free of uniform branches.
template <bool RES, bool O32, int O16, bool ST = false>
__device__ __forceinline__ void epi_block(uint32_t stg, int lane, int row0, int M, float alpha, float4 bb, int act, int fp16,
                                          const float4 (&resv)[8], float* o32, int ldo32, uint16_t* o16, int ldo16,
                                          bool do_stats, float (&cs)[8], int s2d_H = 0, int s2d_W = 0, int s2d_B = 0, int N = 0) {
  const int rsub = lane >> 3;
  const int cc = (lane & 7) * 4;
  // All eight shared-memory reads first, then the arithmetic and the stores: ld_shared_f4 is an `asm volatile` with a memory clobber, so
  // in a single loop the compiler must keep every global store between two of them and the in-order issue serialises
  // {ld.shared -> ~12 dependent ALU ops -> st.global} eight times per chunk (measured ~250 clk per iteration, profiles/r01_epilogue_store_bound.txt).
  // Hoisted, the eight loads pipeline and the eight rows' arithmetic overlaps; the registers are those of the (now dead) TMEM fragment.
  // Batches of EB rows.  Measured (tools/bench_epilogue.py, B200): with 16-bit / fp32 outputs and no residual, hoisting takes 15-18 % off
  // output-bound launches (QKV 48.8 -> 41.3 us, 32768x320x320 26.0 -> 21.4 us); with a residual the eight prefetched residual rows already fill the
  // register budget and the hoisted variant was 20 % SLOWER (30.0 -> 35.9 us), so those keep one row at a time.
  constexpr int EB = (RES || ST) ? 1 : EPI_BATCH;  // (the statistics variant carries 8 more live accumulators: hoisting spills there)
#pragma unroll
  for (int it0 = 0; it0 < 8; it0 += EB) {
  float4 vv[EB];
#pragma unroll
  for (int u = 0; u < EB; ++u) vv[u] = ld_shared_f4(stg + uint32_t(((it0 + u) * 4 + rsub) * STG_LD + cc) * 4);
#pragma unroll
  for (int u = 0; u < EB; ++u) {
    const int it = it0 + u;
    const int r = it * 4 + rsub;
    float4 v = vv[u];
    v.x = fmaf(v.x, alpha, bb.x); v.y = fmaf(v.y, alpha, bb.y); v.z = fmaf(v.z, alpha, bb.z); v.w = fmaf(v.w, alpha, bb.w);
    if constexpr (RES) { v.x += resv[it].x; v.y += resv[it].y; v.z += resv[it].z; v.w += resv[it].w; }
    if (act == ACT_SILU) { v.x = silu_f(v.x); v.y = silu_f(v.y); v.z = silu_f(v.z); v.w = silu_f(v.w); }
    else if (act == ACT_RELU) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
    if (row0 + r < M) {
      if constexpr (O32) *reinterpret_cast<float4*>(o32 + size_t(r) * ldo32) = v;
      if constexpr (O16 == 1) *reinterpret_cast<uint2*>(o16 + size_t(r) * ldo16) = pack4_16(v.x, v.y, v.z, v.w, fp16);
      if constexpr (O16 == 2) {  // the consumer is a stride-2 conv: write its space-to-depth operand [4][B][H/2][W/2][N] directly
        // H and W are powers of two (checked on the host): s2d_H / s2d_W carry log2(H) / log2(W)
        const int m = row0 + r;
        const int x = m & ((1 << s2d_W) - 1), y = (m >> s2d_W) & ((1 << s2d_H) - 1), bimg = m >> (s2d_W + s2d_H);
        const int ph = (y & 1) * 2 + (x & 1);
        const long off = ((((long(ph) * s2d_B + bimg) << (s2d_H - 1)) + (y >> 1)) << (s2d_W - 1)) + (x >> 1);
        const long offN = off * long(N);
        *reinterpret_cast<uint2*>(o16 + offN) = pack4_16(v.x, v.y, v.z, v.w, fp16);
      }
      if (do_stats) {  // GroupNorm statistics of the consumer, fused here: per-column sum / sum of squares of what is stored
        cs[0] += v.x; cs[1] += v.y; cs[2] += v.z; cs[3] += v.w;
        cs[4] = fmaf(v.x, v.x, cs[4]); cs[5] = fmaf(v.y, v.y, cs[5]); cs[6] = fmaf(v.z, v.z, cs[6]); cs[7] = fmaf(v.w, v.w, cs[7]);
      }
    }
  }
  }  // batches
  if (do_stats) {  // fold the 4 row sub-groups of this warp: lanes 0..7 end up with the totals of their 4 columns over 32 rows
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      cs[i] += __shfl_xor_sync(0xffffffffu, cs[i], 8);
      cs[i] += __shfl_xor_sync(0xffffffffu, cs[i], 16);
    }
  }
}

// Column (sum, sum of squares) of a 32x32 block held one row per lane: recursive halving -- at step `off` a lane keeps the half of its
// columns selected by its own bit and receives the partner's partial sums of that half -- leaves lane l with the totals of column l
// after 31 shuffles per quantity (fixed order: bit-reproducible, no atomics).
__device__ __forceinline__ void colstats_rows32(const float (&v)[32], int lane, float& sum, float& sumsq) {
  float a[16], q[16];
  {
    const bool up = (lane & 16) != 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float keep = up ? v[k + 16] : v[k], send = up ? v[k] : v[k + 16];
      const float r = __shfl_xor_sync(0xffffffffu, send, 16);
      a[k] = keep + r;
      q[k] = fmaf(keep, keep, r * r);
    }
  }
#pragma unroll
  for (int off = 8; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int k = 0; k < off; ++k) {
      const float keep = up ? a[k + off] : a[k], send = up ? a[k] : a[k + off];
      a[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      const float keepq = up ? q[k + off] : q[k], sendq = up ? q[k] : q[k + off];
      q[k] = keepq + __shfl_xor_sync(0xffffffffu, sendq, off);
    }
  }
  sum = a[0];
  sumsq = q[0];
}

// TMA-store epilogue of one 32x32 block, in the row-per-thread layout tcgen05.ld delivers (thread = row, v[j] = column j, bias and
// activation already applied): the tile is written to a swizzled staging buffer (conflict-free: the 8 lanes of a quarter-warp cover all
// 32 banks) and leaves the SM as ONE bulk tensor store -- or, for `hs += GEMM` (in-place fp32 residual), one bulk reduce-add executed at
// the L2, so the residual never enters the SM.  No ld.shared, no per-thread global loads / stores: the serial chain per chunk is
// tcgen05.ld -> FMAs -> st.shared -> fence -> issue, and the next chunk starts while the TMA engine drains this one.
// `buf` toggles between the EPI_NBUF staging tiles; the elected lane (elect.sync is deterministic for a full mask) owns the bulk groups.
template <bool H16, bool WAIT = true>
__device__ __forceinline__ void tma_epi_tile(const float (&v)[32], uint32_t stg, int& buf, int lane, const CUtensorMap* tm, int mode, int col, int row,
                                             int fp16) {
  const uint32_t sb = stg + uint32_t(buf) * TMA_TILE_BYTES;
  if constexpr (WAIT) { if (elect_one()) bulk_wait_read<EPI_NBUF - 1>(); }  // the store that last used this buffer has read it
  __syncwarp();
  if constexpr (H16) {  // 32 rows x 64 B, SWIZZLE_64B: 16-byte unit index ^= address bits [7,9) = (row >> 1) & 3
    const uint32_t rowp = sb + uint32_t(lane) * 64u;
    const uint32_t sw = uint32_t(lane >> 1) & 3u;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t a = pack2_16(v[8 * u + 0], v[8 * u + 1], fp16), b = pack2_16(v[8 * u + 2], v[8 * u + 3], fp16);
      const uint32_t c = pack2_16(v[8 * u + 4], v[8 * u + 5], fp16), d = pack2_16(v[8 * u + 6], v[8 * u + 7], fp16);
      asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(rowp + ((uint32_t(u) ^ sw) << 4)), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
    }
  } else {  // 32 rows x 128 B, SWIZZLE_128B: 16-byte unit index ^= address bits [7,10) = row & 7
    const uint32_t rowp = sb + uint32_t(lane) * 128u;
    const uint32_t sw = uint32_t(lane) & 7u;
#pragma unroll
    for (int u = 0; u < 8; ++u) st_shared_f4(rowp + ((uint32_t(u) ^ sw) << 4), v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]);
  }
  fence_proxy_async();  // this thread's generic-proxy writes -> visible to the async proxy (TMA)
  __syncwarp();
  if (elect_one()) {
    if (mode == TMA_EPI_RED) tma_reduce_add_2d(tm, sb, col, row);
    else tma_store_2d(tm, sb, col, row);
    bulk_commit();
  }
  buf = (buf + 1 == EPI_NBUF) ? 0 : buf + 1;
}

// Persistent, warp-specialised kernel: one CTA per SM walks the tile list (tile = blockIdx.x + i*gridDim.x, N fastest).
//   warp 0      TMA producer: fills the STAGES-deep smem ring (A box + W box per 64-wide K chunk)
//   warp 1      TMEM allocator + single-thread tcgen05.mma issuer; two accumulator stages in TMEM so the MMAs of tile
//               i+1 overlap the epilogue of tile i
//   warps 2..5  epilogue: tcgen05.ld (thread = row) -> per-warp smem transpose -> coalesced fused epilogue
//               (bias / time-embedding row bias / fp32 residual / SiLU / ReLU / GEGLU) -> fp32 and/or 16-bit stores
template <int BN, int MT, int EPI, bool PAIR>
// Registers: 10 warps are allocated as 12 (granularity of 4 warps), so 65536 / 384 -> 168 registers per thread is the ceiling
// for this block size (measured: a 186-register build reports maxThreadsPerBlock = 256 and fails to launch).
__global__ void __launch_bounds__(kThreads, 1) gemm_tc_kernel(const __grid_constant__ GemmParams p) {
  using C = Cfg<BN, MT, PAIR>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = smem_base;
  const uint32_t sB = smem_base + C::STAGES * C::A_BYTES;
  const uint32_t sEpi = sB + C::STAGES * C::B_STAGE_BYTES;
  const uint32_t sBar = sEpi + C::EPI_BYTES;  // full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2], tmem_addr
  auto full_bar = [&](int s) { return sBar + 8u * s; };
  auto empty_bar = [&](int s) { return sBar + 8u * (C::STAGES + s); };
  auto tmem_full_bar = [&](int a) { return sBar + 8u * (2 * C::STAGES + a); };
  auto tmem_empty_bar = [&](int a) { return sBar + 8u * (2 * C::STAGES + 2 + a); };
  const uint32_t tmem_slot = sBar + 8u * (2 * C::STAGES + 4);
  auto res_bar = [&](int w) { return sBar + 8u * (2 * C::STAGES + 5 + w); };  // one per epilogue warp (residual tile landed)
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_chunks = p.kchunks[0] + (p.nseg > 1 ? p.kchunks[1] : 0);
  // persistent tile walk: a CTA (or a CTA pair) starts at its index and strides by the number of CTAs (pairs)
  const int rank = PAIR ? int(cluster_ctarank()) : 0;
  const int walker = PAIR ? int(blockIdx.x >> 1) : int(blockIdx.x);
  const int walkers = PAIR ? int(gridDim.x >> 1) : int(gridDim.x);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tmA[0]);
    if (p.nseg > 1) prefetch_tmap(&p.tmA[1]);
    prefetch_tmap(&p.tmB);
    if (p.tma_epi) prefetch_tmap(&p.tmO);
    if (p.tma_epi == TMA_EPI_RES_H16) prefetch_tmap(&p.tmR);
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tmem_full_bar(a), 1);
      mbar_init(tmem_empty_bar(a), PAIR ? 2 * kEpiWarps : kEpiWarps);  // one arrival per epilogue warp (of both CTAs of a pair)
    }
    for (int w = 0; w < kEpiWarps; ++w) mbar_init(res_bar(w), 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (PAIR) { tmem_alloc_pair(tmem_slot, C::TMEM_COLS); tmem_relinquish_pair(); }
    else { tmem_alloc(tmem_slot, C::TMEM_COLS); tmem_relinquish(); }
  }
  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all();  // the peer's barriers must be initialised before remote arrivals / TMA bytes reach them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // programmatic dependent launch: everything above (barrier init, TMEM allocation, tensor-map prefetch) overlapped the tail of the
  // previous kernel; nothing below may touch global memory before that kernel has completed
  pdl_trigger();
  pdl_wait();

  if (warp == 0) {
    // ===================== TMA producer =====================
    // elect_one(), not lane == 0: behind elect.sync the compiler knows a single lane is active and feeds the uniform-datapath
    // instructions (UTMALDG / UTCHMMA / UTCBAR) directly instead of wrapping each one in a per-lane "waterfall" loop
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
#ifdef GEMM_INSTR
      long long pw = 0, pt0 = clock64();
#define GI(acc, ...) { const long long t0_ = clock64(); __VA_ARGS__; acc += clock64() - t0_; }
#else
#define GI(acc, ...) __VA_ARGS__
#endif
      for (int t = walker; t < p.num_tiles; t += walkers) {
        const int mn = t / p.splits, sp = t - mn * p.splits;
        const int tile_n = mn % p.n_tiles;
        const int m0 = ((mn / p.n_tiles) * (PAIR ? 2 : 1) + rank) * (BM * MT);
        const int n0 = tile_n * BN + rank * C::B_ROWS;
        const int kc0 = (total_chunks * sp) / p.splits, kc1 = (total_chunks * (sp + 1)) / p.splits;
        int x0[MT], y0[MT], b0[MT];
#pragma unroll
        for (int s = 0; s < MT; ++s) {
          const int ms = m0 + s * BM;
          if (p.pix >= BM) {
            b0[s] = ms / p.pix;
            const int rem = ms - b0[s] * p.pix;
            y0[s] = rem / p.W;
            x0[s] = rem - y0[s] * p.W;
          } else {
            b0[s] = ms / p.pix;
            y0[s] = 0;
            x0[s] = 0;
          }
        }
        for (int kc = kc0; kc < kc1; ++kc) {
          const int seg = (kc < p.kchunks[0]) ? 0 : 1;
          const int lk = seg ? kc - p.kchunks[0] : kc;
          const int tap = lk / p.cpt[seg];
          const int cc = lk - tap * p.cpt[seg];
          GI(pw, mbar_wait(empty_bar(stage), phase ^ 1u));
          if constexpr (PAIR) {  // both CTAs' bytes are counted on the leader's barrier; only the leader arms it
            if (rank == 0) mbar_arrive_expect_tx(full_bar(stage), 2 * C::STAGE_BYTES);
#pragma unroll
            for (int s = 0; s < MT; ++s)
              tma_load_4d_pair(sA + stage * C::A_BYTES + s * A_STAGE_BYTES, &p.tmA[seg], full_bar(stage), cc * BK, x0[s] + p.dx[seg][tap],
                               y0[s] + p.dy[seg][tap], b0[s] + p.boff[seg][tap]);
            tma_load_2d_pair(sB + stage * C::B_STAGE_BYTES, &p.tmB, full_bar(stage), kc * BK, n0);
          } else {
            mbar_arrive_expect_tx(full_bar(stage), C::STAGE_BYTES);
#pragma unroll
            for (int s = 0; s < MT; ++s)
              tma_load_4d(sA + stage * C::A_BYTES + s * A_STAGE_BYTES, &p.tmA[seg], full_bar(stage), cc * BK, x0[s] + p.dx[seg][tap],
                          y0[s] + p.dy[seg][tap], b0[s] + p.boff[seg][tap]);
            tma_load_2d(sB + stage * C::B_STAGE_BYTES, &p.tmB, full_bar(stage), kc * BK, n0);
          }
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
#ifdef GEMM_INSTR
      if (blockIdx.x == 5) printf("producer: total %lld clk, waiting for empty slots %lld\n", clock64() - pt0, pw);
#endif
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread; in a pair only the leader CTA issues) =====================
    if (rank == 0 && elect_one()) {
      const uint32_t idesc = make_idesc_16(PAIR ? 2 * BM : BM, BN, p.fp16);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
#ifdef GEMM_INSTR
      long long w_full = 0, w_acc = 0, t_issue = 0, t_commit = 0, mt0 = clock64(), n_mma = 0, n_chunks = 0, n_tiles_done = 0;
#endif
      for (int t = walker; t < p.num_tiles; t += walkers) {
        GI(w_acc, mbar_wait(tmem_empty_bar(acc), acc_phase ^ 1u));  // epilogue has drained this accumulator stage
        tc_fence_after();
        const uint32_t tacc = tmem_base + uint32_t(acc * MT * C::ACC_STRIDE);
        const int sp = t % p.splits;
        const int kc0 = (total_chunks * sp) / p.splits, kc1 = (total_chunks * (sp + 1)) / p.splits;
        for (int kc = kc0; kc < kc1; ++kc) {
          GI(w_full, mbar_wait(full_bar(stage), phase));
          tc_fence_after();
          const uint64_t bdesc = make_smem_desc_sw128(sB + stage * C::B_STAGE_BYTES);
#ifdef GEMM_INSTR
          const long long ti0 = clock64();
          n_mma += MT * (BK / 16); ++n_chunks;
#endif
#pragma unroll
          for (int s = 0; s < MT; ++s) {
            const uint64_t adesc = make_smem_desc_sw128(sA + stage * C::A_BYTES + s * A_STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              // advance 32 B (16 elements) along K inside the 128 B swizzle row: +2 in the (addr >> 4) field
              if constexpr (PAIR)
                umma_f16_ss_pair(tacc + uint32_t(s * C::ACC_STRIDE), adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), idesc,
                                 (kc > kc0 || k > 0) ? 1u : 0u);
              else
                umma_bf16_ss(tacc + uint32_t(s * C::ACC_STRIDE), adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), idesc,
                             (kc > kc0 || k > 0) ? 1u : 0u);
            }
          }
#ifdef GEMM_INSTR
          t_issue += clock64() - ti0;
#endif
          // frees the smem slot (in both CTAs of a pair) when these MMAs retire
          if constexpr (PAIR) { GI(t_commit, umma_commit_pair(empty_bar(stage))); }
          else { GI(t_commit, umma_commit(empty_bar(stage))); }
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if constexpr (PAIR) umma_commit_pair(tmem_full_bar(acc));  // accumulator complete -> epilogue (of both CTAs)
        else umma_commit(tmem_full_bar(acc));
        if (++acc == C::NACC) {
          acc = 0;
          acc_phase ^= 1u;
        }
#ifdef GEMM_INSTR
        ++n_tiles_done;
#endif
      }
#ifdef GEMM_INSTR
      if (blockIdx.x == 5)
        printf("mma: total %lld clk, %lld tiles %lld chunks %lld mmas (BN=%d MT=%d) | wait full %lld wait acc %lld issue %lld commit %lld | ideal tensor clk %lld\n",
               clock64() - mt0, n_tiles_done, n_chunks, n_mma, BN, MT, w_full, w_acc, t_issue, t_commit, n_mma * BN / 2);
#endif
    }
  } else {
    // ===================== epilogue (warps 2..9) =====================
    const int q = warp & 3;                 // TMEM lane quarter this warp may access
    const int par = (warp - 2) >> 2;        // which half of the 32-column chunks this warp takes
    const uint32_t stg = sEpi + uint32_t(warp - 2) * STG_WARP_BYTES;
    // kernel parameters -> registers once (the asm volatile memory clobbers would otherwise force constant re-loads)
    const float alpha = p.alpha;
    const int fp16 = p.fp16, act = p.act, M = p.M, N = p.N, vec_ok = p.vec_ok, n_tiles = p.n_tiles;
    const float* const bias = p.bias;
    const float* const rowbias = p.rowbias;
    const int rows_per_img = p.rows_per_img, ld_rowbias = p.ld_rowbias;
    const float* const residual = p.residual;
    uint16_t* const out16 = reinterpret_cast<uint16_t*>(p.out_bf16);
    const int ldr = p.ldr, ldo32 = p.ldo32, ldo16 = p.ldo16;
    const int mode = (residual ? 4 : 0) | (p.out_f32 ? 2 : 0) | (out16 ? 1 : 0);
    constexpr bool STATS = (EPI & EPI_STATS) != 0;
    constexpr bool S2D = (EPI & EPI_S2D) != 0;  // separate instantiation: its extra live values would otherwise spill in every variant
    constexpr bool do_stats = STATS;  // compile-time: the statistics-free variant keeps the tighter rolled chunk loop
    // TMA-store epilogue (plain variant only: statistics / space-to-depth outputs keep the coalesced path)
    constexpr bool TMA = (EPI & EPI_TMA) != 0;  // separate instantiation: neither path pays for the other's live registers
    const int tma_epi = TMA ? p.tma_epi : 0;
    int tbuf = 0;
    uint32_t res_phase = 0;
    const uint32_t rbar = res_bar(warp - 2);
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t r[32];
#ifdef GEMM_INSTR
    long long e_wait = 0, e_work = 0, e_tiles = 0, e_ldtm = 0, e_tr = 0, e_blk = 0, e_chunks = 0;
    const long long e_t0 = clock64();
#endif
    float* const out32_base = p.out_f32;
    const int splits = p.splits;
    const long split_stride = p.split_stride;
    for (int t = walker; t < p.num_tiles; t += walkers) {
      const int mn = t / splits;
      const int tile_n = mn % n_tiles;
      const int m0 = ((mn / n_tiles) * (PAIR ? 2 : 1) + rank) * (BM * MT);
      const int n0 = tile_n * BN;
      float* const out32 = out32_base ? out32_base + long(t - mn * splits) * split_stride : nullptr;
#ifdef GEMM_INSTR
      const long long ei0 = clock64();
#endif
      mbar_wait(tmem_full_bar(acc), acc_phase);
      tc_fence_after();
#ifdef GEMM_INSTR
      const long long ei1 = clock64();
      e_wait += ei1 - ei0;
#endif
#pragma unroll 1
      for (int sub = 0; sub < MT; ++sub) {  // M sub-tiles of this CTA tile
      const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t((acc * MT + sub) * C::ACC_STRIDE);
      const int row0 = m0 + sub * BM + q * 32;  // first row of this warp's 32-row block

      if constexpr (BN < 32) {
        // narrow tile (latent head, N = 4 of 16): one row per thread, scalar stores
        if (par == 0) {
          const int m = row0 + lane;
          __syncwarp();
          tmem_ld16(taddr, r);
          tmem_ld_wait();
          if (m < M) {
            const float* rb = rowbias ? rowbias + size_t(m / rows_per_img) * ld_rowbias : nullptr;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int n = n0 + j;
              if (n >= N) continue;
              float v = __uint_as_float(r[j]) * alpha;
              if (bias) v += __ldg(bias + n);
              if (rb) v += __ldg(rb + n);
              if (residual) v += residual[size_t(m) * ldr + n];
              if (act == ACT_SILU) v = silu_f(v);
              else if (act == ACT_RELU) v = fmaxf(v, 0.0f);
              if (out32) out32[size_t(m) * ldo32 + n] = v;
              if (out16) out16[size_t(m) * ldo16 + n] = cvt_16(v, fp16);
            }
          }
        }
      } else if (act == ACT_GEGLU) {
        // weight rows are tile-interleaved: columns [0,64) of this tile = value, [64,128) = gate, for output cols [64*tile_n, +64)
        if constexpr (BN == 128) {
          uint32_t g[32];
          const int on0 = tile_n * 64;
          const int half = par;
          __syncwarp();
          tmem_ld32(taddr + half * 32, r);
          tmem_ld32(taddr + 64 + half * 32, g);
          tmem_ld_wait();
          if constexpr (TMA) {  // value * gelu(gate) in the row-per-thread layout -> one 16-bit tile store
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 bh = make_float4(0.f, 0.f, 0.f, 0.f), bg = bh;
              if (bias) {
                bh = __ldg(reinterpret_cast<const float4*>(bias + n0 + half * 32 + j));
                bg = __ldg(reinterpret_cast<const float4*>(bias + n0 + 64 + half * 32 + j));
              }
              v[j + 0] = fmaf(__uint_as_float(r[j + 0]), alpha, bh.x) * gelu_erf_f(fmaf(__uint_as_float(g[j + 0]), alpha, bg.x));
              v[j + 1] = fmaf(__uint_as_float(r[j + 1]), alpha, bh.y) * gelu_erf_f(fmaf(__uint_as_float(g[j + 1]), alpha, bg.y));
              v[j + 2] = fmaf(__uint_as_float(r[j + 2]), alpha, bh.z) * gelu_erf_f(fmaf(__uint_as_float(g[j + 2]), alpha, bg.z));
              v[j + 3] = fmaf(__uint_as_float(r[j + 3]), alpha, bh.w) * gelu_erf_f(fmaf(__uint_as_float(g[j + 3]), alpha, bg.w));
            }
            if (row0 < M) tma_epi_tile<true>(v, stg, tbuf, lane, &p.tmO, TMA_EPI_H16, on0 + half * 32, row0, fp16);
          } else {
          // value * gelu(gate) in the row-per-thread layout, then transpose through smem for coalesced 16-bit stores
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float v[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float h = __uint_as_float(r[j + e]) * alpha;
              float gt = __uint_as_float(g[j + e]) * alpha;
              if (bias) {
                h += __ldg(bias + n0 + half * 32 + j + e);
                gt += __ldg(bias + n0 + 64 + half * 32 + j + e);
              }
              v[e] = h * gelu_erf_f(gt);
            }
            st_shared_f4(stg + uint32_t(lane * STG_LD + j) * 4, v[0], v[1], v[2], v[3]);
          }
          __syncwarp();
          const int cc = (lane & 7) * 4;
          float nostats[8];
          const float4 nores[8] = {};
          epi_block<false, false, 1>(stg, lane, row0, M, 1.0f, make_float4(0.f, 0.f, 0.f, 0.f), ACT_NONE, fp16, nores, nullptr, 0,
                                     out16 + size_t(row0) * ldo16 + on0 + half * 32 + cc, ldo16, false, nostats);
          }  // !TMA
        }
      } else {
        float cs1[8];  // column statistics of the current chunk (STATS variant only)
#pragma unroll 1
        for (int c = par * 32; c < BN; c += 64) {
          if constexpr (TMA) {  // (N % 32 == 0 on this path: a chunk is either inside the matrix or entirely outside)
            if (n0 + c >= N) break;
            __syncwarp();
            const int n = n0 + c;
            if (tma_epi == TMA_EPI_RES_H16 && row0 < M) {  // the residual tile of this chunk: TMA load into staging tile 0 (its latency overlaps the TMEM load)
              if (elect_one()) {
                bulk_wait_read<0>();  // (also frees staging tile 1 of the previous chunk's store)
                mbar_arrive_expect_tx(rbar, TMA_TILE_BYTES);
                tma_load_2d(stg, &p.tmR, rbar, n, row0);
              }
              __syncwarp();
            }
            tmem_ld32(taddr + c, r);
            const float* rb = rowbias ? rowbias + size_t(min(row0, M - 1) / rows_per_img) * ld_rowbias + n : nullptr;
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {  // bias (+ time-embedding row bias): uniform addresses, issued under the TMEM load
              float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
              if (bias) b4 = __ldg(reinterpret_cast<const float4*>(bias + n + j));
              if (rb) {
                const float4 t4 = __ldg(reinterpret_cast<const float4*>(rb + j));
                b4.x += t4.x; b4.y += t4.y; b4.z += t4.z; b4.w += t4.w;
              }
              v[j] = b4.x; v[j + 1] = b4.y; v[j + 2] = b4.z; v[j + 3] = b4.w;
            }
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              float x = fmaf(__uint_as_float(r[j]), alpha, v[j]);
              if (act == ACT_SILU) x = silu_f(x);
              else if (act == ACT_RELU) x = fmaxf(x, 0.f);
              v[j] = x;
            }
            if (tma_epi == TMA_EPI_RES_H16) {  // v += residual (swizzled staging tile 0, rows past M zero-filled by TMA) -> 16-bit tile in staging tile 1
              if (row0 < M) {
                mbar_wait(rbar, res_phase);
                res_phase ^= 1u;
                const uint32_t rowp = stg + uint32_t(lane) * 128u;
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                  const float4 r4 = ld_shared_f4(rowp + ((uint32_t(u) ^ (uint32_t(lane) & 7u)) << 4));
                  v[4 * u] += r4.x; v[4 * u + 1] += r4.y; v[4 * u + 2] += r4.z; v[4 * u + 3] += r4.w;
                }
                int one = 1;  // staging tile 1
                tma_epi_tile<true, false>(v, stg, one, lane, &p.tmO, TMA_EPI_H16, n, row0, fp16);
              }
              continue;
            }
            if (row0 < M) {
              if (tma_epi == TMA_EPI_H16) tma_epi_tile<true>(v, stg, tbuf, lane, &p.tmO, tma_epi, n, row0, fp16);
              else tma_epi_tile<false>(v, stg, tbuf, lane, &p.tmO, tma_epi, n, row0, fp16);
              if constexpr (STATS) {  // GroupNorm statistics of the consumer: (sum, sumsq) of the fp32 values per column over this warp's 32 rows
                if (row0 + lane >= M) {
#pragma unroll
                  for (int j = 0; j < 32; ++j) v[j] = 0.f;
                }
                float cs, cq;
                colstats_rows32(v, lane, cs, cq);
                *reinterpret_cast<float2*>(p.colstats + (size_t(row0 >> 5) * N + n + lane) * 2) = make_float2(cs, cq);
              }
            }
          } else {
          if constexpr (STATS) {
#pragma unroll
            for (int i = 0; i < 8; ++i) cs1[i] = 0.f;
          }
          // fp32 residual of this chunk: issued before the TMEM load / transpose so its HBM / L2 latency overlaps them
          // (in-place residual == out_f32 stays safe: these are this chunk's own elements, loaded before its stores)
          float4 resv[8];
          if (residual && vec_ok && n0 + c + 32 <= N) {
            if (p.res16) {  // 16-bit residual stream (8 bytes per lane and row)
              const uint16_t* resp = reinterpret_cast<const uint16_t*>(residual) + size_t(row0) * ldr + n0 + c + (lane & 7) * 4;
              uint2 raw16[8];
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                const int rr = it * 4 + (lane >> 3);
                raw16[it] = (row0 + rr < M) ? *reinterpret_cast<const uint2*>(resp + size_t(rr) * ldr) : make_uint2(0u, 0u);
              }
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                float2 lo, hi;
                if (fp16) { lo = __half22float2(*reinterpret_cast<const __half2*>(&raw16[it].x)); hi = __half22float2(*reinterpret_cast<const __half2*>(&raw16[it].y)); }
                else { lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw16[it].x)); hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw16[it].y)); }
                resv[it] = make_float4(lo.x, lo.y, hi.x, hi.y);
              }
            } else {
              const float* resp = residual + size_t(row0) * ldr + n0 + c + (lane & 7) * 4;
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                const int rr = it * 4 + (lane >> 3);
                resv[it] = (row0 + rr < M) ? *reinterpret_cast<const float4*>(resp + size_t(rr) * ldr) : make_float4(0.f, 0.f, 0.f, 0.f);
              }
            }
          }
          __syncwarp();  // previous chunk's smem reads are done; warp converged for the aligned tcgen05.ld
#ifdef GEMM_INSTR
          const long long ec0 = clock64();
#endif
          tmem_ld32(taddr + c, r);
          tmem_ld_wait();
#ifdef GEMM_INSTR
          const long long ec1 = clock64();
          e_ldtm += ec1 - ec0;
#endif
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            st_shared_f4(stg + uint32_t(lane * STG_LD + j) * 4, __uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                         __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
          __syncwarp();
#ifdef GEMM_INSTR
          const long long ec2 = clock64();
          e_tr += ec2 - ec1;
          ++e_chunks;
#endif
          const int cc = (lane & 7) * 4;
          const int n = n0 + c + cc;
          if (vec_ok && n0 + c + 32 <= N) {
            float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (bias) bb = __ldg(reinterpret_cast<const float4*>(bias + n));
            if (rowbias) {  // a 32-row block never straddles images (rows_per_img % 32 == 0, checked on the host)
              const int img = min(row0, M - 1) / rows_per_img;
              const float4 t4 = __ldg(reinterpret_cast<const float4*>(rowbias + size_t(img) * ld_rowbias + n));
              bb.x += t4.x; bb.y += t4.y; bb.z += t4.z; bb.w += t4.w;
            }
            float* o32p = out32 ? out32 + size_t(row0) * ldo32 + n : nullptr;
            if constexpr (S2D) {  // 16-bit output in space-to-depth layout (row offsets computed per row inside)
              const int s2d_W = p.s2d_W, s2d_H = p.s2d_H, s2d_B = p.s2d_B;
              uint16_t* o16p = out16 + n;
              if (residual) epi_block<true, true, 2, STATS>(stg, lane, row0, M, alpha, bb, act, fp16, resv, o32p, ldo32, o16p, ldo16, do_stats, cs1, s2d_H, s2d_W, s2d_B, N);
              else if (out32) epi_block<false, true, 2, STATS>(stg, lane, row0, M, alpha, bb, act, fp16, resv, o32p, ldo32, o16p, ldo16, do_stats, cs1, s2d_H, s2d_W, s2d_B, N);
              else epi_block<false, false, 2, STATS>(stg, lane, row0, M, alpha, bb, act, fp16, resv, o32p, ldo32, o16p, ldo16, do_stats, cs1, s2d_H, s2d_W, s2d_B, N);
            } else {
              uint16_t* o16p = out16 ? out16 + size_t(row0) * ldo16 + n : nullptr;
              switch (mode) {
                case 1: epi_block<false, false, 1, STATS>(stg, lane, row0, M, alpha, bb, act, fp16, resv, o32p, ldo32, o16p, ldo16, do_stats, cs1); break;
                case 2: epi_block<false, true, 0, STATS>(stg, lane, row0, M, alpha, bb, act, fp16, resv, o32p, ldo32, o16p, ldo16, do_stats, cs1); break;
                case 3: epi_block<false, true, 1, STATS>(stg, lane, row0, M, alpha, bb, act, fp16, resv, o32p, ldo32, o16p, ldo16, do_stats, cs1); break;
                case 5: epi_block<true, false, 1, STATS>(stg, lane, row0, M, alpha, bb, act, fp16, resv, o32p, ldo32, o16p, ldo16, do_stats, cs1); break;
                case 6: epi_block<true, true, 0, STATS>(stg, lane, row0, M, alpha, bb, act, fp16, resv, o32p, ldo32, o16p, ldo16, do_stats, cs1); break;
                default: epi_block<true, true, 1, STATS>(stg, lane, row0, M, alpha, bb, act, fp16, resv, o32p, ldo32, o16p, ldo16, do_stats, cs1); break;
              }
            }
#ifdef GEMM_INSTR
            e_blk += clock64() - ec2;
#endif
            if (do_stats && lane < 8 && row0 < M) {
              // one (sum, sumsq) pair per column for this warp's 32-row block: 8 lanes x 32 B = 256 contiguous bytes, written by
              // exactly one warp -> no atomics, no cross-warp synchronisation, bit-reproducible
              float4* dst = reinterpret_cast<float4*>(p.colstats + (size_t(row0 >> 5) * N + n) * 2);
              dst[0] = make_float4(cs1[0], cs1[4], cs1[1], cs1[5]);
              dst[1] = make_float4(cs1[2], cs1[6], cs1[3], cs1[7]);
            }
          } else {
#pragma unroll 1
            for (int it = 0; it < 8; ++it) {
              const int rr = it * 4 + (lane >> 3);
              const int m = row0 + rr;
              const float4 v4 = ld_shared_f4(stg + uint32_t(rr * STG_LD + cc) * 4);
              const float vv[4] = {v4.x, v4.y, v4.z, v4.w};
              if (m < M) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const int ne = n + e;
                  if (ne >= N) continue;
                  float v = vv[e] * alpha;
                  if (bias) v += __ldg(bias + ne);
                  if (rowbias) v += __ldg(rowbias + size_t(m / rows_per_img) * ld_rowbias + ne);
                  if (residual) v += residual[size_t(m) * ldr + ne];
                  if (act == ACT_SILU) v = silu_f(v);
                  else if (act == ACT_RELU) v = fmaxf(v, 0.0f);
                  if (out32) out32[size_t(m) * ldo32 + ne] = v;
                  if (out16) out16[size_t(m) * ldo16 + ne] = cvt_16(v, fp16);
                }
              }
            }
          }
          }  // !TMA
        }
      }
      }  // sub-tiles
#ifdef GEMM_INSTR
      e_work += clock64() - ei1;
      ++e_tiles;
#endif
      // release this accumulator stage back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR) mbar_arrive_leader(tmem_empty_bar(acc));  // the issuing thread lives in the leader CTA
        else mbar_arrive(tmem_empty_bar(acc));
      }
      if (++acc == C::NACC) {
        acc = 0;
        acc_phase ^= 1u;
      }
    }
    if (tma_epi) {  // all bulk stores of this warp are complete (smem read and global writes) before the CTA may exit
      if (elect_one()) bulk_wait_all();
      __syncwarp();
    }
#ifdef GEMM_INSTR
    if (blockIdx.x == 4 && lane == 0 && (warp == 2 || warp == 6))
      printf("epilogue warp %d: total %lld clk, %lld tiles %lld chunks | waiting for the accumulator %lld, draining it %lld (tcgen05.ld %lld, transpose %lld, "
             "bias + epi_block %lld)\n", warp, clock64() - e_t0, e_tiles, e_chunks, e_wait, e_work, e_ldtm, e_tr, e_blk);
#endif
  }

  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all();  // the peer may still be reading this CTA's smem / arriving on its barriers
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if constexpr (PAIR) tmem_dealloc_pair(tmem_base, C::TMEM_COLS);
    else tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static const char* encode_map(CUtensorMap* tm, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                              const cuuint32_t* box, CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_UINT16,
                              CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return "cuTensorMapEncodeTiled unavailable (no CUDA driver)";
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(tm, dt, rank, const_cast<void*>(ptr), dims, strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    static thread_local char buf[160];
    snprintf(buf, sizeof(buf), "cuTensorMapEncodeTiled failed (CUresult %d, rank %d, dims %llu/%llu)", int(r), rank,
             (unsigned long long)dims[0], (unsigned long long)dims[1]);
    return buf;
  }
  return nullptr;
}

static int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

// N-tile choice: fewest waves of the persistent grid, preferring wide tiles (a 128xBN UMMA reads (128+BN)*32 B of smem per
// 128*BN*16 MACs, so BN >= 160 keeps the tensor pipe ahead of the 128 B/clk smem port; BN = 64 cannot).
static int pick_bn(const GemmDesc& d) {
  if (d.act == ACT_GEGLU) return 128;
  const int N = d.N;
  if (N <= 16) return 16;
  if (N <= 32) return 32;
  if (N <= 64) return 64;
  const int m_tiles = (d.M + BM - 1) / BM;
  const int cand[5] = {256, 192, 160, 128, 64};
  const double eff[5] = {1.0, 1.0, 1.0, 1.08, 1.5};
  int best = 128;
  double best_cost = 1e30;
  for (int i = 0; i < 5; ++i) {
    const int bn = cand[i];
    if (bn > N && bn != 128 && !(bn == 64)) continue;
    const long tiles = long(m_tiles) * ((N + bn - 1) / bn);
    const long waves = (tiles + num_sms() - 1) / num_sms();
    const double cost = double(waves) * (bn * eff[i] + 24.0);
    if (cost < best_cost - 1e-9) {
      best_cost = cost;
      best = bn;
    }
  }
  return best;
}

int gemm_auto_tiles(const GemmDesc& d) {
  const int bn = d.bn ? d.bn : pick_bn(d);
  const int Ncols = (d.act == ACT_GEGLU) ? 2 * d.N : d.N;
  return ((d.M + BM - 1) / BM) * ((Ncols + bn - 1) / bn);
}

const char* gemm_prepare(const GemmDesc& d, GemmLaunch* out) {
  GemmLaunch& L = *out;
  L.d = d;
  if (d.nseg < 1 || d.nseg > 2) return "gemm: nseg must be 1 or 2";
  if (d.M <= 0 || d.N <= 0) return "gemm: empty problem";
  if (!d.out_f32 && !d.out_bf16) return "gemm: no output";
  if (d.act == ACT_GEGLU && (!d.out_bf16 || d.out_f32 || d.residual || d.rowbias)) return "gemm: GEGLU epilogue writes bf16 only";
  if (d.act == ACT_GEGLU && d.N % 64 != 0) return "gemm: GEGLU needs N % 64 == 0";
  if (d.rowbias && d.rows_per_img % 32 != 0) return "gemm: rows_per_img must be a multiple of 32 when a row bias is given";
  if (d.s2d_W > 0) {
    if (!d.out_f32 && d.residual) return "gemm: a space-to-depth-only output cannot take an fp32 residual";
    if (!d.out_bf16 || (d.s2d_W & 1) || (d.s2d_H & 1) || d.M % (d.s2d_H * d.s2d_W) != 0 || d.N % 32 != 0 || d.act == ACT_GEGLU)
      return "gemm: space-to-depth output needs a 16-bit output, even H/W, M = B*H*W and N % 32 == 0";
  }
  if (d.res16) {
    if (!d.residual) return "gemm: res16 without a residual";
    if (d.N % 32 != 0 || d.ldr % 4 != 0 || (reinterpret_cast<uintptr_t>(d.residual) & 7) != 0)
      return "gemm: a 16-bit residual needs N % 32 == 0, ldr % 4 == 0 and an 8B-aligned pointer (vector epilogue only)";
  }
  if (d.colstats) {
    if (d.stat_rows != 32) return "gemm: stat_rows must be 32";
    if (d.N % 32 != 0 || d.act == ACT_GEGLU) return "gemm: column statistics need N % 32 == 0 and a plain epilogue";
  }
  L.bn = d.bn ? d.bn : pick_bn(d);
  const GemmASeg& s0 = d.seg[0];
  const int pix = s0.H * s0.W;
  if (d.M % pix != 0 && !(s0.H == 1)) return "gemm: M must be a multiple of H*W";
  // M-tile box over (W, H, B)
  if (s0.H == 1 && s0.Bt == 1) {  // plain [M,K] matrix: rows past M are zero-filled by TMA and masked in the epilogue
    L.box_w = BM; L.box_h = 1; L.box_b = 1;
  } else if (s0.W >= BM) {
    if (s0.W % BM != 0) return "gemm: W must be a multiple of 128 when W >= 128";
    L.box_w = BM; L.box_h = 1; L.box_b = 1;
  } else {
    if (BM % s0.W != 0) return "gemm: W must divide 128";
    L.box_w = s0.W;
    int rows = BM / s0.W;
    if (s0.H >= rows) {
      if (s0.H % rows != 0) return "gemm: H must be a multiple of 128/W";
      L.box_h = rows; L.box_b = 1;
    } else {
      if (rows % s0.H != 0) return "gemm: H*W must divide 128";
      L.box_h = s0.H; L.box_b = rows / s0.H;
    }
  }
  int ktot = 0;
  for (int s = 0; s < d.nseg; ++s) {
    const GemmASeg& sg = d.seg[s];
    if (sg.C % BK != 0 || sg.C <= 0) return "gemm: segment channels must be a positive multiple of 64";
    if (sg.ntaps < 1 || sg.ntaps > 9) return "gemm: ntaps out of range";
    if (s > 0 && (sg.H != s0.H || sg.W != s0.W)) return "gemm: segments must share the output grid";
    const int ld = sg.ld ? sg.ld : sg.C;
    if (ld % 8 != 0) return "gemm: channel pitch must be a multiple of 8";
    if ((reinterpret_cast<uintptr_t>(sg.ptr) & 15) != 0) return "gemm: A pointer must be 16B aligned";
    L.cpt[s] = sg.C / BK;
    L.kchunks[s] = sg.ntaps * L.cpt[s];
    ktot += sg.ntaps * sg.C;
    cuuint64_t dims[4] = {cuuint64_t(sg.C), cuuint64_t(sg.W), cuuint64_t(sg.H), cuuint64_t(sg.Bt)};
    cuuint64_t strides[3] = {cuuint64_t(ld) * 2, cuuint64_t(sg.W) * ld * 2, cuuint64_t(sg.H) * sg.W * ld * 2};
    cuuint32_t box[4] = {cuuint32_t(BK), cuuint32_t(L.box_w), cuuint32_t(L.box_h), cuuint32_t(L.box_b)};
    if (const char* e = encode_map(&L.tmA[s], sg.ptr, 4, dims, strides, box)) return e;
  }
  const int Ncols = (d.act == ACT_GEGLU) ? 2 * d.N : d.N;
  const int n_tiles = (Ncols + L.bn - 1) / L.bn;
  // 256-row CTA tiles (two M sub-tiles sharing each W box) for the 128-wide N tile when there is enough work to keep every SM
  // busy with the larger tiles
  L.mt = 1;
  if (L.bn == 128 && d.mt != 1) {
    const long tiles2 = long((d.M + 2 * BM - 1) / (2 * BM)) * n_tiles;
    if (d.mt == 2 || tiles2 >= 2L * num_sms()) L.mt = 2;
  }
  int m_tiles = (d.M + BM * L.mt - 1) / (BM * L.mt);
  // CTA pairs: worthwhile when every pair still gets at least one full tile; needs an even CTA count
  L.pair = 0;
  {
    const bool shape_ok = L.bn >= 128 && num_sms() % 2 == 0;
    const long pair_tiles = long((m_tiles + 1) / 2) * n_tiles;
    if (shape_ok && d.pair >= 0 && (d.pair == 1 || pair_tiles >= num_sms() / 2)) L.pair = 1;
  }
  if (L.pair) m_tiles = (m_tiles + 1) / 2;  // tiles of the pair
  {
    const int Nw = d.Nw ? d.Nw : d.N;
    if ((reinterpret_cast<uintptr_t>(d.w) & 15) != 0) return "gemm: W pointer must be 16B aligned";
    cuuint64_t dims[2] = {cuuint64_t(ktot), cuuint64_t(Nw)};
    const int ldw = d.ldw ? d.ldw : ktot;
    if (ldw % 8 != 0 || ldw < ktot) return "gemm: weight pitch must be >= Ktot and a multiple of 8";
    cuuint64_t strides[1] = {cuuint64_t(ldw) * 2};
    cuuint32_t box[2] = {cuuint32_t(BK), cuuint32_t(L.pair ? L.bn / 2 : L.bn)};  // a pair's CTAs stage half of the W tile each
    if (const char* e = encode_map(&L.tmB, d.w, 2, dims, strides, box)) return e;
  }
  L.splits = 1;
  L.split_stride = 0;
  if (d.splits > 1) {  // split-K: raw fp32 partials, reduced (with the fused epilogue) by splitk_reduce
    if (d.bias || d.rowbias || d.residual || d.out_bf16 || d.act != ACT_NONE || d.colstats || d.alpha != 1.0f || !d.out_f32)
      return "gemm: a split-K launch writes raw fp32 partials only";
    L.splits = d.splits;
    L.split_stride = d.split_stride;
  }
  L.num_tiles = n_tiles * m_tiles * L.splits;
  // TMA-store epilogue: single-output launches whose 32-column chunks tile N exactly.  fp32 output -> bulk tensor store; in-place fp32
  // residual (hs += GEMM, no activation) -> bulk reduce-add at the L2; 16-bit output (also GEGLU) -> 16-bit tile store; fused GroupNorm
  // column statistics ride along (EPI_TMA | EPI_STATS), except with the reduce-add, whose sums never enter the SM.  Space-to-depth,
  // split-K, two outputs and out-of-place / 16-bit residuals keep the coalesced epilogue.  MADM_GEMM_TMA_EPI=0 disables.
  L.tma_epi = TMA_EPI_NONE;
  {
    const char* env = getenv("MADM_GEMM_TMA_EPI");
    const bool on = !(env && strcmp(env, "0") == 0);
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    const bool plain = on && L.bn >= 32 && L.splits == 1 && d.s2d_W == 0 && d.N % 32 == 0 && (!d.bias || al16(d.bias)) &&
                       (!d.rowbias || (al16(d.rowbias) && (d.ld_rowbias ? d.ld_rowbias : d.N) % 4 == 0));
    if (plain && d.act == ACT_GEGLU) {
      if (al16(d.out_bf16) && d.ldo16 % 8 == 0) L.tma_epi = TMA_EPI_H16;
    } else if (plain && d.out_f32 && !d.out_bf16 && al16(d.out_f32) && d.ldo32 % 4 == 0) {
      if (!d.residual) L.tma_epi = TMA_EPI_F32;
      else if (!d.res16 && d.residual == d.out_f32 && d.ldr == d.ldo32 && d.act == ACT_NONE && !d.colstats) L.tma_epi = TMA_EPI_RED;
    } else if (plain && d.out_bf16 && !d.out_f32 && !d.residual && al16(d.out_bf16) && d.ldo16 % 8 == 0) {
      L.tma_epi = TMA_EPI_H16;
    } else if (plain && d.out_bf16 && !d.out_f32 && d.residual && !d.res16 && !d.colstats && d.act == ACT_NONE && al16(d.out_bf16) && d.ldo16 % 8 == 0 &&
               al16(d.residual) && d.ldr % 4 == 0 && EPI_NBUF >= 2) {
      L.tma_epi = TMA_EPI_RES_H16;  // out16 = 16-bit(GEMM + fp32 residual), residual out of place: the transformer's FF out-projection
    }
    if (L.tma_epi == TMA_EPI_RES_H16) {
      cuuint64_t dims[2] = {cuuint64_t(d.N), cuuint64_t(d.M)};
      cuuint64_t strides[1] = {cuuint64_t(d.ldr) * 4};
      cuuint32_t box[2] = {32, 32};
      if (const char* e = encode_map(&L.tmR, d.residual, 2, dims, strides, box, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, CU_TENSOR_MAP_SWIZZLE_128B)) return e;
    }
    if (L.tma_epi) {
      const bool h16 = L.tma_epi == TMA_EPI_H16 || L.tma_epi == TMA_EPI_RES_H16;
      cuuint64_t dims[2] = {cuuint64_t(d.N), cuuint64_t(d.M)};
      cuuint64_t strides[1] = {h16 ? cuuint64_t(d.ldo16) * 2 : cuuint64_t(d.ldo32) * 4};
      cuuint32_t box[2] = {32, 32};
      const void* base = h16 ? static_cast<const void*>(d.out_bf16) : static_cast<const void*>(d.out_f32);
      if (const char* e = encode_map(&L.tmO, base, 2, dims, strides, box, h16 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                                     h16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B))
        return e;
    }
  }
  if (L.pair) {
    const int pairs = L.num_tiles < num_sms() / 2 ? L.num_tiles : num_sms() / 2;
    L.grid = dim3(unsigned(2 * pairs));
  } else {
    L.grid = dim3(unsigned(L.num_tiles < num_sms() ? L.num_tiles : num_sms()));
  }
  switch (L.bn) {
    case 16: L.smem = Cfg<16, 1>::SMEM; break;
    case 32: L.smem = Cfg<32, 1>::SMEM; break;
    case 64: L.smem = Cfg<64, 1>::SMEM; break;
    case 128: L.smem = L.mt == 2 ? (L.pair ? Cfg<128, 2, true>::SMEM : Cfg<128, 2>::SMEM) : (L.pair ? Cfg<128, 1, true>::SMEM : Cfg<128, 1>::SMEM); break;
    case 160: L.smem = L.pair ? Cfg<160, 1, true>::SMEM : Cfg<160, 1>::SMEM; break;
    case 192: L.smem = L.pair ? Cfg<192, 1, true>::SMEM : Cfg<192, 1>::SMEM; break;
    case 256: L.smem = L.pair ? Cfg<256, 1, true>::SMEM : Cfg<256, 1>::SMEM; break;
    default: return "gemm: unsupported N tile";
  }
  return nullptr;
}

template <int BN, int MT, int EPI, bool PAIR>
static const char* launch_bn_s(const GemmLaunch& L, const GemmParams& p, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(gemm_tc_kernel<BN, MT, EPI, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             int(Cfg<BN, MT, PAIR>::SMEM)) != cudaSuccess)
      return "gemm: cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed";
    attr_set = true;
  }
  if constexpr (PAIR) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = L.grid;
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = Cfg<BN, MT, PAIR>::SMEM;
    cfg.stream = stream;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (pdl_train_scope()) {
      at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[1].val.programmaticStreamSerializationAllowed = 1;
      cfg.numAttrs = 2;
    }
    const cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, MT, EPI, PAIR>, p);
    if (e == cudaSuccess) return nullptr;
    static thread_local char buf[160];
    snprintf(buf, sizeof(buf), "gemm: cluster launch failed (%s)", cudaGetErrorString(e));
    return buf;
  } else {
    const cudaError_t e = launch_k(gemm_tc_kernel<BN, MT, EPI, PAIR>, L.grid, dim3(kThreads), Cfg<BN, MT, PAIR>::SMEM, stream, p);
    if (e == cudaSuccess) return nullptr;
    static thread_local char buf[160];
    cudaFuncAttributes fa{};
    cudaFuncGetAttributes(&fa, gemm_tc_kernel<BN, MT, EPI, PAIR>);
    snprintf(buf, sizeof(buf), "gemm: kernel launch failed (%s; %d regs, max %d threads, %d B smem)", cudaGetErrorString(e), fa.numRegs,
             fa.maxThreadsPerBlock, int(Cfg<BN, MT, PAIR>::SMEM));
    return buf;
  }
}
template <int BN, int MT, bool PAIR>
static const char* launch_epi(const GemmLaunch& L, const GemmParams& p, cudaStream_t stream) {
  const int epi = (p.s2d_W > 0 ? EPI_S2D : 0) | (p.colstats ? EPI_STATS : 0);
  if constexpr (BN >= 32) {  // (tma_epi is only chosen for launches without a space-to-depth output, see gemm_prepare)
    if (p.tma_epi) return p.colstats ? launch_bn_s<BN, MT, EPI_TMA | EPI_STATS, PAIR>(L, p, stream) : launch_bn_s<BN, MT, EPI_TMA, PAIR>(L, p, stream);
  }
  switch (epi) {
    case 0: return launch_bn_s<BN, MT, 0, PAIR>(L, p, stream);
    case 1: return launch_bn_s<BN, MT, 1, PAIR>(L, p, stream);
    case 2: return launch_bn_s<BN, MT, 2, PAIR>(L, p, stream);
    default: return launch_bn_s<BN, MT, 3, PAIR>(L, p, stream);
  }
}
template <int BN>
static const char* launch_bn(const GemmLaunch& L, const GemmParams& p, cudaStream_t stream) {
  if constexpr (BN == 128) {
    if (L.mt == 2) return L.pair ? launch_epi<BN, 2, true>(L, p, stream) : launch_epi<BN, 2, false>(L, p, stream);
  }
  if constexpr (BN >= 128) {
    if (L.pair) return launch_epi<BN, 1, true>(L, p, stream);
  }
  return launch_epi<BN, 1, false>(L, p, stream);
}

const char* gemm_launch(const GemmLaunch& L, cudaStream_t stream) {
  const GemmDesc& d = L.d;
  GemmParams p;
  p.tmA[0] = L.tmA[0];
  p.tmA[1] = L.tmA[d.nseg > 1 ? 1 : 0];
  p.tmB = L.tmB;
  p.tma_epi = L.tma_epi;
  if (L.tma_epi) p.tmO = L.tmO; else p.tmO = L.tmB;
  p.tmR = L.tma_epi == TMA_EPI_RES_H16 ? L.tmR : L.tmB;
  p.nseg = d.nseg;
  for (int s = 0; s < 2; ++s) {
    p.kchunks[s] = s < d.nseg ? L.kchunks[s] : 0;
    p.cpt[s] = s < d.nseg ? L.cpt[s] : 1;
    for (int t = 0; t < 9; ++t) {
      p.dx[s][t] = d.seg[s].dx[t];
      p.dy[s][t] = d.seg[s].dy[t];
      p.boff[s][t] = d.seg[s].b_off[t];
    }
  }
  p.M = d.M;
  p.N = (d.act == ACT_GEGLU) ? 2 * d.N : d.N;
  p.W = d.seg[0].W;
  p.pix = d.seg[0].H * d.seg[0].W;
  p.box_w = L.box_w; p.box_h = L.box_h; p.box_b = L.box_b;
  p.bias = d.bias;
  p.rowbias = d.rowbias;
  p.rows_per_img = d.rows_per_img > 0 ? d.rows_per_img : 1;
  p.ld_rowbias = d.ld_rowbias ? d.ld_rowbias : d.N;
  p.residual = d.residual; p.ldr = d.ldr; p.res16 = d.res16;
  p.out_f32 = d.out_f32; p.ldo32 = d.ldo32;
  p.out_bf16 = reinterpret_cast<__nv_bfloat16*>(d.out_bf16); p.ldo16 = d.ldo16;
  p.act = d.act;
  p.alpha = d.alpha;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  p.vec_ok = (d.N % 8 == 0) && (!d.bias || al16(d.bias)) && (!d.rowbias || (al16(d.rowbias) && p.ld_rowbias % 4 == 0)) &&
             (!d.residual || (al16(d.residual) && d.ldr % 4 == 0)) && (!d.out_f32 || (al16(d.out_f32) && d.ldo32 % 4 == 0)) &&
             (!d.out_bf16 || (al16(d.out_bf16) && d.ldo16 % 8 == 0));
  if (d.res16 && !p.vec_ok) return "gemm: a 16-bit residual needs the vector epilogue (16B-aligned operands)";
  if (d.act == ACT_GEGLU && !p.vec_ok) return "gemm: GEGLU epilogue needs 16B-aligned outputs";
  if (d.s2d_W > 0 && !p.vec_ok) return "gemm: space-to-depth output needs 16B-aligned operands";
  p.n_tiles = (p.N + L.bn - 1) / L.bn;
  p.fp16 = d.fp16;
  p.num_tiles = L.num_tiles;
  p.colstats = d.colstats;
  p.stat_rows = d.stat_rows;
  p.splits = L.splits;
  p.split_stride = L.split_stride;
  p.s2d_H = 0; p.s2d_W = 0; p.s2d_B = 0;
  if (d.s2d_W > 0) {  // the kernel takes log2(H), log2(W)
    int lh = 0, lw = 0;
    while ((1 << lh) < d.s2d_H) ++lh;
    while ((1 << lw) < d.s2d_W) ++lw;
    if ((1 << lh) != d.s2d_H || (1 << lw) != d.s2d_W) return "gemm: space-to-depth output needs power-of-two H and W";
    p.s2d_H = lh; p.s2d_W = lw; p.s2d_B = d.M / (d.s2d_H * d.s2d_W);
  }
  switch (L.bn) {
    case 16: return launch_bn<16>(L, p, stream);
    case 32: return launch_bn<32>(L, p, stream);
    case 64: return launch_bn<64>(L, p, stream);
    case 128: return launch_bn<128>(L, p, stream);
    case 160: return launch_bn<160>(L, p, stream);
    case 192: return launch_bn<192>(L, p, stream);
    case 256: return launch_bn<256>(L, p, stream);
  }
  return "gemm: unsupported N tile";
}

}  // namespace madm
