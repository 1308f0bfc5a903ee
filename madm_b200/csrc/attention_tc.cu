// tcgen05 / TMEM flash attention for the SD-1.4 UNet (self: n in {4096,1024,256,64}; cross: 77 keys; 8 heads, d in {40,80,160}).
//
// One CTA = NQT (2, or 1 for d = 160) tiles of 128 query rows of one (image, head).  Per 128-key tile and query tile:
//   S = Q K^T          tcgen05.mma 128x128xd   (Q, K tiles K-major in 128B-swizzled smem, loaded by 4-D TMA boxes over the
//                                               [d, heads, tokens, batch] view; head-dim columns past d are zero-filled by TMA)
//   softmax            4 warps, thread = query row: one tcgen05.ld round trip pulls the fp32 score row into registers, online
//                      max in registers (no shuffles), p = 2^(s*c - m*c) as one FFMA + MUFU, packed to 16 bits
//   O_tile = P V       tcgen05.mma 128xdx128   (V tile used as an MN-major B operand: no transpose pass).  d = 40: P is handed
//                      over through TMEM (tcgen05.st, A operand from tensor memory) and column d of V is set to 1, so the MMA
//                      also accumulates the softmax denominator.  d = 80 / 160: P goes through swizzled smem.
//   O = O*corr + O_tile in registers (fp32), deferred by one tile so the P V latency is hidden behind the next tile's softmax.
// Warp roles: warp 0 TMA producer (double-buffered K/V), warps 1..NQT MMA issuers (one per query tile, also TMEM allocator),
// then one softmax / output warpgroup per query tile.
#include "cvt.cuh"
#include "kernels.h"
#include "launch.cuh"
#include "ptx.cuh"

#include <stdio.h>

namespace madm {

static constexpr int FA_BM = 128;     // queries per CTA
static constexpr int FA_BN = 128;     // keys per tile
static constexpr int FA_TILE = 128 * 128;  // bytes of one [128 rows][64 x 16-bit] swizzled sub-tile

template <int D, int NQT>
struct FaCfg {
  static constexpr int KC = (D + 63) / 64;          // 64-wide head-dim chunks
  static constexpr int DV = (D + 15) / 16 * 16;     // P V output columns (UMMA N)
  static constexpr int KSTEPS = (D + 15) / 16;      // 16-wide k-steps of Q K^T that carry data
  // d <= 80: the softmax thread pulls its whole 128-score row into registers with one TMEM round trip and releases the S
  // buffer immediately, so one S buffer per query tile suffices.  d = 160 keeps its registers for the O accumulator and
  // re-reads S in two passes from two S buffers.
  static constexpr bool REG_S = D <= 80;
  // d = 40 pads its P V tile to 48 columns: column d of the V tile is set to 1 so that the MMA accumulates the softmax
  // denominator (the row sum of exactly the rounded P it multiplies) for free; no per-score add in the softmax warps.
  static constexpr bool ONES = REG_S && DV > D;
  static constexpr int NSB = REG_S ? 1 : 2;         // S buffers per query tile
  // d = 40 also has the TMEM room (2 x 128 S + 2 x 64 P + 2 x 64 O = 512 columns) to hand P to the P V MMA through tensor
  // memory (A operand from TMEM): the 16-bit P tile never touches shared memory, whose port is the bottleneck of the narrow
  // (N = 48) P V MMAs -- each k-step would re-read 4 KB of P for 1.5 KB of V.
  static constexpr bool P_TMEM = ONES && NQT == 2;
  static constexpr int Q_BYTES = NQT * KC * FA_TILE;
  static constexpr int KV_BYTES = KC * FA_TILE;     // per stage, per operand
  static constexpr int P_BYTES = P_TMEM ? 0 : NQT * 2 * FA_TILE;
  static constexpr int STAGES = (Q_BYTES + P_BYTES + 4 * KV_BYTES + 2048 <= 227 * 1024) ? 2 : 1;  // K/V ring depth
  static constexpr size_t SMEM = Q_BYTES + 2 * STAGES * KV_BYTES + P_BYTES + 1024 + 512;
  static constexpr int S_COLS = NQT * NSB * 128;    // S buffers first, then (P_TMEM) one 64-column P tile, then one O tile per query tile
  static constexpr int P_COLS = P_TMEM ? NQT * 64 : 0;
  static constexpr int O_BASE = S_COLS + P_COLS;
  static constexpr int O_STRIDE = (DV + 31) / 32 * 32;
  static constexpr int TMEM_NEED = O_BASE + NQT * O_STRIDE;
  static constexpr int TMEM_COLS = TMEM_NEED <= 256 ? 256 : 512;
  static constexpr int THREADS = 32 * (1 + NQT) + NQT * 128;  // TMA producer, one MMA issuer per query tile, softmax warpgroups
  static_assert(TMEM_NEED <= 512, "TMEM budget");
  static_assert(SMEM <= 227 * 1024, "smem budget");
};

struct FaParams {
  CUtensorMap tmQ, tmK, tmV;
  uint16_t* O;
  int ldo;
  long o_bs;
  int Nq, Nk;
  float scale_log2;
  int fp16;
  float* lse;  // optional [B, heads, Nq]: natural-log log-sum-exp of the scaled scores of every query row (consumed by the backward pass)
};

__device__ __forceinline__ float fa_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// NQT query tiles (128 rows each) per CTA share every K/V tile; each query tile has its own softmax warpgroup, S / O tiles in
// TMEM and P buffer, so the softmax of one tile overlaps the MMAs (and the softmax) of the other.
template <int D, int NQT, bool FP16>
__global__ void __launch_bounds__(FaCfg<D, NQT>::THREADS, 1) fa_tc_kernel(const __grid_constant__ FaParams p) {
  using C = FaCfg<D, NQT>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sQ = base;
  const uint32_t sK = sQ + C::Q_BYTES;
  const uint32_t sV = sK + C::STAGES * C::KV_BYTES;
  const uint32_t sP = sV + C::STAGES * C::KV_BYTES;
  const uint32_t sBar = sP + C::P_BYTES;
  // barriers: q_full | k_full[2] k_empty[2] v_full[2] v_empty[2] | per group g: s_full[2] s_empty[2] pv_go pv_done
  const uint32_t q_full = sBar;
  auto k_full = [&](int s) { return sBar + 8u * (1 + s); };
  auto k_empty = [&](int s) { return sBar + 8u * (3 + s); };
  auto v_full = [&](int s) { return sBar + 8u * (5 + s); };
  auto v_empty = [&](int s) { return sBar + 8u * (7 + s); };
  auto gbar = [&](int g, int i) { return sBar + 8u * (9 + g * 8 + i); };
  auto s_full = [&](int g, int a) { return gbar(g, a); };
  auto s_empty = [&](int g, int a) { return gbar(g, 2 + a); };
  // pv_go(j):   softmax -> issuer: P(j) is posted, V(j) has landed and O(j-1) has been consumed, so P V(j) may run
  // pv_done(j): issuer -> softmax (tcgen05.commit): P V(j) has retired, i.e. the P buffer is free and the O tile holds P V(j)
  auto pv_go = [&](int g) { return gbar(g, 4); };
  auto pv_done = [&](int g) { return gbar(g, 5); };
  const uint32_t tmem_slot = sBar + 8u * (9 + 16);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * (FA_BM * NQT), h = blockIdx.y, b = blockIdx.z;
  const int ntiles = (p.Nk + FA_BN - 1) / FA_BN;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tmQ); prefetch_tmap(&p.tmK); prefetch_tmap(&p.tmV);
    mbar_init(q_full, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(k_full(s), 1); mbar_init(k_empty(s), NQT); mbar_init(v_full(s), 1); mbar_init(v_empty(s), NQT);
    }
    for (int g = 0; g < NQT; ++g) {
      for (int a = 0; a < 2; ++a) { mbar_init(s_full(g, a), 1); mbar_init(s_empty(g, a), 4); }
      mbar_init(pv_go(g), 4); mbar_init(pv_done(g), 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, C::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  pdl_trigger();  // programmatic dependent launch: the prologue above overlapped the previous kernel's tail
  pdl_wait();

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {  // elect.sync (not lane == 0) lets the compiler issue UTMALDG / UTCHMMA without per-lane waterfall loops
      mbar_arrive_expect_tx(q_full, C::Q_BYTES);
#pragma unroll
      for (int g = 0; g < NQT; ++g)
#pragma unroll
        for (int kc = 0; kc < C::KC; ++kc)
          tma_load_4d(sQ + (g * C::KC + kc) * FA_TILE, &p.tmQ, q_full, kc * 64, h, q0 + g * FA_BM, b);
      int stage = 0;
      uint32_t phase = 0;
      for (int j = 0; j < ntiles; ++j) {
        mbar_wait(k_empty(stage), phase ^ 1u);
        mbar_arrive_expect_tx(k_full(stage), C::KV_BYTES);
#pragma unroll
        for (int kc = 0; kc < C::KC; ++kc) tma_load_4d(sK + stage * C::KV_BYTES + kc * FA_TILE, &p.tmK, k_full(stage), kc * 64, h, j * FA_BN, b);
        mbar_wait(v_empty(stage), phase ^ 1u);
        mbar_arrive_expect_tx(v_full(stage), C::KV_BYTES);
#pragma unroll
        for (int kc = 0; kc < C::KC; ++kc) tma_load_4d(sV + stage * C::KV_BYTES + kc * FA_TILE, &p.tmV, v_full(stage), kc * 64, h, j * FA_BN, b);
        if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp <= NQT) {
    // ===================== MMA issuers: one warp per query tile =====================
    // A single thread issues ~60-70 clk per tcgen05.mma (descriptor set-up on the uniform datapath, barrier polls, commits);
    // with 22 small MMAs per 128-key step that thread, not the tensor pipe, bounded the kernel.  Each query tile therefore has
    // its own issuer, and every smem descriptor is computed once up front.
    if (elect_one()) {
      const int g = warp - 1;
      const uint32_t idesc_s = make_idesc_16(FA_BM, FA_BN, FP16 ? 1 : 0);
      const uint32_t idesc_o = make_idesc_16(FA_BM, C::DV, FP16 ? 1 : 0) | (1u << 16);  // B (= V) is MN-major
      uint64_t qd[C::KSTEPS], kd[C::STAGES][C::KSTEPS], vd[C::STAGES], pd[2];
#pragma unroll
      for (int ks = 0; ks < C::KSTEPS; ++ks) {
        const int kc = ks >> 2, k = ks & 3;
        qd[ks] = make_smem_desc_sw128(sQ + (g * C::KC + kc) * FA_TILE) + uint64_t(2 * k);
#pragma unroll
        for (int st = 0; st < C::STAGES; ++st) kd[st][ks] = make_smem_desc_sw128(sK + st * C::KV_BYTES + kc * FA_TILE) + uint64_t(2 * k);
      }
#pragma unroll
      for (int st = 0; st < C::STAGES; ++st) vd[st] = make_smem_desc_sw128_mn(sV + st * C::KV_BYTES, FA_TILE);
      pd[0] = make_smem_desc_sw128(sP + (g * 2) * FA_TILE);
      pd[1] = make_smem_desc_sw128(sP + (g * 2 + 1) * FA_TILE);
      const uint32_t tmem_og = tmem + C::O_BASE + g * C::O_STRIDE;
      const uint32_t tmem_pg = tmem + C::S_COLS + g * 64;
      auto issue_s = [&](int j) {  // S_g = Q_g K(j)^T; K(j) is released once every issuer has committed its MMAs
        const int stage = j % C::STAGES;
        const int sb = j % C::NSB;
        mbar_wait(k_full(stage), (j / C::STAGES) & 1);
        mbar_wait(s_empty(g, sb), ((j / C::NSB) & 1) ^ 1u);
        tc_fence_after();
        const uint32_t ts = tmem + uint32_t((g * C::NSB + sb) * 128);
#pragma unroll
        for (int ks = 0; ks < C::KSTEPS; ++ks) umma_bf16_ss(ts, qd[ks], stage == 0 ? kd[0][ks] : kd[C::STAGES - 1][ks], idesc_s, ks != 0);
        umma_commit(s_full(g, sb));
        umma_commit(k_empty(stage));
      };
      mbar_wait(q_full, 0);
      issue_s(0);
      for (int j = 0; j < ntiles; ++j) {
        if (j + 1 < ntiles) issue_s(j + 1);
        // O_g tile = P_g(j) V(j)
        const int stage = j % C::STAGES;
        int keys = p.Nk - j * FA_BN;
        if (keys > FA_BN) keys = FA_BN;
        const int ksteps = (keys + 15) >> 4;
        mbar_wait(pv_go(g), j & 1);
        tc_fence_after();
        const uint64_t vds = stage == 0 ? vd[0] : vd[C::STAGES - 1];
#pragma unroll
        for (int kk = 0; kk < FA_BN / 16; ++kk) {
          if (kk < ksteps) {
            const uint64_t bd = vds + uint64_t(kk * (2048 >> 4));
            if constexpr (C::P_TMEM) umma_f16_ts(tmem_og, tmem_pg + kk * 8, bd, idesc_o, kk != 0);
            else umma_bf16_ss(tmem_og, pd[kk >> 2] + uint64_t(2 * (kk & 3)), bd, idesc_o, kk != 0);
          }
        }
        umma_commit(pv_done(g));
        umma_commit(v_empty(stage));
      }
    }
  } else {
    // ===================== softmax / output (one warpgroup per query tile, thread = query row) =====================
    const int g = (warp - (1 + NQT)) >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_base = uint32_t(q * 32) << 16;
    const uint32_t sPg = sP + uint32_t(g * 2) * FA_TILE;
    const uint32_t tmem_o = tmem + lane_base + C::O_BASE + g * C::O_STRIDE;
    const uint32_t tmem_p = tmem + lane_base + C::S_COLS + g * 64;
    const float sl = p.scale_log2;
    constexpr int fp16 = FP16 ? 1 : 0;
    constexpr int OC = C::ONES ? D + 1 : D;  // live accumulator columns: the head dim (+ the denominator column); d = 40: 41 of the 48 MMA columns
    float o_acc[C::DV];
#pragma unroll
    for (int i = 0; i < C::DV; ++i) o_acc[i] = 0.f;
    float m_run = -INFINITY, l_run = 0.f, corr_prev = 1.f;
    uint32_t r[32];

    auto o_update = [&](float corr) {  // O = O*corr + (P V) of the tile whose pv_done has been observed
      tc_fence_after();
      constexpr int OB = (C::DV % 48 == 0) ? 48 : 32;  // columns per TMEM round trip (all their loads in flight, one wait)
#pragma unroll
      for (int c0 = 0; c0 < C::DV; c0 += OB) {
        uint32_t ro[OB];
        __syncwarp();
        if (c0 + 0 < C::DV) tmem_ld16_at<0>(tmem_o + c0, ro);
        if (c0 + 16 < C::DV) tmem_ld16_at<16>(tmem_o + c0 + 16, ro);
        if constexpr (OB == 48) { if (c0 + 32 < C::DV) tmem_ld16_at<32>(tmem_o + c0 + 32, ro); }
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < OB; ++i)
          if (c0 + i < OC) o_acc[c0 + i] = fmaf(o_acc[c0 + i], corr, __uint_as_float(ro[i]));  // (columns past OC are head-dim padding: never kept)
      }
      tc_fence_before();
    };

    for (int j = 0; j < ntiles; ++j) {
      const int sb = j % C::NSB;
      mbar_wait(s_full(g, sb), (j / C::NSB) & 1);
      tc_fence_after();
      const uint32_t ts = tmem + lane_base + uint32_t((g * C::NSB + sb) * 128);
      const int kvalid = p.Nk - j * FA_BN;  // keys >= kvalid are masked (only the last tile can be ragged)
      const bool ragged = kvalid < FA_BN;
      float corr, rs = 0.f;
      if constexpr (C::REG_S && C::P_TMEM) {
        // whole score row -> registers (4 loads in flight, one wait), then hand the S buffer back to the MMA warp
        uint32_t sc[4][32];
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 4; ++c) tmem_ld32(ts + c * 32, sc[c]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty(g, sb));
        if (ragged) {
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c * 32 + i >= kvalid) sc[c][i] = 0xff800000u;  // -inf
        }
        float mx0 = m_run, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          mx0 = fmaxf(mx0, __uint_as_float(sc[0][i]));
          mx1 = fmaxf(mx1, __uint_as_float(sc[1][i]));
          mx2 = fmaxf(mx2, __uint_as_float(sc[2][i]));
          mx3 = fmaxf(mx3, __uint_as_float(sc[3][i]));
        }
        const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
        corr = fa_ex2((m_run - mx) * sl);
        m_run = mx;
        const float ms = -mx * sl;
        {  // every softmax thread observes V(j) before P(j) is posted, so the issuer needs no wait of its own on v_full
          const int stage = j % C::STAGES;
          mbar_wait(v_full(stage), (j / C::STAGES) & 1);
          if constexpr (C::ONES) {
            // V(j)[key = row][column D] = 1 (the TMA zero-filled the head-dim padding); published with P below.  Every query
            // tile writes it (same value, same place): its own issuer must not depend on another tile's progress.
            const uint32_t addr = sV + stage * C::KV_BYTES + uint32_t(D >> 6) * FA_TILE + uint32_t(row) * 128 +
                                  uint32_t((((D & 63) >> 3) ^ (row & 7)) << 4) + uint32_t((D & 7) * 2);
            const uint16_t one = FP16 ? 0x3C00 : 0x3F80;
            asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(one) : "memory");
          }
        }
        float rs1 = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float p0 = fa_ex2(fmaf(__uint_as_float(sc[c][i]), sl, ms));
            const float p1 = fa_ex2(fmaf(__uint_as_float(sc[c][i + 1]), sl, ms));
            pk[i >> 1] = pack2_16(p0, p1, fp16);
            if constexpr (!C::ONES) { rs += p0; rs1 += p1; }
          }
          if (c == 0) {  // the first quarter of the exponentials is computed before the P buffer has to be free
            if (j > 0) mbar_wait(pv_done(g), (j - 1) & 1);
            if constexpr (C::P_TMEM) { tc_fence_after(); __syncwarp(); }
          }
          if constexpr (C::P_TMEM) {
            tmem_st16(tmem_p + c * 16, pk);  // keys [32c, 32c+32) of this row = 16 packed columns of the A operand
          } else {
            const uint32_t chunk_base = sPg + uint32_t(c >> 1) * FA_TILE + uint32_t(row) * 128;
            const int u0 = (c & 1) * 4;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const uint32_t addr = chunk_base + uint32_t(((u0 + u) ^ (row & 7)) << 4);
              asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(pk[4 * u]), "r"(pk[4 * u + 1]), "r"(pk[4 * u + 2]),
                           "r"(pk[4 * u + 3]) : "memory");
            }
          }
        }
        if constexpr (C::P_TMEM) { tmem_st_wait(); tc_fence_before(); }
        rs += rs1;
      } else if constexpr (C::REG_S) {
        // d = 80 (P through shared memory): two TMEM passes.  Pass 1: row maximum, two quarters (64 columns) per round trip.  Pass 2
        // re-reads the scores quarter by quarter (TMEM reads are cheap) instead of keeping all 128 next to the 80-column O accumulator:
        // that spilled at the 168-register cap (measured: 74 -> 64 us per launch at n = 1024, B = 8).  For d = 40 the single-pass
        // variant above stays faster (445 vs 480 us): it releases the only S buffer right after the load, so the next Q K^T overlaps.
        uint32_t sa[32], sb2[32];
        float mx0 = m_run, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int hlf = 0; hlf < 2; ++hlf) {
          __syncwarp();
          tmem_ld32(ts + hlf * 64, sa);
          tmem_ld32(ts + hlf * 64 + 32, sb2);
          tmem_ld_wait();
          if (ragged) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if (hlf * 64 + i >= kvalid) sa[i] = 0xff800000u;  // -inf
              if (hlf * 64 + 32 + i >= kvalid) sb2[i] = 0xff800000u;
            }
          }
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            mx0 = fmaxf(mx0, __uint_as_float(sa[i]));
            mx1 = fmaxf(mx1, __uint_as_float(sa[i + 1]));
            mx2 = fmaxf(mx2, __uint_as_float(sb2[i]));
            mx3 = fmaxf(mx3, __uint_as_float(sb2[i + 1]));
          }
        }
        const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
        corr = fa_ex2((m_run - mx) * sl);
        m_run = mx;
        const float ms = -mx * sl;
        {  // every softmax thread observes V(j) before P(j) is posted, so the issuer needs no wait of its own on v_full
          const int stage = j % C::STAGES;
          mbar_wait(v_full(stage), (j / C::STAGES) & 1);
          if constexpr (C::ONES) {  // (d = 40 with one query tile per CTA) V(j)[key = row][column D] = 1: the P V MMA accumulates the denominator
            const uint32_t addr = sV + stage * C::KV_BYTES + uint32_t(D >> 6) * FA_TILE + uint32_t(row) * 128 +
                                  uint32_t((((D & 63) >> 3) ^ (row & 7)) << 4) + uint32_t((D & 7) * 2);
            const uint16_t one = FP16 ? 0x3C00 : 0x3F80;
            asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(one) : "memory");
          }
        }
        float rs1 = 0.f;
        // Pass 2: p = 2^(s*c - m*c), quarter by quarter; the next quarter's scores are in flight while this one's exponentials run.
        __syncwarp();
        tmem_ld32(ts, sa);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t (&cur)[32] = (c & 1) ? sb2 : sa;
          uint32_t (&nxt)[32] = (c & 1) ? sa : sb2;
          tmem_ld_wait();
          if (c < 3) {
            __syncwarp();
            tmem_ld32(ts + (c + 1) * 32, nxt);
          } else {  // all of S(j) has been read: hand the buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(s_empty(g, sb));
          }
          if (ragged) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c * 32 + i >= kvalid) cur[i] = 0xff800000u;  // -inf -> p = 0
          }
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float p0 = fa_ex2(fmaf(__uint_as_float(cur[i]), sl, ms));
            const float p1 = fa_ex2(fmaf(__uint_as_float(cur[i + 1]), sl, ms));
            pk[i >> 1] = pack2_16(p0, p1, fp16);
            if constexpr (!C::ONES) { rs += p0; rs1 += p1; }
          }
          if (c == 0 && j > 0) mbar_wait(pv_done(g), (j - 1) & 1);  // the first quarter is computed before the P buffer has to be free
          const uint32_t chunk_base = sPg + uint32_t(c >> 1) * FA_TILE + uint32_t(row) * 128;
          const int u0 = (c & 1) * 4;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint32_t addr = chunk_base + uint32_t(((u0 + u) ^ (row & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(pk[4 * u]), "r"(pk[4 * u + 1]), "r"(pk[4 * u + 2]),
                         "r"(pk[4 * u + 3]) : "memory");
          }
        }
        rs += rs1;
      } else {
        // pass 1: row max
        float mx = m_run;
#pragma unroll 1
        for (int c = 0; c < FA_BN; c += 32) {
          __syncwarp();
          tmem_ld32(ts + c, r);
          tmem_ld_wait();
          if (c + 32 <= kvalid) {
#pragma unroll
            for (int i = 0; i < 32; ++i) mx = fmaxf(mx, __uint_as_float(r[i]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c + i < kvalid) mx = fmaxf(mx, __uint_as_float(r[i]));
          }
        }
        corr = fa_ex2((m_run - mx) * sl);
        m_run = mx;
        const float ms = -mx * sl;
        mbar_wait(v_full(j % C::STAGES), (j / C::STAGES) & 1);
        if (j > 0) mbar_wait(pv_done(g), (j - 1) & 1);  // P buffer consumed by the previous P V, whose O tile is now complete
        // pass 2: p = 2^(s*sl - m*sl), row sum, 16-bit P into swizzled smem
#pragma unroll 1
        for (int c = 0; c < FA_BN; c += 32) {
          __syncwarp();
          tmem_ld32(ts + c, r);
          tmem_ld_wait();
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float p0 = fa_ex2(fmaf(__uint_as_float(r[i]), sl, ms));
            float p1 = fa_ex2(fmaf(__uint_as_float(r[i + 1]), sl, ms));
            if (c + i >= kvalid) p0 = 0.f;
            if (c + i + 1 >= kvalid) p1 = 0.f;
            rs += p0 + p1;
            pk[i >> 1] = pack2_16(p0, p1, fp16);
          }
          // 32 keys = 4 x 16-byte units of this row; unit index XOR (row & 7) inside the 128-byte swizzle row
          const uint32_t chunk_base = sPg + uint32_t(c >> 6) * FA_TILE + uint32_t(row) * 128;
          const int u0 = (c & 63) >> 3;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint32_t addr = chunk_base + uint32_t(((u0 + u) ^ (row & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(pk[4 * u]), "r"(pk[4 * u + 1]), "r"(pk[4 * u + 2]),
                         "r"(pk[4 * u + 3]) : "memory");
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty(g, sb));
      }
      l_run = l_run * corr + rs;
      // P ready (generic -> async proxy fence before the MMA reads it)
      fence_proxy_async();
      // deferred accumulation of the previous tile's P V (its MMA ran while this tile's softmax was computed)
      if (j > 0) o_update(corr_prev);
      corr_prev = corr;
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(pv_go(g));
    }
    mbar_wait(pv_done(g), (ntiles - 1) & 1);
    o_update(corr_prev);
    // normalise and store this row
    const int m = q0 + g * FA_BM + row;
    if (m < p.Nq) {
      const float den = C::ONES ? o_acc[C::ONES ? D : 0] : l_run;
      const float inv = 1.0f / den;
      if (p.lse) p.lse[(size_t(b) * gridDim.y + h) * p.Nq + m] = (m_run * p.scale_log2 + log2f(den)) * 0.6931471805599453f;
      uint16_t* op = p.O + size_t(b) * p.o_bs + size_t(m) * p.ldo + h * D;
#pragma unroll
      for (int c = 0; c < D; c += 8) {
        uint4 v;
        v.x = pack2_16(o_acc[c] * inv, o_acc[c + 1] * inv, fp16);
        v.y = pack2_16(o_acc[c + 2] * inv, o_acc[c + 3] * inv, fp16);
        v.z = pack2_16(o_acc[c + 4] * inv, o_acc[c + 5] * inv, fp16);
        v.w = pack2_16(o_acc[c + 6] * inv, o_acc[c + 7] * inv, fp16);
        *reinterpret_cast<uint4*>(op + c) = v;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, C::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------ host side
const char* attention_head_map(CUtensorMap* tm, const char* op, const void* ptr, int d, int heads, int ntok, int B, int ld, long bstride, int box_rows) {
  cuuint64_t dims[4] = {cuuint64_t(d), cuuint64_t(heads), cuuint64_t(ntok), cuuint64_t(B)};
  cuuint64_t strides[3] = {cuuint64_t(d) * 2, cuuint64_t(ld) * 2, cuuint64_t(bstride) * 2};
  if (B == 1) strides[2] = cuuint64_t(ntok) * ld * 2;
  cuuint32_t box[4] = {64, 1, cuuint32_t(box_rows), 1};
  return encode_tensor_map(tm, op, ptr, 4, dims, strides, box);
}

const char* flash_attention_tc_prepare(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o, int ldo, int B,
                                       int heads, int d, int Nq, int Nk, long q_bs, long kv_bs, long o_bs, float scale, int fp16,
                                       FaLaunch* L, float* lse) {
  if (d != 40 && d != 80 && d != 160) return "attention: unsupported head dim (40, 80, 160)";
  if (ldq % 8 || ldk % 8 || ldv % 8 || ldo % 8 || q_bs % 8 || kv_bs % 8) return "attention: pitches must be multiples of 8 elements";
  if ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(o)) & 15)
    return "attention: pointers must be 16-byte aligned";
  if (Nq < 1 || Nk < 1) return "attention: empty problem";
  static_assert(sizeof(FaParams) <= sizeof(L->params), "FaLaunch::params too small");
  FaParams* p = reinterpret_cast<FaParams*>(L->params);
  if (const char* e = attention_head_map(&p->tmQ, "attention", q, d, heads, Nq, B, ldq, q_bs, 128)) return e;
  if (const char* e = attention_head_map(&p->tmK, "attention", k, d, heads, Nk, B, ldk, kv_bs, 128)) return e;
  if (const char* e = attention_head_map(&p->tmV, "attention", v, d, heads, Nk, B, ldv, kv_bs, 128)) return e;
  p->O = reinterpret_cast<uint16_t*>(o);
  p->ldo = ldo; p->o_bs = o_bs; p->Nq = Nq; p->Nk = Nk;
  p->scale_log2 = scale * 1.4426950408889634f;
  p->fp16 = fp16;
  p->lse = lse;
  L->d = d;
  L->nqt = (d <= 80 && Nq >= 2 * FA_BM) ? 2 : 1;  // two query tiles per CTA when there are enough rows (d=160: TMEM/regs allow one)
  L->grid = dim3((Nq + FA_BM * L->nqt - 1) / (FA_BM * L->nqt), heads, B);
  return nullptr;
}

template <int D, int NQT, bool FP16>
static const char* fa_launch_t(const FaLaunch& L, cudaStream_t st) {
  using C = FaCfg<D, NQT>;
  static bool attr = false;
  if (!attr) {
    if (cudaFuncSetAttribute(fa_tc_kernel<D, NQT, FP16>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(C::SMEM)) != cudaSuccess)
      return "attention: cudaFuncSetAttribute failed";
    attr = true;
  }
  if (launch_k(fa_tc_kernel<D, NQT, FP16>, L.grid, dim3(C::THREADS), C::SMEM, st, *reinterpret_cast<const FaParams*>(L.params)) != cudaSuccess)
    return "fa_tc launch failed";
  return cudaGetLastError() == cudaSuccess ? nullptr : "attention: launch failed";
}
template <int D, int NQT>
static const char* fa_launch_d(const FaLaunch& L, cudaStream_t st) {
  return reinterpret_cast<const FaParams*>(L.params)->fp16 ? fa_launch_t<D, NQT, true>(L, st) : fa_launch_t<D, NQT, false>(L, st);
}

const char* flash_attention_tc_launch(const FaLaunch& L, cudaStream_t st) {
  switch (L.d) {
    case 40: return L.nqt == 2 ? fa_launch_d<40, 2>(L, st) : fa_launch_d<40, 1>(L, st);
    case 80: return L.nqt == 2 ? fa_launch_d<80, 2>(L, st) : fa_launch_d<80, 1>(L, st);
    case 160: return fa_launch_d<160, 1>(L, st);
  }
  return "attention: unsupported head dim";
}

}  // namespace madm
