// Backward of softmax(Q K^T * scale) V per (image, head) for the LoRA training step (SURVEY §8 row f-3; the reference back-propagates
// through diffusers' Attention processors, modeling/meta_arch/mtmadise.py:240-302 under engine/train_loop.py:277-302).
// Flash-style: the probability matrix is never stored.  Three kernels, all deterministic (no atomics):
//   attn_bwd_prep : L[i] = logsumexp_j(scale * q_i.k_j) (one more pass over K with an online max / sum) and D[i] = sum_c dO[i,c] O[i,c]
//   attn_bwd_dkv  : one CTA per 64-key block, loops over the query blocks:  P = exp(scale*S - L), dS = P * (dO V^T - D) * scale,
//                   dV += P^T dO, dK += dS^T Q   (accumulators stay in registers for the whole loop)
//   attn_bwd_dq   : one CTA per 64-query block, loops over the key blocks:   dQ += dS K
// Tiles are 64 x 64 with the head dim padded to a multiple of 16 in shared memory (d = 40 -> 48); products run on the tensor cores through
// warp-level wmma (16x16x16, fp32 accumulate) on the context's 16-bit operand dtype.  This is the first backward of the path: it is sized
// for the training step's 2 images per GPU, where attention backward is ~1.3 TFLOP per step, not for the tcgen05 peak of the forward kernel.
#include "kernels.h"
#include "launch.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <mma.h>

namespace madm {

namespace {

using namespace nvcuda;

constexpr int AB = 64;        // block of queries / keys
constexpr int AB_THREADS = 256;
constexpr int SLD = AB + 4;   // fp32 score tile pitch
constexpr int PLD = AB + 8;   // 16-bit probability tile pitch
// The probability and dS tiles are rounded to 16 bits for the second set of products.  With thousands of keys P ~ 1/n and
// dS = P * (dP - D) * scale sits around 1e-8 .. 1e-5: in fp16 that is the subnormal range (or below it).  Both tiles are therefore
// stored pre-multiplied by a power of two and the fp32 accumulators are divided by it when the results are written (exact exponent shifts).
constexpr float kPScale = 256.0f;     // P <= 1
constexpr float kDsScale = 16384.0f;

struct AttnBwdParams {
  const uint16_t *q, *k, *v, *o, *dout;
  uint16_t *dq, *dk, *dv;
  int ldq, ldk, ldv, ldo, lddo, lddq, lddk, lddv;
  long q_bs, k_bs, v_bs, o_bs, do_bs, dq_bs, dk_bs, dv_bs;
  int heads, d, Nq, Nk;
  float scale;
  float *L, *D;  // [B, heads, Nq]
  // few keys (cross-attention, 77): the query loop of the dK / dV kernel is split over qsplit CTAs per key block, each writing an fp32
  // partial [qsplit][B][heads][kv blocks * 64][DP] that attn_bwd_kv_reduce sums in fixed order
  int qsplit;
  float *part_k, *part_v;
  float* L2out;  // tcgen05 path: log2-domain log-sum-exp L * log2(e), written by the L / D pass (replaces L when that pass computes it itself)
};

template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ __half from_float<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <typename T> __device__ __forceinline__ float to_float(T v);
template <> __device__ __forceinline__ float to_float<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_float<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

// rows [row0, row0 + 64) x head columns [0, d) of a [*, ld] matrix -> dst[64][DP + 8]; rows >= nrows and columns >= d are zero
template <typename T, int DP>
__device__ __forceinline__ void load_tile(T* dst, const uint16_t* src, int ld, int row0, int nrows, int d) {
  constexpr int LD = DP + 8;
  for (int i = threadIdx.x; i < AB * (DP / 8); i += AB_THREADS) {
    const int r = i / (DP / 8), c8 = (i % (DP / 8)) * 8;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (row0 + r < nrows && c8 < d) v = *reinterpret_cast<const uint4*>(src + size_t(row0 + r) * ld + c8);
    *reinterpret_cast<uint4*>(dst + r * LD + c8) = v;
  }
}

// the same through cp.async (16-byte copies, zero fill where load_tile writes zeros): the tile of the NEXT loop iteration is in flight
// while the current one is consumed
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
  const unsigned s = unsigned(__cvta_generic_to_shared(smem));
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem, bool valid) {
  const unsigned s = unsigned(__cvta_generic_to_shared(smem));
  const int sz = valid ? 4 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(s), "l"(gmem), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <typename T, int DP>
__device__ __forceinline__ void load_tile_async(T* dst, const uint16_t* src, int ld, int row0, int nrows, int d) {
  constexpr int LD = DP + 8;
  for (int i = threadIdx.x; i < AB * (DP / 8); i += AB_THREADS) {
    const int r = i / (DP / 8), c8 = (i % (DP / 8)) * 8;
    const bool ok = row0 + r < nrows && c8 < d;
    cp_async16(dst + r * LD + c8, ok ? src + size_t(row0 + r) * ld + c8 : src, ok);
  }
}

// S = A B^T for two 64 x DP tiles: warp w computes the 16-row band w/2 and two 16-column tiles; results -> out[64][SLD] (fp32)
template <typename T, int DP>
__device__ __forceinline__ void tile_abt(const T* A, const T* Bm, float* out) {
  constexpr int LD = DP + 8;
  const int warp = threadIdx.x >> 5, r = warp >> 1, c0 = (warp & 1) * 2;
  wmma::fragment<wmma::accumulator, 16, 16, 16, float> acc[2];
  wmma::fill_fragment(acc[0], 0.0f);
  wmma::fill_fragment(acc[1], 0.0f);
#pragma unroll
  for (int kk = 0; kk < DP / 16; ++kk) {
    wmma::fragment<wmma::matrix_a, 16, 16, 16, T, wmma::row_major> fa;
    wmma::load_matrix_sync(fa, A + (r * 16) * LD + kk * 16, LD);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      wmma::fragment<wmma::matrix_b, 16, 16, 16, T, wmma::col_major> fb;  // B^T: element (c, key) at Bm[key][c]
      wmma::load_matrix_sync(fb, Bm + ((c0 + j) * 16) * LD + kk * 16, LD);
      wmma::mma_sync(acc[j], fa, fb, acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) wmma::store_matrix_sync(out + (r * 16) * SLD + (c0 + j) * 16, acc[j], SLD, wmma::mem_row_major);
}

// fp32 staging [64][DP + 4] -> 16-bit global rows [row0, row0+64) x [0, d)
template <typename T, int DP>
__device__ __forceinline__ void write_tile(const float* stage, uint16_t* dst, int ld, int row0, int nrows, int d, float mul) {
  constexpr int FLD = DP + 4;
  for (int i = threadIdx.x; i < AB * (d / 2); i += AB_THREADS) {
    const int r = i / (d / 2), c = (i % (d / 2)) * 2;
    if (row0 + r < nrows) {
      T a = from_float<T>(stage[r * FLD + c] * mul), b = from_float<T>(stage[r * FLD + c + 1] * mul);
      uint32_t w = uint32_t(*reinterpret_cast<uint16_t*>(&a)) | (uint32_t(*reinterpret_cast<uint16_t*>(&b)) << 16);
      *reinterpret_cast<uint32_t*>(dst + size_t(row0 + r) * ld + c) = w;
    }
  }
}

// ------------------------------------------------------------------------------------------------ L and D
template <typename T, int DP>
__global__ void __launch_bounds__(AB_THREADS) attn_bwd_prep_kernel(const AttnBwdParams p) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int LD = DP + 8;
  T* Qs = reinterpret_cast<T*>(smem_raw);
  T* Ks = Qs + AB * LD;
  float* Sf = reinterpret_cast<float*>(Ks + AB * LD);
  const int ib = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int i0 = ib * AB;
  const uint16_t* q = p.q + size_t(b) * p.q_bs + h * p.d;
  const uint16_t* k = p.k + size_t(b) * p.k_bs + h * p.d;
  load_tile<T, DP>(Qs, q, p.ldq, i0, p.Nq, p.d);
  const int row = threadIdx.x >> 2, part = threadIdx.x & 3;
  float m = -1e30f, l = 0.f;
  for (int j0 = 0; j0 < p.Nk; j0 += AB) {
    __syncthreads();  // previous tile's readers are done (and Qs is visible on the first pass)
    load_tile<T, DP>(Ks, k, p.ldk, j0, p.Nk, p.d);
    __syncthreads();
    tile_abt<T, DP>(Qs, Ks, Sf);
    __syncthreads();
    float mx = -1e30f;
    float sv[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const int col = part * 16 + c;
      sv[c] = (j0 + col < p.Nk) ? Sf[row * SLD + col] * p.scale : -1e30f;
      mx = fmaxf(mx, sv[c]);
    }
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    const float mn = fmaxf(m, mx);
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < 16; ++c) s += (sv[c] > -1e29f) ? __expf(sv[c] - mn) : 0.f;
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    l = l * __expf(m - mn) + s;
    m = mn;
  }
  // D = sum over the head's channels of dO * O
  float dsum = 0.f;
  if (i0 + row < p.Nq) {
    const uint16_t* orow = p.o + size_t(b) * p.o_bs + size_t(i0 + row) * p.ldo + h * p.d;
    const uint16_t* drow = p.dout + size_t(b) * p.do_bs + size_t(i0 + row) * p.lddo + h * p.d;
    for (int c = part; c < p.d; c += 4)
      dsum += to_float<T>(*reinterpret_cast<const T*>(orow + c)) * to_float<T>(*reinterpret_cast<const T*>(drow + c));
  }
  dsum += __shfl_xor_sync(0xffffffffu, dsum, 1);
  dsum += __shfl_xor_sync(0xffffffffu, dsum, 2);
  if (part == 0 && i0 + row < p.Nq) {
    const size_t o = (size_t(b) * p.heads + h) * p.Nq + i0 + row;
    if (p.L2out) p.L2out[o] = (m + __logf(l)) * 1.4426950408889634f;
    else p.L[o] = m + __logf(l);
    p.D[o] = dsum;
  }
}

// D only (the forward kernel supplied L): one warp-quarter per row as above, no Q K^T pass
__global__ void __launch_bounds__(AB_THREADS) attn_bwd_d_kernel(const AttnBwdParams p, int fp16) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  const int ib = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int row = threadIdx.x >> 2, part = threadIdx.x & 3;
  const int i = ib * AB + row;
  float dsum = 0.f;
  if (i < p.Nq) {
    const uint16_t* orow = p.o + size_t(b) * p.o_bs + size_t(i) * p.ldo + h * p.d;
    const uint16_t* drow = p.dout + size_t(b) * p.do_bs + size_t(i) * p.lddo + h * p.d;
    for (int c = part * 2; c < p.d; c += 8) {
      const uint32_t a = *reinterpret_cast<const uint32_t*>(orow + c), g = *reinterpret_cast<const uint32_t*>(drow + c);
      float2 fa, fg;
      if (fp16) { fa = __half22float2(*reinterpret_cast<const __half2*>(&a)); fg = __half22float2(*reinterpret_cast<const __half2*>(&g)); }
      else { fa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&a)); fg = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&g)); }
      dsum = fmaf(fa.x, fg.x, dsum); dsum = fmaf(fa.y, fg.y, dsum);
    }
  }
  dsum += __shfl_xor_sync(0xffffffffu, dsum, 1);
  dsum += __shfl_xor_sync(0xffffffffu, dsum, 2);
  if (part == 0 && i < p.Nq) {
    const size_t o = (size_t(b) * p.heads + h) * p.Nq + i;
    p.D[o] = dsum;
    if (p.L2out) p.L2out[o] = p.L[o] * 1.4426950408889634f;
  }
}

// shared by the two main kernels: P (optional) and dS tiles from the fp32 S / dP tiles
template <typename T>
__device__ __forceinline__ void softmax_grad_tile(const float* Sf, const float* dPf, const float* Ls, const float* Ds, int i0, int j0, int Nq, int Nk,
                                                  float scale, T* Ps, T* dSs) {
  for (int i = threadIdx.x; i < AB * AB; i += AB_THREADS) {
    const int r = i >> 6, c = i & 63;
    float pv = 0.f, ds = 0.f;
    if (i0 + r < Nq && j0 + c < Nk) {
      pv = __expf(Sf[r * SLD + c] * scale - Ls[r]);
      ds = pv * (dPf[r * SLD + c] - Ds[r]) * scale;
    }
    if (Ps) Ps[r * PLD + c] = from_float<T>(pv * kPScale);
    dSs[r * PLD + c] = from_float<T>(ds * kDsScale);
  }
}

template <int DP> struct AttnSmem {
  static constexpr int LD = DP + 8;
  static constexpr size_t TILE = size_t(AB) * LD * 2;                                  // one 16-bit 64 x DP tile
  static constexpr size_t DKV = 6 * TILE + 2 * AB * SLD * 4 + 2 * AB * PLD * 2 + 4 * AB * 4;  // K, V, 2 x (Q, dO), S, dP, P, dS, 2 x (L, D)
  static constexpr size_t DQ = 6 * TILE + 2 * AB * SLD * 4 + 1 * AB * PLD * 2 + 2 * AB * 4;   // Q, dO, 2 x (K, V), S, dP, dS, L, D
  static constexpr size_t PREP = 2 * TILE + AB * SLD * 4;
  static_assert(2 * TILE >= size_t(AB) * (DP + 4) * 4, "fp32 output staging must fit in two operand tiles");
};

// ------------------------------------------------------------------------------------------------ dK, dV
template <typename T, int DP>
__global__ void __launch_bounds__(AB_THREADS) attn_bwd_dkv_kernel(const AttnBwdParams p) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int LD = DP + 8, NT = DP / 16, NTH = (NT + 1) / 2, FLD = DP + 4;
  T* Ks = reinterpret_cast<T*>(smem_raw);
  T* Vs = Ks + AB * LD;
  T* Qb = Vs + AB * LD;            // [2][64][LD]
  T* dOb = Qb + 2 * AB * LD;       // [2][64][LD]
  float* Sf = reinterpret_cast<float*>(dOb + 2 * AB * LD);
  float* dPf = Sf + AB * SLD;
  T* Ps = reinterpret_cast<T*>(dPf + AB * SLD);
  T* dSs = Ps + AB * PLD;
  float* Lb = reinterpret_cast<float*>(dSs + AB * PLD);  // [2][64]
  float* Db = Lb + 2 * AB;                                // [2][64]
  const int jb = blockIdx.x / p.qsplit, qs = blockIdx.x % p.qsplit, h = blockIdx.y, b = blockIdx.z;
  const int j0 = jb * AB;
  const int warp = threadIdx.x >> 5, r = warp >> 1, tc = warp & 1;
  const uint16_t* q = p.q + size_t(b) * p.q_bs + h * p.d;
  const uint16_t* k = p.k + size_t(b) * p.k_bs + h * p.d;
  const uint16_t* v = p.v + size_t(b) * p.v_bs + h * p.d;
  const uint16_t* dout = p.dout + size_t(b) * p.do_bs + h * p.d;
  const float* Lg = p.L + (size_t(b) * p.heads + h) * p.Nq;
  const float* Dg = p.D + (size_t(b) * p.heads + h) * p.Nq;
  load_tile<T, DP>(Ks, k, p.ldk, j0, p.Nk, p.d);
  load_tile<T, DP>(Vs, v, p.ldv, j0, p.Nk, p.d);
  wmma::fragment<wmma::accumulator, 16, 16, 16, float> accK[NTH], accV[NTH];
#pragma unroll
  for (int i = 0; i < NTH; ++i) { wmma::fill_fragment(accK[i], 0.0f); wmma::fill_fragment(accV[i], 0.0f); }
  const int qblocks = (p.Nq + AB - 1) / AB, per = (qblocks + p.qsplit - 1) / p.qsplit;
  const int i_begin = qs * per * AB, i_end = min(p.Nq, (qs + 1) * per * AB);
  auto prefetch = [&](int i0, int buf) {  // Q / dO tiles and L / D of the query block starting at i0 -> buffer `buf`
    load_tile_async<T, DP>(Qb + buf * AB * LD, q, p.ldq, i0, p.Nq, p.d);
    load_tile_async<T, DP>(dOb + buf * AB * LD, dout, p.lddo, i0, p.Nq, p.d);
    if (threadIdx.x < AB) {
      const bool ok = i0 + threadIdx.x < p.Nq;
      cp_async4(Lb + buf * AB + threadIdx.x, ok ? Lg + i0 + threadIdx.x : Lg, ok);
      cp_async4(Db + buf * AB + threadIdx.x, ok ? Dg + i0 + threadIdx.x : Dg, ok);
    }
    cp_async_commit();
  };
  int buf = 0;
  if (i_begin < i_end) prefetch(i_begin, 0);
  for (int i0 = i_begin; i0 < i_end; i0 += AB, buf ^= 1) {
    cp_async_wait_all();
    __syncthreads();  // this block's tiles have landed; every reader of the other buffer / of P, dS (previous iteration) is done
    if (i0 + AB < i_end) prefetch(i0 + AB, buf ^ 1);
    const T* Qs = Qb + buf * AB * LD;
    const T* dOs = dOb + buf * AB * LD;
    const float* Ls = Lb + buf * AB;
    const float* Ds = Db + buf * AB;
    tile_abt<T, DP>(Qs, Ks, Sf);     // S  = Q K^T
    tile_abt<T, DP>(dOs, Vs, dPf);   // dP = dO V^T
    __syncthreads();
    softmax_grad_tile<T>(Sf, dPf, Ls, Ds, i0, j0, p.Nq, p.Nk, p.scale, Ps, dSs);
    __syncthreads();
    // dV += P^T dO, dK += dS^T Q : this warp's key band r, head-dim tiles tc, tc + 2, ...
#pragma unroll
    for (int kk = 0; kk < AB / 16; ++kk) {
      wmma::fragment<wmma::matrix_a, 16, 16, 16, T, wmma::col_major> fp, fs;  // element (key, query) at Ps[query][key]
      wmma::load_matrix_sync(fp, Ps + (kk * 16) * PLD + r * 16, PLD);
      wmma::load_matrix_sync(fs, dSs + (kk * 16) * PLD + r * 16, PLD);
#pragma unroll
      for (int i = 0; i < NTH; ++i) {
        const int t = tc + 2 * i;
        if (t < NT) {
          wmma::fragment<wmma::matrix_b, 16, 16, 16, T, wmma::row_major> fo, fq;
          wmma::load_matrix_sync(fo, dOs + (kk * 16) * LD + t * 16, LD);
          wmma::load_matrix_sync(fq, Qs + (kk * 16) * LD + t * 16, LD);
          wmma::mma_sync(accV[i], fp, fo, accV[i]);
          wmma::mma_sync(accK[i], fs, fq, accK[i]);
        }
      }
    }
  }
  if (p.qsplit > 1) {  // fp32 partials straight from the accumulators; attn_bwd_kv_reduce finishes
    const int kvrows = ((p.Nk + AB - 1) / AB) * AB;
    const size_t base = (((size_t(qs) * gridDim.z + b) * p.heads + h) * kvrows + j0) * DP;
#pragma unroll
    for (int i = 0; i < NTH; ++i) {
      const int t = tc + 2 * i;
      if (t < NT) {
        wmma::store_matrix_sync(p.part_k + base + size_t(r * 16) * DP + t * 16, accK[i], DP, wmma::mem_row_major);
        wmma::store_matrix_sync(p.part_v + base + size_t(r * 16) * DP + t * 16, accV[i], DP, wmma::mem_row_major);
      }
    }
    return;
  }
  // ---- results: fp32 staging over the (now idle) K / V tiles, then 16-bit rows
  float* stage = reinterpret_cast<float*>(smem_raw);
  uint16_t* dk = p.dk + size_t(b) * p.dk_bs + h * p.d;
  uint16_t* dv = p.dv + size_t(b) * p.dv_bs + h * p.d;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NTH; ++i) { const int t = tc + 2 * i; if (t < NT) wmma::store_matrix_sync(stage + (r * 16) * FLD + t * 16, accK[i], FLD, wmma::mem_row_major); }
  __syncthreads();
  write_tile<T, DP>(stage, dk, p.lddk, j0, p.Nk, p.d, 1.0f / kDsScale);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NTH; ++i) { const int t = tc + 2 * i; if (t < NT) wmma::store_matrix_sync(stage + (r * 16) * FLD + t * 16, accV[i], FLD, wmma::mem_row_major); }
  __syncthreads();
  write_tile<T, DP>(stage, dv, p.lddv, j0, p.Nk, p.d, 1.0f / kPScale);
}

// ------------------------------------------------------------------------------------------------ dQ
template <typename T, int DP>
__global__ void __launch_bounds__(AB_THREADS) attn_bwd_dq_kernel(const AttnBwdParams p) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int LD = DP + 8, NT = DP / 16, NTH = (NT + 1) / 2, FLD = DP + 4;
  T* Kb = reinterpret_cast<T*>(smem_raw);  // [2][64][LD]
  T* Vb = Kb + 2 * AB * LD;                 // [2][64][LD]
  T* Qs = Vb + 2 * AB * LD;
  T* dOs = Qs + AB * LD;
  float* Sf = reinterpret_cast<float*>(dOs + AB * LD);
  float* dPf = Sf + AB * SLD;
  T* dSs = reinterpret_cast<T*>(dPf + AB * SLD);
  float* Ls = reinterpret_cast<float*>(dSs + AB * PLD);
  float* Ds = Ls + AB;
  const int ib = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int i0 = ib * AB;
  const int warp = threadIdx.x >> 5, r = warp >> 1, tc = warp & 1;
  const uint16_t* q = p.q + size_t(b) * p.q_bs + h * p.d;
  const uint16_t* k = p.k + size_t(b) * p.k_bs + h * p.d;
  const uint16_t* v = p.v + size_t(b) * p.v_bs + h * p.d;
  const uint16_t* dout = p.dout + size_t(b) * p.do_bs + h * p.d;
  load_tile<T, DP>(Qs, q, p.ldq, i0, p.Nq, p.d);
  load_tile<T, DP>(dOs, dout, p.lddo, i0, p.Nq, p.d);
  if (threadIdx.x < AB) {
    const bool ok = i0 + threadIdx.x < p.Nq;
    const size_t o = (size_t(b) * p.heads + h) * p.Nq + i0 + threadIdx.x;
    Ls[threadIdx.x] = ok ? p.L[o] : 0.f;
    Ds[threadIdx.x] = ok ? p.D[o] : 0.f;
  }
  wmma::fragment<wmma::accumulator, 16, 16, 16, float> accQ[NTH];
#pragma unroll
  for (int i = 0; i < NTH; ++i) wmma::fill_fragment(accQ[i], 0.0f);
  auto prefetch = [&](int j0, int buf) {
    load_tile_async<T, DP>(Kb + buf * AB * LD, k, p.ldk, j0, p.Nk, p.d);
    load_tile_async<T, DP>(Vb + buf * AB * LD, v, p.ldv, j0, p.Nk, p.d);
    cp_async_commit();
  };
  int buf = 0;
  prefetch(0, 0);
  const T* Ks = Kb;
  for (int j0 = 0; j0 < p.Nk; j0 += AB, buf ^= 1) {
    cp_async_wait_all();
    __syncthreads();  // K / V of this block landed (and Q, dO, L, D on the first pass); the other buffer's readers are done
    if (j0 + AB < p.Nk) prefetch(j0 + AB, buf ^ 1);
    Ks = Kb + buf * AB * LD;
    const T* Vs = Vb + buf * AB * LD;
    tile_abt<T, DP>(Qs, Ks, Sf);
    tile_abt<T, DP>(dOs, Vs, dPf);
    __syncthreads();
    softmax_grad_tile<T>(Sf, dPf, Ls, Ds, i0, j0, p.Nq, p.Nk, p.scale, static_cast<T*>(nullptr), dSs);
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < AB / 16; ++kk) {  // dQ += dS K : query band r, head-dim tiles tc, tc + 2, ...
      wmma::fragment<wmma::matrix_a, 16, 16, 16, T, wmma::row_major> fs;
      wmma::load_matrix_sync(fs, dSs + (r * 16) * PLD + kk * 16, PLD);
#pragma unroll
      for (int i = 0; i < NTH; ++i) {
        const int t = tc + 2 * i;
        if (t < NT) {
          wmma::fragment<wmma::matrix_b, 16, 16, 16, T, wmma::row_major> fk;
          wmma::load_matrix_sync(fk, Ks + (kk * 16) * LD + t * 16, LD);
          wmma::mma_sync(accQ[i], fs, fk, accQ[i]);
        }
      }
    }
  }
  float* stage = reinterpret_cast<float*>(smem_raw);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NTH; ++i) { const int t = tc + 2 * i; if (t < NT) wmma::store_matrix_sync(stage + (r * 16) * FLD + t * 16, accQ[i], FLD, wmma::mem_row_major); }
  __syncthreads();
  write_tile<T, DP>(stage, p.dq + size_t(b) * p.dq_bs + h * p.d, p.lddq, i0, p.Nq, p.d, 1.0f / kDsScale);
}

// dk / dv = sum over the query splits of the fp32 partials (fixed order), unscaled, rounded to 16 bits
template <typename T, int DP>
__global__ void attn_bwd_kv_reduce_kernel(const AttnBwdParams p, int B) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  const int kvrows = ((p.Nk + AB - 1) / AB) * AB;
  const long total = long(B) * p.heads * p.Nk * (p.d / 2);
  const long i = long(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = int(i % (p.d / 2)) * 2;
  long rest = i / (p.d / 2);
  const int j = int(rest % p.Nk); rest /= p.Nk;
  const int h = int(rest % p.heads), b = int(rest / p.heads);
  float k0 = 0.f, k1 = 0.f, v0 = 0.f, v1 = 0.f;
  for (int s = 0; s < p.qsplit; ++s) {
    const size_t o = (((size_t(s) * B + b) * p.heads + h) * kvrows + j) * DP + c;
    k0 += p.part_k[o]; k1 += p.part_k[o + 1]; v0 += p.part_v[o]; v1 += p.part_v[o + 1];
  }
  auto put = [&](uint16_t* dst, float a, float bb) {
    T x = from_float<T>(a), y = from_float<T>(bb);
    *reinterpret_cast<uint32_t*>(dst) = uint32_t(*reinterpret_cast<uint16_t*>(&x)) | (uint32_t(*reinterpret_cast<uint16_t*>(&y)) << 16);
  };
  put(p.dk + size_t(b) * p.dk_bs + size_t(j) * p.lddk + h * p.d + c, k0 * (1.0f / kDsScale), k1 * (1.0f / kDsScale));
  put(p.dv + size_t(b) * p.dv_bs + size_t(j) * p.lddv + h * p.d + c, v0 * (1.0f / kPScale), v1 * (1.0f / kPScale));
}

template <typename T, int DP>
const char* launch_all(const AttnBwdLaunch& L, cudaStream_t st) {
  static bool attr = false;
  if (!attr) {
    if (cudaFuncSetAttribute(attn_bwd_dkv_kernel<T, DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(AttnSmem<DP>::DKV)) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_dq_kernel<T, DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(AttnSmem<DP>::DQ)) != cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_prep_kernel<T, DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(AttnSmem<DP>::PREP)) != cudaSuccess)
      return "attention_bwd: cudaFuncSetAttribute failed";
    attr = true;
  }
  const AttnBwdParams& p = *reinterpret_cast<const AttnBwdParams*>(L.params);
  if (L.have_lse) launch_k(attn_bwd_d_kernel, L.gq, dim3(AB_THREADS), 0, st, p, L.fp16);
  else launch_k(attn_bwd_prep_kernel<T, DP>, L.gq, dim3(AB_THREADS), AttnSmem<DP>::PREP, st, p);
  if (p.L2out) {  // large self-attention: the tcgen05 / TMEM kernels (attention_bwd_tc.cu) take over after the L / D pass
    if (cudaGetLastError() != cudaSuccess) return "attention_bwd launch failed";
    return attention_bwd_tc_launch(L, st);
  }
  launch_k(attn_bwd_dkv_kernel<T, DP>, L.gk, dim3(AB_THREADS), AttnSmem<DP>::DKV, st, p);
  if (p.qsplit > 1) {
    const long total = long(L.B) * p.heads * p.Nk * (p.d / 2);
    launch_k(attn_bwd_kv_reduce_kernel<T, DP>, dim3(unsigned((total + 255) / 256)), dim3(256), 0, st, p, L.B);
  }
  launch_k(attn_bwd_dq_kernel<T, DP>, L.gq, dim3(AB_THREADS), AttnSmem<DP>::DQ, st, p);
  return cudaGetLastError() == cudaSuccess ? nullptr : "attention_bwd launch failed";
}

}  // namespace

// query splits of the dK / dV kernel: only when there are too few key blocks to fill the GPU (cross-attention: 77 keys = 2 blocks)
static int attn_qsplit(int B, int heads, int Nq, int Nk) {
  const int kvb = (Nk + AB - 1) / AB, qb = (Nq + AB - 1) / AB;
  if (kvb * heads * B >= 148 || qb < 4) return 1;
  int s = (296 + kvb * heads * B - 1) / (kvb * heads * B);
  if (s > 16) s = 16;
  if (s > qb) s = qb;
  return s < 1 ? 1 : s;
}
static int attn_dp(int d) { return d == 40 ? 48 : d; }

size_t attention_bwd_scratch_floats(int B, int heads, int d, int Nq, int Nk) {
  size_t n = size_t(2) * B * heads * Nq;
  const int qs = attn_qsplit(B, heads, Nq, Nk);
  if (qs > 1) n += size_t(2) * qs * B * heads * (((Nk + AB - 1) / AB) * AB) * attn_dp(d) + 16;
  return n;
}

const char* attention_bwd_prepare(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, const void* o, int ldo, const void* dout,
                                  int lddo, void* dq, int lddq, void* dk, int lddk, void* dv, int lddv, int B, int heads, int d, int Nq, int Nk, long q_bs,
                                  long k_bs, long v_bs, long o_bs, long do_bs, long dq_bs, long dk_bs, long dv_bs, float scale, float* scratch, int fp16,
                                  AttnBwdLaunch* L, const float* lse) {
  if (d != 40 && d != 80 && d != 160) return "attention_bwd: head dim must be 40, 80 or 160";
  const int lds[8] = {ldq, ldk, ldv, ldo, lddo, lddq, lddk, lddv};
  for (int i = 0; i < 8; ++i) if (lds[i] % 8 != 0) return "attention_bwd: row pitches must be multiples of 8 elements";
  const void* ptrs[8] = {q, k, v, o, dout, dq, dk, dv};
  for (int i = 0; i < 8; ++i) if (reinterpret_cast<uintptr_t>(ptrs[i]) & 15) return "attention_bwd: pointers must be 16-byte aligned";
  static_assert(sizeof(AttnBwdParams) <= sizeof(L->params), "AttnBwdLaunch::params too small");
  AttnBwdParams& p = *reinterpret_cast<AttnBwdParams*>(L->params);
  p.q = static_cast<const uint16_t*>(q); p.k = static_cast<const uint16_t*>(k); p.v = static_cast<const uint16_t*>(v);
  p.o = static_cast<const uint16_t*>(o); p.dout = static_cast<const uint16_t*>(dout);
  p.dq = static_cast<uint16_t*>(dq); p.dk = static_cast<uint16_t*>(dk); p.dv = static_cast<uint16_t*>(dv);
  p.ldq = ldq; p.ldk = ldk; p.ldv = ldv; p.ldo = ldo; p.lddo = lddo; p.lddq = lddq; p.lddk = lddk; p.lddv = lddv;
  p.q_bs = q_bs; p.k_bs = k_bs; p.v_bs = v_bs; p.o_bs = o_bs; p.do_bs = do_bs; p.dq_bs = dq_bs; p.dk_bs = dk_bs; p.dv_bs = dv_bs;
  p.heads = heads; p.d = d; p.Nq = Nq; p.Nk = Nk; p.scale = scale;
  p.L = lse ? const_cast<float*>(lse) : scratch; p.D = scratch + size_t(B) * heads * Nq;
  p.qsplit = attn_qsplit(B, heads, Nq, Nk);
  p.part_k = p.part_v = nullptr;
  p.L2out = attention_bwd_tc_supported(d, Nq, Nk) ? scratch : nullptr;  // (scratch[0, B*heads*Nq) is free when the forward supplied the log-sum-exp)
  if (p.qsplit > 1) {
    float* base = scratch + size_t(2) * B * heads * Nq;
    base = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(base) + 31) & ~uintptr_t(31));  // wmma stores need 32-byte alignment
    const size_t one = size_t(p.qsplit) * B * heads * (((Nk + AB - 1) / AB) * AB) * attn_dp(d);
    p.part_k = base; p.part_v = base + one;
  }
  L->gq = dim3((Nq + AB - 1) / AB, heads, B);
  L->gk = dim3(((Nk + AB - 1) / AB) * p.qsplit, heads, B);
  L->B = B;
  L->fp16 = fp16;
  L->dp = attn_dp(d);
  L->have_lse = lse != nullptr;
  if (p.L2out)
    return attention_bwd_tc_prepare(q, ldq, k, ldk, v, ldv, dout, lddo, dq, lddq, dk, lddk, dv, lddv, B, heads, d, Nq, Nk, q_bs, k_bs, v_bs, do_bs, dq_bs,
                                    dk_bs, dv_bs, scale, p.L2out, p.D, L);
  return nullptr;
}

const char* attention_bwd_launch(const AttnBwdLaunch& L, cudaStream_t st) {
  if (L.fp16) {
    if (L.dp == 48) return launch_all<__half, 48>(L, st);
    if (L.dp == 80) return launch_all<__half, 80>(L, st);
    return launch_all<__half, 160>(L, st);
  }
  if (L.dp == 48) return launch_all<__nv_bfloat16, 48>(L, st);
  if (L.dp == 80) return launch_all<__nv_bfloat16, 80>(L, st);
  return launch_all<__nv_bfloat16, 160>(L, st);
}

}  // namespace madm
