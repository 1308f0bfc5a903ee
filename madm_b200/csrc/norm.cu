// HBM-bound normalisation kernels over the fp32 NHWC residual stream: GroupNorm(32) statistics + apply
// (+SiLU / ReLU, dual-source channel concat, optional raw bf16 copy), LayerNorm, row softmax, and the fused
// relu(GN(a)+GN(b)) -> NCHW fp32 output of the feature projections.  All loads/stores are 16-byte vectorised and
// coalesced along the channel axis; statistics are accumulated in fp32 (sum, sum of squares) per (image, group).
#include "cvt.cuh"
#include "kernels.h"
#include "launch.cuh"

namespace madm {

__device__ __forceinline__ float act_apply(float v, int act) {
  if (act == ACT_SILU) return __fdividef(v, 1.0f + __expf(-v));  // MUFU ex2 + rcp; the result is rounded to 16 bits anyway
  if (act == ACT_RELU) return fmaxf(v, 0.0f);
  return v;
}


// ---------------------------------------------------------------------------------------------- GroupNorm statistics
// V consecutive channels of one pixel: V = 4 from an fp32 tensor (one 16-byte load) or V = 8 from a 16-bit tensor (one
// 16-byte load), so both variants keep the same number of bytes in flight per thread.
template <bool IN16>
struct GnVec {
  static constexpr int V = IN16 ? 8 : 4;
};

template <bool IN16>
__device__ __forceinline__ void ldv(const void* base, size_t elem_off, int fp16, float (&v)[GnVec<IN16>::V]) {
  if constexpr (!IN16) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + elem_off));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(base) + elem_off));
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 f;
      if (fp16) f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
      else f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
      v[2 * i] = f.x; v[2 * i + 1] = f.y;
    }
  }
}

template <int V>
__device__ __forceinline__ void stv16(uint16_t* dst, const float (&v)[V], int fp16) {
  if constexpr (V == 4) {
    *reinterpret_cast<uint2*>(dst) = pack4_16(v[0], v[1], v[2], v[3], fp16);
  } else {
    uint4 o;
    o.x = pack2_16(v[0], v[1], fp16); o.y = pack2_16(v[2], v[3], fp16);
    o.z = pack2_16(v[4], v[5], fp16); o.w = pack2_16(v[6], v[7], fp16);
    *reinterpret_cast<uint4*>(dst) = o;
  }
}

// grid = (slabs, B); block = Q*P threads, Q = C/V channel vectors, P pixel lanes.  Thread (q, pl) owns channels Vq..Vq+V-1
// and walks pixels pl, pl+P, ... of its slab (4 loads in flight), so its per-channel partial sums stay in registers.
template <bool IN16>
__global__ void gn_stats_kernel(const void* __restrict__ x0, int C0, const void* __restrict__ x1, int C1, int HW,
                                int pix_per_cta, int P, int fp16, float* __restrict__ partial /*[B,slabs,32,2]*/) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  constexpr int V = GnVec<IN16>::V;
  extern __shared__ float sm[];  // [2][P][C]
  const int C = C0 + C1;
  const int Q = C / V;
  const int q = threadIdx.x % Q;
  const int pl = threadIdx.x / Q;
  const int b = blockIdx.y;
  const int p_begin = blockIdx.x * pix_per_cta;
  const int p_end = min(HW, p_begin + pix_per_cta);
  const int c = q * V;
  const void* src;
  int ld, cc;
  if (c < C0) { src = x0; ld = C0; cc = c; }
  else        { src = x1; ld = C1; cc = c - C0; }
  const size_t img_off = size_t(b) * HW * ld + cc;
  float s[V], ss[V];
#pragma unroll
  for (int t = 0; t < V; ++t) s[t] = ss[t] = 0.f;
  int p = p_begin + pl;
  for (; p + 3 * P < p_end; p += 4 * P) {
    float v[4][V];
#pragma unroll
    for (int u = 0; u < 4; ++u) ldv<IN16>(src, img_off + size_t(p + u * P) * ld, fp16, v[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int t = 0; t < V; ++t) { s[t] += v[u][t]; ss[t] += v[u][t] * v[u][t]; }
  }
  for (; p < p_end; p += P) {
    float v[V];
    ldv<IN16>(src, img_off + size_t(p) * ld, fp16, v);
#pragma unroll
    for (int t = 0; t < V; ++t) { s[t] += v[t]; ss[t] += v[t] * v[t]; }
  }
  float* sm_s = sm;
  float* sm_ss = sm + P * C;
#pragma unroll
  for (int t = 0; t < V; ++t) {
    sm_s[pl * C + c + t] = s[t];
    sm_ss[pl * C + c + t] = ss[t];
  }
  __syncthreads();
  const int cpg = C / 32;
  if (threadIdx.x < 64) {
    const int g = threadIdx.x & 31;
    const float* base = (threadIdx.x < 32) ? sm_s : sm_ss;
    float acc = 0.f;
    for (int pp = 0; pp < P; ++pp)
      for (int k = 0; k < cpg; ++k) acc += base[pp * C + g * cpg + k];
    // one slot per (image, slab, group, moment): no atomics, so the statistics are bit-reproducible run to run and
    // independent of the batch size (the slab geometry depends on HW and C only)
    partial[((size_t(b) * gridDim.x + blockIdx.x) * 32 + g) * 2 + (threadIdx.x < 32 ? 0 : 1)] = acc;
  }
}

// fixed-order reduction of the per-slab partial sums -> smem[64] = {sum_g, sumsq_g}
__device__ __forceinline__ void gn_reduce_partials(const float* __restrict__ partial, int b, int slabs, float* red /*[64]*/) {
  if (threadIdx.x < 64) {
    const float* p = partial + size_t(b) * slabs * 64 + threadIdx.x;
    float acc = 0.f;
    for (int sidx = 0; sidx < slabs; ++sidx) acc += p[size_t(sidx) * 64];
    red[threadIdx.x] = acc;
  }
  __syncthreads();
}

// the same sums for the short-lived CTAs of the apply pass: up to 4 lane groups take interleaved slabs (independent loads in
// flight instead of one serial chain), combined in a fixed order that depends on the block size (i.e. on C) only
__device__ __forceinline__ void gn_reduce_partials_wide(const float* __restrict__ partial, int b, int slabs, float* red /*[64]*/,
                                                        float* tmp /*[4*64]*/) {
  const int ng = min(4, int(blockDim.x >> 6));
  const int lg = threadIdx.x >> 6, j = threadIdx.x & 63;
  if (lg < ng) {
    const float* p = partial + size_t(b) * slabs * 64 + j;
    float a0 = 0.f, a1 = 0.f;
    int sidx = lg;
    for (; sidx + ng < slabs; sidx += 2 * ng) { a0 += p[size_t(sidx) * 64]; a1 += p[size_t(sidx + ng) * 64]; }
    if (sidx < slabs) a0 += p[size_t(sidx) * 64];
    tmp[lg * 64 + j] = a0 + a1;
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    float acc = tmp[threadIdx.x];
    for (int g = 1; g < ng; ++g) acc += tmp[g * 64 + threadIdx.x];
    red[threadIdx.x] = acc;
  }
  __syncthreads();
}

// Statistics fused into the producing GEMM's epilogue arrive as per-column (sum, sumsq) pairs per block of 32 rows:
// cs[block][c][2].  grid = (S chunks of blocks, B): thread <-> channel (coalesced rows), fixed-order accumulation over the
// chunk's blocks, then per-group sums -> out[b][chunk][32][2], i.e. the same "slab partial" format gn_stats_kernel writes.
// The input may be the channel concat of two producers.
__global__ void gn_colstats_reduce_kernel(const float* __restrict__ cs0, int C0, const float* __restrict__ cs1, int C1, int nb,
                                          int blocks_per_chunk, float* __restrict__ out /*[B,S,32,2]*/) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  extern __shared__ float sm[];  // [C][2]
  const int chunk = blockIdx.x, S = gridDim.x, b = blockIdx.y;
  const int C = C0 + C1, cpg = C / 32;
  const int blk0 = chunk * blocks_per_chunk;
  const int blk1 = min(nb, blk0 + blocks_per_chunk);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float* src = (c < C0) ? cs0 + (size_t(b) * nb * C0 + c) * 2 : cs1 + (size_t(b) * nb * C1 + (c - C0)) * 2;
    const size_t stride = size_t(c < C0 ? C0 : C1) * 2;
    float s = 0.f, ss = 0.f;
    int blk = blk0;
    for (; blk + 3 < blk1; blk += 4) {
      const float2 v0 = __ldg(reinterpret_cast<const float2*>(src + size_t(blk) * stride));
      const float2 v1 = __ldg(reinterpret_cast<const float2*>(src + size_t(blk + 1) * stride));
      const float2 v2 = __ldg(reinterpret_cast<const float2*>(src + size_t(blk + 2) * stride));
      const float2 v3 = __ldg(reinterpret_cast<const float2*>(src + size_t(blk + 3) * stride));
      s += (v0.x + v1.x) + (v2.x + v3.x);
      ss += (v0.y + v1.y) + (v2.y + v3.y);
    }
    for (; blk < blk1; ++blk) {
      const float2 v = __ldg(reinterpret_cast<const float2*>(src + size_t(blk) * stride));
      s += v.x;
      ss += v.y;
    }
    sm[2 * c] = s;
    sm[2 * c + 1] = ss;
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int g = threadIdx.x >> 1, mom = threadIdx.x & 1;
    float acc = 0.f;
    for (int k = 0; k < cpg; ++k) acc += sm[2 * (g * cpg + k) + mom];
    out[((size_t(b) * S + chunk) * 32 + g) * 2 + mom] = acc;
  }
}

__global__ void gn_finalize_kernel(const float* __restrict__ partial, int slabs, float* __restrict__ stats /*[B,32,2]*/) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  __shared__ float red[64];
  gn_reduce_partials(partial, blockIdx.x, slabs, red);
  if (threadIdx.x < 64) stats[size_t(blockIdx.x) * 64 + threadIdx.x] = red[threadIdx.x];
}

// ---------------------------------------------------------------------------------------------- GroupNorm apply
// Same (slab, image) x (channel vector, pixel lane) decomposition as the statistics kernel: each thread keeps the scale /
// shift of its channels in registers and streams its pixels with 4 loads in flight:
// y = act(x*scale + shift) -> 16-bit (and optionally the un-normalised x -> 16-bit for a 1x1 shortcut conv).
template <bool IN16>
__global__ void gn_apply_kernel(const void* __restrict__ x0, int C0, const void* __restrict__ x1, int C1, int HW,
                                int pix_per_cta, int P, const float* __restrict__ partial, int slabs, const float* __restrict__ gamma,
                                const float* __restrict__ beta, float eps, int act, int fp16, uint16_t* __restrict__ y,
                                uint16_t* __restrict__ raw) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  constexpr int V = GnVec<IN16>::V;
  __shared__ float red[64];
  __shared__ float red_tmp[4 * 64];
  const int C = C0 + C1;
  const int Q = C / V;
  const int q = threadIdx.x % Q;
  const int pl = threadIdx.x / Q;
  const int b = blockIdx.y;
  const int cpg = C / 32;
  gn_reduce_partials_wide(partial, b, slabs, red, red_tmp);
  const int c = q * V;
  const float inv_n = 1.0f / (float(HW) * float(cpg));
  float sc[V], sh[V];
#pragma unroll
  for (int t = 0; t < V; ++t) {
    const int g = (c + t) / cpg;
    const float mean = red[g * 2] * inv_n;
    const float var = fmaxf(red[g * 2 + 1] * inv_n - mean * mean, 0.0f);
    const float rstd = rsqrtf(var + eps);
    const float ga = gamma ? gamma[c + t] : 1.0f;
    const float be = beta ? beta[c + t] : 0.0f;
    sc[t] = rstd * ga;
    sh[t] = be - mean * rstd * ga;
  }
  const void* src;
  int ld, cc;
  if (c < C0) { src = x0; ld = C0; cc = c; }
  else        { src = x1; ld = C1; cc = c - C0; }
  const size_t img_off = size_t(b) * HW * ld + cc;
  const size_t out_off = size_t(b) * HW * C + c;
  const int p_begin = blockIdx.x * pix_per_cta;
  const int p_end = min(HW, p_begin + pix_per_cta);
  int p = p_begin + pl;
  for (; p + 3 * P < p_end; p += 4 * P) {
    float v[4][V];
#pragma unroll
    for (int u = 0; u < 4; ++u) ldv<IN16>(src, img_off + size_t(p + u * P) * ld, fp16, v[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const size_t o = out_off + size_t(p + u * P) * C;
      if (raw) stv16<V>(raw + o, v[u], fp16);
#pragma unroll
      for (int t = 0; t < V; ++t) v[u][t] = act_apply(v[u][t] * sc[t] + sh[t], act);
      stv16<V>(y + o, v[u], fp16);
    }
  }
  for (; p < p_end; p += P) {
    float v[V];
    ldv<IN16>(src, img_off + size_t(p) * ld, fp16, v);
    const size_t o = out_off + size_t(p) * C;
    if (raw) stv16<V>(raw + o, v, fp16);
#pragma unroll
    for (int t = 0; t < V; ++t) v[t] = act_apply(v[t] * sc[t] + sh[t], act);
    stv16<V>(y + o, v, fp16);
  }
}

// Slab geometry depends on (HW, C) only, never on the batch size: image i of a batch-8 call reduces in exactly the same
// order as a batch-1 call on that image.
static void gn_geometry(int HW, int C, int V, int* P, int* threads, int* ppc, int* slabs) {
  const int Q = C / V;
  int p = (256 + Q - 1) / Q;
  if (p < 1) p = 1;
  while (Q * p > 1024) --p;
  *P = p;
  *threads = Q * p;
  long per = (HW + 73) / 74;  // up to 74 slabs per image: 592 CTAs (4 per SM) at the benchmark batch of 8
  if (per < 4L * p) per = 4L * p;
  per = ((per + p - 1) / p) * p;
  if (per > HW) per = HW;
  *ppc = int(per);
  *slabs = (HW + int(per) - 1) / int(per);
}

// the slab count must not depend on the input dtype (the partial-sum buffers are sized before it is known): the pixel-lane
// count P of the fp32 geometry is used for both
int groupnorm_slabs(int HW, int C) {
  int P, threads, ppc, slabs;
  gn_geometry(HW, C, 4, &P, &threads, &ppc, &slabs);
  return slabs;
}
static void gn_launch_geometry(int HW, int C, int in16, int* P, int* threads, int* ppc, int* slabs) {
  int P4, t4;
  gn_geometry(HW, C, 4, &P4, &t4, ppc, slabs);  // slabs / pixels per CTA: dtype independent
  const int V = in16 ? 8 : 4;
  const int Q = C / V;
  int p = (256 + Q - 1) / Q;
  while (Q * p > 1024) --p;
  *P = p;
  *threads = Q * p;
}

const char* groupnorm_stats(const void* x0, int C0, const void* x1, int C1, int B, int HW, int in16, int fp16, float* partial,
                            cudaStream_t st) {
  const int C = C0 + C1;
  if (C % 32 != 0 || C % 4 != 0) return "groupnorm: C must be a multiple of 32";
  if (C0 % 4 != 0 || C1 % 4 != 0) return "groupnorm: source channel counts must be multiples of 4";
  if (C / 4 > 1024) return "groupnorm: C too large";
  if (in16 && C % 8 != 0) return "groupnorm: C must be a multiple of 8 for 16-bit inputs";
  int P, threads, ppc, slabs;
  gn_launch_geometry(HW, C, in16, &P, &threads, &ppc, &slabs);
  const size_t smem = size_t(2) * P * C * sizeof(float);
  if (in16) launch_k(gn_stats_kernel<true>, dim3(slabs, B), dim3(threads), smem, st, x0, C0, x1, C1, HW, ppc, P, fp16, partial);
  else launch_k(gn_stats_kernel<false>, dim3(slabs, B), dim3(threads), smem, st, x0, C0, x1, C1, HW, ppc, P, fp16, partial);
  return cudaGetLastError() == cudaSuccess ? nullptr : "groupnorm_stats launch failed";
}

const char* groupnorm_finalize_slabs(const float* partial, int B, int slabs, float* stats, cudaStream_t st) {
  launch_k(gn_finalize_kernel, dim3(B), dim3(64), 0, st, partial, slabs, stats);
  return cudaGetLastError() == cudaSuccess ? nullptr : "groupnorm_finalize launch failed";
}

const char* groupnorm_finalize(const float* partial, int B, int HW, int C, float* stats, cudaStream_t st) {
  launch_k(gn_finalize_kernel, dim3(B), dim3(64), 0, st, partial, groupnorm_slabs(HW, C), stats);
  return cudaGetLastError() == cudaSuccess ? nullptr : "groupnorm_finalize launch failed";
}

int groupnorm_colstats_chunks(int nblocks) {
  int S = nblocks / 8;
  if (S < 1) S = 1;
  if (S > 32) S = 32;
  return S;
}

const char* groupnorm_colstats_reduce(const float* cs0, int C0, const float* cs1, int C1, int B, int nblocks, float* out, cudaStream_t st) {
  const int C = C0 + C1;
  if (C % 32 != 0) return "groupnorm: C must be a multiple of 32";
  const int S = groupnorm_colstats_chunks(nblocks);
  const int bpc = (nblocks + S - 1) / S;
  launch_k(gn_colstats_reduce_kernel, dim3(S, B), dim3(256), size_t(C) * 2 * sizeof(float), st, cs0, C0, cs1, C1, nblocks, bpc, out);
  return cudaGetLastError() == cudaSuccess ? nullptr : "groupnorm_colstats_reduce launch failed";
}

const char* groupnorm_apply(const void* x0, int C0, const void* x1, int C1, int B, int HW, int in16, const float* partial,
                            int stats_slabs, const float* gamma, const float* beta, float eps, int act, void* y, void* raw, int fp16,
                            cudaStream_t st) {
  const int C = C0 + C1;
  int P, threads, ppc, slabs;
  gn_launch_geometry(HW, C, in16, &P, &threads, &ppc, &slabs);
  const int pslabs = stats_slabs > 0 ? stats_slabs : slabs;  // number of partial-sum slabs behind `partial`
  // The apply pass is elementwise, so its own split is free to differ from the statistics slabs: many short CTAs
  // (at most 16 rounds of the 4-deep unrolled loop each) instead of one wave of long ones -- with 3 resident CTAs per SM the
  // 592-CTA statistics geometry ran 1.33 waves (a 2/3-empty tail).
  {
    long want = (long(HW) * B + 148L * 8 - 1) / (148L * 8);  // ~8 CTAs per SM on small tensors ...
    want = (want + 4L * P - 1) / (4L * P) * (4L * P);
    if (want < 4L * P) want = 4L * P;
    if (want > 64L * P) want = 64L * P;                      // ... at most 16 rounds per CTA on large ones
    ppc = int(want);
  }
  if (ppc > HW) ppc = HW;
  slabs = (HW + ppc - 1) / ppc;
  if (in16)
    launch_k(gn_apply_kernel<true>, dim3(slabs, B), dim3(threads), 0, st, x0, C0, x1, C1, HW, ppc, P, partial, pslabs, gamma, beta, eps, act, fp16,
             reinterpret_cast<uint16_t*>(y), reinterpret_cast<uint16_t*>(raw));
  else
    launch_k(gn_apply_kernel<false>, dim3(slabs, B), dim3(threads), 0, st, x0, C0, x1, C1, HW, ppc, P, partial, pslabs, gamma, beta, eps, act, fp16,
             reinterpret_cast<uint16_t*>(y), reinterpret_cast<uint16_t*>(raw));
  return cudaGetLastError() == cudaSuccess ? nullptr : "groupnorm_apply launch failed";
}

// ---------------------------------------------------------------------------------------------- LayerNorm (warp per row)
template <bool IN16>
__global__ void layernorm_kernel(const void* __restrict__ x, int M, int C, const float* __restrict__ gamma,
                                 const float* __restrict__ beta, float eps, int fp16, uint16_t* __restrict__ y) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const int Q = C >> 2;
  float4 v[10];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int q = i * 32 + lane;
    if (q < Q) {
      if constexpr (IN16) {  // 16-bit stream: 4 values = 8 bytes
        const uint2 u = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(x) + size_t(row) * C) + q);
        float2 lo, hi;
        if (fp16) { lo = __half22float2(*reinterpret_cast<const __half2*>(&u.x)); hi = __half22float2(*reinterpret_cast<const __half2*>(&u.y)); }
        else { lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x)); hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y)); }
        v[i] = make_float4(lo.x, lo.y, hi.x, hi.y);
      } else {
        v[i] = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + size_t(row) * C) + q);
      }
      s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / float(C);
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int q = i * 32 + lane;
    if (q < Q) {
      const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      ss += a * a + b * b + c * c + d * d;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float rstd = rsqrtf(ss / float(C) + eps);
  uint16_t* yr = y + size_t(row) * C;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int q = i * 32 + lane;
    if (q < Q) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + q);
      const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + q);
      *reinterpret_cast<uint2*>(yr + q * 4) =
          pack4_16((v[i].x - mean) * rstd * g.x + b.x, (v[i].y - mean) * rstd * g.y + b.y,
                   (v[i].z - mean) * rstd * g.z + b.z, (v[i].w - mean) * rstd * g.w + b.w, fp16);
    }
  }
}

const char* layernorm(const void* x, int in16, int M, int C, const float* gamma, const float* beta, float eps, void* y, int fp16, cudaStream_t st) {
  if (C % 4 != 0 || C > 1280) return "layernorm: C must be a multiple of 4 and <= 1280";
  const int rows_per_cta = 8;
  const unsigned grid = (M + rows_per_cta - 1) / rows_per_cta;
  if (in16) launch_k(layernorm_kernel<true>, dim3(grid), dim3(rows_per_cta * 32), 0, st, x, M, C, gamma, beta, eps, fp16, reinterpret_cast<uint16_t*>(y));
  else launch_k(layernorm_kernel<false>, dim3(grid), dim3(rows_per_cta * 32), 0, st, x, M, C, gamma, beta, eps, fp16, reinterpret_cast<uint16_t*>(y));
  return cudaGetLastError() == cudaSuccess ? nullptr : "layernorm launch failed";
}

// ---------------------------------------------------------------------------------------------- row softmax fp32 -> bf16
// one CTA (256 threads) per row; L <= 256*32.
__global__ void softmax_rows_kernel(const float* __restrict__ s, int L, int fp16, uint16_t* __restrict__ p) {
  __shared__ float red[8];
  const float* sr = s + size_t(blockIdx.x) * L;
  uint16_t* pr = p + size_t(blockIdx.x) * L;
  float v[32];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int j = i * 256 + threadIdx.x;
    v[i] = (j < L) ? sr[j] : -INFINITY;
    mx = fmaxf(mx, v[i]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) mx = fmaxf(mx, red[i]);
  __syncthreads();
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    v[i] = __expf(v[i] - mx);
    sum += v[i];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
  __syncthreads();
  sum = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) sum += red[i];
  const float inv = 1.0f / sum;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int j = i * 256 + threadIdx.x;
    if (j < L) pr[j] = cvt_16(v[i] * inv, fp16);
  }
}

const char* softmax_rows(const float* s, int R, int L, void* p, int fp16, cudaStream_t st) {
  if (L > 256 * 32) return "softmax_rows: row too long";
  softmax_rows_kernel<<<R, 256, 0, st>>>(s, L, fp16, reinterpret_cast<uint16_t*>(p));
  return cudaGetLastError() == cudaSuccess ? nullptr : "softmax_rows launch failed";
}

// ---------------------------------------------------------------------------------------------- projection tail
// out[b, c, p] (NCHW fp32) = relu( GN(a)[b,p,c] + (GN(s) or s)[b,p,c] ); 32x32 (pixel x channel) tiles through smem.
__global__ void gn_add_relu_nchw_kernel(const float* __restrict__ a, const float* __restrict__ stats_a,
                                        const float* __restrict__ ga, const float* __restrict__ ba,
                                        const float* __restrict__ s, const float* __restrict__ stats_s,
                                        const float* __restrict__ gs, const float* __restrict__ bs, float eps, int HW, int C,
                                        float* __restrict__ out, int out_fp16) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int c0 = blockIdx.y * 32;
  const int p0 = blockIdx.x * 32;
  const int cpg = C / 32;
  const float inv_n = 1.0f / (float(HW) * float(cpg));
  const int tx = threadIdx.x;  // 0..31
  const int ty = threadIdx.y;  // 0..7
  // read: channel fastest
  const int c = c0 + tx;
  const int g = c / cpg;
  float sca, sha, scs = 1.f, shs = 0.f;
  {
    const float mean = stats_a[(size_t(b) * 32 + g) * 2] * inv_n;
    const float var = fmaxf(stats_a[(size_t(b) * 32 + g) * 2 + 1] * inv_n - mean * mean, 0.f);
    const float rstd = rsqrtf(var + eps);
    sca = rstd * ga[c];
    sha = ba[c] - mean * sca;
  }
  if (stats_s) {
    const float mean = stats_s[(size_t(b) * 32 + g) * 2] * inv_n;
    const float var = fmaxf(stats_s[(size_t(b) * 32 + g) * 2 + 1] * inv_n - mean * mean, 0.f);
    const float rstd = rsqrtf(var + eps);
    scs = rstd * gs[c];
    shs = bs[c] - mean * scs;
  }
  for (int r = ty; r < 32; r += 8) {
    const int p = p0 + r;
    float v = 0.f;
    if (p < HW) {
      const size_t i = (size_t(b) * HW + p) * C + c;
      v = fmaxf(a[i] * sca + sha + s[i] * scs + shs, 0.f);
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {  // r = channel within tile, tx = pixel
    const int p = p0 + tx;
    if (p < HW) {
      const size_t o = (size_t(b) * C + c0 + r) * HW + p;
      if (out_fp16) reinterpret_cast<__half*>(out)[o] = __float2half_rn(tile[tx][r]);
      else out[o] = tile[tx][r];
    }
  }
}

const char* gn_add_relu_nchw(const float* a, const float* stats_a, const float* ga, const float* ba, const float* s,
                             const float* stats_s, const float* gs, const float* bs, float eps, int B, int HW, int C,
                             float* out, cudaStream_t st, int out_fp16) {
  if (C % 32 != 0) return "gn_add_relu_nchw: C must be a multiple of 32";
  dim3 grid((HW + 31) / 32, C / 32, B);
  gn_add_relu_nchw_kernel<<<grid, dim3(32, 8), 0, st>>>(a, stats_a, ga, ba, s, stats_s, gs, bs, eps, HW, C, out, out_fp16);
  return cudaGetLastError() == cudaSuccess ? nullptr : "gn_add_relu_nchw launch failed";
}

// ---------------------------------------------------------------------------------------------- 3-channel input of the s0 projection
// Bottleneck(3 -> Cb -> Cout) on the decoded image (SURVEY §8 a-11): its two 1x1 convs have K = 3.  They are not GEMMs: a 1x1 conv of a
// 3-channel image is 3 FMAs per output, and the GroupNorm statistics of y_c = w_c . x follow from the image's first and second moments,
//     sum_p y_c = w_c . (sum_p x),     sum_p y_c^2 = w_c^T (sum_p x x^T) w_c,
// so `conv1 -> GN -> ReLU` is ONE elementwise pass writing the 16-bit operand of conv2 (no conv output, no statistics pass), and the
// shortcut branch `conv -> GN` is recomputed from the image inside the block's final pass instead of being stored as a 1 GB fp32 tensor.
static constexpr int kMomSlabs = 64;  // partial moment sums per image: [B][64][12] (9 used), reduced in fixed order by the consumers

__global__ void __launch_bounds__(256) image_moments_kernel(const float4* __restrict__ img4, int HW, float* __restrict__ partial) {
  const int b = blockIdx.y, slab = blockIdx.x;
  const int per = (HW + kMomSlabs - 1) / kMomSlabs;
  const int p0 = slab * per, p1 = min(HW, p0 + per);
  float m[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // x y z xx xy xz yy yz zz
  for (int p = p0 + threadIdx.x; p < p1; p += 256) {
    const float4 v = __ldg(img4 + size_t(b) * HW + p);
    m[0] += v.x; m[1] += v.y; m[2] += v.z;
    m[3] = fmaf(v.x, v.x, m[3]); m[4] = fmaf(v.x, v.y, m[4]); m[5] = fmaf(v.x, v.z, m[5]);
    m[6] = fmaf(v.y, v.y, m[6]); m[7] = fmaf(v.y, v.z, m[7]); m[8] = fmaf(v.z, v.z, m[8]);
  }
  __shared__ float red[9][256];
#pragma unroll
  for (int k = 0; k < 9; ++k) red[k][threadIdx.x] = m[k];
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {  // fixed-order tree
    if (threadIdx.x < s) {
#pragma unroll
      for (int k = 0; k < 9; ++k) red[k][threadIdx.x] += red[k][threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x < 9) partial[(size_t(b) * kMomSlabs + slab) * 12 + threadIdx.x] = red[threadIdx.x][0];
}

// Per image and channel: GroupNorm(32) of y = W x (W fp32 [C][3]) folded into y_norm_c = a . x + d  ->  coef[b][c] = (a0, a1, a2, d).
// grid = B, block = C threads.  The moments are reduced in fixed order, the statistics evaluated in double.
__global__ void c3_gn_coeffs_kernel(const float* __restrict__ partial, const float* __restrict__ w, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, float eps, int HW, int C, float4* __restrict__ coef) {
  __shared__ double mom[9];
  const int b = blockIdx.x, c = threadIdx.x;
  if (c < 9) {
    double acc = 0.0;
    for (int sl = 0; sl < kMomSlabs; ++sl) acc += double(partial[(size_t(b) * kMomSlabs + sl) * 12 + c]);
    mom[c] = acc / double(HW);
  }
  __syncthreads();
  if (c >= C) return;
  const double* mu = mom;       // E[x]
  const double* S = mom + 3;    // E[x x^T]: xx xy xz yy yz zz
  const int cpg = C / 32, g0 = (c / cpg) * cpg;
  double m1 = 0.0, m2 = 0.0;
  for (int k = g0; k < g0 + cpg; ++k) {
    const double wx = w[k * 3], wy = w[k * 3 + 1], wz = w[k * 3 + 2];
    m1 += wx * mu[0] + wy * mu[1] + wz * mu[2];
    m2 += wx * wx * S[0] + 2.0 * wx * wy * S[1] + 2.0 * wx * wz * S[2] + wy * wy * S[3] + 2.0 * wy * wz * S[4] + wz * wz * S[5];
  }
  const double mean = m1 / cpg;
  const double var = fmax(m2 / cpg - mean * mean, 0.0);
  const double sc = double(gamma[c]) / sqrt(var + double(eps));
  coef[size_t(b) * C + c] = make_float4(float(sc * w[c * 3]), float(sc * w[c * 3 + 1]), float(sc * w[c * 3 + 2]), float(double(beta[c]) - mean * sc));
}

// out16[b, p, c] = relu(a_c . x + d_c)  = relu(GN(conv1x1(x)))  for the 3-channel image x (img4: fp32 [B*HW][4], 3 used)
__global__ void __launch_bounds__(256) c3_conv_gn_relu_kernel(const float4* __restrict__ img4, const float4* __restrict__ coef, int HW, int C,
                                                              int pix_per_cta, int fp16, uint16_t* __restrict__ out16) {
  const int b = blockIdx.y;
  const int Q = C >> 3, q = threadIdx.x % Q, pl = threadIdx.x / Q, P = 256 / Q;
  float4 cf[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) cf[t] = __ldg(coef + size_t(b) * C + q * 8 + t);
  const int p0 = blockIdx.x * pix_per_cta, p1 = min(HW, p0 + pix_per_cta);
  for (int p = p0 + pl; p < p1; p += P) {
    const float4 x = __ldg(img4 + size_t(b) * HW + p);
    float o[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) o[t] = fmaxf(fmaf(cf[t].x, x.x, fmaf(cf[t].y, x.y, fmaf(cf[t].z, x.z, cf[t].w))), 0.f);
    uint4 pk;
    pk.x = pack2_16(o[0], o[1], fp16); pk.y = pack2_16(o[2], o[3], fp16); pk.z = pack2_16(o[4], o[5], fp16); pk.w = pack2_16(o[6], o[7], fp16);
    *reinterpret_cast<uint4*>(out16 + (size_t(b) * HW + p) * C + q * 8) = pk;
  }
}

const char* image_moments(const float* img4, int B, int HW, float* partial, cudaStream_t st) {
  image_moments_kernel<<<dim3(kMomSlabs, B), 256, 0, st>>>(reinterpret_cast<const float4*>(img4), HW, partial);
  return cudaGetLastError() == cudaSuccess ? nullptr : "image_moments launch failed";
}
int image_moments_floats(int B) { return B * kMomSlabs * 12; }

const char* c3_gn_coeffs(const float* mom, const float* w, const float* gamma, const float* beta, float eps, int B, int HW, int C, float* coef,
                         cudaStream_t st) {
  if (C % 32 != 0 || C > 1024) return "c3_gn_coeffs: C must be a multiple of 32, at most 1024";
  c3_gn_coeffs_kernel<<<B, C < 32 ? 32 : C, 0, st>>>(mom, w, gamma, beta, eps, HW, C, reinterpret_cast<float4*>(coef));
  return cudaGetLastError() == cudaSuccess ? nullptr : "c3_gn_coeffs launch failed";
}

const char* c3_conv_gn_relu(const float* img4, const float* coef, int B, int HW, int C, void* out16, int fp16, cudaStream_t st) {
  if (C % 32 != 0 || C > 1024 || 256 % (C / 8) != 0) return "c3_conv_gn_relu: C must be a multiple of 32 with C/8 dividing 256";
  const int ppc = 1024;
  c3_conv_gn_relu_kernel<<<dim3((HW + ppc - 1) / ppc, B), 256, 0, st>>>(reinterpret_cast<const float4*>(img4), reinterpret_cast<const float4*>(coef),
                                                                       HW, C, ppc, fp16, reinterpret_cast<uint16_t*>(out16));
  return cudaGetLastError() == cudaSuccess ? nullptr : "c3_conv_gn_relu launch failed";
}

// Final pass of the bottleneck with the shortcut branch recomputed from the 3-channel image:
// out[b, c, p] = relu(GN(a)[b, p, c] + (as_c . x[b, p] + ds_c))  ->  fp32 NCHW   (coef_s = the shortcut's folded conv + GroupNorm)
__global__ void gn_add_relu_nchw_c3_kernel(const float* __restrict__ a, const float* __restrict__ stats_a, const float* __restrict__ ga,
                                           const float* __restrict__ ba, const float4* __restrict__ img4, const float4* __restrict__ coef_s, float eps,
                                           int HW, int C, float* __restrict__ out) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int c0 = blockIdx.y * 32;
  const int p0 = blockIdx.x * 32;
  const int cpg = C / 32;
  const float inv_n = 1.0f / (float(HW) * float(cpg));
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int c = c0 + tx;
  const int g = c / cpg;
  float sca, sha;
  {
    const float mean = stats_a[(size_t(b) * 32 + g) * 2] * inv_n;
    const float var = fmaxf(stats_a[(size_t(b) * 32 + g) * 2 + 1] * inv_n - mean * mean, 0.f);
    const float rstd = rsqrtf(var + eps);
    sca = rstd * ga[c];
    sha = ba[c] - mean * sca;
  }
  const float4 cs = __ldg(coef_s + size_t(b) * C + c);
  const float sh = sha + cs.w;
  for (int r = ty; r < 32; r += 8) {
    const int p = p0 + r;
    float v = 0.f;
    if (p < HW) {
      const float4 x = __ldg(img4 + size_t(b) * HW + p);
      v = fmaxf(fmaf(a[(size_t(b) * HW + p) * C + c], sca, fmaf(cs.x, x.x, fmaf(cs.y, x.y, fmaf(cs.z, x.z, sh)))), 0.f);
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int p = p0 + tx;
    if (p < HW) out[(size_t(b) * C + c0 + r) * HW + p] = tile[tx][r];
  }
}

const char* gn_add_relu_nchw_c3(const float* a, const float* stats_a, const float* ga, const float* ba, const float* img4, const float* coef_s, float eps,
                                int B, int HW, int C, float* out, cudaStream_t st) {
  if (C % 32 != 0) return "gn_add_relu_nchw_c3: C must be a multiple of 32";
  dim3 grid((HW + 31) / 32, C / 32, B);
  gn_add_relu_nchw_c3_kernel<<<grid, dim3(32, 8), 0, st>>>(a, stats_a, ga, ba, reinterpret_cast<const float4*>(img4),
                                                          reinterpret_cast<const float4*>(coef_s), eps, HW, C, out);
  return cudaGetLastError() == cudaSuccess ? nullptr : "gn_add_relu_nchw_c3 launch failed";
}

// ---- backward of one K = 3 branch z_c = GN(w_c . x)_c (-> ReLU) of the s0 projection (training path), again without its [B*HW, C] input.
// With u_c = w_c . x, group g of cpg channels, mean mu_g, rstd r_g (from the image moments, as in the forward), N = HW * cpg, and the
// per-image sums S_c = sum_p g_c, G_c = sum_p g_c x (g_c = dL/dz_c, masked by the ReLU):
//     sum_p g_c xhat_c     = r_g (w_c . G_c - mu_g S_c)                          =: T_c        -> d gamma_c, and d beta_c = S_c
//     sum_p xhat_c x       = r_g HW (E[x x^T] w_c - mu_g E[x])
//     d w_c = r_g (gamma_c G_c - m1_g HW E[x] - m2_g sum_p xhat_c x),   m1_g = sum_{k in g} gamma_k S_k / N,  m2_g = sum_{k in g} gamma_k T_k / N
// (the GroupNorm input gradient r_g (gamma_c g_c - m1_g - xhat_c m2_g) contracted with x).  So one streaming pass over dy and the image
// (partials kernel: S_c and G_c per (image, slab), 4 sums per channel) and a small finish kernel that reduces them in fixed order and
// applies the chain rule in double.
static constexpr int kC3BwdSlabs = 128;  // partial sums per image: [B][128][C][4]

__global__ void __launch_bounds__(256) c3_gn_bwd_partials_kernel(const uint16_t* __restrict__ dy16, const float4* __restrict__ img4,
                                                                 const float4* __restrict__ coef, int HW, int C, int relu, int fp16,
                                                                 float4* __restrict__ partial) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  extern __shared__ float4 red[];  // [256 / (C/8)][C]
  const int b = blockIdx.y, slab = blockIdx.x;
  const int Q = C >> 3, q = threadIdx.x % Q, pl = threadIdx.x / Q, P = 256 / Q;
  float4 cf[8], acc[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    cf[t] = __ldg(coef + size_t(b) * C + q * 8 + t);
    acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int per = (HW + kC3BwdSlabs - 1) / kC3BwdSlabs;
  const int p0 = slab * per, p1 = min(HW, p0 + per);
  for (int p = p0 + pl; p < p1; p += P) {
    const float4 x = __ldg(img4 + size_t(b) * HW + p);
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(dy16 + (size_t(b) * HW + p) * C + q * 8));
    const uint32_t w4[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int t2 = 0; t2 < 4; ++t2) {
      float2 d;
      if (fp16) d = __half22float2(*reinterpret_cast<const __half2*>(&w4[t2]));
      else d = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w4[t2]));
      const float dd[2] = {d.x, d.y};
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int t = 2 * t2 + h;
        float g = dd[h];
        // the forward's expression (c3_conv_gn_relu_kernel), so the ReLU mask is the forward's
        if (relu && !(fmaf(cf[t].x, x.x, fmaf(cf[t].y, x.y, fmaf(cf[t].z, x.z, cf[t].w))) > 0.f)) g = 0.f;
        acc[t].x += g;
        acc[t].y = fmaf(g, x.x, acc[t].y);
        acc[t].z = fmaf(g, x.y, acc[t].z);
        acc[t].w = fmaf(g, x.z, acc[t].w);
      }
    }
  }
#pragma unroll
  for (int t = 0; t < 8; ++t) red[pl * C + q * 8 + t] = acc[t];
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += 256) {  // fixed order over the pixel lanes
    float4 s = red[c];
    for (int l = 1; l < P; ++l) {
      const float4 v = red[l * C + c];
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    partial[(size_t(b) * kC3BwdSlabs + slab) * C + c] = s;
  }
}

// One CTA of C threads (thread = channel) walks the images in order; outputs are written (not accumulated), multiplied by `scale`.
__global__ void c3_gn_bwd_finish_kernel(const float4* __restrict__ partial, const float* __restrict__ mom_partial, const float* __restrict__ w,
                                        const float* __restrict__ gamma, float eps, int B, int HW, int C, float scale, float* __restrict__ dw,
                                        float* __restrict__ dgamma, float* __restrict__ dbeta) {
  pdl_trigger();  // programmatic dependent launch (launch.cuh): no global access before pdl_wait()
  pdl_wait();
  __shared__ double mom[9];
  __shared__ double gs[1024], gt[1024];
  const int c = threadIdx.x;
  const int cpg = C / 32, g0 = (c / cpg) * cpg;
  const double wc[3] = {w[c * 3], w[c * 3 + 1], w[c * 3 + 2]};
  const double gam = gamma[c];
  const double invN = 1.0 / (double(HW) * cpg);
  double aw[3] = {0.0, 0.0, 0.0}, ag = 0.0, ab = 0.0;
  for (int b = 0; b < B; ++b) {
    if (c < 9) {  // the image's moments, reduced as c3_gn_coeffs_kernel does
      double m = 0.0;
      for (int sl = 0; sl < kMomSlabs; ++sl) m += double(mom_partial[(size_t(b) * kMomSlabs + sl) * 12 + c]);
      mom[c] = m / double(HW);
    }
    double S = 0.0, G[3] = {0.0, 0.0, 0.0};
    const float4* pp = partial + size_t(b) * kC3BwdSlabs * C + c;
#pragma unroll 4
    for (int sl = 0; sl < kC3BwdSlabs; ++sl) {
      const float4 v = pp[size_t(sl) * C];
      S += v.x; G[0] += v.y; G[1] += v.z; G[2] += v.w;
    }
    __syncthreads();
    const double* mu = mom;     // E[x]
    const double* Sx = mom + 3;  // E[x x^T]: xx xy xz yy yz zz
    double m1 = 0.0, m2 = 0.0;
    for (int k = g0; k < g0 + cpg; ++k) {
      const double wx = w[k * 3], wy = w[k * 3 + 1], wz = w[k * 3 + 2];
      m1 += wx * mu[0] + wy * mu[1] + wz * mu[2];
      m2 += wx * wx * Sx[0] + 2.0 * wx * wy * Sx[1] + 2.0 * wx * wz * Sx[2] + wy * wy * Sx[3] + 2.0 * wy * wz * Sx[4] + wz * wz * Sx[5];
    }
    const double mean = m1 / cpg;
    const double r = 1.0 / sqrt(fmax(m2 / cpg - mean * mean, 0.0) + double(eps));
    const double T = r * (wc[0] * G[0] + wc[1] * G[1] + wc[2] * G[2] - mean * S);
    gs[c] = gam * S;
    gt[c] = gam * T;
    __syncthreads();
    double s1 = 0.0, s2 = 0.0;
    for (int k = g0; k < g0 + cpg; ++k) { s1 += gs[k]; s2 += gt[k]; }
    s1 *= invN; s2 *= invN;
    const double Sw[3] = {Sx[0] * wc[0] + Sx[1] * wc[1] + Sx[2] * wc[2], Sx[1] * wc[0] + Sx[3] * wc[1] + Sx[4] * wc[2],
                          Sx[2] * wc[0] + Sx[4] * wc[1] + Sx[5] * wc[2]};
#pragma unroll
    for (int j = 0; j < 3; ++j) aw[j] += r * (gam * G[j] - s1 * HW * mu[j] - s2 * r * HW * (Sw[j] - mean * mu[j]));
    ag += T;
    ab += S;
    __syncthreads();  // mom / gs / gt are rewritten for the next image
  }
  if (dw) { dw[c * 3] = float(aw[0] * scale); dw[c * 3 + 1] = float(aw[1] * scale); dw[c * 3 + 2] = float(aw[2] * scale); }
  if (dgamma) dgamma[c] = float(ag * scale);
  if (dbeta) dbeta[c] = float(ab * scale);
}

size_t c3_gn_bwd_scratch_floats(int B, int C) { return size_t(B) * kC3BwdSlabs * C * 4; }

const char* c3_gn_bwd(const float* img4, const float* mom, const float* coef, const float* w, const float* gamma, float eps, int relu, int B, int HW,
                      int C, const void* dy16, int fp16, float scale, float* dw, float* dgamma, float* dbeta, float* partial, cudaStream_t st) {
  if (C % 32 != 0 || C > 1024 || 256 % (C / 8) != 0) return "c3_gn_bwd: C must be a multiple of 32 with C/8 dividing 256";
  const size_t smem = size_t(256 / (C / 8)) * C * sizeof(float4);
  if (launch_k(c3_gn_bwd_partials_kernel, dim3(kC3BwdSlabs, B), dim3(256), smem, st, static_cast<const uint16_t*>(dy16),
               reinterpret_cast<const float4*>(img4), reinterpret_cast<const float4*>(coef), HW, C, relu, fp16,
               reinterpret_cast<float4*>(partial)) != cudaSuccess)
    return "c3_gn_bwd partials launch failed";
  if (launch_k(c3_gn_bwd_finish_kernel, dim3(1), dim3(C), 0, st, reinterpret_cast<const float4*>(partial), mom, w, gamma, eps, B, HW, C, scale, dw,
               dgamma, dbeta) != cudaSuccess)
    return "c3_gn_bwd finish launch failed";
  return nullptr;
}

}  // namespace madm
