// Host-side interface of the tcgen05 implicit-GEMM kernel family (gemm_tc.cu).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace madm {

enum Act : int { ACT_NONE = 0, ACT_SILU = 1, ACT_GEGLU = 2, ACT_RELU = 3 };

// One K-segment of the A operand: an NHWC bf16 activation tensor read through `ntaps` shifted TMA boxes
// (implicit im2col).  K extent of the segment = ntaps * C.  A plain [M,K] matrix is {B=1,H=1,W=M,C=K,ntaps=1}.
struct GemmASeg {
  const void* ptr = nullptr;  // bf16, [Bt, H, W, ld] with C <= ld used channels
  int Bt = 1;                 // images in the tensor (for stride-2 phase tensors: 4*B, see taps[].b_off)
  int H = 1, W = 1, C = 0;    // C % 64 == 0
  int ld = 0;                 // channel pitch in elements (0 -> C)
  int ntaps = 1;              // 1 (1x1 / linear) or 9 (3x3)
  int8_t dx[9] = {0}, dy[9] = {0};
  int b_off[9] = {0};         // image offset added per tap (space-to-depth phase * B)
};

struct GemmDesc {
  GemmASeg seg[2];
  int nseg = 1;
  int M = 0;                  // output rows = B*H*W of the output grid (== grid of seg[0])
  int N = 0;                  // output columns (weights rows)
  const void* w = nullptr;    // bf16 [Nw, Ktot] K-major; Ktot = sum_seg ntaps*C ; Nw >= N (Nw = 2N for GEGLU-interleaved)
  int Nw = 0;
  int ldw = 0;                // weight row pitch in elements (0 -> Ktot)
  const float* bias = nullptr;      // [N] (GEGLU: [2N] tile-interleaved) or null
  const float* rowbias = nullptr;   // [nimg, N] added per image (time-embedding projection) or null
  int rows_per_img = 1;             // H*W of the output grid (for rowbias)
  int ld_rowbias = 0;               // row pitch of rowbias (0 -> N)
  const float* residual = nullptr;  // fp32 [M, ldr] or null (may alias out_f32); with res16 a 16-bit [M, ldr] tensor (may alias out_bf16)
  int ldr = 0;
  int res16 = 0;
  float* out_f32 = nullptr;         // fp32 [M, ldo32] or null
  int ldo32 = 0;
  void* out_bf16 = nullptr;         // bf16 [M, ldo16] or null
  int ldo16 = 0;
  int act = ACT_NONE;
  float alpha = 1.0f;               // scales the accumulator before bias
  int bn = 0;                       // N tile (0 = auto)
  int fp16 = 0;                     // operand / 16-bit output dtype: 0 = bf16, 1 = fp16
  int s2d_H = 0, s2d_W = 0;         // >0: write out_bf16 in space-to-depth layout [4][B][H/2][W/2][N] (operand of a stride-2 conv)
  int pair = 0;                     // CTA pairs (cta_group::2): 0 auto, 1 force, -1 never
  int mt = 0;                       // M sub-tiles per CTA tile for the 128-wide N tile: 0 auto, 1, or 2 (256-row tiles)
  int splits = 1;                   // split-K factor (>1: raw fp32 partial outputs at out_f32 + split * split_stride)
  long split_stride = 0;
  float* colstats = nullptr;        // optional [ceil(M/32)][N][2] per-column (sum, sumsq) of the outputs per 32-row block (fused GN statistics)
};

// Kernel parameters, filled once by gemm_prepare (tensor maps encoded) and passed as they are on every launch
struct GemmParams {
  CUtensorMap tmA[2];
  CUtensorMap tmB;
  CUtensorMap tmR;   // TMA_EPI_RES_H16: the out-of-place fp32 residual (box 32 x 32, 128B swizzle), loaded per chunk into the warp's staging
  CUtensorMap tmO;   // output tensor map of the TMA-store epilogue (box 32 columns x 32 rows; fp32 with 128B swizzle or 16-bit with 64B swizzle)
  int tma_epi;       // TMA_EPI_*: 0 = coalesced-store epilogue, else the epilogue hands 32x32 tiles to cp(.reduce).async.bulk.tensor
  int nseg;
  int kchunks[2];    // 64-wide K chunks per segment
  int cpt[2];        // chunks per tap
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
};

struct GemmLaunch {  // prepared launch: the kernel parameters and the instantiation that runs them
  GemmParams p;
  int bn = 128;
  int mt = 1;
  int pair = 0;              // launched as cta_group::2 pairs (cluster of 2): tiles are 2*mt*128 rows
  dim3 grid;
  size_t smem = 0;
};

// Returns nullptr on success, else a static error string.  gemm_prepare runs every check; gemm_launch only launches.
const char* gemm_prepare(const GemmDesc& d, GemmLaunch* out);
const char* gemm_launch(const GemmLaunch& l, cudaStream_t stream);

// Encodes a tiled TMA tensor map (the driver's cuTensorMapEncodeTiled, looked up once).  Returns nullptr on success, else an error string
// that starts with `op` (the calling operator's name).
const char* encode_tensor_map(CUtensorMap* tm, const char* op, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                              const cuuint32_t* box, CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_UINT16,
                              CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B);

}  // namespace madm
