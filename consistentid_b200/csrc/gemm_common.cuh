// tcgen05 GEMM / implicit-GEMM 3x3 convolution for the ConsistentID UNet hot path (sm_100a).
//
//   C[M, N] = epilogue( A[M, K] * B[N, K]^T )        16-bit inputs (fp16 | bf16), fp32 accumulate in TMEM
//
// Shared argument block / constants of the GEMM kernels (the kernel itself: gemm_tc2.cuh).
//
// A-operand addressing modes:
//   GEMM        2-D map {K, M}; optional second source along K (virtual channel concat: 1x1 shortcut on cat([h, skip]))
//   CONV3x3     4-D map {C, W, H, N} over an NHWC activation: tap (ky,kx) = the same box shifted by (kx-1, ky-1);
//               TMA zero-fills out-of-bounds rows/cols = the conv's zero padding
//   CONV3x3 s2  5-D map {C, W/2, H/2, 4, N} over a phase-split copy of the input (see phase_split kernel)
#pragma once
#include "common.cuh"

namespace cid {

enum EpiMode : int { EPI_STORE = 0, EPI_GEGLU = 1, EPI_QKV = 2, EPI_GELU = 3, EPI_QUICK_GELU = 4, EPI_STORE_TMA = 5, EPI_STORE_TMA2 = 6 };   // EPI_STORE_TMA2: the same with two staging tiles (residual prefetched a tile ahead)   // EPI_STORE_TMA: kernel-internal flavour (store epilogue staged through smem + TMA)   // EPI_GELU: C = gelu_erf(acc + bias) (CLIP MLP fc1)   // EPI_QUICK_GELU: C = quick_gelu(acc + bias) (OpenAI CLIP text MLP fc1)
enum AMode : int { A_GEMM = 0, A_CONV = 1, A_CONV_S2 = 2 };

struct GemmArgs {
  int M, N;
  int kblocks_a1, kblocks_a2;  // 64-wide k-blocks per tap taken from A1 / A2
  int taps;                    // 1 or 9
  int a_mode;
  int W, H, NB;                // conv: OUTPUT geometry
  int TW, TH, TN;              // conv tile (pixels) TW*TH*TN <= 128
  int tiles_x, tiles_y;
  void* C;
  long long ldc;
  const void* bias;
  const void* residual;
  long long ldr;
  const void* rowbias;         // [M / rows_per_group, ld_rowbias]
  int rows_per_group;
  long long ld_rowbias;
  int epi;
  int is_bf16;
  void* Vt;                    // EPI_QKV: V^T [B*heads, hdim, ntok]
  int n_split, heads, hdim, ntok;
  float out_scale;
  // GroupNorm statistics of the OUTPUT, fused into the epilogue (EPI_STORE only): per (sample, channel) sum and sum of squares of the stored
  // values are accumulated into chan_stats[(row / stats_rows) * N + col][2] (fp32, zeroed by the caller).  Every 128-row tile must lie inside
  // one sample (checked on the host).  NULL: off.
  float* chan_stats;
  int stats_rows;
  // LayerNorm folded into the GEMMs on either side of it (no standalone LayerNorm pass):
  //   producer  row_stats != NULL (EPI_STORE): per ROW sum and sum of squares of the stored values are added to row_stats[row][2] (fp32, zeroed
  //             by the caller; the row's N columns may be spread over several tiles / warps);
  //   consumer  ln_stats != NULL (any flavour): A holds the UN-normalised rows x, B = W . diag(gamma), bias = b + W . beta, ln_colsum[c] =
  //             sum_k B[c, k]; the epilogue forms  LN(x) W^T + b = rstd_r (x_r . B_c - mean_r colsum_c) + bias_c  with mean / rstd of row r
  //             from ln_stats[r] = {sum, sum of squares} over ln_width elements.
  float* row_stats;
  const float* ln_stats;
  const float* ln_colsum;
  float ln_eps;
  int ln_width;
  long long* trace;        // debug builds (-DCID_GEMM_TRACE, tools/trace_gemm.py): per-tile phase timestamps of the first 16 CTAs
};

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_THREADS = 192;

template <int BN, int STAGES>
struct GemmSmem {
  static constexpr int A_BYTES = GEMM_BM * 128;
  static constexpr int B_BYTES = BN * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;  // + barriers + alignment slack
};

// exact (erf) GELU, erf by Abramowitz-Stegun 7.1.28: erf(t) = 1 - (1 + a1 t + ... + a6 t^6)^-16, |err| <= 3e-7
// (far below 16-bit output rounding) - ~15 instructions instead of erff's ~40, the GEGLU epilogue is ALU-bound
__device__ __forceinline__ float gelu_erf(float x) {
  const float t = fabsf(x) * 0.70710678118654752f;
  float p = fmaf(t, 0.0000430638f, 0.0002765672f);
  p = fmaf(t, p, 0.0001520143f);
  p = fmaf(t, p, 0.0092705272f);
  p = fmaf(t, p, 0.0422820123f);
  p = fmaf(t, p, 0.0705230784f);
  p = fmaf(t, p, 1.0f);
  p = p * p; p = p * p; p = p * p; p = p * p;
  float rp;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rp) : "f"(p));
  const float e = 1.0f - rp;
  return 0.5f * x * (1.0f + copysignf(e, x));
}
// QuickGELU of the OpenAI CLIP checkpoints (hidden_act "quick_gelu"): x * sigmoid(1.702 x), fp32
__device__ __forceinline__ float quick_gelu(float x) { return x / (1.0f + __expf(-1.702f * x)); }

}  // namespace cid
