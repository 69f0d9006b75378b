// tcgen05 attention kernels for the ConsistentID processors (sm_100a).
//
//  attn_self_kernel   Consistent_AttProcessor core (attention.py:152-159): softmax(scale * Q K^T) V per (sample, head),
//                     flash-style over 128-key tiles, never materialising the [2B*H, N, N] matrix the reference writes.
//  attn_cross_kernel  Consistent_IPAttProcessor core (attention.py:259-279): ONE Q K_cat^T MMA over
//                     K_cat = [77 text keys | pad | 4 id keys | pad] (96 rows), TWO independent softmaxes
//                     (text range / id range), two P V MMAs into separate accumulators, mixed in the epilogue as
//                     O_text / l_text + scale * O_ip / l_ip.
//
// Layouts (all 16-bit, K-major for UMMA):
//   Q, K   [B, N, H, d] views of the projection outputs (row pitch = projection width) - 4-D TMA maps {d, N, H, B},
//          box {64, 128|96}: head dims 40/80/160 are zero-filled by TMA up to the 64-element swizzle row.
//   V^T    [B*H, d, Nkv] (keys contiguous; written transposed by the QKV GEMM epilogue) - 3-D map {Nkv, d, B*H}.
//   P      written by the softmax warps into 128B-swizzled smem (A operand of the second MMA).
// TMEM: S [128 x 128 fp32] at column 0, P*V partial at column 128 (self) / O_text, O_ip (cross).
#pragma once
#include "common.cuh"

namespace cid {

struct AttnArgs {
  int B, H, Nq, Nkv, d;
  float scale_log2;      // d^-0.5 * log2(e)
  void* O;               // [B, Nq, H*d], row pitch ldo elements
  long long ldo;
  int is_bf16;
  int n_text, ip_off, n_ip;   // cross: key ranges [0, n_text) and [ip_off, ip_off + n_ip)
  float ip_scale;
  int vt4d;              // V^T map is the 4-D {64 keys, d, N/64, B*H} view: both 64-key chunks of a tile in ONE TMA instruction
  int causal;            // self (attn_self5_kernel only): query row q sees keys 0..q (CLIP text encoder); 0 for every other caller
  long long* trace;      // debug builds (-DCID_ATTN_TRACE, tools/trace_attn.py): per-tile phase timestamps of the CTAs with blockIdx.y == z == 0
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// write 8 consecutive 16-bit values (one 16-byte chunk) of row r, element column col (multiple of 8, < 64) of a
// [rows x 64] K-major tile stored with the 128-byte swizzle (chunk index XOR (row & 7))
__device__ __forceinline__ void st_sw128(uint8_t* tile, int r, int col, uint4 v) {
  const int chunk = (col >> 3) ^ (r & 7);
  *reinterpret_cast<uint4*>(tile + r * 128 + chunk * 16) = v;
}

constexpr int ATTN_THREADS = 192;

template <int D_PAD>
struct AttnCfg {
  static constexpr int NCH = (D_PAD + 63) / 64;                 // 64-wide head-dim chunks
  static constexpr int STAGES = (D_PAD <= 80) ? 2 : 1;
  static constexpr int Q_BYTES = NCH * 16384;
  static constexpr int K_BYTES = NCH * 16384;                   // per stage
  static constexpr int V_CHUNK = D_PAD * 128;                   // one 64-key chunk of V^T
  static constexpr int V_BYTES = 2 * V_CHUNK;                   // per stage
  static constexpr int P_BYTES = 2 * 16384;
  static constexpr int OFF_K = Q_BYTES;
  static constexpr int OFF_V = OFF_K + STAGES * K_BYTES;
  static constexpr int OFF_P = OFF_V + STAGES * V_BYTES;
  static constexpr int OFF_BAR = OFF_P + P_BYTES;
  static constexpr int TOTAL = OFF_BAR + 256;
  static constexpr int TMEM_COLS = (128 + D_PAD <= 256) ? 256 : 512;
  static constexpr int MIN_CTAS = (TOTAL <= 115000 && TMEM_COLS == 256) ? 2 : 1;
};

__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
// p = 2^x for two fp32 inputs, packed 16-bit result (low half = x0)
template <int BF>
__device__ __forceinline__ uint32_t ex2_pack(float x0, float x1) {
  uint32_t h, p;
  if (BF) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(x1), "f"(x0));
    asm("ex2.approx.ftz.bf16x2 %0, %1;" : "=r"(p) : "r"(h));
  } else {
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(x1), "f"(x0));
    asm("ex2.approx.f16x2 %0, %1;" : "=r"(p) : "r"(h));
  }
  return p;
}
// K-major, NO swizzle, LBO = SBO = 0: all 8x16-byte core matrices alias the 128 bytes at `saddr`
__device__ __forceinline__ uint64_t make_desc_alias128(uint32_t saddr) {
  uint64_t d = 0;
  d |= uint64_t((saddr & 0x3FFFF) >> 4);
  d |= uint64_t(1) << 46;                        // descriptor version; layout type 0 = SWIZZLE_NONE
  return d;
}

// one 32-column chunk of scores -> 16 packed probabilities
template <int BF>
__device__ __forceinline__ void exp_chunk(const uint32_t (&v)[32], float c, float nmc, uint32_t (&pk)[16]) {
#pragma unroll
  for (int i = 0; i < 32; i += 2)
    pk[i >> 1] = ex2_pack<BF>(fmaf(__uint_as_float(v[i]), c, nmc), fmaf(__uint_as_float(v[i + 1]), c, nmc));
}
template <int BF>
__device__ __forceinline__ void exp_chunk_masked(const uint32_t (&v)[32], float c, float nmc, int nvalid, uint32_t (&pk)[16]) {
#pragma unroll
  for (int i = 0; i < 32; i += 2) {
    const float x0 = (i < nvalid) ? fmaf(__uint_as_float(v[i]), c, nmc) : -INFINITY;
    const float x1 = (i + 1 < nvalid) ? fmaf(__uint_as_float(v[i + 1]), c, nmc) : -INFINITY;
    pk[i >> 1] = ex2_pack<BF>(x0, x1);
  }
}

template <int D_PAD>
struct Attn2Cfg : AttnCfg<D_PAD> {
  static constexpr int TMEM_COLS = (128 + D_PAD + 16 <= 256) ? 256 : 512;
  static constexpr int MIN_CTAS = (AttnCfg<D_PAD>::TOTAL <= 115000 && TMEM_COLS == 256) ? 2 : 1;
  static constexpr int OFF_ONES = AttnCfg<D_PAD>::OFF_BAR + 128;      // 128-byte all-ones tile inside the barrier block
};

}  // namespace cid
