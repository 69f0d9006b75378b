// HBM-bound kernels of the ConsistentID UNet hot path (sm_100a): GroupNorm statistics / apply(+SiLU, + virtual
// channel concat), LayerNorm, nearest-2x upsample, stride-2 phase split, layout converters, sinusoidal timestep
// embedding, skinny (M <= 64 rows) linears for the time-embedding MLPs, cross-attention K/V packing and the fused
// CFG-combine + scheduler step.  All activations are NHWC / [tokens, C] row-major, 16-bit; 128-bit vector accesses.
#pragma once
#include "common.cuh"

namespace cid {

// x * sigmoid(x) with one MUFU.EX2 + one MUFU.RCP (the IEEE division of `x / (1 + e)` costs ~10 extra instructions per element and made
// the GroupNorm+SiLU pass ALU-bound: 21 M elements per level-0 tensor); relative error ~2 ulp of fp32, far below the 16-bit output rounding
// (x * sigmoid(x) as h + h * tanh(h) with ONE MUFU op (tanh.approx) instead of ex2 + rcp was measured: -4 % on the GroupNorm-apply launches
// (1.50 -> 1.44 ms per SD1.5 iteration) - the kernel is not MUFU-bound - so the more accurate form stays.)
__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.f + __expf(-x)); }

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8], int bf) {
  float2 a = unpack16(u.x, bf), b = unpack16(u.y, bf), c = unpack16(u.z, bf), d = unpack16(u.w, bf);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8], int bf) {
  return make_uint4(pack16(f[0], f[1], bf), pack16(f[2], f[3], bf), pack16(f[4], f[5], bf), pack16(f[6], f[7], bf));
}

// ------------------------------------------------------------------------------------------------ GroupNorm
// Statistics over x = cat([x1 (C1 ch), x2 (C2 ch)], channel) in NHWC; sums[n, g, {sum, sumsq}] (fp32, pre-zeroed).
// grid (slabs, NB); each block streams a slab of pixels with 16-byte loads, keeps per-channel partial sums in
// registers, reduces them through smem to per-group sums and issues 2 atomics per group.
__global__ void __launch_bounds__(256)
gn_stats_kernel(const uint16_t* __restrict__ x1, int C1, const uint16_t* __restrict__ x2, int C2, int HW, int groups,
                float* __restrict__ sums, int bf) {
  griddep_wait();                  // PDL (no-op for a normal launch)
  __shared__ float sh[2 * 2048];                 // per-channel partial sums of this block's channel chunk
  const int C = C1 + C2, V = C / 8;              // 8-channel vectors per pixel
  const int n = blockIdx.y;
  const int vbeg = blockIdx.z * 256;             // this block covers vectors [vbeg, vbeg + Vb) (<= 2048 channels)
  const int Vb = min(V - vbeg, 256);
  const int cbeg = vbeg * 8, Cb = Vb * 8;
  const int tpp = blockDim.x / Vb;               // pixels processed in parallel
  const int vec = vbeg + threadIdx.x % Vb, prow = threadIdx.x / Vb;
  for (int i = threadIdx.x; i < 2 * 2048; i += blockDim.x) sh[i] = 0.f;
  __syncthreads();
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { s[i] = 0.f; q[i] = 0.f; }
  if (prow < tpp) {
    const int c0 = vec * 8;
    const bool first = c0 < C1;
    const uint16_t* src = first ? x1 + (size_t)n * HW * C1 + c0 : x2 + (size_t)n * HW * C2 + (c0 - C1);
    const int pitch = first ? C1 : C2;
    // 4 independent 16-byte loads in flight per thread (the pass is pure HBM streaming)
    const int pstride = gridDim.x * tpp;
    int p = blockIdx.x * tpp + prow;
    for (; p + 3 * pstride < HW; p += 4 * pstride) {
      uint4 u[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) u[k] = *reinterpret_cast<const uint4*>(src + (size_t)(p + k * pstride) * pitch);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float f[8]; unpack8(u[k], f, bf);
#pragma unroll
        for (int i = 0; i < 8; ++i) { s[i] += f[i]; q[i] += f[i] * f[i]; }
      }
    }
    for (; p < HW; p += pstride) {
      uint4 u = *reinterpret_cast<const uint4*>(src + (size_t)p * pitch);
      float f[8]; unpack8(u, f, bf);
#pragma unroll
      for (int i = 0; i < 8; ++i) { s[i] += f[i]; q[i] += f[i] * f[i]; }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) { atomicAdd(&sh[c0 - cbeg + i], s[i]); atomicAdd(&sh[2048 + c0 - cbeg + i], q[i]); }
  }
  __syncthreads();
  const int cpg = C / groups;
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    const int lo = max(g * cpg, cbeg), hi = min((g + 1) * cpg, cbeg + Cb);
    if (lo >= hi) continue;
    float a = 0.f, b = 0.f;
    for (int c = lo; c < hi; ++c) { a += sh[c - cbeg]; b += sh[2048 + c - cbeg]; }
    atomicAdd(&sums[((size_t)n * groups + g) * 2], a);
    atomicAdd(&sums[((size_t)n * groups + g) * 2 + 1], b);
  }
}

// Streaming part of the GroupNorm apply kernels: y = [silu](x * scale[c] + shift[c]) over one sample, per-channel affine in smem
// (aff[0..C) scale, aff[C..2C) shift).  Four 16-byte loads are in flight per thread before the first one is consumed.
__device__ __forceinline__ void gn_stream(const uint16_t* __restrict__ x1n, int C1, const uint16_t* __restrict__ x2n, int C2,
                                          uint16_t* __restrict__ yn, const float* aff, long long per_sample, int do_silu, int bf) {
  const int C = C1 + C2;
  const unsigned V = unsigned(C / 8), n = unsigned(per_sample);            // (a sample has < 2^32 vectors: 32-bit index math)
  const unsigned stride = gridDim.x * blockDim.x;
  constexpr int U = 4;
  for (unsigned i0 = blockIdx.x * blockDim.x + threadIdx.x; i0 < n; i0 += U * stride) {
    uint4 u[U];
    int c0[U];
    size_t pix[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const unsigned i = i0 + k * stride;
      if (i < n && i >= i0) {
        const unsigned px = i / V;
        pix[k] = px;
        c0[k] = int(i - px * V) * 8;
        u[k] = (c0[k] < C1) ? *reinterpret_cast<const uint4*>(x1n + pix[k] * C1 + c0[k])
                            : *reinterpret_cast<const uint4*>(x2n + pix[k] * C2 + (c0[k] - C1));
      }
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      if (i0 + k * stride < n && i0 + k * stride >= i0) {
        float f[8]; unpack8(u[k], f, bf);
        const float4 s0 = *reinterpret_cast<const float4*>(aff + c0[k]), s1 = *reinterpret_cast<const float4*>(aff + c0[k] + 4);
        const float4 h0 = *reinterpret_cast<const float4*>(aff + C + c0[k]), h1 = *reinterpret_cast<const float4*>(aff + C + c0[k] + 4);
        const float sc[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
        const float sh[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float v = fmaf(f[e], sc[e], sh[e]);
          f[e] = do_silu ? silu_f(v) : v;
        }
        *reinterpret_cast<uint4*>(yn + pix[k] * C + c0[k]) = pack8(f, bf);
      }
    }
  }
}

// y = [silu]((x - mean) * rstd * gamma + beta), x = cat([x1, x2]) NHWC -> y NHWC with C = C1 + C2 channels
__global__ void __launch_bounds__(256)
gn_apply_kernel(const uint16_t* __restrict__ x1, int C1, const uint16_t* __restrict__ x2, int C2, int HW, int groups,
                const float* __restrict__ sums, const uint16_t* __restrict__ gamma, const uint16_t* __restrict__ beta,
                float eps, int do_silu, uint16_t* __restrict__ y, float* __restrict__ zero_next, int bf) {
  griddep_wait();                  // PDL (no-op for a normal launch)
  // grid (slabs, NB): a block serves ONE sample, so the per-channel affine (scale = rstd*gamma, shift = beta - mean*scale)
  // is built once in smem and the streaming loop is one FMA (+ SiLU) per element.
  extern __shared__ float aff[];                 // [2 * C]
  const int C = C1 + C2, V = C / 8, cpg = C / groups;
  const int n = blockIdx.y;
  const float inv_n = 1.f / (float(HW) * float(cpg));
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int g = c / cpg;
    const float sm = sums[((size_t)n * groups + g) * 2], sq = sums[((size_t)n * groups + g) * 2 + 1];
    const float mean = sm * inv_n;
    const float rstd = rsqrtf(fmaxf(sq * inv_n - mean * mean, 0.f) + eps);
    const float sc = rstd * load16(gamma, c, bf);
    aff[c] = sc;
    aff[C + c] = load16(beta, c, bf) - mean * sc;
  }
  // the statistics buffer the NEXT GroupNorm accumulates into (its last reader finished before this grid started)
  if (zero_next != nullptr && blockIdx.x == 0)
    for (int i = threadIdx.x; i < groups * 2; i += blockDim.x) zero_next[(size_t)n * groups * 2 + i] = 0.f;
  __syncthreads();
  const long long per_sample = (long long)HW * V;
  const uint16_t* x1n = x1 + (size_t)n * HW * C1;
  const uint16_t* x2n = x2 ? x2 + (size_t)n * HW * C2 : nullptr;
  uint16_t* yn = y + (size_t)n * HW * C;
  gn_stream(x1n, C1, x2n, C2, yn, aff, per_sample, do_silu, bf);
}

// Same apply, statistics given PER CHANNEL by the producers' epilogues (gemm_tc2.cuh "fused GroupNorm statistics"): sums1[n, c, {sum, sumsq}]
// for the C1 channels of x1, sums2 likewise for x2 (virtual concat: the 32 groups do not align with the concat boundary, SURVEY Appendix D).
// Each block folds the channel sums of its sample into group statistics (smem), then streams like gn_apply_kernel.
__global__ void __launch_bounds__(256)
gn_apply_ch_kernel(const uint16_t* __restrict__ x1, int C1, const float* __restrict__ sums1, const uint16_t* __restrict__ x2, int C2,
                   const float* __restrict__ sums2, int HW, int groups, const uint16_t* __restrict__ gamma, const uint16_t* __restrict__ beta,
                   float eps, int do_silu, uint16_t* __restrict__ y, int bf) {
  griddep_wait();
  extern __shared__ float aff[];                 // [2 * C] affine | [2 * C] channel sums | [2 * groups] group mean / rstd
  const int C = C1 + C2, V = C / 8, cpg = C / groups;
  float* chs = aff + 2 * C;
  float* grp = aff + 4 * C;
  const int n = blockIdx.y;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float* src = (c < C1) ? sums1 + ((size_t)n * C1 + c) * 2 : sums2 + ((size_t)n * C2 + (c - C1)) * 2;
    chs[2 * c] = src[0]; chs[2 * c + 1] = src[1];
  }
  __syncthreads();
  const float inv_n = 1.f / (float(HW) * float(cpg));
  for (int gi = threadIdx.x; gi < groups; gi += blockDim.x) {
    float sm = 0.f, sq = 0.f;
    for (int c = gi * cpg; c < (gi + 1) * cpg; ++c) { sm += chs[2 * c]; sq += chs[2 * c + 1]; }
    const float mean = sm * inv_n;
    grp[2 * gi] = mean;
    grp[2 * gi + 1] = rsqrtf(fmaxf(sq * inv_n - mean * mean, 0.f) + eps);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int gi = c / cpg;
    const float sc = grp[2 * gi + 1] * load16(gamma, c, bf);
    aff[c] = sc;
    aff[C + c] = load16(beta, c, bf) - grp[2 * gi] * sc;
  }
  __syncthreads();
  const long long per_sample = (long long)HW * V;
  const uint16_t* x1n = x1 + (size_t)n * HW * C1;
  const uint16_t* x2n = x2 ? x2 + (size_t)n * HW * C2 : nullptr;
  uint16_t* yn = y + (size_t)n * HW * C;
  gn_stream(x1n, C1, x2n, C2, yn, aff, per_sample, do_silu, bf);
}

// ------------------------------------------------------------------------------------------------ GroupNorm, small tensors: ONE pass
// One CTA per (sample, group): its HW x (C / groups) slab (5-40 KB at the 8x8 / 16x16 levels) is loaded once into registers (up to VPT
// 16-byte vectors per thread), mean and variance (two-pass over the registers, fp32) reduced across the block, affine + SiLU applied, stored.
// Replaces gn_stats + gn_apply where the statistics cannot ride on the producer's epilogue (a 128-row tile spans two samples at HW = 64):
// two launches of ~20 us each - block prologues and a grid-wide dependency for 2.6 MB of data - become one short launch.
// Needs groups that do not straddle the concat boundary and 8-channel vectors that do not straddle groups (host-checked).
constexpr int GN_SMALL_THREADS = 512;
template <int VPT>
__global__ void __launch_bounds__(GN_SMALL_THREADS)
gn_small_kernel(const uint16_t* __restrict__ x1, int C1, const uint16_t* __restrict__ x2, int C2, int HW, int groups,
                const uint16_t* __restrict__ gamma, const uint16_t* __restrict__ beta, float eps, int do_silu, uint16_t* __restrict__ y, int bf) {
  griddep_wait();
  __shared__ float red[2][GN_SMALL_THREADS / 32];
  const int C = C1 + C2, cpg = C / groups, vpp = cpg / 8;              // vectors per pixel inside the group
  const int n = blockIdx.y, gi = blockIdx.x, c0 = gi * cpg;
  const int total = HW * vpp;
  const bool first = c0 < C1;
  const uint16_t* src = first ? x1 + (size_t)n * HW * C1 + c0 : x2 + (size_t)n * HW * C2 + (c0 - C1);
  const int pitch = first ? C1 : C2;
  float f[VPT][8];
  int pix[VPT], vec[VPT];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < VPT; ++j) {
    const int idx = threadIdx.x + j * GN_SMALL_THREADS;
    pix[j] = idx / vpp; vec[j] = idx - pix[j] * vpp;
    if (idx < total) {
      unpack8(__ldg(reinterpret_cast<const uint4*>(src + (size_t)pix[j] * pitch + vec[j] * 8)), f[j], bf);
#pragma unroll
      for (int e = 0; e < 8; ++e) s += f[j][e];
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) f[j][e] = 0.f;
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  auto block_sum = [&](float v, int slot) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[slot][warp] = v;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < GN_SMALL_THREADS / 32; ++w) t += red[slot][w];
    return t;
  };
  const float inv_n = 1.f / (float(HW) * float(cpg));
  const float mean = block_sum(s, 0) * inv_n;
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < VPT; ++j) {
    if (threadIdx.x + j * GN_SMALL_THREADS < total) {
#pragma unroll
      for (int e = 0; e < 8; ++e) { const float d = f[j][e] - mean; q = fmaf(d, d, q); }
    }
  }
  const float rstd = rsqrtf(block_sum(q, 1) * inv_n + eps);
  uint16_t* yn = y + (size_t)n * HW * C + c0;
#pragma unroll
  for (int j = 0; j < VPT; ++j) {
    if (threadIdx.x + j * GN_SMALL_THREADS < total) {
      float g8[8], b8[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(gamma + c0 + vec[j] * 8)), g8, bf);
      unpack8(__ldg(reinterpret_cast<const uint4*>(beta + c0 + vec[j] * 8)), b8, bf);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float v = fmaf((f[j][e] - mean) * rstd, g8[e], b8[e]);
        f[j][e] = do_silu ? silu_f(v) : v;
      }
      *reinterpret_cast<uint4*>(yn + (size_t)pix[j] * C + vec[j] * 8) = pack8(f[j], bf);
    }
  }
}

// ------------------------------------------------------------------------------------------------ LayerNorm
// LPR lanes share a row (8 / 16 / 32 for C <= 320 / 640 / 2048), i.e. a warp normalises 32 / LPR rows at once and every lane has up to VPL
// independent 16-byte loads in flight (5 for the UNet widths 320 / 640 / 1280) - the one-row-per-warp first version had at most two and ran
// at 40 % of the HBM bandwidth.  Warps loop over row groups (grid-stride).  Two-pass variance in fp32.
template <int LPR, int VPL>
__global__ void __launch_bounds__(256, 3)
layernorm_kernel(const uint16_t* __restrict__ x, const uint16_t* __restrict__ gamma, const uint16_t* __restrict__ beta,
                 uint16_t* __restrict__ y, long long rows, int C, float eps, int bf) {
  griddep_wait();                  // PDL (no-op for a normal launch)
  constexpr int RPW = 32 / LPR;                                   // rows per warp
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sub = lane % LPR, rsel = lane / LPR;
  const int V = C / 8;
  const float inv_c = 1.f / float(C);
  const long long wstride = (long long)gridDim.x * (blockDim.x >> 5) * RPW;
  for (long long row = ((long long)blockIdx.x * (blockDim.x >> 5) + warp) * RPW + rsel; row < rows; row += wstride) {   // (rsel keeps LPR-groups together)
    float f[VPL][8];
    uint4 u[VPL];
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const int v = sub + j * LPR;
      if (v < V) u[j] = *reinterpret_cast<const uint4*>(x + row * C + v * 8);
    }
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const int v = sub + j * LPR;
      if (v < V) {
        unpack8(u[j], f[j], bf);
#pragma unroll
        for (int k = 0; k < 8; ++k) s += f[j][k];
      }
    }
#pragma unroll
    for (int o = LPR / 2; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s * inv_c;
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const int v = sub + j * LPR;
      if (v < V) {
#pragma unroll
        for (int k = 0; k < 8; ++k) { const float d = f[j][k] - mean; q += d * d; }
      }
    }
#pragma unroll
    for (int o = LPR / 2; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = rsqrtf(q * inv_c + eps);
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      const int v = sub + j * LPR;
      if (v < V) {
        float g8[8], b8[8], o8[8];                        // gamma / beta: a few hundred bytes, L1-resident after the first row group
        unpack8(__ldg(reinterpret_cast<const uint4*>(gamma + v * 8)), g8, bf); unpack8(__ldg(reinterpret_cast<const uint4*>(beta + v * 8)), b8, bf);
#pragma unroll
        for (int k = 0; k < 8; ++k) o8[k] = (f[j][k] - mean) * rstd * g8[k] + b8[k];
        *reinterpret_cast<uint4*>(y + row * C + v * 8) = pack8(o8, bf);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ resampling / layout
// nearest 2x: x [NB, H, W, C] -> y [NB, 2H, 2W, C]
__global__ void __launch_bounds__(256)
upsample2x_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int NB, int H, int W, int V, long long total_out_vec) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total_out_vec; i += (long long)gridDim.x * blockDim.x) {
    const int v = int(i % V);
    long long p = i / V;
    const int ox = int(p % (2 * W)); p /= (2 * W);
    const int oy = int(p % (2 * H));
    const int n = int(p / (2 * H));
    y[i] = x[(((long long)n * H + (oy >> 1)) * W + (ox >> 1)) * V + v];
  }
}
// stride-2 phase split: x [NB, H, W, C] -> y [NB, 4 (py*2+px), H/2, W/2, C]; y[n,ph,y',x'] = x[n, 2y'+py, 2x'+px]
__global__ void __launch_bounds__(256)
phase_split_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int NB, int H, int W, int V, long long total_vec) {
  const int H2 = H / 2, W2 = W / 2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total_vec; i += (long long)gridDim.x * blockDim.x) {
    const int v = int(i % V);
    long long p = i / V;
    const int xx = int(p % W2); p /= W2;
    const int yy = int(p % H2); p /= H2;
    const int ph = int(p % 4);
    const int n = int(p / 4);
    y[i] = x[(((long long)n * H + (2 * yy + (ph >> 1))) * W + (2 * xx + (ph & 1))) * V + v];
  }
}
// NCHW [NB, Cin, H, W] (16-bit) -> NHWC with CP (>= Cin, multiple of 8) channels, zero padded, times `scale`
__global__ void __launch_bounds__(256)
nchw_to_nhwc_pad_kernel(const uint16_t* __restrict__ x, uint16_t* __restrict__ y, int NB, int Cin, int HW, int CP,
                        const float* __restrict__ scale_ptr, int bf) {
  const float sc = scale_ptr ? *scale_ptr : 1.f;
  const long long total = (long long)NB * HW * (CP / 8);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = int(i % (CP / 8));
    const long long pix = i / (CP / 8);
    const int n = int(pix / HW), p = int(pix % HW);
    float f[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = v * 8 + k;
      f[k] = (c < Cin) ? load16(x, ((size_t)n * Cin + c) * HW + p, bf) * sc : 0.f;
    }
    *reinterpret_cast<uint4*>(y + pix * CP + v * 8) = pack8(f, bf);
  }
}
// [NB*HW, ld] rows (first Cout columns valid) -> NCHW [NB, Cout, H, W]
__global__ void __launch_bounds__(256)
rows_to_nchw_kernel(const uint16_t* __restrict__ x, int ld, uint16_t* __restrict__ y, int NB, int Cout, int HW) {
  const long long total = (long long)NB * Cout * HW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int p = int(i % HW);
    const int c = int((i / HW) % Cout);
    const int n = int(i / ((long long)HW * Cout));
    y[i] = x[((size_t)n * HW + p) * ld + c];
  }
}
// y += x (16-bit, vectorised); used for ControlNet residual injection
__global__ void __launch_bounds__(256)
add_inplace_kernel(uint4* __restrict__ y, const uint4* __restrict__ x, long long total_vec, int bf) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total_vec; i += (long long)gridDim.x * blockDim.x) {
    float a[8], b[8]; unpack8(y[i], a, bf); unpack8(x[i], b, bf);
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] += b[k];
    y[i] = pack8(a, bf);
  }
}

// y = silu(y) (ControlNet conditioning-embedding convs)
__global__ void __launch_bounds__(256)
silu_inplace_kernel(uint4* __restrict__ y, long long total_vec, int bf) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total_vec; i += (long long)gridDim.x * blockDim.x) {
    float a[8]; unpack8(y[i], a, bf);
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = silu_f(a[k]);
    y[i] = pack8(a, bf);
  }
}
// CLIP text embeddings: out[b*Lp + i] = tok[ids[b, i]] + pos[i] for i < L, zero rows for L <= i < Lp (fp32 sum, one rounding, as the 16-bit
// torch add); an id outside [0, V) contributes a zero token row and is never dereferenced
__global__ void __launch_bounds__(256)
embed_tokens_kernel(const long long* __restrict__ ids, int L, int Lp, const uint4* __restrict__ tok, long long V, const uint4* __restrict__ pos,
                    uint4* __restrict__ out, int CV, long long total_vec, int bf) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total_vec; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / CV;
    const int c = int(i - row * CV);
    const int b = int(row / Lp), t = int(row - (long long)b * Lp);
    if (t >= L) { out[i] = make_uint4(0u, 0u, 0u, 0u); continue; }
    const long long id = ids[(long long)b * L + t];
    float a[8], p[8];
    unpack8(pos[(long long)t * CV + c], p, bf);
    if (id >= 0 && id < V) {
      unpack8(tok[id * CV + c], a, bf);
#pragma unroll
      for (int k = 0; k < 8; ++k) a[k] += p[k];
      out[i] = pack8(a, bf);
    } else {
      out[i] = pack8(p, bf);
    }
  }
}

// inpaint latent blending after a scheduler step (pipelines/StableDIffusionControlNetInpaint_ConsistentID.py:437-449):
//   x = (1 - m) * (ca * image_latents + cn * noise) + m * x,   {ca, cn} = blend_table[step] = add_noise coefficients of the
//   NEXT timestep ((1, 0) on the last step).  x: fp32 master latents [B,4,HW]; mask [B,1,HW] (1 = repaint).
__global__ void __launch_bounds__(256)
inpaint_blend_kernel(float* __restrict__ x, uint16_t* __restrict__ x16, const float* __restrict__ img, const float* __restrict__ noise,
                     const float* __restrict__ mask, int B, int HW, const float* __restrict__ blend_table, const int* __restrict__ step_ptr, int bf) {
  const float ca = blend_table[2 * (*step_ptr)], cn = blend_table[2 * (*step_ptr) + 1];
  const long long total = (long long)B * 4 * HW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int p = int(i % HW);
    const int b = int(i / (4LL * HW));
    const float m = mask[(size_t)b * HW + p];
    const float v = (1.f - m) * (ca * img[i] + cn * noise[i]) + m * x[i];
    x[i] = v;
    store16(x16, i, v, bf);
  }
}

// ------------------------------------------------------------------------------------------------ embeddings
// diffusers get_timestep_embedding(flip_sin_to_cos=True, downscale_freq_shift=0): out[r] = [cos(t*f), sin(t*f)], f_i = 1e4^(-i/half)
// t values: t_ptr[r * t_stride] (t_stride 0 -> one scalar broadcast to all rows).  Output rounded to 16-bit at
// out[r*ld + col0 ..], like `t_emb.to(sample.dtype)`.
__global__ void __launch_bounds__(128)
timestep_embed_kernel(const float* __restrict__ t_ptr, int t_stride, int rows, int dim, uint16_t* __restrict__ out,
                      long long ld, int col0, int bf) {
  const int half = dim / 2;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < rows * half; i += gridDim.x * blockDim.x) {
    const int r = i / half, k = i % half;
    const float t = t_ptr[(size_t)r * t_stride];
    const float freq = expf(-9.210340371976184f * float(k) / float(half));   // ln(10000)
    const float e = t * freq;
    store16(out, (size_t)r * ld + col0 + k, cosf(e), bf);
    store16(out, (size_t)r * ld + col0 + half + k, sinf(e), bf);
  }
}

// y[M, N] (+)= act_in(x)[M, K] . W[N, K]^T + b     for tiny M (time-embedding MLPs, per-resnet temb projections, embedding producers)
// act_in: 0 identity, 1 SiLU, 2 GELU(erf).  One warp per output column; x staged in smem in 16-row slabs with 16-byte copies; the weight
// stream is software-pipelined - four 16-byte loads per lane are in flight before the FMAs of the first one start (the embedding producers
// stream 250-600 MB of weights through this kernel on <= 10 rows; the un-pipelined first version was bound by the load -> FMA chain).
__global__ void __launch_bounds__(256)
skinny_linear2_kernel(const uint16_t* __restrict__ x, long long ldx, const uint16_t* __restrict__ w, const uint16_t* __restrict__ bias,
                      uint16_t* __restrict__ y, long long ldy, int M, int N, int K, int act_in, int accumulate, int bf, int slab) {
  extern __shared__ uint16_t xs[];               // [slab][K], slab <= 16
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col = blockIdx.x * (blockDim.x >> 5) + warp;
  const int V = K / 8;
  const bool x_vec = (ldx % 8 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  for (int m0 = 0; m0 < M; m0 += slab) {
    const int mrows = min(slab, M - m0);
    __syncthreads();
    for (int r = 0; r < mrows; ++r) {
      const uint16_t* xr = x + (size_t)(m0 + r) * ldx;
      for (int v = threadIdx.x; v < V; v += blockDim.x) {
        float f[8];
        if (x_vec) unpack8(*reinterpret_cast<const uint4*>(xr + v * 8), f, bf);
        else {
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = load16(xr, v * 8 + e, bf);
        }
        if (act_in == 1) {
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = silu_f(f[e]);
        } else if (act_in == 2) {
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = 0.5f * f[e] * (1.f + erff(f[e] * 0.70710678118654752f));
        }
        *reinterpret_cast<uint4*>(xs + (size_t)r * K + v * 8) = pack8(f, bf);
      }
    }
    __syncthreads();
    if (col < N) {
      float acc[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) acc[r] = 0.f;
      const uint16_t* wr = w + (size_t)col * K;
      for (int k0 = lane * 8; k0 < K; k0 += 1024) {
        uint4 wv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int k = k0 + u * 256;
          wv[u] = (k < K) ? *reinterpret_cast<const uint4*>(wr + k) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int k = k0 + u * 256;
          if (k < K) {
            float wf[8]; unpack8(wv[u], wf, bf);
#pragma unroll
            for (int r = 0; r < 16; ++r) {
              if (r < mrows) {
                float xf[8]; unpack8(*reinterpret_cast<const uint4*>(xs + (size_t)r * K + k), xf, bf);
#pragma unroll
                for (int e = 0; e < 8; ++e) acc[r] += wf[e] * xf[e];
              }
            }
          }
        }
      }
#pragma unroll
      for (int r = 0; r < 16; ++r) {
#pragma unroll
        for (int o = 16; o; o >>= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
      }
      if (lane == 0) {
        const float bv = bias ? load16(bias, col, bf) : 0.f;
        for (int r = 0; r < mrows; ++r) {
          float v = acc[r] + bv;
          const size_t o = (size_t)(m0 + r) * ldy + col;
          if (accumulate) v += load16(y, o, bf);
          store16(y, o, v, bf);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ cross-attn K/V packing
// K_cat[b, 96, C]: rows [0,77) = text keys, [80,84) = id keys, rest 0.   Vt_cat[b*H + h, d, 96]: same columns, transposed.
__global__ void __launch_bounds__(256)
pack_cross_kv_kernel(const uint16_t* __restrict__ k_text, const uint16_t* __restrict__ v_text, const uint16_t* __restrict__ k_ip,
                     const uint16_t* __restrict__ v_ip, uint16_t* __restrict__ k_cat, uint16_t* __restrict__ vt_cat,
                     int B, int C, int heads, int n_text, int n_ip, int ip_off, int krows) {
  const long long total = (long long)B * krows * C;
  const int d = C / heads;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % C);
    const int row = int((i / C) % krows);
    const int b = int(i / ((long long)C * krows));
    uint16_t kv = 0, vv = 0;
    if (row < n_text) { kv = k_text[((size_t)b * n_text + row) * C + c]; vv = v_text[((size_t)b * n_text + row) * C + c]; }
    else if (row >= ip_off && row < ip_off + n_ip) {
      kv = k_ip[((size_t)b * n_ip + (row - ip_off)) * C + c]; vv = v_ip[((size_t)b * n_ip + (row - ip_off)) * C + c];
    }
    k_cat[i] = kv;
    const int h = c / d, dd = c % d;
    vt_cat[(((size_t)b * heads + h) * d + dd) * krows + row] = vv;
  }
}

// ------------------------------------------------------------------------------------------------ CFG + scheduler step
// One fused pass per denoising step (pipline_StableDiffusion_ConsistentID.py:537-540, 560-571):
//   eps   = eps_u + g * (eps_c - eps_u)                      eps rows: [2B*HW, ld_eps], first 4 columns valid
//   x0    = kx * x + ke * eps                                (kept for multistep solvers)
//   x'    = cx * x + ce * eps + cp * x0_prev                 (DDIM / Euler / DPM-Solver++(2M) are all of this form)
//   next UNet input (both CFG halves, NHWC, CP channels, zero padded) = x' * in_scale_next
// coef[step] = {cx, ce, cp, kx, ke, in_scale_next, 0, 0}; step index read from device memory (CUDA-graph friendly).
// Master latents x are fp32 [B, 4, HW] (NCHW); a 16-bit copy is written for the API surface.
__global__ void __launch_bounds__(256)
cfg_sched_step_kernel(const uint16_t* __restrict__ eps, int ld_eps, float* __restrict__ x, float* __restrict__ x0_prev,
                      uint16_t* __restrict__ x16, uint16_t* __restrict__ next_in, int CP, int B, int HW, float guidance,
                      const float* __restrict__ coef_table, const int* __restrict__ step_ptr, int bf) {
  const float* cf = coef_table + 8 * (*step_ptr);
  const float cx = cf[0], ce = cf[1], cp = cf[2], kx = cf[3], ke = cf[4], sc = cf[5];
  const long long total = (long long)B * HW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = int(i / HW), p = int(i % HW);
    const uint2 eu = *reinterpret_cast<const uint2*>(eps + ((size_t)b * HW + p) * ld_eps);
    const uint2 ec = *reinterpret_cast<const uint2*>(eps + ((size_t)(B + b) * HW + p) * ld_eps);
    float2 u01 = unpack16(eu.x, bf), u23 = unpack16(eu.y, bf), c01 = unpack16(ec.x, bf), c23 = unpack16(ec.y, bf);
    const float uu[4] = {u01.x, u01.y, u23.x, u23.y}, cc[4] = {c01.x, c01.y, c23.x, c23.y};
    float nx[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) nx[k] = 0.f;
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
      const size_t o = ((size_t)b * 4 + ch) * HW + p;
      const float e = uu[ch] + guidance * (cc[ch] - uu[ch]);
      const float xv = x[o];
      const float x0 = kx * xv + ke * e;
      const float xn = cx * xv + ce * e + cp * x0_prev[o];
      x0_prev[o] = x0;
      x[o] = xn;
      store16(x16, o, xn, bf);
      nx[ch] = xn * sc;
    }
    if (next_in) {
      const uint4 v = pack8(nx, bf);
      uint4* d0 = reinterpret_cast<uint4*>(next_in + ((size_t)b * HW + p) * CP);
      uint4* d1 = reinterpret_cast<uint4*>(next_in + ((size_t)(B + b) * HW + p) * CP);
      d0[0] = v; d1[0] = v;                      // channels >= 8 stay zero (buffer zeroed once at allocation)
    }
  }
}

// first-step helper: fp32 master latents [B,4,HW] -> UNet input NHWC (both CFG halves), times in_scale of step 0
__global__ void __launch_bounds__(256)
latents_to_input_kernel(const float* __restrict__ x, uint16_t* __restrict__ next_in, int CP, int B, int HW,
                        const float* __restrict__ coef_table, const int* __restrict__ step_ptr, int nsteps, int vec4_only, int bf) {
  int st = step_ptr ? *step_ptr : 0;
  if (st >= nsteps) st = nsteps - 1;
  const float sc = coef_table[8 * st + 6];       // in_scale of the step about to run
  const long long total = (long long)B * HW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = int(i / HW), p = int(i % HW);
    float nx[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) nx[k] = 0.f;
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) nx[ch] = x[((size_t)b * 4 + ch) * HW + p] * sc;
    const uint4 v = pack8(nx, bf);
    if (vec4_only) {                             // 9-channel inpaint UNet: channels 4..8 (mask, masked latents) are static, keep them
      reinterpret_cast<uint2*>(next_in + ((size_t)b * HW + p) * CP)[0] = make_uint2(v.x, v.y);
      reinterpret_cast<uint2*>(next_in + ((size_t)(B + b) * HW + p) * CP)[0] = make_uint2(v.x, v.y);
    } else {
      reinterpret_cast<uint4*>(next_in + ((size_t)b * HW + p) * CP)[0] = v;
      reinterpret_cast<uint4*>(next_in + ((size_t)(B + b) * HW + p) * CP)[0] = v;
    }
  }
}

// end-of-step bookkeeping inside the CUDA graph: step += 1; t = timesteps[step] (clamped)
__global__ void advance_step_kernel(int* __restrict__ step, float* __restrict__ t_dev, const float* __restrict__ ts_table, int n) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const int s = *step + 1;
    *step = s;
    *t_dev = ts_table[s < n ? s : n - 1];
  }
}

}  // namespace cid
