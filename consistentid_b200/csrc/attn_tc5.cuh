// attn_self5_kernel - flash self-attention, v5 (same operands / results as v3 / v4).
//
// Measured (tools/microbench_softmax.cu, profiles/r02_microbench_softmax.txt): tcgen05.ld moves ~800-960 B/clk/SM (a whole 128 x 128
// fp32 score tile in < 100 cycles) - reading S is NOT a limiter; the exponentials are: 15.9 ex2/clk/SM whatever the packing
// (ex2.approx.f16x2 is two MUFU.EX2 in SASS), i.e. >= 1030 cycles per score tile, more than twice the tensor-pipe time of the tile.
// v3 / v4 nevertheless take ~2000 cycles per tile: between two tiles the softmax warps of BOTH co-resident CTAs wait for tensor
// results at the same moments (P is single-buffered, so tile j+1 cannot write its probabilities before P.V_j has drained P_j; the
// CTAs share the MUFU fairly, finish together, and then both sit behind the same serial MMA queue).  v5 removes those waits:
//   * P is DOUBLE-buffered in shared memory: the softmax of tile j+1 writes P[(j+1)&1] while P.V_j still reads P[j&1]; the only wait
//     left on P.V is two tiles back (never blocks in steady state) or the rare O / l rescale;
//   * the whole 128-score row is pulled into registers at once (4 x tcgen05.ld.x32, < 100 cycles) and S is released immediately, so
//     S_{j+1} = Q K_{j+1}^T runs under the exponentials of tile j;
//   * the smem for the second P buffer comes from the K / V rings: one stage each for head dims <= 64 (two CTAs per SM; K_{j+1} is
//     fetched as soon as S_j has been issued, V_{j+1} as soon as P.V_j retires - both a full softmax time before they are needed).
// Row max first, exact per tile (64 max3), lazy rescaling of O / l in TMEM as in v3 (FlashAttention-4).
#pragma once
#include "attn_common.cuh"

namespace cid {

#ifndef CID_TMEM_ST_DEFINED
#define CID_TMEM_ST_DEFINED
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

constexpr float ATTN_RESCALE_THRESHOLD = 8.0f;      // log2 units: P <= 2^8, exact range of fp16 / bf16
#endif

template <int D_PAD>
struct Attn5Cfg {
  static constexpr int NCH = (D_PAD + 63) / 64;                 // 64-wide head-dim chunks
  static constexpr int Q_BYTES = NCH * 16384;
  static constexpr int K_BYTES = NCH * 16384;                   // per stage
  static constexpr int V_CHUNK = D_PAD * 128;                   // one 64-key chunk of V^T
  static constexpr int V_BYTES = 2 * V_CHUNK;                   // per stage
  static constexpr int P_BYTES = 2 * 16384;                     // per buffer, two buffers
  static constexpr int TMEM_COLS = (128 + D_PAD + 16 <= 256) ? 256 : 512;
  // two CTAs per SM (head dims <= 64) leave ~113 KB each: one K / V stage; otherwise two stages when they fit
  // (228 KB per SM, 1 KB reserved per CTA: two CTAs fit when each asks for <= 115 200 bytes)
  static constexpr bool SMALL = TMEM_COLS == 256 && (Q_BYTES + K_BYTES + V_BYTES + 2 * P_BYTES + 384 <= 115200);
  static constexpr int STAGES = SMALL ? 1 : ((Q_BYTES + 2 * (K_BYTES + V_BYTES) + 2 * P_BYTES + 384 <= 227 * 1024) ? 2 : 1);
  static constexpr int OFF_K = Q_BYTES;
  static constexpr int OFF_V = OFF_K + STAGES * K_BYTES;
  static constexpr int OFF_P = OFF_V + STAGES * V_BYTES;
  static constexpr int OFF_BAR = OFF_P + 2 * P_BYTES;
  static constexpr int OFF_ONES = OFF_BAR + 128;                // 128-byte all-ones tile (row sums by MMA)
  static constexpr int TOTAL = OFF_BAR + 256 + 128;
  static constexpr int MIN_CTAS = SMALL ? 2 : 1;
};

constexpr int ATTN5_THREADS = 224;       // warp 0 TMA (Q, K), warp 1 MMA, warps 2-5 softmax, warp 6 TMA (V^T)

template <int D_PAD, int BF>
__global__ void __launch_bounds__(ATTN5_THREADS, Attn5Cfg<D_PAD>::MIN_CTAS)
attn_self5_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                  const __grid_constant__ CUtensorMap tmVt, const AttnArgs a) {
  using C = Attn5Cfg<D_PAD>;
  constexpr int STAGES = C::STAGES;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t sbase = smem_u32(smem_raw);
  if ((sbase & 1023u) != 0) { if (threadIdx.x == 0) printf("cid: attn smem base not 1024-aligned\n"); __trap(); }
  const uint32_t bar0 = sbase + C::OFF_BAR;
  const uint32_t q_full = bar0;
  auto k_full = [&](int s) { return bar0 + 8u * (1 + s); };
  auto k_empty = [&](int s) { return bar0 + 8u * (1 + STAGES + s); };
  auto v_full = [&](int s) { return bar0 + 8u * (1 + 2 * STAGES + s); };
  auto v_empty = [&](int s) { return bar0 + 8u * (1 + 3 * STAGES + s); };
  const uint32_t s_full = bar0 + 8u * (1 + 4 * STAGES);
  const uint32_t s_free = s_full + 8u;
  auto p_full = [&](int b) { return s_full + 16u + 8u * b; };      // P[b] written by the 128 softmax threads
  auto pv_full = [&](int b) { return s_full + 32u + 8u * b; };     // the P.V that read P[b] (and everything before it) retired
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_raw + C::OFF_BAR + 8 * (7 + 4 * STAGES));
  static_assert(8 * (8 + 4 * 2) <= 128, "barrier block overlaps the ones tile");

  const int warp = warp_id(), lane = lane_id();
  const int q0 = blockIdx.x * 128, h = blockIdx.y, b = blockIdx.z;
  // causal: key tiles above the diagonal are skipped by all three roles alike (a disagreement on T would leave an mbarrier waiting forever)
  const int T = a.causal ? min((a.Nkv + 127) / 128, int(blockIdx.x) + 1) : (a.Nkv + 127) / 128;

  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmVt); }
  if (warp == 1) {
    if (lane == 0) {
      mbar_init(q_full, 1);
      for (int s = 0; s < STAGES; ++s) { mbar_init(k_full(s), 1); mbar_init(k_empty(s), 1); mbar_init(v_full(s), 1); mbar_init(v_empty(s), 1); }
      mbar_init(s_full, 1); mbar_init(s_free, 128);
      for (int i = 0; i < 2; ++i) { mbar_init(p_full(i), 128); mbar_init(pv_full(i), 1); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc<C::TMEM_COLS>(smem_u32(const_cast<uint32_t*>(tmem_slot)));
  }
  if (warp == 2) {
    reinterpret_cast<uint32_t*>(smem_raw + C::OFF_ONES)[lane] = BF ? 0x3F803F80u : 0x3C003C00u;
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_S = tmem, tmem_O = tmem + 128, tmem_L = tmem + 128 + D_PAD;
  griddep_wait();                  // PDL: the prologue above overlaps the predecessor's tail

  // Producer / issuer warps are WARP-CONVERGED with the single-thread instructions under elect_one() (see gemm_tc2.cuh).
  if (warp == 0) {
    // ============================================================ TMA producer: Q, then the K stream
    if (elect_one()) {
      mbar_expect_tx(q_full, C::Q_BYTES);
#pragma unroll
      for (int ch = 0; ch < C::NCH; ++ch) tma_load_4d(sbase + ch * 16384, &tmQ, q_full, ch * 64, q0, h, b);
    }
    __syncwarp();
    int stage = 0; uint32_t phase = 0;
    for (int j = 0; j < T; ++j) {
      mbar_wait(k_empty(stage), phase ^ 1u);
      const uint32_t kb = k_full(stage), dst = sbase + C::OFF_K + stage * C::K_BYTES;
      if (elect_one()) {
        mbar_expect_tx(kb, C::K_BYTES);
#pragma unroll
        for (int ch = 0; ch < C::NCH; ++ch) tma_load_4d(dst + ch * 16384, &tmK, kb, ch * 64, j * 128, h, b);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
  } else if (warp == 6) {
    // ============================================================ TMA producer: the V^T stream (own warp: a K tile must never queue behind
    // the V tile of the previous key block, whose buffer is only released when P.V retires, late in the tile)
    int stage = 0; uint32_t phase = 0;
    const int bh = b * a.H + h;
    for (int j = 0; j < T; ++j) {
      mbar_wait(v_empty(stage), phase ^ 1u);
      const uint32_t vb = v_full(stage), dst = sbase + C::OFF_V + stage * C::V_BYTES;
      if (elect_one()) {
        mbar_expect_tx(vb, C::V_BYTES);
        tma_load_3d(dst, &tmVt, vb, j * 128, 0, bh);
        tma_load_3d(dst + C::V_CHUNK, &tmVt, vb, j * 128 + 64, 0, bh);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
    if (elect_one()) griddep_launch_dependents();
    __syncwarp();
  } else if (warp == 1) {
    // ============================================================ MMA issuer
    const uint32_t idesc_s = make_idesc(128, 128, BF);
    const uint32_t idesc_pv = make_idesc(128, D_PAD, BF);
    const uint32_t idesc_l = make_idesc(128, 16, BF);
    const uint64_t ones_desc = make_desc_alias128(sbase + C::OFF_ONES);
    const uint32_t q_lo = desc_lo(sbase), k_lo = desc_lo(sbase + C::OFF_K), v_lo = desc_lo(sbase + C::OFF_V), p_lo = desc_lo(sbase + C::OFF_P);
    auto issue_S = [&](int stage) {
      const uint32_t kl = k_lo + uint32_t(stage * C::K_BYTES) / 16;
      const uint32_t ke = k_empty(stage);
      if (elect_one()) {
#pragma unroll
        for (int ch = 0; ch < C::NCH; ++ch) {
          const int ksteps = (D_PAD - ch * 64 >= 64) ? 4 : (D_PAD - ch * 64) / 16;
#pragma unroll
          for (int kk = 0; kk < ksteps; ++kk)
            umma_ss(tmem_S, desc_make(q_lo + ch * 1024 + kk * 2), desc_make(kl + ch * 1024 + kk * 2), idesc_s, (ch | kk) ? 1u : 0u);
        }
        umma_commit(s_full);
        umma_commit(ke);
      }
      __syncwarp();
    };
    mbar_wait(q_full, 0);
    int stage = 0; uint32_t phase = 0;
    int nstage = 0; uint32_t nphase = 0;
    mbar_wait(k_full(0), 0);
    tc_fence_after();
    issue_S(0);
    if (++nstage == STAGES) { nstage = 0; nphase ^= 1u; }
    for (int j = 0; j < T; ++j) {
      if (j + 1 < T) {
        mbar_wait(k_full(nstage), nphase);
        mbar_wait(s_free, uint32_t(j & 1));              // the softmax warps hold S_j in registers
        tc_fence_after();
        issue_S(nstage);
        if (++nstage == STAGES) { nstage = 0; nphase ^= 1u; }
      }
      const int pb = j & 1;
      mbar_wait(p_full(pb), uint32_t((j >> 1) & 1));     // P_j in smem buffer pb, O / l rescaled if needed
      mbar_wait(v_full(stage), phase);
      tc_fence_after();
      const uint32_t vl = v_lo + uint32_t(stage * C::V_BYTES) / 16;
      const uint32_t pl = p_lo + uint32_t(pb * C::P_BYTES) / 16;
      const uint32_t acc0 = j > 0 ? 1u : 0u;
      const uint32_t pvb = pv_full(pb), veb = v_empty(stage);
      if (elect_one()) {
#pragma unroll
        for (int kc = 0; kc < 2; ++kc)
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            const uint64_t pdesc = desc_make(pl + kc * 1024 + kk * 2);
            const uint32_t acc = (kc | kk) ? 1u : acc0;
            umma_ss(tmem_O, pdesc, desc_make(vl + kc * (C::V_CHUNK / 16) + kk * 2), idesc_pv, acc);
            umma_ss(tmem_L, pdesc, ones_desc, idesc_l, acc);
          }
        umma_commit(pvb);
        umma_commit(veb);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
  } else {
    // ============================================================ softmax + output (warps 2..5, one query row per thread)
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_off = uint32_t(quarter * 32) << 16;
    const float c = a.scale_log2;
    float m_use = -INFINITY;                              // row max baked into O, l and used for P
    // parity of the latest completed phase of pv_full(b) after tile t's P.V: ((t >> 1) & 1)
    auto wait_pv = [&](int t) { mbar_wait(pv_full(t & 1), uint32_t((t >> 1) & 1)); };

#ifdef CID_ATTN_TRACE
    const bool tr = a.trace != nullptr && blockIdx.y == 0 && blockIdx.z == 0 && warp == 2 && lane == 0 && blockIdx.x < 64;
    auto stamp = [&](int j_, int e) { if (tr && j_ < 64) a.trace[((size_t)blockIdx.x * 64 + j_) * 8 + e] = clock64(); };
    if (tr) { unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); a.trace[((size_t)blockIdx.x * 64) * 8 + 7] = smid; }
#else
    auto stamp = [&](int, int) {};
#endif
    for (int j = 0; j < T; ++j) {
      // keys of this tile the row may see: the ragged tail, and under the causal mask keys <= the row's own index (only the diagonal tile
      // cuts: j < blockIdx.x gives >= 129); every row keeps key j * 128 at least, so no row sums to l = 0
      int kvalid = a.Nkv - j * 128;
      if (a.causal) kvalid = min(kvalid, q0 + r - j * 128 + 1);
      stamp(j, 0);
      mbar_wait(s_full, uint32_t(j & 1));
      tc_fence_after();
      stamp(j, 1);
      uint32_t v[128];
      {
        uint32_t (&v0)[32] = *reinterpret_cast<uint32_t (*)[32]>(&v[0]);
        uint32_t (&v1)[32] = *reinterpret_cast<uint32_t (*)[32]>(&v[32]);
        uint32_t (&v2)[32] = *reinterpret_cast<uint32_t (*)[32]>(&v[64]);
        uint32_t (&v3)[32] = *reinterpret_cast<uint32_t (*)[32]>(&v[96]);
        tmem_ld_x32(tmem_S + lane_off + 0, v0);
        tmem_ld_x32(tmem_S + lane_off + 32, v1);
        tmem_ld_x32(tmem_S + lane_off + 64, v2);
        tmem_ld_x32(tmem_S + lane_off + 96, v3);
        tmem_ld_wait();
      }
      tc_fence_before();
      mbar_arrive(s_free);                                // S_j lives in registers now: S_{j+1} may be computed
      stamp(j, 2);
      if (kvalid < 128) {
#pragma unroll
        for (int i = 0; i < 128; ++i) if (i >= kvalid) v[i] = 0xff800000u;       // -inf
      }
      // (eight independent max chains: one 64-deep dependent chain of 3-input max cost ~500 cycles per tile in the phase trace)
      float m8[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) m8[q] = max3(__uint_as_float(v[q * 16]), __uint_as_float(v[q * 16 + 1]), __uint_as_float(v[q * 16 + 2]));
#pragma unroll
      for (int i = 3; i < 15; i += 2) {
#pragma unroll
        for (int q = 0; q < 8; ++q) m8[q] = max3(m8[q], __uint_as_float(v[q * 16 + i]), __uint_as_float(v[q * 16 + i + 1]));
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) m8[q] = fmaxf(m8[q], __uint_as_float(v[q * 16 + 15]));
      const float mx = fmaxf(max3(max3(m8[0], m8[1], m8[2]), max3(m8[3], m8[4], m8[5]), m8[6]), m8[7]);
      const float m_new = fmaxf(m_use, mx);
      const bool need = (m_new - m_use) * c > ATTN_RESCALE_THRESHOLD;            // also true on the first tile (m_use = -inf)
      if (j > 0 && __any_sync(0xffffffffu, need)) {
        wait_pv(j - 1);                                   // every P.V issued so far retired: O / l quiescent
        tc_fence_after();
        const float f = need ? fast_exp2((m_use - m_new) * c) : 1.0f;
#pragma unroll
        for (int cc = 0; cc < D_PAD + 16; cc += 16) {     // O columns then the 16 row-sum columns (contiguous in TMEM)
          uint32_t t[16];
          tmem_ld_x16(tmem_O + lane_off + cc, t);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) t[i] = __float_as_uint(__uint_as_float(t[i]) * f);
          tmem_st_x16(tmem_O + lane_off + cc, t);
        }
        tmem_st_wait();
      }
      if (need) m_use = m_new;
      const float nmc = -m_use * c;
      stamp(j, 3);
      if (j >= 2) wait_pv(j - 2);                         // P[j & 1] was last read by P.V_{j-2}: long retired in steady state
      stamp(j, 4);
      uint8_t* sP = smem_raw + C::OFF_P + (j & 1) * C::P_BYTES;
      // P = 2^((s - m_use) c), packed, straight into the swizzled A-operand tile
#pragma unroll
      for (int cc = 0; cc < 128; cc += 32) {
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 32; i += 2)
          pk[i >> 1] = ex2_pack<BF>(fmaf(__uint_as_float(v[cc + i]), c, nmc), fmaf(__uint_as_float(v[cc + i + 1]), c, nmc));
        uint8_t* tile = sP + (cc >> 6) * 16384;
        const int col = cc & 63;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          st_sw128(tile, r, col + q * 8, make_uint4(pk[q * 4], pk[q * 4 + 1], pk[q * 4 + 2], pk[q * 4 + 3]));
      }
      stamp(j, 5);
      fence_proxy_async();
      tc_fence_before();
      mbar_arrive(p_full(j & 1));
      stamp(j, 6);
    }
    // ---- normalise and store
    wait_pv(T - 1);
    tc_fence_after();
    float l;
    {
      uint32_t t[16];
      tmem_ld_x16(tmem_L + lane_off, t);
      tmem_ld_wait();
      l = __uint_as_float(t[0]);
    }
    const float inv = 1.f / l;
    const bool row_ok = q0 + r < a.Nq;
    uint16_t* dst = reinterpret_cast<uint16_t*>(a.O) + ((long long)b * a.Nq + q0 + r) * a.ldo + h * a.d;
#pragma unroll
    for (int cc = 0; cc < D_PAD; cc += 16) {
      uint32_t t[16];
      tmem_ld_x16(tmem_O + lane_off + cc, t);
      tmem_ld_wait();
      if (row_ok) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          if (cc + q * 8 < a.d) {
            uint4 u;
            u.x = pack16(__uint_as_float(t[q * 8 + 0]) * inv, __uint_as_float(t[q * 8 + 1]) * inv, BF);
            u.y = pack16(__uint_as_float(t[q * 8 + 2]) * inv, __uint_as_float(t[q * 8 + 3]) * inv, BF);
            u.z = pack16(__uint_as_float(t[q * 8 + 4]) * inv, __uint_as_float(t[q * 8 + 5]) * inv, BF);
            u.w = pack16(__uint_as_float(t[q * 8 + 6]) * inv, __uint_as_float(t[q * 8 + 7]) * inv, BF);
            *reinterpret_cast<uint4*>(dst + cc + q * 8) = u;
          }
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc<C::TMEM_COLS>(tmem); }
}

}  // namespace cid
