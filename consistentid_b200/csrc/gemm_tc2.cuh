// Persistent tcgen05 GEMM / implicit-GEMM conv3x3 (arguments: gemm_common.cuh).
//
// One CTA per SM loops over output tiles (tile = blockIdx.x + i*gridDim.x, N-tile fastest so CTAs running at the same
// time share the activation (A) tile in L2).  Roles (320 threads):
//   warp 0      TMA producer - keeps the STAGES-deep smem ring full ACROSS tile boundaries
//   warp 1      TMEM allocator (512 columns = two accumulators) + tcgen05.mma issuer; alternates accumulators so the
//               main loop of tile i+1 overlaps the epilogue of tile i
//   warps 2-17  epilogue: four warps per TMEM lane quarter, each draining a quarter of the tile's columns in 16-column
//               tcgen05.ld chunks; residual rows are prefetched into registers BEFORE waiting for the accumulator and the
//               bias slice of the tile is staged once in smem, so no global-load latency sits between TMEM and the stores
//
// Tail balancing (split-K): a launch of T tiles on G CTAs runs floor(T/G) whole-tile rounds; the remaining T mod G tiles would keep
// G - (T mod G) SMs idle for a full tile time (M=4096/1024 levels of SD1.5: 160 or 40 tiles, SDXL N=1280 GEMMs: 320 tiles = 2.16
// waves).  When the K loop is long enough each tail tile is cut into `ksplit` K-ranges handled by different CTAs: every unit publishes
// its fp32 partial accumulator to a workspace ([chunk][row][16] floats, coalesced), bumps the tile's arrival counter, and the LAST
// arriver adds the other partials into its own TMEM accumulator (tcgen05.ld -> add -> tcgen05.st) and runs the normal fused epilogue.
// No unit ever waits for another one, so there is no ordering requirement between CTAs.
#pragma once
#include <type_traits>
#include "elementwise.cuh"
#include "gemm_common.cuh"

namespace cid {

// 16 epilogue warps: four per TMEM lane quarter, each draining a quarter of the tile's columns.  The epilogue of the small-K GEMMs is
// latency-bound (ncu, profiles/r02_ncu_outproj_sd15_*: IPC 0.07 per warp - residual loads, TMEM loads, instruction fetch), not issue-bound:
// with eight warps (two per scheduler) a 128 x 160 tile took ~14 k cycles against 1.7 k of tensor work.
#ifndef CID_GEMM_EPI_WARPS
#define CID_GEMM_EPI_WARPS 16                                // (8 = the round-1 layout, kept for A/B builds: tools/build_variant.sh epi8 -DCID_GEMM_EPI_WARPS=8)
#endif
constexpr int GEMM2_EPI_WARPS = CID_GEMM_EPI_WARPS;
constexpr int GEMM2_EPI_THREADS = GEMM2_EPI_WARPS * 32;
constexpr int GEMM2_THREADS = 64 + GEMM2_EPI_THREADS;
constexpr int GEMM2_PARTS = GEMM2_EPI_WARPS / 4;            // column ranges per lane quarter

template <int BN, int STAGES, int TMA_OUT = 0>            // TMA_OUT: number of 128 x BN staging tiles of the TMA-store flavours (0, 1 or 2)
struct Gemm2Smem {
  static constexpr int A_BYTES = GEMM_BM * 128;
  static constexpr int B_BYTES = BN * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
  static constexpr int BIAS_OFF = BAR_OFF + 256;             // 2 x BN floats
  static constexpr int FLAG_OFF = BIAS_OFF + 2 * BN * 4;     // split-K "last arriver" flag
  static constexpr int STAT_OFF = FLAG_OFF + 16;             // 2 x [sum | sumsq] x BN floats: per-tile column statistics (fused GroupNorm stats)
  static constexpr int CS_OFF = STAT_OFF + 2 * 2 * BN * 4;   // 2 x BN floats: column sums of the gamma-scaled weights (folded LayerNorm)
  // TMA-store flavour: the 128 x BN 16-bit output tile (and, before it, the residual tile) staged as BN/32 boxes of [128 rows x 64 B], 64B-swizzled
  static constexpr int OUT_OFF = (CS_OFF + 2 * BN * 4 + 1023) / 1024 * 1024;
  static constexpr int OUT_TILE = GEMM_BM * BN * 2;
  static constexpr int OUT_BYTES = TMA_OUT * OUT_TILE;
  static constexpr int TOTAL = OUT_OFF + OUT_BYTES + 1024;
};

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(GEMM2_EPI_THREADS) : "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st16_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Column sums over the 32 rows held by the lanes of a warp: in v[16] (one row per lane), out: the sum of column
// col_of_lane(lane) in every lane (lanes 2k and 2k+1 hold the same column).  16 shuffles instead of 16 x 5.
__device__ __forceinline__ int colsum_col_of_lane(int lane) { return ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1); }
__device__ __forceinline__ float warp_colsum16(float (&s)[16], int lane) {
  {
    const bool hi = lane & 16;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float send = hi ? s[i] : s[i + 8], keep = hi ? s[i + 8] : s[i];
      s[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
  }
  {
    const bool hi = lane & 8;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float send = hi ? s[i] : s[i + 4], keep = hi ? s[i + 4] : s[i];
      s[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
  }
  {
    const bool hi = lane & 4;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float send = hi ? s[i] : s[i + 2], keep = hi ? s[i + 2] : s[i];
      s[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
  }
  {
    const bool hi = lane & 2;
    const float send = hi ? s[0] : s[1], keep = hi ? s[1] : s[0];
    s[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  return s[0] + __shfl_xor_sync(0xffffffffu, s[0], 1);
}

// Work list of one CTA: `full_iters` whole tiles (tile = blockIdx.x + i*gridDim.x), then at most one tail item: a whole tail tile
// (ksplit <= 1, blockIdx.x < tail_tiles) or K-range `split` of tail tile blockIdx.x / ksplit.
struct GemmSched {
  int full_iters, tail_tiles, ksplit;
  float* ws;        // split-K partials: [tail tile][split][BN/16 chunks][128 rows][16] fp32
  int* counters;    // [tail tile] arrival counters, zero between launches
};
struct GemmWork { int tile, kb0, kb1, split, tail_idx; };

// EPI (epilogue flavour: EPI_STORE covers the plain / GELU / fused-statistics stores, EPI_GEGLU, EPI_QKV) and BF (0 fp16, 1 bf16) are
// compile-time: the generic kernel was 41 k SASS instructions at BN = 256 (every flavour x both 16-bit types, fully unrolled) and ncu showed
// instruction-fetch stalls (`no_instruction` 2.0-3.5 per issue) on the epilogue-bound GEMMs; a specialised instance holds only its own path.
// LEAN (TMA-store flavours): the epilogue is compiled WITHOUT the per-sample row bias, the fused GroupNorm statistics and the GELU - the profile of
// the transformer GEMMs (bias, residual, output scale, LayerNorm row statistics / folded LayerNorm).  With every optional feature compiled in, a
// 16-column chunk of the drain was ~1 000 SASS instructions, much of it if-converted (executed, then discarded by FSEL): ~2 500 cycles of
// drain per 128x160 tile on the K = C GEMMs whose epilogue is their critical path (profiles/r02_trace_gemm_epilogue_dbl.txt).
template <int BN, int STAGES, int EPI, int BF, bool LEAN = false>
__global__ void __launch_bounds__(GEMM2_THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
                const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC, const GemmArgs g, const int n_tiles,
                const GemmSched sched) {
  constexpr bool TMAO = EPI == EPI_STORE_TMA || EPI == EPI_STORE_TMA2;   // store flavour with the output (and residual) tile staged through shared memory
  constexpr bool DBL = EPI == EPI_STORE_TMA2;                  // two staging tiles: tile i works in buffer i & 1, the residual of tile i+1 is copied a tile ahead
  constexpr bool STOREF = EPI == EPI_STORE || TMAO;
  static_assert(BN % 32 == 0 || BN == 16, "column split");
  constexpr int ACC_STRIDE = 256;                              // TMEM column offset between the two accumulators
  using SM = Gemm2Smem<BN, STAGES, DBL ? 2 : (TMAO ? 1 : 0)>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + SM::BAR_OFF;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto acc_full = [&](int b) { return bar_base + 8u * (2 * STAGES + b); };
  auto acc_empty = [&](int b) { return bar_base + 8u * (2 * STAGES + 2 + b); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_gen + SM::BAR_OFF + 8 * (2 * STAGES + 4));
  float* bias_s = reinterpret_cast<float*>(smem_gen + SM::BIAS_OFF);
  float* stat_s = reinterpret_cast<float*>(smem_gen + SM::STAT_OFF);
  float* cs_s = reinterpret_cast<float*>(smem_gen + SM::CS_OFF);

  const int warp = warp_id();
  const int lane = lane_id();
  const int kb_per_tap = g.kblocks_a1 + g.kblocks_a2;
  const int num_kb = g.taps * kb_per_tap;
  const int n_work = sched.full_iters + ((int)blockIdx.x < (sched.ksplit > 1 ? sched.tail_tiles * sched.ksplit : sched.tail_tiles) ? 1 : 0);
  auto get_work = [&](int it) -> GemmWork {
    if (it < sched.full_iters) return GemmWork{int(blockIdx.x) + it * int(gridDim.x), 0, num_kb, -1, 0};
    const int base = sched.full_iters * int(gridDim.x);
    if (sched.ksplit <= 1) return GemmWork{base + int(blockIdx.x), 0, num_kb, -1, 0};
    const int t = int(blockIdx.x) / sched.ksplit, sp = int(blockIdx.x) - t * sched.ksplit;
    return GemmWork{base + t, sp * num_kb / sched.ksplit, (sp + 1) * num_kb / sched.ksplit, sp, t};
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA1);
    if (g.kblocks_a2 > 0) tma_prefetch_desc(&tmA2);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
      for (int b = 0; b < 2; ++b) { mbar_init(acc_full(b), 1); mbar_init(acc_empty(b), GEMM2_EPI_THREADS); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc<512>(smem_u32(const_cast<uint32_t*>(tmem_slot)));
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // prologue above touched only shared memory / TMEM / descriptors: it may overlap the predecessor's tail (PDL)
  griddep_wait();
#ifdef CID_GEMM_TRACE
  // role 0 = epilogue thread 0, 1 = MMA warp, 2 = producer; [role][cta < 16][tile iteration < 64][8 events]
  auto gstamp = [&](int role, int it_, int e, long long val = -1) {
    if (g.trace != nullptr && blockIdx.x < 16 && it_ < 64) g.trace[(((size_t)role * 16 + blockIdx.x) * 64 + it_) * 8 + e] = val < 0 ? clock64() : val;
  };
#else
  auto gstamp = [&](int, int, int, long long = -1) {};
#endif

  auto tile_origin = [&](int mt, int& tn0, int& ty0, int& tx0) {
    const int tx = mt % g.tiles_x;
    const int rest = mt / g.tiles_x;
    tx0 = tx * g.TW; ty0 = (rest % g.tiles_y) * g.TH; tn0 = (rest / g.tiles_y) * g.TN;
  };

  // Role code is WARP-CONVERGED: all 32 lanes run the loops and poll the mbarriers, the single-thread instructions (TMA, tcgen05.mma,
  // tcgen05.commit) sit in `if (elect_one())` blocks whose operands were computed outside, by the whole warp.  Writing the roles as
  // `if (lane == 0) { ...loop... }` makes every TMA / MMA operand a per-thread value: the compiler then has to move it to the uniform
  // datapath with R2UR and wraps each UTMALDG / UTCHMMA in an ELECT + BRA.U.ANY retry loop - ~90 cycles per MMA issue and ~225 per TMA
  // issue (what round 1 measured as "the cost of a TMA instruction"); converged, the same instructions issue back to back.
  if (warp == 0) {
    // ================================================================ TMA producer
    const uint32_t a_bytes = (g.a_mode == A_GEMM) ? uint32_t(SM::A_BYTES) : uint32_t(g.TW * g.TH * g.TN * 128);
    int stage = 0; uint32_t phase = 0;
    for (int it = 0; it < n_work; ++it) {
      const GemmWork w = get_work(it);
      const int tile = w.tile;
      const int nt = tile % n_tiles, mt = tile / n_tiles;
      int tn0 = 0, ty0 = 0, tx0 = 0;
      if (g.a_mode != A_GEMM) tile_origin(mt, tn0, ty0, tx0);
      if (lane == 0) gstamp(2, it, 0);
      for (int kb = w.kb0; kb < w.kb1; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1u);
        if (lane == 0 && kb == w.kb0) gstamp(2, it, 1);
        const uint32_t sa = smem_base + stage * SM::STAGE_BYTES;
        const uint32_t sb = sa + SM::A_BYTES;
        const uint32_t fb = full_bar(stage);
        const int tap = kb / kb_per_tap;
        const int cb = kb - tap * kb_per_tap;
        const int ky = tap / 3, kx = tap - ky * 3;
        if (elect_one()) {
          mbar_expect_tx(fb, a_bytes + uint32_t(SM::B_BYTES));
          if (g.a_mode == A_GEMM) {
            if (cb < g.kblocks_a1) tma_load_2d(sa, &tmA1, fb, cb * GEMM_BK, mt * GEMM_BM);
            else tma_load_2d(sa, &tmA2, fb, (cb - g.kblocks_a1) * GEMM_BK, mt * GEMM_BM);
          } else if (g.a_mode == A_CONV) {
            tma_load_4d(sa, &tmA1, fb, cb * GEMM_BK, tx0 + kx - 1, ty0 + ky - 1, tn0);
          } else {
            const int py = (ky == 1) ? 0 : 1, dy = (ky == 0) ? -1 : 0;
            const int px = (kx == 1) ? 0 : 1, dx = (kx == 0) ? -1 : 0;
            tma_load_5d(sa, &tmA1, fb, cb * GEMM_BK, tx0 + dx, ty0 + dy, py * 2 + px, tn0);
          }
          tma_load_2d(sb, &tmB, fb, kb * GEMM_BK, nt * BN);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
      if (lane == 0) gstamp(2, it, 2);
    }
    if (elect_one()) griddep_launch_dependents();   // all loads of this CTA are in flight: the successor's prologue may overlap the remaining MMAs + epilogue
    __syncwarp();
  } else if (warp == 1) {
    // ================================================================ MMA issuer
    const uint32_t idesc = make_idesc(GEMM_BM, BN, BF);
    int stage = 0; uint32_t phase = 0;
    const uint32_t a_lo0 = desc_lo(smem_base);
    for (int it = 0; it < n_work; ++it) {
      const GemmWork w = get_work(it);
      const int ab = it & 1;
      const uint32_t aphase = uint32_t(it >> 1) & 1u;
      if (lane == 0) gstamp(1, it, 0);
      mbar_wait(acc_empty(ab), aphase ^ 1u);              // epilogue has drained this accumulator (first use: free)
      tc_fence_after();
      if (lane == 0) gstamp(1, it, 1);
      const uint32_t tmem_acc = tmem_base + ab * ACC_STRIDE;
      for (int kb = w.kb0; kb < w.kb1; ++kb) {
        mbar_wait(full_bar(stage), phase);
        tc_fence_after();
        if (lane == 0 && kb == w.kb0) gstamp(1, it, 2);
        const uint32_t a_lo = a_lo0 + uint32_t(stage) * uint32_t(SM::STAGE_BYTES / 16);
        const uint32_t b_lo = a_lo + uint32_t(SM::A_BYTES / 16);
        const uint32_t eb = empty_bar(stage), af = acc_full(ab);
        const uint32_t first = (kb == w.kb0) ? 0u : 1u;
        const bool last = kb == w.kb1 - 1;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k)
            umma_ss(tmem_acc, desc_make(a_lo + k * 2), desc_make(b_lo + k * 2), idesc, k ? 1u : first);
          umma_commit(eb);
          if (last) umma_commit(af);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
      if (lane == 0) gstamp(1, it, 3);
    }
  } else {
    // ================================================================ epilogue (warps 2..9)
    constexpr int bf = BF;
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int part = ew >> 2;                              // which share of the tile's columns this warp drains (GEMM2_PARTS per lane quarter)
    const int r = quarter * 32 + lane;
    const int et = threadIdx.x - 64;                       // 0 .. GEMM2_EPI_THREADS - 1
    constexpr bool geglu = EPI == EPI_GEGLU;
    // column range [c_beg, c_end) in 16-column chunks (GEGLU: over the value half only)
    constexpr int NCHUNK = BN / 16;
    constexpr int NCHUNK_G = (BN / 2) / 16 > 0 ? (BN / 2) / 16 : 1;
    const int nch = geglu ? NCHUNK_G : NCHUNK;
    const int ch_beg = part * nch / GEMM2_PARTS;
    const int ch_end = (part + 1) * nch / GEMM2_PARTS;
    constexpr int MAXCH = (NCHUNK + GEMM2_PARTS - 1) / GEMM2_PARTS;
    // global row of this thread's accumulator row in tile `tile_`
    auto my_row = [&](int tile_, long long& grow_) -> bool {
      const int mt_ = tile_ / n_tiles;
      if (g.a_mode == A_GEMM) { grow_ = (long long)mt_ * GEMM_BM + r; return grow_ < g.M; }
      int tn0, ty0, tx0;
      tile_origin(mt_, tn0, ty0, tx0);
      const int per_img = g.TW * g.TH;
      const int dn = r / per_img, rem = r - dn * per_img;
      const int dy = rem / g.TW, dx = rem - dy * g.TW;
      const int n = tn0 + dn, y = ty0 + dy, x = tx0 + dx;
      grow_ = ((long long)n * g.H + y) * g.W + x;
      return (dn < g.TN) && (n < g.NB) && (y < g.H) && (x < g.W);
    };
    // global row of accumulator row 0 of tile `tile_` (the statistics' sample index: all rows of a tile share it, host-checked)
    auto my_row_base = [&](int tile_) -> long long {
      const int mt_ = tile_ / n_tiles;
      if (g.a_mode == A_GEMM) return (long long)mt_ * GEMM_BM;
      int tn0, ty0, tx0;
      tile_origin(mt_, tn0, ty0, tx0);
      return ((long long)tn0 * g.H + ty0) * g.W + tx0;
    };
    volatile int* last_flag = reinterpret_cast<volatile int*>(smem_gen + SM::FLAG_OFF);
    // TMA-store flavour: staging tile + the coalesced residual loader (chunk q of the tile = row q / (BN/8), 16-byte column chunk q % (BN/8))
    uint8_t* const stage_base = smem_gen + SM::OUT_OFF;
    constexpr int NPF = TMAO ? (GEMM_BM * BN / 8) / GEMM2_EPI_THREADS : 1;
    static_assert(!TMAO || (GEMM_BM * BN / 8) % GEMM2_EPI_THREADS == 0, "tile chunks must divide over the epilogue threads");
    // Residual tile -> staging tile with cp.async (LDGSTS): coalesced 16-byte chunks (consecutive threads = consecutive bytes of a row), global
    // memory straight into the swizzled shared-memory slots, NO registers.  (The first version held the chunks in registers one tile ahead;
    // under the 96-register cap nvcc homed them in local memory, and the spill store right behind each load waited for the data: 2 400 exposed
    // cycles per tile plus 1 400 for the register -> shared copy, profiles/r02_trace_gemm_epilogue_before.txt.)
    auto copy_res_tile_async = [&](int tile_, int buf) {
      const long long r0 = my_row_base(tile_);
      const int c0 = (tile_ % n_tiles) * BN;
#pragma unroll
      for (int i = 0; i < NPF; ++i) {
        const int q = et + i * GEMM2_EPI_THREADS, rr = q / (BN / 8), c16 = q - rr * (BN / 8);
        const long long gr = r0 + rr;
        const int gc = c0 + c16 * 8;
        const bool ok = gr < g.M && gc + 8 <= g.N;
        const uint16_t* src = reinterpret_cast<const uint16_t*>(g.residual) + (ok ? gr * g.ldr + gc : 0);
        const uint32_t dst = smem_base + SM::OUT_OFF + buf * SM::OUT_TILE + (c16 >> 2) * (GEMM_BM * 64) + rr * 64 + (((c16 & 3) ^ ((rr >> 1) & 3)) << 4);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(ok ? 16 : 0) : "memory");   // src-size 0: zero fill
      }
    };
    if constexpr (DBL) {                                    // first tile's residual: nothing to overlap it with, exposed once per CTA
      if (g.residual != nullptr && n_work > 0) copy_res_tile_async(get_work(0).tile, 0);
    }
    for (int it = 0; it < n_work; ++it) {
      const GemmWork w = get_work(it);
      const int tile = w.tile;
      const int ab = it & 1;
      const uint32_t aphase = uint32_t(it >> 1) & 1u;
      const int nt = tile % n_tiles, mt = tile / n_tiles;
      const int n0 = nt * BN;
      if (et == 0) gstamp(0, it, 0);
      long long grow;
      const bool row_ok = my_row(tile, grow);
      (void)mt;
      const int ob = DBL ? (it & 1) : 0;                     // staging tile of this work item
      uint8_t* const stage_out = stage_base + ob * SM::OUT_TILE;
      if constexpr (DBL) { if (et == 0) { gstamp(0, it, 1); gstamp(0, it, 2); } }
      if constexpr (TMAO && !DBL) {
        // ---- single staging tile: once the previous tile's TMA store has finished reading it, this tile's residual is copied into it
        // asynchronously; the copy's latency overlaps only the staging loops below (~2 400 exposed cycles per tile, r02_trace_gemm_*)
        if (et == 0) gstamp(0, it, 1);
        if (et == 0 && it > 0) bulk_wait_read_all();
        epi_bar_sync();
        if (et == 0) gstamp(0, it, 2);
        if (g.residual != nullptr) copy_res_tile_async(tile, 0);
      }
      // stage this tile's bias slice (fp32) in smem; buffer alternates with the accumulator
      float* bs = bias_s + ab * BN;
      for (int j = et; j < BN; j += GEMM2_EPI_THREADS) bs[j] = (g.bias && n0 + j < g.N) ? load16(g.bias, n0 + j, bf) : 0.f;
      // folded LayerNorm (consumer side): v = acc * lnA + lnB * colsum[c] + bias[c] with lnA = rstd_r, lnB = -rstd_r mean_r (1, 0 when off)
      float* cs = cs_s + ab * BN;
      float lnA = 1.f, lnB = 0.f;
      const bool has_ln = g.ln_stats != nullptr;
      if (has_ln) {
        for (int j = et; j < BN; j += GEMM2_EPI_THREADS) cs[j] = (n0 + j < g.N) ? g.ln_colsum[n0 + j] : 0.f;
        if (row_ok) {
          const float2 st2 = *reinterpret_cast<const float2*>(g.ln_stats + 2 * grow);
          const float inv_w = 1.f / float(g.ln_width);
          const float mean = st2.x * inv_w;
          lnA = rsqrtf(fmaxf(st2.y * inv_w - mean * mean, 0.f) + g.ln_eps);
          lnB = -lnA * mean;
        }
      } else {
        for (int j = et; j < BN; j += GEMM2_EPI_THREADS) cs[j] = 0.f;
      }
      float rsum = 0.f, rsq = 0.f;                           // producer side: this thread's share of its row's LayerNorm statistics
      const bool do_stats = !LEAN && STOREF && g.chan_stats != nullptr;
      float* st = stat_s + ab * 2 * BN;
      if (do_stats) for (int j = et; j < 2 * BN; j += GEMM2_EPI_THREADS) st[j] = 0.f;
      // prefetch residual rows for this thread's chunks (latency overlaps the wait for the accumulator; prefetching a whole
      // tile ahead was measured: no gain at BN=160, register spills at BN=256)
      constexpr int RES_REGS = TMAO ? 1 : MAXCH;
      uint4 res[RES_REGS][2];
      const bool use_res = g.residual != nullptr && !geglu && row_ok;
      const uint16_t* rrow = use_res ? reinterpret_cast<const uint16_t*>(g.residual) + grow * g.ldr + n0 : nullptr;
      const bool res_vec = use_res && ((reinterpret_cast<uintptr_t>(rrow) & 15) == 0) && (n0 + BN <= g.N);
      if constexpr (!TMAO) {
#pragma unroll
        for (int c = 0; c < MAXCH; ++c) {
          const int ch = ch_beg + c;
          if (res_vec && ch < ch_end) {
            res[c][0] = reinterpret_cast<const uint4*>(rrow + ch * 16)[0];
            res[c][1] = reinterpret_cast<const uint4*>(rrow + ch * 16)[1];
          }
        }
      } else {
        if (g.residual != nullptr) asm volatile("cp.async.wait_all;" ::: "memory");      // this thread's residual chunks (of THIS tile) have landed
        if constexpr (DBL) { if (et == 0 && it > 0) bulk_wait_read_all(); }             // the other staging tile: tile it-1's TMA store has read it
      }
      epi_bar_sync();                                       // bias slice (and the staged residual tile) visible to all epilogue threads
      if constexpr (DBL) {
        // two staging tiles: the NEXT tile's residual goes into the other one now - a whole tile ahead of its use, nothing exposed
        if (g.residual != nullptr && it + 1 < n_work) copy_res_tile_async(get_work(it + 1).tile, ob ^ 1);
      }
      if (et == 0) gstamp(0, it, 3);
      mbar_wait(acc_full(ab), aphase);
      tc_fence_after();
      if (et == 0) gstamp(0, it, 4);
      const uint32_t t_row = tmem_base + ab * ACC_STRIDE + (uint32_t(quarter * 32) << 16);

      bool run_epilogue = true;
      bool released = false;                               // acc_empty already signalled for this tile
      if (w.split >= 0) {
        // ---- split-K tail unit: publish the partial accumulator; the last arriver of the tile folds the others in and finishes
        constexpr int SLOT = GEMM_BM * BN;                                  // floats per partial
        float* tile_ws = sched.ws + (size_t)w.tail_idx * sched.ksplit * SLOT;
        float* mine = tile_ws + (size_t)w.split * SLOT;
        const int nsets = geglu ? 2 : 1;                                    // GEGLU threads own a value chunk and the matching gate chunk
        for (int set = 0; set < nsets; ++set) {
#pragma unroll
          for (int c = 0; c < MAXCH; ++c) {
            const int ch = ch_beg + c;
            if (ch < ch_end) {
              const int colc = ch + set * (BN / 32);                          // 16-column chunk index inside the tile
              uint32_t a[16];
              tmem_ld_x16(t_row + colc * 16, a);
              tmem_ld_wait();
              float4* dst = reinterpret_cast<float4*>(mine + ((size_t)colc * GEMM_BM + r) * 16);
#pragma unroll
              for (int j = 0; j < 4; ++j)
                dst[j] = make_float4(__uint_as_float(a[4 * j]), __uint_as_float(a[4 * j + 1]), __uint_as_float(a[4 * j + 2]), __uint_as_float(a[4 * j + 3]));
            }
          }
        }
        __threadfence();
        epi_bar_sync();
        if (et == 0) {
          const int old = atomicAdd(sched.counters + w.tail_idx, 1);
          const int last = (old == sched.ksplit - 1) ? 1 : 0;
          if (last) sched.counters[w.tail_idx] = 0;                         // every unit of this tile has arrived: re-arm for the next launch
          *last_flag = last;
        }
        epi_bar_sync();
        run_epilogue = (*last_flag != 0);
        if (run_epilogue) {
          __threadfence();
          for (int set = 0; set < nsets; ++set) {
#pragma unroll
            for (int c = 0; c < MAXCH; ++c) {
              const int ch = ch_beg + c;
              if (ch < ch_end) {
                const int colc = ch + set * (BN / 32);
                uint32_t a[16];
                tmem_ld_x16(t_row + colc * 16, a);
                tmem_ld_wait();
                for (int sp = 0; sp < sched.ksplit; ++sp) {
                  if (sp == w.split) continue;
                  const float4* src = reinterpret_cast<const float4*>(tile_ws + (size_t)sp * SLOT + ((size_t)colc * GEMM_BM + r) * 16);
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float4 p = __ldcg(src + j);
                    a[4 * j] = __float_as_uint(__uint_as_float(a[4 * j]) + p.x);
                    a[4 * j + 1] = __float_as_uint(__uint_as_float(a[4 * j + 1]) + p.y);
                    a[4 * j + 2] = __float_as_uint(__uint_as_float(a[4 * j + 2]) + p.z);
                    a[4 * j + 3] = __float_as_uint(__uint_as_float(a[4 * j + 3]) + p.w);
                  }
                }
                tmem_st16(t_row + colc * 16, a);
              }
            }
          }
          tmem_st16_wait();
        }
      }

      if (!run_epilogue) {
        // partial published; nothing else to do for this unit
      } else if (BN >= 32 && geglu) {
        constexpr int HALF = BN / 2;
        const int out_col0 = nt * HALF;
#pragma unroll
        for (int c = 0; c < MAXCH; ++c) {
          const int ch = ch_beg + c;
          if (ch < ch_end) {
            uint32_t a[16], b[16];
            tmem_ld_x16(t_row + ch * 16, a);
            tmem_ld_x16(t_row + HALF + ch * 16, b);
            tmem_ld_wait();
            if (row_ok) {
              uint32_t packed[8];
#pragma unroll
              for (int q = 0; q < 4; ++q) {                // 16-byte reads of the bias / column-sum slices (value and gate halves)
                const float4 bv = *reinterpret_cast<const float4*>(bs + ch * 16 + q * 4), bg = *reinterpret_cast<const float4*>(bs + HALF + ch * 16 + q * 4);
                const float4 cv = *reinterpret_cast<const float4*>(cs + ch * 16 + q * 4), cg = *reinterpret_cast<const float4*>(cs + HALF + ch * 16 + q * 4);
                const int j = q * 4;
                const float v0 = fmaf(__uint_as_float(a[j]), lnA, fmaf(lnB, cv.x, bv.x)), v1 = fmaf(__uint_as_float(a[j + 1]), lnA, fmaf(lnB, cv.y, bv.y));
                const float v2 = fmaf(__uint_as_float(a[j + 2]), lnA, fmaf(lnB, cv.z, bv.z)), v3 = fmaf(__uint_as_float(a[j + 3]), lnA, fmaf(lnB, cv.w, bv.w));
                const float g0 = fmaf(__uint_as_float(b[j]), lnA, fmaf(lnB, cg.x, bg.x)), g1 = fmaf(__uint_as_float(b[j + 1]), lnA, fmaf(lnB, cg.y, bg.y));
                const float g2 = fmaf(__uint_as_float(b[j + 2]), lnA, fmaf(lnB, cg.z, bg.z)), g3 = fmaf(__uint_as_float(b[j + 3]), lnA, fmaf(lnB, cg.w, bg.w));
                packed[q * 2] = pack16(v0 * gelu_erf(g0), v1 * gelu_erf(g1), bf);
                packed[q * 2 + 1] = pack16(v2 * gelu_erf(g2), v3 * gelu_erf(g3), bf);
              }
              uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(g.C) + grow * g.ldc + out_col0 + ch * 16);
              dst[0] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
              dst[1] = make_uint4(packed[4], packed[5], packed[6], packed[7]);
            }
          }
        }
      } else {
        // software-pipelined drain: the tcgen05.ld of chunk c+1 is in flight while chunk c is converted and stored
        // (measured: +5 % on the bias/residual epilogues, -7 % on the scattered transposed-V stores of the QKV epilogue, which keeps the
        // plain load -> wait -> store order)
        uint32_t acc2[2][16];
        constexpr bool pipelined = EPI != EPI_QKV;
        if (pipelined && ch_beg < ch_end) tmem_ld_x16(t_row + ch_beg * 16, acc2[0]);
#pragma unroll
        for (int c = 0; c < MAXCH; ++c) {
          const int ch = ch_beg + c;
          if (ch < ch_end) {
            if (!pipelined) tmem_ld_x16(t_row + ch * 16, acc2[c & 1]);
            tmem_ld_wait();
            if (pipelined && ch + 1 < ch_end) tmem_ld_x16(t_row + (ch + 1) * 16, acc2[(c + 1) & 1]);
            const uint32_t (&a)[16] = acc2[c & 1];
            const int col0 = n0 + ch * 16;
            const bool full = (col0 + 16 <= g.N);
            const bool active = row_ok && col0 < g.N;
            float v[16];
            if (active) {
              // bias (and, with a folded LayerNorm, column-sum) slices as 16-byte shared-memory reads: the scalar form issued 32 LDS per
              // chunk and thread - 1 280 warp-level LDS per 128x160 tile on the single LSU, about half of the drain (r02_trace_gemm_*)
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float4 b4 = *reinterpret_cast<const float4*>(bs + ch * 16 + q * 4);
                v[q * 4 + 0] = b4.x; v[q * 4 + 1] = b4.y; v[q * 4 + 2] = b4.z; v[q * 4 + 3] = b4.w;
              }
              if (has_ln) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const float4 c4 = *reinterpret_cast<const float4*>(cs + ch * 16 + q * 4);
                  v[q * 4 + 0] = fmaf(lnB, c4.x, v[q * 4 + 0]); v[q * 4 + 1] = fmaf(lnB, c4.y, v[q * 4 + 1]);
                  v[q * 4 + 2] = fmaf(lnB, c4.z, v[q * 4 + 2]); v[q * 4 + 3] = fmaf(lnB, c4.w, v[q * 4 + 3]);
                }
              }
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = fmaf(__uint_as_float(a[j]), lnA, v[j]);
              if (!LEAN && g.rowbias) {
                const uint16_t* rb = reinterpret_cast<const uint16_t*>(g.rowbias) + (grow / g.rows_per_group) * g.ld_rowbias + col0;
                if (full && ((reinterpret_cast<uintptr_t>(rb) & 15) == 0)) {
                  float f0[8], f1[8];
                  unpack8(reinterpret_cast<const uint4*>(rb)[0], f0, bf); unpack8(reinterpret_cast<const uint4*>(rb)[1], f1, bf);
#pragma unroll
                  for (int j = 0; j < 8; ++j) { v[j] += f0[j]; v[8 + j] += f1[j]; }
                } else {
#pragma unroll
                  for (int j = 0; j < 16; ++j) if (full || col0 + j < g.N) v[j] += load16(rb, j, bf);
                }
              }
              if (EPI == EPI_QKV && col0 >= g.n_split) {
                const int b = int(grow / g.ntok), tok = int(grow - (long long)b * g.ntok);
          const size_t vC = (size_t)g.heads * g.hdim;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                  const int vc = col0 + j - g.n_split;
                  if (full || col0 + j < g.N) {
                    store16(g.Vt, ((size_t)b * vC + vc) * g.ntok + tok, v[j], bf);   // (b*heads + h)*hdim + dd == b*C + vc
                  }
                }
              } else {
                uint8_t* srow = nullptr;                   // TMA flavour: this thread's 32-byte slot pair in the staging tile
                int sw0 = 0, sw1 = 0;
                if constexpr (TMAO) {
                  srow = stage_out + (ch >> 1) * (GEMM_BM * 64) + r * 64;
                  const int k0 = (ch & 1) * 2, sx = (r >> 1) & 3;
                  sw0 = ((k0 ^ sx) << 4); sw1 = (((k0 + 1) ^ sx) << 4);
                  if (g.residual != nullptr) {
                    float f0[8], f1[8];
                    unpack8(*reinterpret_cast<const uint4*>(srow + sw0), f0, bf); unpack8(*reinterpret_cast<const uint4*>(srow + sw1), f1, bf);
#pragma unroll
                    for (int j = 0; j < 8; ++j) { v[j] += f0[j]; v[8 + j] += f1[j]; }
                  }
                } else if (use_res) {
                  if (res_vec) {
                    float f0[8], f1[8];
                    unpack8(res[c][0], f0, bf); unpack8(res[c][1], f1, bf);
#pragma unroll
                    for (int j = 0; j < 8; ++j) { v[j] += f0[j]; v[8 + j] += f1[j]; }
                  } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) if (full || col0 + j < g.N) v[j] += load16(rrow, ch * 16 + j, bf);
                  }
                }
                if (g.out_scale != 1.0f) {
#pragma unroll
                  for (int j = 0; j < 16; ++j) v[j] *= g.out_scale;
                }
                if (!LEAN && STOREF && g.epi == EPI_GELU) {
#pragma unroll
                  for (int j = 0; j < 16; ++j) v[j] = gelu_erf(v[j]);
                } else if (!LEAN && STOREF && g.epi == EPI_QUICK_GELU) {
#pragma unroll
                  for (int j = 0; j < 16; ++j) v[j] = quick_gelu(v[j]);
                }
                if (STOREF && g.row_stats != nullptr) {
#pragma unroll
                  for (int j = 0; j < 16; ++j) if (full || col0 + j < g.N) { rsum += v[j]; rsq = fmaf(v[j], v[j], rsq); }
                }
                uint16_t* crow = reinterpret_cast<uint16_t*>(g.C) + grow * g.ldc + col0;
                if constexpr (TMAO) {
                  float lo[8], hi[8];
#pragma unroll
                  for (int j = 0; j < 8; ++j) { lo[j] = v[j]; hi[j] = v[8 + j]; }
                  *reinterpret_cast<uint4*>(srow + sw0) = pack8(lo, bf);
                  *reinterpret_cast<uint4*>(srow + sw1) = pack8(hi, bf);
                } else if (full && ((reinterpret_cast<uintptr_t>(crow) & 15) == 0)) {
                  float lo[8], hi[8];
#pragma unroll
                  for (int j = 0; j < 8; ++j) { lo[j] = v[j]; hi[j] = v[8 + j]; }
                  reinterpret_cast<uint4*>(crow)[0] = pack8(lo, bf);
                  reinterpret_cast<uint4*>(crow)[1] = pack8(hi, bf);
                } else {
#pragma unroll
                  for (int j = 0; j < 16; ++j) if (full || col0 + j < g.N) store16(crow, j, v[j], bf);
                }
              }
            }
            if (do_stats && col0 < g.N) {                   // warp-uniform: every lane joins the shuffles, inactive rows / columns add 0
              float s1[16], s2[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float x = (active && (full || col0 + j < g.N)) ? v[j] : 0.f;
                s1[j] = x; s2[j] = x * x;
              }
              const float cs = warp_colsum16(s1, lane), cq = warp_colsum16(s2, lane);
              if ((lane & 1) == 0) {
                const int cc = ch * 16 + colsum_col_of_lane(lane);
                atomicAdd(&st[cc], cs); atomicAdd(&st[BN + cc], cq);
              }
            }
          }
        }
        // this thread's accumulator reads are complete: hand the TMEM buffer back NOW (the issuer can start tile it+2 while the statistics,
        // the final barrier and the TMA store of this tile are still under way; thread 0's TMA issue alone cost ~800 cycles of that)
        tc_fence_before();
        mbar_arrive(acc_empty(ab));
        released = true;
        if (STOREF && g.row_stats != nullptr && row_ok && ch_beg < ch_end) {
          atomicAdd(g.row_stats + 2 * grow, rsum); atomicAdd(g.row_stats + 2 * grow + 1, rsq);
        }
        if (et == 0) gstamp(0, it, 5);
        if constexpr (TMAO) fence_proxy_async();            // this thread's staging-tile writes -> visible to the TMA (async proxy)
        if (do_stats || TMAO) epi_bar_sync();
        if (et == 0) gstamp(0, it, 6);
        if constexpr (TMAO) {
          if (et == 0) {
            const int row0 = int(my_row_base(tile));
#pragma unroll
            for (int bx = 0; bx < BN / 32; ++bx)
              if (n0 + bx * 32 < g.N) tma_store_2d(&tmC, smem_base + SM::OUT_OFF + ob * SM::OUT_TILE + bx * (GEMM_BM * 64), n0 + bx * 32, row0);
            bulk_commit();
          }
        }
        if (do_stats) {
          // the four row quarters of this tile were combined in smem: one global reduction per column and statistic
          const long long srow = my_row_base(tile);
          float* dst = g.chan_stats + ((srow / g.stats_rows) * g.N + n0) * 2;
          for (int j = et; j < BN; j += GEMM2_EPI_THREADS)
            if (n0 + j < g.N) { atomicAdd(dst + 2 * j, st[j]); atomicAdd(dst + 2 * j + 1, st[BN + j]); }
        }
      }
      if (!released) {
        tc_fence_before();
        mbar_arrive(acc_empty(ab));                         // this thread no longer reads accumulator `ab`
      }
      if (et == 0) gstamp(0, it, 7);
    }
    if constexpr (TMAO) { if (et == 0) bulk_wait_all(); }   // every TMA store of this CTA has landed before the grid can be considered complete
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace cid
