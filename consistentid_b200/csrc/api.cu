// libcidb200.so - C-ABI entry points (include/cidb200.h) for the ConsistentID denoising hot path on sm_100a.
// Host side: argument checking, TMA tensor-map encoding (driver entry point resolved at run time so the
// library links without libcuda), kernel selection and launch on the caller's stream.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <mutex>
#include <utility>

#include <cudaTypedefs.h>

#include "../../include/cidb200.h"
#include "attn_cross.cuh"
#include "attn_cross2.cuh"         // persistent / pipelined flavour for head dims <= 80
#include "attn_tc5.cuh"           // one 128-row query tile per CTA: head dims > 80 and short sequences
#ifndef CID_ATTN_NO_V6
#include "attn_tc6.cuh"           // two query tiles per CTA, P in tensor memory (aliasing S): head dim 80, >= 256 queries
#include "attn_tc7.cuh"           // ... with P in its own TMEM columns and S_{j+1} issued early: head dims <= 64, >= 256 queries
#define CID_ATTN_V6 1
#endif
#include "elementwise.cuh"
#include "embed.cuh"
#include "gemm_tc2.cuh"

using namespace cid;

namespace {

thread_local char g_err[512] = "";
int fail(int code, const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
  return code;
}
#define CID_CHECK_LAUNCH(name)                                                                   \
  do {                                                                                           \
    cudaError_t e__ = cudaGetLastError();                                                        \
    if (e__ != cudaSuccess) return fail(CID_ERR_CUDA, "%s launch: %s", name, cudaGetErrorString(e__)); \
  } while (0)

// Programmatic dependent launch (see common.cuh): kernels that call griddep_wait() before touching global memory are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization so their prologue overlaps the predecessor's tail.
template <typename... KArgs, typename... Args>
void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(std::forward<Args>(args))...);   // error picked up by CID_CHECK_LAUNCH
}

PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
std::once_flag g_encode_once;
void resolve_encode() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
      qres == cudaDriverEntryPointSuccess)
    g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
}

// rank-R tiled map over 16-bit elements, 128B swizzle; dims[0] is the contiguous dimension.
int make_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
             const cuuint32_t* box, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  std::call_once(g_encode_once, resolve_encode);
  if (!g_encode) return fail(CID_ERR_DRIVER, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return fail(CID_ERR_ARG, "TMA base %p not 16-byte aligned", base);
  for (int i = 0; i + 1 < rank; ++i)
    if (strides_bytes[i] % 16 != 0) return fail(CID_ERR_ARG, "TMA stride[%d]=%llu not a multiple of 16 bytes", i, (unsigned long long)strides_bytes[i]);
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, rank, const_cast<void*>(base), dims, strides_bytes, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(CID_ERR_DRIVER, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d)", int(r), rank);
  return 0;
}
int map_2d(CUtensorMap* m, const void* base, long long inner, long long rows, long long pitch_elems, int box_rows) {
  cuuint64_t dims[2] = {cuuint64_t(inner), cuuint64_t(rows)};
  cuuint64_t str[1] = {cuuint64_t(pitch_elems) * 2};
  cuuint32_t box[2] = {64, cuuint32_t(box_rows)};
  return make_map(m, base, 2, dims, str, box);
}

// output map of the TMA-store epilogue: [rows, N] 16-bit, boxes of 32 columns (64 B) x 128 rows, 64B swizzle (gemm_tc2.cuh staging layout)
int map_out(CUtensorMap* m, const void* base, long long cols, long long rows, long long pitch_elems) {
  cuuint64_t dims[2] = {cuuint64_t(cols), cuuint64_t(rows)};
  cuuint64_t str[1] = {cuuint64_t(pitch_elems) * 2};
  cuuint32_t box[2] = {32, 128};
  return make_map(m, base, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B);
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device (per-context) attribute: remember it per (kernel, device) so that one
// process may drive several GPUs through this library.
constexpr int MAX_DEVICES = 64;
int current_device() { int d = 0; return cudaGetDevice(&d) == cudaSuccess && d >= 0 && d < MAX_DEVICES ? d : 0; }
template <typename K>
int set_smem(K kernel, int bytes, const char* name, bool (&done)[MAX_DEVICES]) {
  const int dev = current_device();
  if (done[dev]) return 0;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return fail(CID_ERR_CUDA, "cudaFuncSetAttribute(%s, %d B): %s", name, bytes, cudaGetErrorString(e));
  done[dev] = true;
  return 0;
}

int grid_for(long long work_items, int block) {
  long long g = (work_items + block - 1) / block;
  const long long cap = 148LL * 16;
  return int(g < 1 ? 1 : (g > cap ? cap : g));
}

int g_num_sms[MAX_DEVICES] = {};
int num_sms() {
  const int dev = current_device();
  if (g_num_sms[dev] == 0) {
    int n = 0;
    g_num_sms[dev] = (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) ? n : 148;
  }
  return g_num_sms[dev];
}

// Split-K tail-balancing policy.  Measured (profiles/r01_splitk_sweep.txt): every extra K-range costs the finishing CTA ~3.5 us and a tail
// tile running on an otherwise idle chip is ~1.6x faster than one in a full wave, so splitting pays only for long K loops: >= 48 k-blocks
// (K >= 3072) per unit, at most 4 units.  cid_set_splitk overrides (tests force it on to exercise the path).
constexpr size_t WS_COUNTER_BYTES = 4096;
int g_splitk_min_kb = 48, g_splitk_max = 4;
#ifdef CID_NO_TMA_EPILOGUE
bool g_tma_epilogue = false;      // A/B builds: register epilogue everywhere
#else
bool g_tma_epilogue = true;
#endif
int g_tma_epilogue_max_kb = 24;
#ifdef CID_NO_TMA_EPILOGUE_DBL
bool g_tma_epilogue_dbl = false;
#else
bool g_tma_epilogue_dbl = true;
#endif
bool g_cross2 = true;
#ifdef CID_GEMM_TRACE
long long* g_gemm_trace = nullptr;       // debug builds only (tools/trace_gemm.py)
#endif

// N tile of the store / GELU / QKV flavours (their operand layouts do not depend on the tile; GEGLU's interleaved weight does, so it keeps
// cid_gemm_tile_n).  Picks between the 256- and 160-wide tiles by a wave model: cost = waves x BN x (cost per column), where a tail wave
// counts 1 unless the tail-balancing split applies (1/sp + fix-up), and a 160-wide tile pays ~10 % more per column (more L2->SMEM bytes
// per FLOP).  N = 1280 at 32 row tiles is 160 tiles of 256 (1.08 waves -> 2) but 256 tiles of 160 (1.73 waves -> 2): 0.69x the time.
#ifndef CID_TILE_STATIC
double tile_cost(int bn, int N, int m_tiles, int num_kb, bool ws) {
  const int G = num_sms();
  const int total = ((N + bn - 1) / bn) * m_tiles;
  const int full = total / G, tail = total % G;
  double waves = full;
  if (tail) {
    int sp = 1;
    if (ws && g_splitk_max > 1) {
      sp = G / tail;
      if (sp > num_kb / g_splitk_min_kb) sp = num_kb / g_splitk_min_kb;
      if (sp > g_splitk_max) sp = g_splitk_max;
    }
    waves += sp >= 2 ? 1.0 / sp + 0.15 : 1.0;
  }
  return waves * bn * (bn == 256 ? 1.0 : 1.1);
}
#endif
int pick_tile_n(int N, int epi, int m_tiles, int num_kb, bool ws) {
  const int fixed = cid_gemm_tile_n(N, epi);
#ifndef CID_TILE_STATIC
  if (epi != CID_EPI_GEGLU && fixed == 256 && N % 160 == 0 && tile_cost(160, N, m_tiles, num_kb, ws) < tile_cost(256, N, m_tiles, num_kb, ws))
    return 160;
#endif
  return fixed;
}

template <int BN, int STAGES, int EPI, int BF, bool LEAN = false>
int launch_gemm2(const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& b, const CUtensorMap& c, const GemmArgs& g, int grid,
                 const GemmSched& sched, int n_tiles, cudaStream_t st) {
  using SM = Gemm2Smem<BN, STAGES, EPI == EPI_STORE_TMA2 ? 2 : (EPI == EPI_STORE_TMA ? 1 : 0)>;
  static bool configured[MAX_DEVICES] = {};
  if (int rc = set_smem(gemm_tc2_kernel<BN, STAGES, EPI, BF, LEAN>, SM::TOTAL, "gemm_tc2_kernel", configured)) return rc;
#ifdef CID_GEMM_TRACE
  GemmArgs gt = g; gt.trace = g_gemm_trace;
  launch_pdl(gemm_tc2_kernel<BN, STAGES, EPI, BF, LEAN>, dim3(grid), dim3(GEMM2_THREADS), SM::TOTAL, st, a1, a2, b, c, gt, n_tiles, sched);
#else
  launch_pdl(gemm_tc2_kernel<BN, STAGES, EPI, BF, LEAN>, dim3(grid), dim3(GEMM2_THREADS), SM::TOTAL, st, a1, a2, b, c, g, n_tiles, sched);
#endif
  CID_CHECK_LAUNCH("gemm_tc2_kernel");
  return 0;
}
// STAGES_T: ring depth of the TMA-store flavour (its 128 x BN staging tile comes out of the operand ring's shared memory)
template <int BN, int STAGES, int STAGES_T, int STAGES_T2 = STAGES_T>
int launch_gemm2_any(const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& b, const CUtensorMap* c_out, const GemmArgs& g, int m_tiles,
                     void* ws, size_t ws_bytes, cudaStream_t st) {
  const int n_tiles = (g.N + BN - 1) / BN;
  const int total = n_tiles * m_tiles;
  const int G = num_sms();
  GemmSched sched{};
  int grid;
  if (total >= G) { grid = G; sched.full_iters = total / G; sched.tail_tiles = total % G; }
  else { grid = total; sched.full_iters = 0; sched.tail_tiles = total; }
  sched.ksplit = 1;
  // tail balancing: cut each tail tile into K-ranges so that (almost) every SM gets a share (see gemm_tc2.cuh); needs the caller's workspace
  if (sched.tail_tiles > 0 && ws != nullptr && ws_bytes > WS_COUNTER_BYTES && g_splitk_max > 1) {
    const int num_kb = g.taps * (g.kblocks_a1 + g.kblocks_a2);
    int sp = G / sched.tail_tiles;
    if (sp > num_kb / g_splitk_min_kb) sp = num_kb / g_splitk_min_kb;
    if (sp > g_splitk_max) sp = g_splitk_max;
    const size_t need = WS_COUNTER_BYTES + (size_t)sched.tail_tiles * sp * GEMM_BM * BN * sizeof(float);
    if (sp >= 2 && sched.tail_tiles * sizeof(int) <= WS_COUNTER_BYTES && need <= ws_bytes) {
      sched.ksplit = sp;
      sched.counters = reinterpret_cast<int*>(ws);
      sched.ws = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + WS_COUNTER_BYTES);
      if (sched.tail_tiles * sp > grid) grid = sched.tail_tiles * sp;
    }
  }
  const int flavour = g.epi == EPI_GEGLU ? EPI_GEGLU : (g.epi == EPI_QKV ? EPI_QKV : EPI_STORE);      // EPI_GELU / EPI_QUICK_GELU ride on the store flavour
#define CID_G2(S, E) (g.is_bf16 ? launch_gemm2<BN, S, E, 1>(a1, a2, b, c_out ? *c_out : b, g, grid, sched, n_tiles, st) \
                                : launch_gemm2<BN, S, E, 0>(a1, a2, b, c_out ? *c_out : b, g, grid, sched, n_tiles, st))
  if constexpr (BN >= 32) {
    if (flavour == EPI_GEGLU) return CID_G2(STAGES, EPI_GEGLU);
    if (flavour == EPI_QKV) return CID_G2(STAGES, EPI_QKV);
    // Store epilogue through shared memory + TMA for SHORT K loops only (K <= 1536, where the epilogue is a large share of the tile): its
    // staging tile costs one operand-ring stage, which long K loops miss more than they gain from the coalesced stores.  Measured A/B in
    // profiles/r02_tma_epilogue_ab.txt: 8192x1280x1280 51.6 -> 44.0 us, 65536x320x320 -13 %, but 8192x1280x5120 116 -> 126 us.
    const int num_kb_all = g.taps * (g.kblocks_a1 + g.kblocks_a2);
    if (c_out != nullptr && sched.ksplit == 1 && g_tma_epilogue && num_kb_all <= g_tma_epilogue_max_kb) {
      // K <= 640 with a residual: the epilogue, not the main loop, bounds the tile - two staging tiles (the residual of tile i+1 is copied a
      // whole tile ahead) at the price of a 3-stage operand ring; longer K keeps the deeper ring and one staging tile
      // lean instances (no row bias / GroupNorm statistics / GELU compiled in) for the calls that use none of them: the transformer GEMMs
#ifndef CID_NO_LEAN_EPILOGUE
      const bool lean = g.rowbias == nullptr && g.chan_stats == nullptr && g.epi != EPI_GELU && g.epi != EPI_QUICK_GELU;
#else
      const bool lean = false;
#endif
#define CID_G2L(S, E) (g.is_bf16 ? launch_gemm2<BN, S, E, 1, true>(a1, a2, b, *c_out, g, grid, sched, n_tiles, st) \
                                 : launch_gemm2<BN, S, E, 0, true>(a1, a2, b, *c_out, g, grid, sched, n_tiles, st))
      if constexpr (BN == 160 || BN == 64) {
        if (g.residual != nullptr && num_kb_all <= 10 && g_tma_epilogue_dbl) return lean ? CID_G2L(STAGES_T2, EPI_STORE_TMA2) : CID_G2(STAGES_T2, EPI_STORE_TMA2);
      }
      return lean ? CID_G2L(STAGES_T, EPI_STORE_TMA) : CID_G2(STAGES_T, EPI_STORE_TMA);
#undef CID_G2L
    }
  } else {
    if (flavour != EPI_STORE) return fail(CID_ERR_UNSUPPORTED, "GEGLU / QKV epilogues need an N tile >= 32");
  }
  return CID_G2(STAGES, EPI_STORE);
#undef CID_G2
}

int dispatch_gemm(int bn, const CUtensorMap& a1, const CUtensorMap& a2, const CUtensorMap& b, const CUtensorMap* c_out, const GemmArgs& g,
                  int m_tiles, void* ws, size_t ws_bytes, cudaStream_t st) {
  switch (bn) {
    case 256: return launch_gemm2_any<256, 4, 3>(a1, a2, b, c_out, g, m_tiles, ws, ws_bytes, st);
    case 160: return launch_gemm2_any<160, 5, 4, 3>(a1, a2, b, c_out, g, m_tiles, ws, ws_bytes, st);
    case 64: return launch_gemm2_any<64, 8, 6, 6>(a1, a2, b, c_out, g, m_tiles, ws, ws_bytes, st);
    case 16: return launch_gemm2_any<16, 8, 8>(a1, a2, b, nullptr, g, m_tiles, ws, ws_bytes, st);
  }
  return fail(CID_ERR_UNSUPPORTED, "no GEMM instantiation for tile N %d", bn);
}
int check_ws(const void* ws, size_t ws_bytes, const char* who) {
  if (ws != nullptr && (reinterpret_cast<uintptr_t>(ws) % 256 || ws_bytes < WS_COUNTER_BYTES))
    return fail(CID_ERR_ARG, "%s: workspace must be 256-byte aligned and >= %zu bytes (or NULL)", who, WS_COUNTER_BYTES);
  return 0;
}

#ifdef CID_ATTN_TRACE
long long* g_attn_trace = nullptr;       // debug builds only (tools/trace_attn.py)
#endif
int d_pad_for(int d) {
  if (d <= 0 || d % 8) return -1;
  if (d <= 32) return 32;
  if (d <= 48) return 48;
  if (d <= 64) return 64;
  if (d <= 80) return 80;
  if (d <= 128) return 128;
  if (d <= 160) return 160;
  return -1;
}

template <int D_PAD, int BF>
int launch_attn_self_t(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const AttnArgs& a, cudaStream_t st) {
  using C = Attn5Cfg<D_PAD>;
  static bool configured[MAX_DEVICES] = {};
  if (int rc = set_smem(attn_self5_kernel<D_PAD, BF>, C::TOTAL, "attn_self5_kernel", configured)) return rc;
  dim3 grid((a.Nq + 127) / 128, a.H, a.B);
  launch_pdl(attn_self5_kernel<D_PAD, BF>, dim3(grid), dim3(ATTN5_THREADS), C::TOTAL, st, q, k, v, a);
  CID_CHECK_LAUNCH("attn_self5_kernel");
  return 0;
}
#ifdef CID_ATTN_V6
// two 128-row query tiles per CTA, P in tensor memory, ping-pong softmax warpgroups (attn_tc6.cuh): head dims <= 80, >= 256 queries
template <int D_PAD, int BF>
int launch_attn_self6_t(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const AttnArgs& a, cudaStream_t st) {
  using C = Attn6Cfg<D_PAD>;
  static bool configured[MAX_DEVICES] = {};
  if (int rc = set_smem(attn_self6_kernel<D_PAD, BF>, C::TOTAL, "attn_self6_kernel", configured)) return rc;
  dim3 grid((a.Nq + 255) / 256, a.H, a.B);
  launch_pdl(attn_self6_kernel<D_PAD, BF>, dim3(grid), dim3(ATTN6_THREADS), C::TOTAL, st, q, k, v, a);
  CID_CHECK_LAUNCH("attn_self6_kernel");
  return 0;
}
#endif
#ifdef CID_ATTN_V6
template <int D_PAD, int BF>
int launch_attn_self7_t(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const AttnArgs& a, cudaStream_t st) {
  using C = Attn7Cfg<D_PAD>;
  static bool configured[MAX_DEVICES] = {};
  if (int rc = set_smem(attn_self7_kernel<D_PAD, BF>, C::TOTAL, "attn_self7_kernel", configured)) return rc;
  dim3 grid((a.Nq + 255) / 256, a.H, a.B);
  launch_pdl(attn_self7_kernel<D_PAD, BF>, dim3(grid), dim3(ATTN6_THREADS), C::TOTAL, st, q, k, v, a);
  CID_CHECK_LAUNCH("attn_self7_kernel");
  return 0;
}
#endif
template <int D_PAD>
int launch_attn_self(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const AttnArgs& a, cudaStream_t st) {
#ifdef CID_ATTN_V6
#ifndef CID_ATTN_NO_V7
  if constexpr (D_PAD <= 64) {
    if (a.Nq >= 256) return a.is_bf16 ? launch_attn_self7_t<D_PAD, 1>(q, k, v, a, st) : launch_attn_self7_t<D_PAD, 0>(q, k, v, a, st);
  }
#endif
  if constexpr (D_PAD <= 80) {
    if (a.Nq >= 256) return a.is_bf16 ? launch_attn_self6_t<D_PAD, 1>(q, k, v, a, st) : launch_attn_self6_t<D_PAD, 0>(q, k, v, a, st);
  }
#endif
  return a.is_bf16 ? launch_attn_self_t<D_PAD, 1>(q, k, v, a, st) : launch_attn_self_t<D_PAD, 0>(q, k, v, a, st);
}
template <int D_PAD>
int launch_attn_cross(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const AttnArgs& a, cudaStream_t st) {
  using C = CrossCfg<D_PAD>;
  static bool configured[MAX_DEVICES] = {};
  if (int rc = set_smem(attn_cross_kernel<D_PAD>, C::TOTAL, "attn_cross_kernel", configured)) return rc;
  dim3 grid((a.Nq + 127) / 128, a.H, a.B);
  launch_pdl(attn_cross_kernel<D_PAD>, dim3(grid), dim3(128), C::TOTAL, st, q, k, v, a);
  CID_CHECK_LAUNCH("attn_cross_kernel");
  return 0;
}

template <int D_PAD>
int launch_attn_cross2(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const AttnArgs& a, long long units, cudaStream_t st) {
  using C = Cross2Cfg<D_PAD>;
  static bool configured[2][MAX_DEVICES] = {};
  const int grid = units < num_sms() ? int(units) : num_sms();
  // the CTA allocates all 512 TMEM columns: ask for more than half an SM's shared memory so that two of them never share an SM
  constexpr int SMEM = C::TOTAL > 117 * 1024 ? C::TOTAL : 117 * 1024;
  if (a.is_bf16) {
    if (int rc = set_smem(attn_cross2_kernel<D_PAD, 1>, SMEM, "attn_cross2_kernel", configured[1])) return rc;
    launch_pdl(attn_cross2_kernel<D_PAD, 1>, dim3(grid), dim3(CROSS2_THREADS), SMEM, st, q, k, v, a);
  } else {
    if (int rc = set_smem(attn_cross2_kernel<D_PAD, 0>, SMEM, "attn_cross2_kernel", configured[0])) return rc;
    launch_pdl(attn_cross2_kernel<D_PAD, 0>, dim3(grid), dim3(CROSS2_THREADS), SMEM, st, q, k, v, a);
  }
  CID_CHECK_LAUNCH("attn_cross2_kernel");
  return 0;
}

// Q/K style map: [B, N, H, d] view, row pitch `pitch` elements, box {64, box_rows, 1, 1}
int map_qk(CUtensorMap* m, const void* base, int B, int N, int H, int d, long long pitch, int box_rows) {
  cuuint64_t dims[4] = {cuuint64_t(d), cuuint64_t(N), cuuint64_t(H), cuuint64_t(B)};
  cuuint64_t str[3] = {cuuint64_t(pitch) * 2, cuuint64_t(d) * 2, cuuint64_t(N) * cuuint64_t(pitch) * 2};
  cuuint32_t box[4] = {64, cuuint32_t(box_rows), 1, 1};
  return make_map(m, base, 4, dims, str, box);
}
int map_vt(CUtensorMap* m, const void* base, int BH, int d, int Nkv, int d_pad) {
  cuuint64_t dims[3] = {cuuint64_t(Nkv), cuuint64_t(d), cuuint64_t(BH)};
  cuuint64_t str[2] = {cuuint64_t(Nkv) * 2, cuuint64_t(Nkv) * cuuint64_t(d) * 2};
  cuuint32_t box[3] = {64, cuuint32_t(d_pad), 1};
  return make_map(m, base, 3, dims, str, box);
}

}  // namespace

extern "C" {

int cid_version(void) { return 100; }
const char* cid_last_error(void) { return g_err; }

int cid_gemm_tile_n(int N, int epi) {
  // 256-wide tiles cut the L2->SMEM bytes per FLOP (the limiter of the 128x160 tile) wherever the width allows
  if (N % 256 == 0 && N >= 1024) return 256;
  if (epi == CID_EPI_GEGLU) {
    if (N % 160 == 0) return 160;
    if (N % 64 == 0) return 64;
    return -1;
  }
  if (N % 160 == 0) return 160;
  if (N <= 16) return 16;
  if (N % 64 == 0) return 64;
  return 160;
}

int cid_gemm(const void* A, long long lda, const void* A2, long long lda2, int K1, int K2, const void* B, void* C,
             long long ldc, int M, int N, const void* bias, const void* residual, long long ldr, const void* rowbias,
             int rows_per_group, long long ld_rowbias, int epi, void* Vt, int n_split, int heads, int hdim, int ntok,
             float out_scale, int dtype, void* workspace, unsigned long long ws_bytes, float* chan_stats, int stats_rows,
             float* row_stats, const float* ln_stats, const float* ln_colsum, float ln_eps, void* stream) {
  if (!A || !B || !C || M <= 0 || N <= 0) return fail(CID_ERR_ARG, "cid_gemm: null pointer or empty problem (M=%d N=%d)", M, N);
  if (chan_stats && (epi != CID_EPI_STORE || stats_rows <= 0 || stats_rows % 128 || M % stats_rows))
    return fail(CID_ERR_ARG, "cid_gemm: fused statistics need the plain store epilogue and stats_rows (%d) a multiple of 128 dividing M", stats_rows);
  if (int rc = check_ws(workspace, ws_bytes, "cid_gemm")) return rc;
  if (K1 <= 0 || K1 % 64 || K2 < 0 || K2 % 64) return fail(CID_ERR_ARG, "cid_gemm: K1=%d K2=%d must be multiples of 64", K1, K2);
  if (K2 > 0 && !A2) return fail(CID_ERR_ARG, "cid_gemm: K2 > 0 without A2");
  const int bn = pick_tile_n(N, epi, (M + GEMM_BM - 1) / GEMM_BM, (K1 + K2) / 64, workspace != nullptr);
  if (bn < 0) return fail(CID_ERR_UNSUPPORTED, "cid_gemm: GEGLU needs N %% 64 == 0 (N=%d)", N);
  if (epi == CID_EPI_QKV && (!Vt || n_split % 32 || heads <= 0 || hdim <= 0 || ntok <= 0 || M % ntok))
    return fail(CID_ERR_ARG, "cid_gemm: bad QKV epilogue arguments");
  CUtensorMap ta1, ta2, tb;
  int rc;
  if ((rc = map_2d(&ta1, A, K1, M, lda, 128))) return rc;
  if (K2 > 0) { if ((rc = map_2d(&ta2, A2, K2, M, lda2, 128))) return rc; } else ta2 = ta1;
  if ((rc = map_2d(&tb, B, K1 + K2, N, K1 + K2, bn))) return rc;
  GemmArgs g{};
  g.M = M; g.N = N; g.kblocks_a1 = K1 / 64; g.kblocks_a2 = K2 / 64; g.taps = 1; g.a_mode = A_GEMM;
  g.C = C; g.ldc = ldc; g.bias = bias; g.residual = residual; g.ldr = ldr;
  g.rowbias = rowbias; g.rows_per_group = rows_per_group > 0 ? rows_per_group : 1; g.ld_rowbias = ld_rowbias;
  g.epi = epi; g.is_bf16 = dtype == CID_BF16; g.Vt = Vt; g.n_split = n_split; g.heads = heads; g.hdim = hdim; g.ntok = ntok;
  g.out_scale = out_scale; g.chan_stats = chan_stats; g.stats_rows = stats_rows;
  if (row_stats && epi != CID_EPI_STORE) return fail(CID_ERR_ARG, "cid_gemm: row_stats needs the plain store epilogue");
  if ((ln_stats != nullptr) != (ln_colsum != nullptr)) return fail(CID_ERR_ARG, "cid_gemm: ln_stats and ln_colsum go together");
  if (ln_stats && (reinterpret_cast<uintptr_t>(ln_stats) & 7)) return fail(CID_ERR_ARG, "cid_gemm: ln_stats must be 8-byte aligned");
  g.row_stats = row_stats; g.ln_stats = ln_stats; g.ln_colsum = ln_colsum; g.ln_eps = ln_eps; g.ln_width = K1 + K2;
  // TMA-store epilogue (plain / GELU / QuickGELU store flavours): 16-byte aligned rows of C and of the residual; rowbias constant inside a 128-row tile
  CUtensorMap tc; const CUtensorMap* pc = nullptr;
  if ((epi == CID_EPI_STORE || epi == CID_EPI_GELU || epi == CID_EPI_QUICK_GELU) && bn >= 64 && N % 8 == 0 && ldc % 8 == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0 &&
      (!residual || (ldr % 8 == 0 && (reinterpret_cast<uintptr_t>(residual) & 15) == 0))) {
    if ((rc = map_out(&tc, C, N, M, ldc))) return rc;
    pc = &tc;
  }
  return dispatch_gemm(bn, ta1, ta2, tb, pc, g, (M + 127) / 128, workspace, (size_t)ws_bytes, static_cast<cudaStream_t>(stream));
}

int cid_conv3x3(const void* X, const void* Wt, void* Y, long long ldy, int NB, int H, int W, int Cin, int Cout, int stride2,
                const void* bias, const void* residual, long long ldr, const void* rowbias, long long ld_rowbias,
                float out_scale, int dtype, void* workspace, unsigned long long ws_bytes, float* chan_stats, void* stream) {
  if (!X || !Wt || !Y || NB <= 0 || H <= 0 || W <= 0) return fail(CID_ERR_ARG, "cid_conv3x3: null pointer or empty problem");
  if (int rc0 = check_ws(workspace, ws_bytes, "cid_conv3x3")) return rc0;
  if (Cin % 64 || Cout <= 0) return fail(CID_ERR_ARG, "cid_conv3x3: Cin=%d must be a multiple of 64", Cin);
  GemmArgs g{};
  if (W >= 128) { g.TW = 128; g.TH = 1; g.TN = 1; }
  else {
    g.TW = W; g.TH = 128 / W; if (g.TH > H) g.TH = H;
    g.TN = (g.TH == H) ? (128 / (W * H)) : 1;
    if (g.TN < 1) g.TN = 1;
    if (g.TN > NB) g.TN = NB;
  }
  g.tiles_x = (W + g.TW - 1) / g.TW; g.tiles_y = (H + g.TH - 1) / g.TH;
  const int tiles_n = (NB + g.TN - 1) / g.TN;
  const int m_tiles = g.tiles_x * g.tiles_y * tiles_n;
  const int bn = pick_tile_n(Cout, CID_EPI_STORE, m_tiles, 9 * Cin / 64, workspace != nullptr);
  CUtensorMap ta, tb;
  int rc;
  if (!stride2) {
    cuuint64_t dims[4] = {cuuint64_t(Cin), cuuint64_t(W), cuuint64_t(H), cuuint64_t(NB)};
    cuuint64_t str[3] = {cuuint64_t(Cin) * 2, cuuint64_t(W) * Cin * 2, cuuint64_t(H) * W * Cin * 2};
    cuuint32_t box[4] = {64, cuuint32_t(g.TW), cuuint32_t(g.TH), cuuint32_t(g.TN)};
    if ((rc = make_map(&ta, X, 4, dims, str, box))) return rc;
  } else {
    cuuint64_t dims[5] = {cuuint64_t(Cin), cuuint64_t(W), cuuint64_t(H), 4, cuuint64_t(NB)};
    cuuint64_t str[4] = {cuuint64_t(Cin) * 2, cuuint64_t(W) * Cin * 2, cuuint64_t(H) * W * Cin * 2, cuuint64_t(4) * H * W * Cin * 2};
    cuuint32_t box[5] = {64, cuuint32_t(g.TW), cuuint32_t(g.TH), 1, cuuint32_t(g.TN)};
    if ((rc = make_map(&ta, X, 5, dims, str, box))) return rc;
  }
  if ((rc = map_2d(&tb, Wt, 9LL * Cin, Cout, 9LL * Cin, bn))) return rc;
  g.M = NB * H * W; g.N = Cout; g.kblocks_a1 = Cin / 64; g.kblocks_a2 = 0; g.taps = 9;
  g.a_mode = stride2 ? A_CONV_S2 : A_CONV; g.W = W; g.H = H; g.NB = NB;
  g.C = Y; g.ldc = ldy; g.bias = bias; g.residual = residual; g.ldr = ldr;
  g.rowbias = rowbias; g.rows_per_group = H * W; g.ld_rowbias = ld_rowbias;
  g.epi = EPI_STORE; g.is_bf16 = dtype == CID_BF16; g.out_scale = out_scale;
  if (chan_stats) {
    if (g.TN != 1) return fail(CID_ERR_UNSUPPORTED, "cid_conv3x3: fused statistics need every 128-pixel tile inside one sample (H*W = %d too small)", H * W);
    g.chan_stats = chan_stats; g.stats_rows = H * W;
  }
  // TMA-store epilogue: the 128 pixels of a tile must be 128 CONSECUTIVE rows of Y (full-width row blocks, or 128-pixel strips of wide rows)
  CUtensorMap tc; const CUtensorMap* pc = nullptr;
  const bool rows_contiguous = (g.TW == W && g.TW * g.TH * g.TN == 128 && (H % g.TH) == 0 && (g.TN == 1 || NB % g.TN == 0)) || (W % 128 == 0 && g.TW == 128);
  if (rows_contiguous && bn >= 64 && Cout % 8 == 0 && ldy % 8 == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0 &&
      (!residual || (ldr % 8 == 0 && (reinterpret_cast<uintptr_t>(residual) & 15) == 0))) {
    if ((rc = map_out(&tc, Y, Cout, (long long)NB * H * W, ldy))) return rc;
    pc = &tc;
  }
  return dispatch_gemm(bn, ta, ta, tb, pc, g, m_tiles, workspace, (size_t)ws_bytes, static_cast<cudaStream_t>(stream));
}

static int attn_self_impl(const void* Q, long long q_pitch, const void* K, long long k_pitch, const void* Vt, void* O, long long ldo,
                          int B, int H, int N, int n_valid, int d, int dtype, int causal, void* stream);
int cid_attn_self(const void* Q, long long q_pitch, const void* K, long long k_pitch, const void* Vt, void* O, long long ldo,
                  int B, int H, int N, int d, int dtype, void* stream) {
  return attn_self_impl(Q, q_pitch, K, k_pitch, Vt, O, ldo, B, H, N, N, d, dtype, 0, stream);
}
int cid_attn_self_causal(const void* Q, long long q_pitch, const void* K, long long k_pitch, const void* Vt, void* O, long long ldo,
                         int B, int H, int N, int d, int dtype, void* stream) {
  return attn_self_impl(Q, q_pitch, K, k_pitch, Vt, O, ldo, B, H, N, N, d, dtype, 1, stream);
}
int cid_attn_self_ragged(const void* Q, long long q_pitch, const void* K, long long k_pitch, const void* Vt, void* O, long long ldo,
                         int B, int H, int N, int n_valid, int d, int dtype, void* stream) {
  if (n_valid <= 0 || n_valid > N) return fail(CID_ERR_ARG, "cid_attn_self_ragged: need 0 < n_valid <= N (got %d, %d)", n_valid, N);
  return attn_self_impl(Q, q_pitch, K, k_pitch, Vt, O, ldo, B, H, N, n_valid, d, dtype, 0, stream);
}
static int attn_self_impl(const void* Q, long long q_pitch, const void* K, long long k_pitch, const void* Vt, void* O, long long ldo,
                          int B, int H, int N, int n_valid, int d, int dtype, int causal, void* stream) {
  if (!Q || !K || !Vt || !O || B <= 0 || H <= 0 || N <= 0) return fail(CID_ERR_ARG, "cid_attn_self: null pointer or empty problem");
  const int dp = d_pad_for(d);
  if (dp < 0) return fail(CID_ERR_UNSUPPORTED, "cid_attn_self: head dim %d unsupported (multiple of 8, <= 160)", d);
  if (N % 8) return fail(CID_ERR_UNSUPPORTED, "cid_attn_self: N=%d must be a multiple of 8", N);
  CUtensorMap tq, tk, tv; int rc;
  if ((rc = map_qk(&tq, Q, B, N, H, d, q_pitch, 128))) return rc;
  if ((rc = map_qk(&tk, K, B, N, H, d, k_pitch, 128))) return rc;
  AttnArgs a{}; a.B = B; a.H = H; a.Nq = N; a.Nkv = n_valid; a.d = d; a.scale_log2 = 1.4426950408889634f / sqrtf(float(d));
  a.O = O; a.ldo = ldo; a.is_bf16 = dtype == CID_BF16; a.causal = causal;
#ifdef CID_ATTN_TRACE
  a.trace = g_attn_trace;
#endif
  if ((rc = map_vt(&tv, Vt, B * H, d, N, dp))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (causal) {                    // the causal mask lives in the 128-query-tile kernel only, whatever N (launch_attn_self sends N >= 256 elsewhere)
    switch (dp) {
#define CID_ATTN_CAUSAL(DP) case DP: return a.is_bf16 ? launch_attn_self_t<DP, 1>(tq, tk, tv, a, st) : launch_attn_self_t<DP, 0>(tq, tk, tv, a, st);
      CID_ATTN_CAUSAL(32) CID_ATTN_CAUSAL(48) CID_ATTN_CAUSAL(64) CID_ATTN_CAUSAL(80) CID_ATTN_CAUSAL(128) CID_ATTN_CAUSAL(160)
#undef CID_ATTN_CAUSAL
    }
  }
  switch (dp) {
    case 32: return launch_attn_self<32>(tq, tk, tv, a, st);
    case 48: return launch_attn_self<48>(tq, tk, tv, a, st);
    case 64: return launch_attn_self<64>(tq, tk, tv, a, st);
    case 80: return launch_attn_self<80>(tq, tk, tv, a, st);
    case 128: return launch_attn_self<128>(tq, tk, tv, a, st);
    case 160: return launch_attn_self<160>(tq, tk, tv, a, st);
  }
  return fail(CID_ERR_UNSUPPORTED, "cid_attn_self: no instantiation for padded head dim %d", dp);
}

#ifdef CID_ATTN_TRACE
int cid_debug_set_attn_trace(long long* buf) { g_attn_trace = buf; return 0; }
#endif
#ifdef CID_GEMM_TRACE
int cid_debug_set_gemm_trace(long long* buf) { g_gemm_trace = buf; return 0; }
#endif

int cid_attn_cross(const void* Q, long long q_pitch, const void* Kcat, const void* Vtcat, void* O, long long ldo, int B, int H,
                   int N, int d, int n_text, int n_ip, float ip_scale, int dtype, void* stream) {
  if (!Q || !Kcat || !Vtcat || !O || B <= 0 || H <= 0 || N <= 0) return fail(CID_ERR_ARG, "cid_attn_cross: null pointer or empty problem");
  if (n_text <= 0 || n_text > (n_ip > 0 ? 80 : 96) || n_ip < 0 || n_ip > 16) return fail(CID_ERR_UNSUPPORTED, "cid_attn_cross: n_text=%d (<=80, or <=96 without id tokens), n_ip=%d (<=16)", n_text, n_ip);
  const int dp = d_pad_for(d);
  if (dp < 0) return fail(CID_ERR_UNSUPPORTED, "cid_attn_cross: head dim %d unsupported", d);
  CUtensorMap tq, tk, tv; int rc;
  if ((rc = map_qk(&tq, Q, B, N, H, d, q_pitch, 128))) return rc;
  if ((rc = map_qk(&tk, Kcat, B, 96, H, d, (long long)H * d, 96))) return rc;
  if ((rc = map_vt(&tv, Vtcat, B * H, d, 96, dp))) return rc;
  AttnArgs a{}; a.B = B; a.H = H; a.Nq = N; a.Nkv = 96; a.d = d; a.scale_log2 = 1.4426950408889634f / sqrtf(float(d));
  a.O = O; a.ldo = ldo; a.is_bf16 = dtype == CID_BF16; a.n_text = n_text; a.ip_off = 80; a.n_ip = n_ip; a.ip_scale = ip_scale;
#ifdef CID_ATTN_TRACE
  a.trace = g_attn_trace;
#endif
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#ifndef CID_CROSS_V1
  // persistent pipelined flavour wherever there is at least one unit per SM (smaller problems: one short CTA per unit is as good)
  const long long units = (long long)B * H * ((N + 127) / 128);
  // N > 128: with one query tile per (sample, head) the S stream (3 units ahead) would need a third K/V group in the 2-slot ring
  if (dp <= 80 && units >= num_sms() && N > 128 && g_cross2) {
    switch (dp) {
      case 32: return launch_attn_cross2<32>(tq, tk, tv, a, units, st);
      case 48: return launch_attn_cross2<48>(tq, tk, tv, a, units, st);
      case 64: return launch_attn_cross2<64>(tq, tk, tv, a, units, st);
      case 80: return launch_attn_cross2<80>(tq, tk, tv, a, units, st);
    }
  }
#endif
  switch (dp) {
    case 32: return launch_attn_cross<32>(tq, tk, tv, a, st);
    case 48: return launch_attn_cross<48>(tq, tk, tv, a, st);
    case 64: return launch_attn_cross<64>(tq, tk, tv, a, st);
    case 80: return launch_attn_cross<80>(tq, tk, tv, a, st);
    case 128: return launch_attn_cross<128>(tq, tk, tv, a, st);
    case 160: return launch_attn_cross<160>(tq, tk, tv, a, st);
  }
  return fail(CID_ERR_UNSUPPORTED, "cid_attn_cross: no instantiation for padded head dim %d", dp);
}

int cid_pack_cross_kv(const void* k_text, const void* v_text, const void* k_ip, const void* v_ip, void* k_cat, void* vt_cat,
                      int B, int C, int heads, int n_text, int n_ip, void* stream) {
  if (!k_text || !v_text || !k_cat || !vt_cat || (n_ip > 0 && (!k_ip || !v_ip))) return fail(CID_ERR_ARG, "cid_pack_cross_kv: null pointer");
  if (n_text > (n_ip > 0 ? 80 : 96) || n_ip > 16 || C % heads) return fail(CID_ERR_ARG, "cid_pack_cross_kv: bad sizes");
  const long long total = (long long)B * 96 * C;
  pack_cross_kv_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      (const uint16_t*)k_text, (const uint16_t*)v_text, (const uint16_t*)k_ip, (const uint16_t*)v_ip, (uint16_t*)k_cat,
      (uint16_t*)vt_cat, B, C, heads, n_text, n_ip, 80, 96);
  CID_CHECK_LAUNCH("pack_cross_kv_kernel");
  return 0;
}

int cid_gn_stats(const void* x1, int C1, const void* x2, int C2, int NB, int HW, int groups, float* sums, int zero_sums, int dtype, void* stream) {
  const int C = C1 + C2;
  if (!x1 || !sums || C1 % 8 || C2 % 8 || C % groups || (C2 > 0 && !x2)) return fail(CID_ERR_ARG, "cid_gn_stats: bad arguments (C1=%d C2=%d groups=%d)", C1, C2, groups);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (zero_sums) {
    cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(float) * 2 * NB * groups, st);
    if (e != cudaSuccess) return fail(CID_ERR_CUDA, "cid_gn_stats memset: %s", cudaGetErrorString(e));
  }
  const int V = C / 8;
  const int zchunks = (V + 255) / 256;
  int slabs = (148 * 8) / (NB * zchunks); if (slabs < 1) slabs = 1;
  const int tpp = 256 / (V < 256 ? V : 256);
  const int max_slabs = (HW + tpp - 1) / tpp; if (slabs > max_slabs) slabs = max_slabs;
  launch_pdl(gn_stats_kernel, dim3(slabs, NB, zchunks), dim3(256), 0, st, (const uint16_t*)x1, C1, (const uint16_t*)x2, C2, HW, groups, sums, int(dtype == CID_BF16));
  CID_CHECK_LAUNCH("gn_stats_kernel");
  return 0;
}
int cid_gn_apply(const void* x1, int C1, const void* x2, int C2, int NB, int HW, int groups, const float* sums, const void* gamma,
                 const void* beta, float eps, int silu, void* y, float* zero_next, int dtype, void* stream) {
  const int C = C1 + C2;
  if (!x1 || !sums || !gamma || !beta || !y || C1 % 8 || C2 % 8 || C % groups) return fail(CID_ERR_ARG, "cid_gn_apply: bad arguments");
  if (C > 4096) return fail(CID_ERR_UNSUPPORTED, "cid_gn_apply: C=%d > 4096", C);
  int slabs = grid_for((long long)HW * (C / 8), 256) / NB;
  if (slabs < 1) slabs = 1;
  launch_pdl(gn_apply_kernel, dim3(slabs, NB), dim3(256), 2 * C * sizeof(float), static_cast<cudaStream_t>(stream),
             (const uint16_t*)x1, C1, (const uint16_t*)x2, C2, HW, groups, sums, (const uint16_t*)gamma, (const uint16_t*)beta, eps, silu,
             (uint16_t*)y, zero_next, int(dtype == CID_BF16));
  CID_CHECK_LAUNCH("gn_apply_kernel");
  return 0;
}
int cid_gn_apply_ch(const void* x1, int C1, const float* sums1, const void* x2, int C2, const float* sums2, int NB, int HW, int groups,
                    const void* gamma, const void* beta, float eps, int silu, void* y, int dtype, void* stream) {
  const int C = C1 + C2;
  if (!x1 || !sums1 || !gamma || !beta || !y || C1 % 8 || C2 % 8 || C % groups || (C2 > 0 && (!x2 || !sums2))) return fail(CID_ERR_ARG, "cid_gn_apply_ch: bad arguments");
  if (C > 4096 || groups > 256) return fail(CID_ERR_UNSUPPORTED, "cid_gn_apply_ch: C=%d > 4096 or groups=%d > 256", C, groups);
  int slabs = grid_for((long long)HW * (C / 8), 256) / NB;
  if (slabs < 1) slabs = 1;
  launch_pdl(gn_apply_ch_kernel, dim3(slabs, NB), dim3(256), (4 * C + 2 * groups) * sizeof(float), static_cast<cudaStream_t>(stream),
             (const uint16_t*)x1, C1, sums1, (const uint16_t*)x2, C2, sums2, HW, groups, (const uint16_t*)gamma, (const uint16_t*)beta, eps, silu,
             (uint16_t*)y, int(dtype == CID_BF16));
  CID_CHECK_LAUNCH("gn_apply_ch_kernel");
  return 0;
}
int cid_gn_small(const void* x1, int C1, const void* x2, int C2, int NB, int HW, int groups, const void* gamma, const void* beta, float eps,
                 int silu, void* y, int dtype, void* stream) {
  const int C = C1 + C2;
  if (!x1 || !gamma || !beta || !y || groups <= 0 || C % groups || (C2 > 0 && !x2)) return fail(CID_ERR_ARG, "cid_gn_small: bad arguments");
  const int cpg = C / groups;
  if (cpg % 8 || C1 % cpg || (long long)HW * (cpg / 8) > 8LL * GN_SMALL_THREADS)
    return fail(CID_ERR_UNSUPPORTED, "cid_gn_small: needs 8 | C/groups (%d), groups aligned with the concat boundary (C1=%d) and HW*C/groups <= %d elements",
                cpg, C1, 64 * GN_SMALL_THREADS);
  const int total = HW * (cpg / 8);
  const dim3 grid(groups, NB);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define CID_GNS(V) launch_pdl(gn_small_kernel<V>, grid, dim3(GN_SMALL_THREADS), 0, st, (const uint16_t*)x1, C1, (const uint16_t*)x2, C2, HW, groups, \
                              (const uint16_t*)gamma, (const uint16_t*)beta, eps, silu, (uint16_t*)y, int(dtype == CID_BF16))
  if (total <= GN_SMALL_THREADS) CID_GNS(1);
  else if (total <= 2 * GN_SMALL_THREADS) CID_GNS(2);
  else if (total <= 4 * GN_SMALL_THREADS) CID_GNS(4);
  else CID_GNS(8);
#undef CID_GNS
  CID_CHECK_LAUNCH("gn_small_kernel");
  return 0;
}
int cid_layernorm(const void* x, const void* gamma, const void* beta, void* y, long long rows, int C, float eps, int dtype, void* stream) {
  if (!x || !gamma || !beta || !y || C % 8 || C > 2048) return fail(CID_ERR_ARG, "cid_layernorm: C=%d must be a multiple of 8 and <= 2048", C);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int V = C / 8;
  const int lpr = V <= 40 ? 8 : (V <= 80 ? 16 : 32);
  const long long groups = (rows + (32 / lpr) - 1) / (32 / lpr);                 // warp-iterations
  long long blocks = (groups + 7) / 8;
  const long long cap = 148LL * 3;                                                 // 3 resident 256-thread blocks per SM, warps loop
  const unsigned grid = (unsigned)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
#define CID_LN(L, P) launch_pdl(layernorm_kernel<L, P>, dim3(grid), dim3(256), 0, st, (const uint16_t*)x, (const uint16_t*)gamma, (const uint16_t*)beta, (uint16_t*)y, rows, C, eps, int(dtype == CID_BF16))
  if (lpr == 8) CID_LN(8, 5); else if (lpr == 16) CID_LN(16, 5); else CID_LN(32, 8);
#undef CID_LN
  CID_CHECK_LAUNCH("layernorm_kernel");
  return 0;
}
int cid_upsample2x(const void* x, void* y, int NB, int H, int W, int C, void* stream) {
  if (!x || !y || C % 8) return fail(CID_ERR_ARG, "cid_upsample2x: bad arguments");
  const long long total = (long long)NB * 4 * H * W * (C / 8);
  upsample2x_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((const uint4*)x, (uint4*)y, NB, H, W, C / 8, total);
  CID_CHECK_LAUNCH("upsample2x_kernel");
  return 0;
}
int cid_phase_split(const void* x, void* y, int NB, int H, int W, int C, void* stream) {
  if (!x || !y || C % 8 || H % 2 || W % 2) return fail(CID_ERR_ARG, "cid_phase_split: needs even H, W and C %% 8 == 0");
  const long long total = (long long)NB * H * W * (C / 8);
  phase_split_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((const uint4*)x, (uint4*)y, NB, H, W, C / 8, total);
  CID_CHECK_LAUNCH("phase_split_kernel");
  return 0;
}
int cid_nchw_to_nhwc_pad(const void* x, void* y, int NB, int Cin, int HW, int CP, const float* scale_dev, int dtype, void* stream) {
  if (!x || !y || CP % 8 || CP < Cin) return fail(CID_ERR_ARG, "cid_nchw_to_nhwc_pad: bad arguments");
  const long long total = (long long)NB * HW * (CP / 8);
  nchw_to_nhwc_pad_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((const uint16_t*)x, (uint16_t*)y, NB, Cin, HW, CP, scale_dev, dtype == CID_BF16);
  CID_CHECK_LAUNCH("nchw_to_nhwc_pad_kernel");
  return 0;
}
int cid_rows_to_nchw(const void* x, int ld, void* y, int NB, int Cout, int HW, void* stream) {
  if (!x || !y) return fail(CID_ERR_ARG, "cid_rows_to_nchw: null pointer");
  const long long total = (long long)NB * Cout * HW;
  rows_to_nchw_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((const uint16_t*)x, ld, (uint16_t*)y, NB, Cout, HW);
  CID_CHECK_LAUNCH("rows_to_nchw_kernel");
  return 0;
}
int cid_add_inplace(void* y, const void* x, long long n_elems, int dtype, void* stream) {
  if (!x || !y || n_elems % 8) return fail(CID_ERR_ARG, "cid_add_inplace: n_elems must be a multiple of 8");
  add_inplace_kernel<<<grid_for(n_elems / 8, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((uint4*)y, (const uint4*)x, n_elems / 8, dtype == CID_BF16);
  CID_CHECK_LAUNCH("add_inplace_kernel");
  return 0;
}
int cid_silu_inplace(void* y, long long n_elems, int dtype, void* stream) {
  if (!y || n_elems % 8) return fail(CID_ERR_ARG, "cid_silu_inplace: n_elems must be a multiple of 8");
  silu_inplace_kernel<<<grid_for(n_elems / 8, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((uint4*)y, n_elems / 8, dtype == CID_BF16);
  CID_CHECK_LAUNCH("silu_inplace_kernel");
  return 0;
}
int cid_embed_tokens(const long long* ids, int B, int L, int Lp, const void* tok, long long V, const void* pos, void* out, int C, int dtype,
                     void* stream) {
  if (!ids || !tok || !pos || !out || B <= 0 || L <= 0 || Lp < L || V <= 0 || C <= 0 || C % 8)
    return fail(CID_ERR_ARG, "cid_embed_tokens: need B, L, V > 0, Lp >= L and C %% 8 == 0 (B=%d L=%d Lp=%d C=%d)", B, L, Lp, C);
  const long long total = (long long)B * Lp * (C / 8);
  embed_tokens_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      ids, L, Lp, (const uint4*)tok, V, (const uint4*)pos, (uint4*)out, C / 8, total, dtype == CID_BF16);
  CID_CHECK_LAUNCH("embed_tokens_kernel");
  return 0;
}
int cid_inpaint_blend(float* x, void* x16, const float* image_latents, const float* noise, const float* mask, int B, int HW,
                      const float* blend_table, const int* step_dev, int dtype, void* stream) {
  if (!x || !x16 || !image_latents || !noise || !mask || !blend_table || !step_dev) return fail(CID_ERR_ARG, "cid_inpaint_blend: null pointer");
  inpaint_blend_kernel<<<grid_for((long long)B * 4 * HW, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, (uint16_t*)x16, image_latents, noise, mask, B, HW, blend_table, step_dev, dtype == CID_BF16);
  CID_CHECK_LAUNCH("inpaint_blend_kernel");
  return 0;
}
int cid_timestep_embed(const float* t_dev, int t_stride, int rows, int dim, void* out, long long ld, int col0, int dtype, void* stream) {
  if (!t_dev || !out || dim % 2) return fail(CID_ERR_ARG, "cid_timestep_embed: bad arguments");
  timestep_embed_kernel<<<grid_for((long long)rows * dim / 2, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(t_dev, t_stride, rows, dim, (uint16_t*)out, ld, col0, dtype == CID_BF16);
  CID_CHECK_LAUNCH("timestep_embed_kernel");
  return 0;
}
int cid_skinny_linear(const void* x, long long ldx, const void* W, const void* bias, void* y, long long ldy, int M, int N, int K,
                      int silu_in, int accumulate, int dtype, void* stream) {
  if (!x || !W || !y || K % 8 || K > 8192 || M <= 0) return fail(CID_ERR_ARG, "cid_skinny_linear: K=%d must be a multiple of 8 and <= 8192", K);
  const int slab = K <= 4096 ? 16 : 8;           // rows of x staged per pass: slab * K * 2 bytes of shared memory (<= 128 KB)
  static bool configured[MAX_DEVICES] = {};
  if (int rc = set_smem(skinny_linear2_kernel, 16 * 4096 * 2, "skinny_linear2_kernel", configured)) return rc;
  skinny_linear2_kernel<<<(N + 7) / 8, 256, (size_t)slab * K * 2, static_cast<cudaStream_t>(stream)>>>(
      (const uint16_t*)x, ldx, (const uint16_t*)W, (const uint16_t*)bias, (uint16_t*)y, ldy, M, N, K, silu_in, accumulate, dtype == CID_BF16, slab);
  CID_CHECK_LAUNCH("skinny_linear2_kernel");
  return 0;
}
int cid_cfg_sched_step(const void* eps, int ld_eps, float* x, float* x0_prev, void* x16, void* next_in, int CP, int B, int HW,
                       float guidance, const float* coef_table, const int* step_dev, int dtype, void* stream) {
  if (!eps || !x || !x0_prev || !x16 || !coef_table || !step_dev || ld_eps % 4 || (next_in && CP % 8)) return fail(CID_ERR_ARG, "cid_cfg_sched_step: bad arguments");
  cfg_sched_step_kernel<<<grid_for((long long)B * HW, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      (const uint16_t*)eps, ld_eps, x, x0_prev, (uint16_t*)x16, (uint16_t*)next_in, CP, B, HW, guidance, coef_table, step_dev, dtype == CID_BF16);
  CID_CHECK_LAUNCH("cfg_sched_step_kernel");
  return 0;
}
int cid_latents_to_input(const float* x, void* next_in, int CP, int B, int HW, const float* coef_table, const int* step_dev, int nsteps,
                         int keep_ch4_up, int dtype, void* stream) {
  if (!x || !next_in || !coef_table || CP % 8 || nsteps <= 0) return fail(CID_ERR_ARG, "cid_latents_to_input: bad arguments");
  latents_to_input_kernel<<<grid_for((long long)B * HW, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, (uint16_t*)next_in, CP, B, HW, coef_table, step_dev, nsteps, keep_ch4_up, dtype == CID_BF16);
  CID_CHECK_LAUNCH("latents_to_input_kernel");
  return 0;
}

int cid_advance_step(int* step_dev, float* t_dev, const float* ts_table, int n, void* stream) {
  if (!step_dev || !t_dev || !ts_table || n <= 0) return fail(CID_ERR_ARG, "cid_advance_step: bad arguments");
  advance_step_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(step_dev, t_dev, ts_table, n);
  CID_CHECK_LAUNCH("advance_step_kernel");
  return 0;
}

int cid_set_splitk(int max_split, int min_kblocks) {
  if (max_split > 64) return fail(CID_ERR_ARG, "cid_set_splitk: max_split=%d > 64", max_split);
  g_splitk_max = max_split < 0 ? 4 : max_split;               // negative: back to the measured default; 0 / 1 disables splitting
  g_splitk_min_kb = min_kblocks < 0 ? 48 : (min_kblocks == 0 ? 1 : min_kblocks);
  return 0;
}

int cid_layernorm_rows(const void* x, long long ldx, long long x_group_rows, long long x_row0, const void* gamma, const void* beta, void* y,
                       long long ldy, long long y_group_rows, long long y_row0, long long rows, long long rows_per_group, int C, float eps,
                       int dtype, void* stream) {
  if (!x || !gamma || !beta || !y || C <= 0 || C % 8 || ldx % 8 || ldy % 8 || rows_per_group <= 0)
    return fail(CID_ERR_ARG, "cid_layernorm_rows: C=%d, ldx, ldy must be multiples of 8 and rows_per_group > 0", C);
  if (rows <= 0) return 0;
  layernorm_rows_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      (const uint16_t*)x, ldx, x_group_rows, x_row0, (const uint16_t*)gamma, (const uint16_t*)beta, (uint16_t*)y, ldy, y_group_rows, y_row0, rows,
      rows_per_group, C, eps, dtype == CID_BF16);
  CID_CHECK_LAUNCH("layernorm_rows_kernel");
  return 0;
}

int cid_softmax_rows(void* x, long long ld, long long rows, int cols, int dtype, void* stream) {
  if (!x || cols <= 0 || cols % 8 || ld % 8 || ld < cols || rows < 0 || rows > 0x7fffffffLL)
    return fail(CID_ERR_ARG, "cid_softmax_rows: cols=%d and ld must be multiples of 8, ld >= cols", cols);
  if (rows == 0) return 0;
  softmax_rows_kernel<<<(unsigned)rows, 256, 0, static_cast<cudaStream_t>(stream)>>>((uint16_t*)x, ld, cols, dtype == CID_BF16);
  CID_CHECK_LAUNCH("softmax_rows_kernel");
  return 0;
}

int cid_perceiver_attn(const void* q, long long ldq, const void* kv, long long ldkv, void* out, long long ldo, int B, int L, int n_kv, int heads,
                       int dim_head, int dtype, void* stream) {
  if (!q || !kv || !out || dim_head != 64 || B <= 0 || L <= 0 || heads <= 0 || n_kv <= 0 || n_kv > 8192 || ldkv % 8)
    return fail(CID_ERR_ARG, "cid_perceiver_attn: dim_head must be 64, 0 < n_kv <= 8192, ldkv %% 8 == 0 (got dim_head=%d n_kv=%d)", dim_head, n_kv);
  perceiver_attn_kernel<<<(unsigned)(B * L * heads), 128, (size_t)n_kv * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      (const uint16_t*)q, ldq, (const uint16_t*)kv, ldkv, (uint16_t*)out, ldo, L, n_kv, heads, dtype == CID_BF16);
  CID_CHECK_LAUNCH("perceiver_attn_kernel");
  return 0;
}

}  // extern "C"
