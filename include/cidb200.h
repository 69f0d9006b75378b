/* cidb200 - C ABI of the B200-native ConsistentID denoising hot path (libcidb200.so).
 *
 * The reference has NO C ABI for this path: its arithmetic is reached through Python objects
 *   - diffusers AttnProcessor protocol   attention.py:110-117 / :207-215 (processor __call__)
 *   - unet(...).sample                   pipline_StableDiffusion_ConsistentID.py:552-557,
 *                                        pipline_StableDiffusionXL_ConsistentID.py:634-641
 *   - scheduler.scale_model_input/step   pipline_StableDiffusion_ConsistentID.py:540, 569-571
 * and its only native binding is a pybind11 module of dead code (models/BiSeNet/modules/src/inplace_abn.cpp:86-95).
 * This header therefore DEFINES the boundary a replacement binds to; each entry point names the reference
 * lines whose arithmetic it replaces.  INTEGRATION.md shows the ctypes stub on the reference side.
 *
 * Conventions: every pointer is a DEVICE pointer (16-byte aligned) unless stated otherwise; activations are
 * 16-bit (dtype 0 = fp16, 1 = bf16), row-major [rows, channels] == NHWC; `ld*`/pitches are in ELEMENTS;
 * `stream` is a cudaStream_t.  Functions never allocate, free or synchronise; they return 0 on success or a
 * negative cid_status and set a thread-local message readable with cid_last_error().  All of them are
 * CUDA-graph capturable.
 */
#ifndef CIDB200_H
#define CIDB200_H
#ifdef __cplusplus
extern "C" {
#endif

typedef enum { CID_OK = 0, CID_ERR_ARG = -1, CID_ERR_CUDA = -2, CID_ERR_UNSUPPORTED = -3, CID_ERR_DRIVER = -4 } cid_status;
typedef enum { CID_F16 = 0, CID_BF16 = 1 } cid_dtype;
typedef enum { CID_EPI_STORE = 0, CID_EPI_GEGLU = 1, CID_EPI_QKV = 2, CID_EPI_GELU = 3, CID_EPI_QUICK_GELU = 4 } cid_epilogue;

int cid_version(void);
const char* cid_last_error(void);
/* Workspace convention (cid_gemm / cid_conv3x3): `workspace` is caller-owned scratch for the tail balancing (split-K partial accumulators +
 * arrival counters), passed PER CALL: a device buffer, 256-byte aligned, >= 4 KB (24 MB covers every shape of the SD / SDXL UNets), that the
 * caller zero-fills ONCE before first use (the kernels re-arm the counters themselves) and does not share between streams that may run
 * concurrently.  NULL / 0: tiles are never split (same results, idle SMs in the last wave).  The library keeps no pointer to it.
 *
 * Tail-balancing policy: a tail tile is cut into at most max_split K-ranges of at least min_kblocks 64-wide k-blocks each (defaults 4 / 48);
 * max_split <= 1 disables splitting, negative values restore the defaults.  A process-wide POLICY knob, not state: results do not depend on it
 * beyond fp32 summation order. */
int cid_set_splitk(int max_split, int min_kblocks);
/* N-tile width the GEMM will use for (N, epilogue): GEGLU weights must be row-interleaved per tile of this width. */
int cid_gemm_tile_n(int N, int epi);

/* C[M,N] = epi( [A | A2][M, K1+K2] . B[N, K1+K2]^T + bias[N] + rowbias[row / rows_per_group, N] + residual[M,N] ) * out_scale
 * Replaces: attn.to_q/to_k/to_v/to_out (+ LoRA folded) attention.py:138-146,162,236-250,282; BasicTransformerBlock
 * GEGLU / FF linears, Transformer2D proj_in/out, ResnetBlock2D 1x1 conv_shortcut (diffusers 0.23; SURVEY A.3-A.4).
 *   epi = GEGLU : B rows interleaved per tile (value half | gate half); writes C[M, N/2] = v * gelu(g).
 *   epi = QKV   : columns >= n_split are V and are written TRANSPOSED to Vt[(row/ntok)*heads + h, dd, row%ntok].
 *   epi = GELU  : C = gelu_erf(acc + bias (+ residual)) - the fc1 + activation of the CLIP vision MLP (SURVEY 8f-4).
 *   epi = QUICK_GELU : C = q(acc + bias (+ residual)), q(x) = x * sigmoid(1.702 x) in fp32 - the fc1 + activation of the OpenAI CLIP
 *                 ViT-L/14 text MLP (hidden_act "quick_gelu").
 *   chan_stats  : non-NULL (plain store epilogue only) = GroupNorm statistics of the OUTPUT fused into the epilogue: per (sample, column)
 *                 sum and sum of squares are ADDED to chan_stats[(row / stats_rows) * N + col][2] (fp32, zeroed by the caller); stats_rows =
 *                 rows per sample, a multiple of 128.  Consumed by cid_gn_apply_ch: the standalone statistics pass (one re-read of the
 *                 tensor per GroupNorm) disappears.
 *   LayerNorm folded into the GEMMs around it (BasicTransformerBlock norm1/2/3: no standalone LayerNorm pass):
 *   row_stats   : non-NULL (plain store epilogue only) = the PRODUCER side: per-row sum and sum of squares of the stored row are ADDED to
 *                 row_stats[row][2] (fp32, zeroed by the caller);
 *   ln_stats    : non-NULL = the CONSUMER side: A holds the un-normalised rows, B = W . diag(gamma) (16-bit), bias = b + W . beta and
 *                 ln_colsum[c] = sum_k B[c,k] (fp32, of the ROUNDED B); the epilogue forms rstd_r (A_r . B_c - mean_r colsum_c) + bias_c with
 *                 mean / rstd of row r from ln_stats[r] over K1 + K2 elements and ln_eps - exactly LayerNorm(A) W^T + b in fp32. */
int cid_gemm(const void* A, long long lda, const void* A2, long long lda2, int K1, int K2, const void* B,
             void* C, long long ldc, int M, int N, const void* bias, const void* residual, long long ldr,
             const void* rowbias, int rows_per_group, long long ld_rowbias, int epi, void* Vt, int n_split, int heads,
             int hdim, int ntok, float out_scale, int dtype, void* workspace, unsigned long long ws_bytes, float* chan_stats,
             int stats_rows, float* row_stats, const float* ln_stats, const float* ln_colsum, float ln_eps, void* stream);

/* 3x3 convolution, padding 1, as implicit GEMM over NHWC.  X: [NB,H,W,Cin] (stride 1) or the phase-split copy
 * [NB,4,H,W,Cin] of a [NB,2H,2W,Cin] tensor (stride2 = 1; H,W are OUTPUT dims).  Wt: [Cout, 9*Cin] = (ky,kx,c) order.
 * Y[NB*H*W, ldy].  Replaces ResnetBlock2D.conv1/conv2, Downsample2D.conv, Upsample2D.conv, conv_in, conv_out.
 * chan_stats as in cid_gemm (rows per sample = H*W; needs H*W >= 128 so that no 128-pixel tile spans two samples). */
int cid_conv3x3(const void* X, const void* Wt, void* Y, long long ldy, int NB, int H, int W, int Cin, int Cout,
                int stride2, const void* bias, const void* residual, long long ldr, const void* rowbias,
                long long ld_rowbias, float out_scale, int dtype, void* workspace, unsigned long long ws_bytes, float* chan_stats, void* stream);

/* softmax(Q K^T / sqrt(d)) V per (sample, head).  Q,K: [B,N,H,d] views with row pitch q_pitch/k_pitch;
 * Vt: [B*H, d, N] (keys contiguous); O: [B,N,H*d] pitch ldo.  Replaces attention.py:152-159. */
int cid_attn_self(const void* Q, long long q_pitch, const void* K, long long k_pitch, const void* Vt, void* O,
                  long long ldo, int B, int H, int N, int d, int dtype, void* stream);

/* Decoupled text + id cross-attention: O = softmax(Q Kt^T) Vt + ip_scale * softmax(Q Ki^T) Vi, with
 * Kcat [B, 96, H*d] (rows [0,n_text) text, [80,80+n_ip) id, others zero) and Vtcat [B*H, d, 96].
 * Replaces attention.py:259-279.  n_text <= 80 (<= 96 without id tokens), n_ip <= 16.  Head dims <= 80 with at least one 128-query
 * tile per SM and N > 128 run the persistent pipelined kernel (both softmaxes normalised before ONE P.V accumulation: the 16-bit
 * rounding the reference applies to each branch before the mix sits on the probabilities); other shapes the per-tile kernel that
 * rounds each branch as the reference does.  Both are covered by the processor golden vectors. */
int cid_attn_cross(const void* Q, long long q_pitch, const void* Kcat, const void* Vtcat, void* O, long long ldo,
                   int B, int H, int N, int d, int n_text, int n_ip, float ip_scale, int dtype, void* stream);
int cid_pack_cross_kv(const void* k_text, const void* v_text, const void* k_ip, const void* v_ip, void* k_cat,
                      void* vt_cat, int B, int C, int heads, int n_text, int n_ip, void* stream);

/* GroupNorm over cat([x1 (C1), x2 (C2)]) NHWC: stats accumulate into sums[NB, groups, 2] (fp32; zeroed by the call when zero_sums != 0,
 * otherwise the caller guarantees zeros), then y = [silu](gn(x)); gn_apply also zeroes zero_next[NB, groups, 2] when non-NULL - two
 * alternating buffers then need one memset per forward instead of one per GroupNorm.
 * Replaces ResnetBlock2D.norm1/norm2 + nonlinearity, Transformer2D.norm, conv_norm_out + conv_act. */
int cid_gn_stats(const void* x1, int C1, const void* x2, int C2, int NB, int HW, int groups, float* sums, int zero_sums, int dtype,
                 void* stream);
int cid_gn_apply(const void* x1, int C1, const void* x2, int C2, int NB, int HW, int groups, const float* sums,
                 const void* gamma, const void* beta, float eps, int silu, void* y, float* zero_next, int dtype, void* stream);
/* gn_apply with the statistics given per (sample, channel) by the producers' epilogues (cid_gemm / cid_conv3x3 chan_stats): sums1[NB, C1, 2] for
 * x1, sums2[NB, C2, 2] for x2 (NULL when C2 == 0).  Group statistics are formed on the fly (the 32 groups do not align with the concat boundary). */
int cid_gn_apply_ch(const void* x1, int C1, const float* sums1, const void* x2, int C2, const float* sums2, int NB, int HW, int groups,
                    const void* gamma, const void* beta, float eps, int silu, void* y, int dtype, void* stream);
/* GroupNorm(+SiLU) of small tensors in ONE pass (one CTA per (sample, group), the slab held in registers): for tensors whose statistics cannot
 * ride on the producer's epilogue (HW not a multiple of 128: the 8x8 level).  Requires 8 | C/groups, C1 a multiple of C/groups and
 * HW * C/groups <= 32768 elements; CID_ERR_UNSUPPORTED otherwise (use cid_gn_stats + cid_gn_apply). */
int cid_gn_small(const void* x1, int C1, const void* x2, int C2, int NB, int HW, int groups, const void* gamma, const void* beta, float eps,
                 int silu, void* y, int dtype, void* stream);
int cid_layernorm(const void* x, const void* gamma, const void* beta, void* y, long long rows, int C, float eps, int dtype, void* stream);
int cid_upsample2x(const void* x, void* y, int NB, int H, int W, int C, void* stream);
int cid_phase_split(const void* x, void* y, int NB, int H, int W, int C, void* stream);
int cid_nchw_to_nhwc_pad(const void* x, void* y, int NB, int Cin, int HW, int CP, const float* scale_dev, int dtype, void* stream);
int cid_rows_to_nchw(const void* x, int ld, void* y, int NB, int Cout, int HW, void* stream);
int cid_add_inplace(void* y, const void* x, long long n_elems, int dtype, void* stream);

/* diffusers get_timestep_embedding(flip_sin_to_cos=True, freq_shift=0); t read from device memory. */
int cid_timestep_embed(const float* t_dev, int t_stride, int rows, int dim, void* out, long long ld, int col0, int dtype, void* stream);
/* y[M,N] (+)= act(x)[M,K] . W[N,K]^T + b for small M (time_embedding, add_embedding, all time_emb_proj at once; the latent-row linears of the
 * embedding producers).  silu_in selects act: 0 identity, 1 SiLU, 2 GELU(erf). */
int cid_skinny_linear(const void* x, long long ldx, const void* W, const void* bias, void* y, long long ldy, int M, int N,
                      int K, int silu_in, int accumulate, int dtype, void* stream);

/* Fused CFG combine + scheduler step + next-step UNet input (pipline_StableDiffusion_ConsistentID.py:537-540,560-571).
 * coef_table: device [steps, 8] fp32 rows {cx, ce, cp, kx, ke, in_scale_next, in_scale_this, 0}; step index from device. */
int cid_cfg_sched_step(const void* eps, int ld_eps, float* x, float* x0_prev, void* x16, void* next_in, int CP, int B,
                       int HW, float guidance, const float* coef_table, const int* step_dev, int dtype, void* stream);
/* in-graph step bookkeeping: *step_dev += 1; *t_dev = ts_table[min(*step_dev, n-1)] */
int cid_advance_step(int* step_dev, float* t_dev, const float* ts_table, int n, void* stream);
/* fp32 master latents -> scaled, batch-duplicated NHWC UNet input for the step *step_dev (NULL = step 0);
 * keep_ch4_up = 1 writes channels 0-3 only (9-channel inpaint UNet keeps mask / masked-latent channels). */
int cid_latents_to_input(const float* x, void* next_in, int CP, int B, int HW, const float* coef_table, const int* step_dev, int nsteps,
                         int keep_ch4_up, int dtype, void* stream);
/* y = silu(y) */
int cid_silu_inplace(void* y, long long n_elems, int dtype, void* stream);
/* inpaint blend after a scheduler step (pipelines/StableDIffusionControlNetInpaint_ConsistentID.py:437-449):
 * x = (1-m) * (ca*image_latents + cn*noise) + m*x with {ca,cn} = blend_table[*step_dev] */
int cid_inpaint_blend(float* x, void* x16, const float* image_latents, const float* noise, const float* mask, int B, int HW,
                      const float* blend_table, const int* step_dev, int dtype, void* stream);

/* ---- embedding producers (SURVEY.md 8f-1): the modules that write encoder_hidden_states = [77 fused text rows | 4 id rows] ---- */
/* LayerNorm with grouped row mapping: logical row r = g*rows_per_group + i reads x row (g*x_group_rows + x_row0 + i) (pitch ldx) and writes
 * y row (g*y_group_rows + y_row0 + i) (pitch ldy): norm1(x) / norm2(latents) of PerceiverAttention land directly in the concatenated
 * key/value input (functions.py:434-444); also MLP.layernorm / FuseModule.layer_norm (attention.py:21,54) and FeedForward[0]. */
int cid_layernorm_rows(const void* x, long long ldx, long long x_group_rows, long long x_row0, const void* gamma, const void* beta, void* y,
                       long long ldy, long long y_group_rows, long long y_row0, long long rows, long long rows_per_group, int C, float eps,
                       int dtype, void* stream);
/* PerceiverAttention core (functions.py:446-453): per (sample, head, latent) softmax_fp32((q*s)(k*s)^T) v with s = dim_head^-1/4, dim_head 64.
 * q [B*L, ldq]; kv [B*n_kv, ldkv] = to_kv output (K columns [0,heads*64), V columns [heads*64, 2*heads*64)); out [B*L, ldo]. */
int cid_perceiver_attn(const void* q, long long ldq, const void* kv, long long ldkv, void* out, long long ldo, int B, int L, int n_kv, int heads,
                       int dim_head, int dtype, void* stream);

/* cid_attn_self on buffers of N tokens per sample (N % 8 == 0) of which only the first n_valid are real keys: the rest are masked out of the
 * softmax (CLIP ViT-H/14: 257 tokens in 264-row buffers; transformers CLIPAttention behind
 * pipline_StableDiffusion_ConsistentID.py:182-183, 202-203).  Rows >= n_valid of O are computed but meaningless. */
int cid_attn_self_ragged(const void* Q, long long q_pitch, const void* K, long long k_pitch, const void* Vt, void* O, long long ldo,
                         int B, int H, int N, int n_valid, int d, int dtype, void* stream);
/* cid_attn_self with the causal mask of the CLIP text transformer: softmax(Q K^T / sqrt(d) + mask) V where query row q sees keys 0..q, so
 * every row has at least one key.  Same arguments and layouts as cid_attn_self (N % 8 == 0, head dims multiple of 8 up to 160).  Runs the
 * 128-query-tile kernel for every N; key tiles above the diagonal are never loaded.  Rows of a sequence padded from L to N tokens never read
 * the pad keys, but pad V rows must hold finite values (masked probabilities are zeros that still multiply them). */
int cid_attn_self_causal(const void* Q, long long q_pitch, const void* K, long long k_pitch, const void* Vt, void* O, long long ldo,
                         int B, int H, int N, int d, int dtype, void* stream);

/* ---- CLIP text encoder ---- */
/* Token + position embedding gather: out[b*Lp + i, :] = tok[ids[b*L + i], :] + pos[i, :] for i < L, and zero rows for L <= i < Lp.
 * ids: int64 [B, L] device array (what tokenizers return); tok: [V, C], pos: [>= L, C], out: [B*Lp, C], all 16-bit, C % 8 == 0.
 * An id outside [0, V) is never dereferenced: it contributes a zero token row (out = pos[i]). */
int cid_embed_tokens(const long long* ids, int B, int L, int Lp, const void* tok, long long V, const void* pos, void* out, int C, int dtype,
                     void* stream);

/* ---- VAE decode (SURVEY.md 8f-3): everything but this reuses cid_conv3x3 / cid_gemm / cid_gn_* / cid_upsample2x ---- */
/* In-place softmax over each row of x[rows, cols] (pitch ld), fp32 math: probabilities of the single-head d=512 attention of the VAE mid
 * block (diffusers Attention, upcast_softmax), between the Q.K^T and P.V cid_gemm launches. */
int cid_softmax_rows(void* x, long long ld, long long rows, int cols, int dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif
