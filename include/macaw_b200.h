/*
 * macaw_b200.h — C ABI of libmacaw_b200.so, the sm_100a kernel library behind the MM_LLMs forward hot path.
 *
 * The reference (lyuchenyang/Macaw-LLM) has no FFI layer of its own: its hot path is Python calling
 * torch / transformers modules (SURVEY.md §8b).  Each entry point below therefore cites the reference
 * call site(s) whose arithmetic it replaces; the Python host code in macaw-llm_b200/ binds them with
 * ctypes (INTEGRATION.md shows the stub a maintainer of the reference would add).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; mm_last_error() returns a message for the
 *     calling thread.  No exceptions cross this boundary and nothing here calls cudaMalloc.
 *   - all pointers are DEVICE pointers owned by the caller (torch's caching allocator in practice).
 *   - `stream` is a cudaStream_t passed as void*; all calls are asynchronous and never synchronise.
 *   - "bf16" means 16-bit bfloat16 storage, row-major unless a leading dimension says otherwise; all
 *     accumulation is fp32.
 */
#ifndef MACAW_B200_H_
#define MACAW_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------ meta */
const char* mm_last_error(void);
int32_t mm_abi_version(void);
/* Content hash of the kernel sources + this header the library was built from (the loader compares it with the sources
 * on disk and rebuilds on mismatch, so a stale library never meets a newer struct layout). */
const char* mm_build_hash(void);
/* Number of kernel launches issued through this library by the calling process since the last reset. */
int64_t mm_launch_count(void);
void mm_launch_count_reset(void);
/* 16-bit storage format of activations and parameters for the CALLING THREAD: 0 = bf16 (default), 1 = fp16 (IEEE half).
 * Wherever this header says "bf16" for an activation / parameter tensor, the tensor is fp16 while the format is 1.  The
 * reference itself trains and runs in fp16 (train.sh:36 `--fp16 True`, llm_trainer.py:366-368 `.half()`); an fp16 model is
 * computed in fp16 (11-bit significands: storage rounding 8x smaller than bf16), a bf16 model in bf16.  mm_gemm_fwd and
 * mm_align_fwd take their operand formats explicitly; they use this flag for the epilogue's bias / residual tensors. */
void mm_set_act_format(int32_t f16);
int32_t mm_get_act_format(void);

/* ------------------------------------------------------------------------------------------------ GEMM
 * C[b] = epilogue( alpha * A[b] (M x K, K contiguous) * B[b]^T ) for b in [0, batch).
 * Replaces every nn.Linear / Conv-as-matmul / bmm on the path:
 *   LLaMA q/k/v/o/gate/up/down/lm_head   modeling.py:134-140, 159-162, 179-181, 226, 597
 *   alignment MHA in/out projections      modeling.py:986-987, 1007-1008, 1025-1026 -> torch F.multi_head_attention_forward
 *   Conv1d down-samplers, Linear C->E     modeling.py:982-984, 999-1001, 1022-1024
 *   CLIP / Whisper encoder linears, convs  modeling.py:1073, 1082, 1092 -> transformers modeling_clip / modeling_whisper
 * Implementation: persistent, warp-specialised TMA -> tcgen05.mma (TMEM accumulators) kernel.
 */
enum {
  MM_ACT_NONE = 0,
  MM_ACT_GELU = 1,        /* exact erf GELU (Whisper) */
  MM_ACT_QUICK_GELU = 2,  /* x * sigmoid(1.702 x) (CLIP) */
  MM_ACT_SILU = 3
};
enum {
  MM_EPI_STD = 0,    /* bias / activation / residual */
  MM_EPI_SWIGLU = 1, /* B rows interleaved [32 gate | 32 up]; C[:, j] = silu(gate_j) * up_j, N_out = N/2 */
  MM_EPI_ROPE = 2    /* rotate-half RoPE (head_dim 128) on columns < rope_cols, pos = row % rope_T */
};

typedef struct mm_gemm_args {
  /* problem: batch (inner) x batch2 (outer, 0 or 1 = none) independent products */
  int32_t M, N, K, batch, batch2;
  /* A: bf16 [batch][M][K], row stride lda (elements), batch stride a_bs (elements; rows may overlap) */
  const void* A;
  int64_t lda, a_bs, a_bs2;
  /* B: bf16.  b_mn_major == 0: [batch][N][K] (K contiguous, i.e. an nn.Linear weight), row stride ldb.
   *           b_mn_major == 1: [batch][K][N] (N contiguous), row stride ldb.  b_bs == 0 shares B across batch. */
  const void* B;
  int64_t ldb, b_bs, b_bs2;
  int32_t b_mn_major;
  /* C: bf16 (c_fp32 == 0) or fp32 (c_fp32 == 1) [batch][M][N_out], row stride ldc */
  void* C;
  int64_t ldc, c_bs, c_bs2;
  int32_t c_fp32;
  /* epilogue */
  int32_t epi;            /* MM_EPI_* */
  int32_t act;            /* MM_ACT_* (MM_EPI_STD only) */
  float alpha;
  const void* bias;       /* bf16 [N] or NULL; bias_bs = per-batch stride in elements */
  int64_t bias_bs;
  const float* row_scale; /* fp32 [batch2*batch*M] or NULL: multiplies row m of the product before bias */
  const void* residual;   /* bf16, added after activation; row index = m % res_row_mod if res_row_mod > 0 */
  int64_t ldr, r_bs, r_bs2;
  int32_t res_row_mod;
  const float* rope_cos;  /* fp32 [rope_T][64] */
  const float* rope_sin;
  int32_t rope_T, rope_cols;
  const int32_t* rope_pos; /* NULL, or device int added to every row's position (decode steps replayed from a CUDA graph) */
  int32_t c_trans; /* 1: C and residual are addressed transposed (C[n][m], row stride ldc), bias is indexed by m, row_scale by n:
                      lets a caller swap the operands (A = weight rows, B = a handful of activation rows) so that thin
                      decode GEMMs fill the 128-row MMA tile with weights (standard epilogue, batch == 1) */
  /* 16-bit operand formats: 0 = bf16 (default), 1 = fp16 (IEEE half).  A and B must agree: the instruction descriptor has
   * independent format fields, but sm_100a raises an illegal-instruction fault for f16 x bf16 (measured, round 2).
   * The alignment chain runs in fp16 (11-bit significand: one stored stage costs 1.4e-4 norm-wise instead of bf16's
   * 1.1e-3) against fp16 COPIES of its weights and of the embedding table (exact conversions of the bf16 values). */
  int32_t a_fp16, b_fp16;
  int32_t c_fp16; /* 1: C is fp16 (c_fp32 must be 0) */
  /* MM_EPI_STD only: out += bias_rs[b*M + m] * bias[n] (when bias_rs != NULL the bias term is scaled per row) and
   * out += bias2_rs[b*M + m] * bias2[n].  Value-side bias terms of the absorbed alignment attention
   * (functional.py:6531-6537: b_v rides on every real key, bias_v on the appended key). bias2 shares bias_bs. */
  const float* bias_rs;
  const void* bias2;
  const float* bias2_rs;
  /* 1: A is given as [batch][K][M] (M contiguous, row stride lda) — the transpose of a row-major activation.  With
   * b_mn_major this is the weight-gradient product dW[n][k] = sum_m dY[m][n] X[m][k] on the tensors as stored
   * (reference: autograd of every nn.Linear on the path; llm_trainer.py:184-188 -> loss.backward()). */
  int32_t a_mn_major;
  /* RMSNorm statistics without a separate pass over the residual stream (LlamaRMSNorm modeling.py:311-319):
   * sumsq_out (MM_EPI_STD, 16-bit C): fp32 [M][ceil(N/32)] — the epilogue that WRITES the new residual stream also writes,
   * per row and 32-column chunk, the sum of squares of the values as stored.  rs_sumsq (any epilogue): fp32 [M][rs_parts] —
   * the GEMM that CONSUMES the stream derives its per-row scale rsqrt(sum / K + rs_eps) from those partials (fixed
   * summation order: deterministic) instead of reading `row_scale`. */
  float* sumsq_out;
  const float* rs_sumsq;
  int32_t rs_parts;
  float rs_eps;
  /* Stream-K tail (optional; null = plain data-parallel tiles).  When the tile count leaves a partial last wave
   * (e.g. 272 tiles on 148 SMs), the tail's k-blocks are divided evenly over ALL CTAs; partial fp32 accumulators pass
   * through this workspace: 8192 bytes of flags (zero before the first use, self-resetting afterwards) followed by one
   * 128 x 256 fp32 slot per SM — mm_gemm_streamk_workspace_bytes().  One workspace must not be used by GEMMs running
   * CONCURRENTLY on different streams.  Ignored for multicast-pair launches and for launches without one full wave of
   * tiles (the tail pieces run first and hide their hand-over behind the full tiles). */
  void* sk_workspace;
  int64_t sk_workspace_bytes;
} mm_gemm_args;

int32_t mm_gemm_fwd(const mm_gemm_args* args, void* stream);
/* The schedule mm_gemm_fwd would use for `args` on the current device (148 SMs when no device is visible), without
 * touching memory or launching: the host-side decisions — tile width from the cost model, CTA pairs / cta_group::2,
 * rasterisation group, stream-K tail — are a pure function of the shapes, strides, alignments and flags.  Operand
 * pointers are only checked for null / alignment, never dereferenced.  Host logic made testable without a GPU
 * (tests/test_gemm_plan.py) and printable per BASELINE shape (tools/gemm_plan.py -> profiles/r2_gemm_schedules.txt). */
typedef struct mm_gemm_schedule {
  int32_t block_n;             /* tile = 128 x block_n x 64 (pairs: 256 x 256 x 64 per CTA pair) */
  int32_t pairs;               /* 0 = single CTAs, 1 = multicast pairs of cta_group::1 MMAs, 2 = cta_group::2 pairs */
  int32_t m_tiles, n_tiles, k_blocks;
  int64_t units;               /* work units over all batches: tiles, or pair tiles (2 M tiles x 1 N tile) */
  int32_t workers;             /* units in flight: SMs, or SM pairs */
  int32_t grid;                /* CTAs launched (persistent: <= SM count) */
  int32_t waves;               /* ceil(units / workers) */
  int32_t group_m;             /* rasterisation: M units per L2 group */
  int32_t streamk_tiles;       /* tiles of the partial last wave shared over all CTAs (0 = plain tiles) */
  int32_t smem_bytes;          /* dynamic shared memory per CTA */
  int32_t vectorised_epilogue; /* 1 = 128-bit epilogue accesses (all alignments hold) */
} mm_gemm_schedule;
int32_t mm_gemm_plan(const mm_gemm_args* args, mm_gemm_schedule* plan);
/* Stream-K policy of the process: 0 never, 1 when the saved MMA time exceeds the hand-over cost (default; environment
 * MACAW_B200_GEMM_STREAMK), 2 whenever the schedule allows (tests).  mode < 0 only queries.  Returns the previous mode. */
int32_t mm_gemm_streamk_mode(int32_t mode);
/* Pair launches (wide tiles, several waves — the LLaMA GEMMs at batch 32) as ONE cta_group::2 MMA unit (mode 1, default)
 * instead of two cta_group::1 MMAs sharing a multicast B tile (mode 0).  Environment MACAW_B200_GEMM_CG2.  mode < 0 only
 * queries.  Returns the previous mode. */
int32_t mm_gemm_cg2_mode(int32_t mode);
/* bytes of mm_gemm_args.sk_workspace on the current device */
int64_t mm_gemm_streamk_workspace_bytes(void);

/* Sum fp32 partials [splits][M][N] (+ bf16 bias[N]) -> bf16 (or fp16 when out_fp16 != 0) [M][N] (row stride ldo).
 * Split-K tail of the Conv1d down-samplers (modeling.py:982, 999, 1022). */
int32_t mm_splitk_reduce(const float* partial, int32_t splits, int32_t M, int32_t N, const void* bias, void* out,
                         int64_t ldo, int32_t out_fp16, void* stream);

/* ------------------------------------------------------------------------------------------------ attention
 * out[b,t,h,:] = softmax(scale * q k^T + mask) v, flash-style (no T x T tensor in HBM).
 * Replaces: LlamaAttention.forward modeling.py:197-215 (causal + key padding), CLIP / Whisper encoder
 * self-attention (transformers modeling_clip.py / modeling_whisper.py eager attention), and
 * video_long_self_attention modeling.py:1078 (two synthetic keys are materialised by the caller).
 * q/k/v/out: bf16 with element strides (batch, token, head); head_dim contiguous, head_dim in {64, 96, 128}.
 * key_mask: int32 [B][Tk] (1 = attend, 0 = masked) or NULL.  causal: key j visible to query i iff j <= i + (Tk - Tq).
 */
typedef struct mm_attn_args {
  const void *q, *k, *v;
  void* out;
  int32_t B, H, Tq, Tk, head_dim;
  int64_t q_bs, q_ts, q_hs;
  int64_t k_bs, k_ts, k_hs;
  int64_t v_bs, v_ts, v_hs;
  int64_t o_bs, o_ts, o_hs;
  const int32_t* key_mask;
  int32_t causal;
  float scale;
  int32_t impl; /* 0 = tcgen05 kernel (head_dim 64 / 96 / 128); 1 = force the legacy mma.sync kernel (tests only) */
  const int32_t* tk_dev; /* NULL, or device int holding the number of valid keys (<= Tk, which then is the capacity of
                            k / v): lets one captured launch serve a growing KV cache (tcgen05 kernel only) */
} mm_attn_args;
int32_t mm_attn_fwd(const mm_attn_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------ norms
 * LlamaRMSNorm modeling.py:311-319 (fp32 variance);  y = x * rsqrt(mean(x^2) + eps) * w.  x, y bf16 [rows][cols]. */
int32_t mm_rmsnorm_fwd(const void* x, const void* w, void* y, int32_t rows, int32_t cols, float eps, void* stream);
/* rstd[r] = rsqrt(mean(x[r]^2) + eps) (fp32): the row statistic of LlamaRMSNorm.  With the gain folded into the next
 * Linear's weight (W' = W * diag(g)) the norm itself becomes the `row_scale` of that GEMM's epilogue:
 * RMSNorm(x) W^T = rstd * (x W'^T), so the normalised activations are never written to HBM. */
int32_t mm_rms_rstd(const void* x, float* rstd, int32_t rows, int32_t cols, float eps, void* stream);
/* nn.LayerNorm of the CLIP / Whisper encoders (transformers modeling_clip.py:CLIPEncoderLayer, modeling_whisper.py). */
int32_t mm_layernorm_fwd(const void* x, int64_t ldx, const void* w, const void* b, void* y, int64_t ldy, int32_t rows,
                         int32_t cols, float eps, void* stream);

/* ------------------------------------------------------------------------------------------------ gathers / layout
 * embed_tokens lookup modeling.py:971-972, 979-980, 996-997, 1019-1020: out[i,:] = table[ids[i],:] (ids int64). */
int32_t mm_embed_gather(const void* table, int32_t vocab, int32_t dim, const int64_t* ids, int64_t n_ids, void* out,
                        int64_t ldo, void* stream);
/* Splice modeling.py:989-993, 1010-1016, 1028-1034 done in one pass.
 * dst (B, T, E) bf16 with T = 1 + n_prefix + (L-1):  dst[b,0] = text[b,0]; dst[b,1+j] = prefix[b,j]; dst[b,1+n_prefix+j] = text[b,1+j].
 * Also builds the int64 mask/label prefix of modeling.py:1036-1046 (bit-exact): mask_out = [1]*n_prefix ++ mask_in,
 * labels_out = [-100]*n_prefix ++ labels_in.  mask_in/labels_in may be NULL (then the outputs are not written). */
int32_t mm_splice_prefix(const void* text, const void* prefix, void* dst, int32_t B, int32_t L, int32_t n_prefix,
                         int32_t E, const int64_t* mask_in, int64_t* mask_out, const int64_t* labels_in,
                         int64_t* labels_out, void* stream);
/* CLIP patch embedding im2col (transformers modeling_clip.py:CLIPVisionEmbeddings): images (B,3,H,W) bf16 ->
 * rows (B*gh*gw, ldo) with column order (c, py, px); columns >= 3*p*p are zero. */
int32_t mm_patchify(const void* images, int32_t B, int32_t C, int32_t H, int32_t W, int32_t patch, void* out,
                    int64_t ldo, void* stream);
/* (B, C, T) -> (B, T + 2*pad, C) with zero pad rows (Whisper conv stem input, modeling_whisper.py:WhisperEncoder.forward). */
int32_t mm_transpose_pad(const void* x, int32_t B, int32_t C, int32_t T, int32_t pad, void* out, void* stream);
/* y[r,:] = x[r,:] + add[r % add_rows,:]  (bf16; CLIP class/position embeddings, video sinusoid PE modeling.py:1108-1118) */
int32_t mm_add_rows(const void* x, int64_t ldx, const void* add, int64_t lda, int32_t add_rows, void* y, int64_t ldy,
                    int32_t rows, int32_t cols, void* stream);
/* bf16 rows -> fp16 rows (modal features entering the fp16 alignment chain; exact within fp16's normal range) */
int32_t mm_cast_bf16_f16(const void* x, int64_t ldx, void* y, int64_t ldy, int32_t rows, int32_t cols, void* stream);
/* generic strided 2-D copy of bf16 rows (concats, CLS drop) */
int32_t mm_copy_rows(const void* x, int64_t ldx, void* y, int64_t ldy, int32_t rows, int32_t cols, void* stream);

/* ------------------------------------------------------------------------------------------------ fused alignment attention
 * The cross-modal alignment attention of reference modeling.py:986-987 / 1007-1008 / 1025-1026
 * (nn.MultiheadAttention with K = V = the whole embedding table, add_bias_kv, add_zero_attn; torch functional.py:6531-6672)
 * in ABSORBED form (SURVEY.md §7): for the R = H * Nq per-head query rows q~ = (q_h / sqrt(hd)) W_k[h] (fp16, width E)
 *     out[r, :]      = sum_{v < V} P[r, v] * table[v, :]                               (fp16, R x E; "ctx~")
 *     P[r, :]        = softmax over the S = V + 2 keys of { q~[r] . table[v] + row_bias[r] (v < V), extra[r], 0 }
 *     p_sum_real[r]  = sum_{v < V} P[r, v]        p_extra[r] = P of the appended bias_k key
 * ONE persistent kernel: phase 1 streams K-major table tiles through TMA into tcgen05 (S = q~ . table^T) and its
 * epilogue writes the un-normalised probabilities once, in fp16 (no fp32 score tensor, no softmax kernel); phase 2
 * streams the SAME table rows as an MN-major operand (O = P' . table) and normalises in its epilogue.  The caller
 * finishes with ctx_h = ctx~_h W_v[h]^T + p_sum_real * b_v[h] + p_extra * bias_v[h] (mm_gemm_fwd with row-scaled biases).
 * row_bias[r] = q_h . b_k[h] / sqrt(hd) and extra[r] = q_h . bias_k[h] / sqrt(hd) are read at index r * stat_stride.
 * P: scratch fp16 [R][ldp], ldp >= V rounded up to 8.  workspace: mm_align_workspace_bytes(R, V) bytes, 16-byte aligned
 * (zeroed by the call).  mode 0: one cooperative launch with grid-wide barriers between the phases; mode 1: the same
 * kernel launched three times in stream order (phase 1, conditional redo, phase 2). */
typedef struct mm_align_args {
  const void* table; /* fp16 [V][ldt] (exact fp16 copy of the bf16 embedding table) */
  int32_t V, E;
  int64_t ldt;
  const void* qt; /* fp16 [R][ldq] */
  int32_t R;
  int64_t ldq;
  const float* row_bias;
  const float* extra;
  int64_t stat_stride;
  void* out; /* fp16 [R][ldo] */
  int64_t ldo;
  float* p_sum_real;
  float* p_extra;
  void* P;
  int64_t ldp;
  void* workspace;
  int32_t mode;
  float* inv_l; /* optional fp32 [R]: 1 / softmax denominator, so that P = P' * inv_l (kept for the backward pass) */
} mm_align_args;
int32_t mm_align_fwd(const mm_align_args* args, void* stream);
int64_t mm_align_workspace_bytes(int32_t R, int32_t V);

/* ------------------------------------------------------------------------------------------------ alignment softmax
 * Row softmax of the absorbed-form alignment scores (torch F.multi_head_attention_forward: softmax over S = V + 2 keys,
 * functional.py:6531-6537, 6585-6602, 6630-6650).  scores fp32 [R][V] hold q~ . table[v]; the kernel adds row_bias[r]
 * (q_h . b_k[h]; read at row_bias[r * stat_stride], same stride for extra_score) to every real key, includes the bias_k key (score extra_score[r]) and the zero key (score 0) in the
 * normaliser, and writes P bf16 [R][V] (row stride ldp), p_sum_real[r] = sum_v P[r,v] and p_extra[r] = P of the bias_k key. */
int32_t mm_align_softmax(const float* scores, int64_t lds, const float* row_bias, const float* extra_score,
                         int64_t stat_stride, void* P, int64_t ldp, float* p_sum_real, float* p_extra, int32_t R,
                         int32_t V, void* stream);
/* Value-side bias terms of the absorbed form (functional.py:6531-6537: bias_v is appended un-projected; b_v rides on
 * every real key):  ctx[n, h*hd + d] += p_sum_real[h*Nq + n] * b_v[h*hd + d] + p_extra[h*Nq + n] * bias_v[h*hd + d]. */
int32_t mm_align_ctx_fixup(void* ctx, int64_t ldc, const float* p_sum_real, const float* p_extra, const void* b_v,
                           const void* bias_v, int32_t Nq, int32_t E, int32_t head_dim, void* stream);

/* ------------------------------------------------------------------------------------------------ decode (generate branch)
 * Greedy decoding behind inputs['inference'] = True (reference modeling.py:954-960 -> HF generate, vendored KV-cache
 * logic modeling.py:190-195).  mm_kv_append copies the K and V thirds of a fused [q|k|v] activation (rows (b, t),
 * row stride ld_qkv) into a per-layer cache (B, Tmax, 2, E) at time positions t0 .. t0 + T_new - 1.
 * mm_argmax_rows: out[r] = argmax_c logits[r, c] (lowest index on ties), bf16 logits, int64 out. */
int32_t mm_kv_append(const void* qkv, int64_t ld_qkv, int32_t B, int32_t T_new, int32_t E, void* cache, int32_t Tmax,
                     int32_t t0, const int32_t* t0_dev, void* stream); /* t0_dev != NULL overrides t0 with a device int */
int32_t mm_argmax_rows(const void* logits, int64_t ld, int32_t rows, int32_t V, int64_t* out, void* stream);
/* Thin-row companions of the swapped-operand decode GEMMs (mm_gemm_args.c_trans), whose epilogue cannot pair columns:
 * mm_rope_rows: in-place rotate-half RoPE (head_dim 128, apply_rotary_pos_emb modeling.py:83-91) on the first rot_cols
 * columns; position of row r = (*pos_dev if given) + r % rope_T.  mm_swiglu_rows: out[r, j] = silu(gate_j) * up_j from
 * the [32 gate | 32 up]-interleaved product (LlamaMLP modeling.py:139-140). */
/* Split-K tail of a thin (decode) GEMM: part fp32 [splits][N][ldp] holds W_s x_s^T per K slice (mm_gemm_fwd with the
 * operands swapped, batch = splits, fp32 out); out[m][n] = row_scale[m] * sum_s part[s][n][m] (+ residual[m][n]), bf16.
 * Splitting K lets the 32-tile o_proj / down_proj grids of a decode step cover all 148 SMs (weight streaming). */
int32_t mm_thin_reduce(const float* part, int32_t splits, int32_t N, int32_t M, int32_t ldp, const float* row_scale,
                       const void* residual, int64_t ldr, void* out, int64_t ldo, void* stream);
/* Fused tail of a split-K thin GEMM — one launch instead of mm_thin_reduce + mm_rope_rows + mm_kv_append /
 * mm_swiglu_rows / mm_rms_rstd (a decode step is launch-bound: 14 -> 9 kernels per LLaMA layer):
 *   MM_THIN_RES     out = rs * sum_s part + residual; sumsq_out (optional, [M][N/32]) = per-(row, 32-column) sums of squares
 *                   of the stored values, the next RMSNorm's statistic (LlamaRMSNorm modeling.py:311-319)
 *   MM_THIN_SWIGLU  out[m][32q+i] = silu(gate) * up from the [32 gate | 32 up]-interleaved product (modeling.py:139-140)
 *   MM_THIN_QKV     N = 3E: rotate-half RoPE (modeling.py:83-91) on q and k in fp32, q -> out[m][0..E), k / v -> the
 *                   layer's KV cache (B, Tmax, 2, E) at slot t0 (*t0_dev if given), row m = sample m (modeling.py:190-195)
 * rs = row_scale[m] | rsqrt(sum_j rs_sumsq[m][j] / rs_K + rs_eps) | 1. */
enum { MM_THIN_RES = 0, MM_THIN_SWIGLU = 1, MM_THIN_QKV = 2 };
typedef struct mm_thin_args {
  const float* part;       /* [splits][N][ldp] fp32 */
  int32_t splits, N, M, ldp, mode;
  const float* row_scale;  /* [M] or null */
  const float* rs_sumsq;   /* [M][rs_parts] or null */
  int32_t rs_parts, rs_K;
  float rs_eps;
  const void* residual;    /* [M][ldr] 16-bit or null (MM_THIN_RES) */
  int64_t ldr;
  void* out;
  int64_t ldo;
  float* sumsq_out;
  const float* rope_cos;   /* MM_THIN_QKV: (T, 64) fp32 tables; row = *pos_dev (0 if null) */
  const float* rope_sin;
  const int32_t* pos_dev;
  int32_t E;
  void* cache;
  int32_t Tmax, t0;
  const int32_t* t0_dev;
} mm_thin_args;
int32_t mm_thin_fused(const mm_thin_args* args, void* stream);
int32_t mm_rope_rows(void* x, int64_t ld, int32_t rows, int32_t rot_cols, const float* cos_t, const float* sin_t,
                     int32_t rope_T, const int32_t* pos_dev, void* stream);
int32_t mm_swiglu_rows(const void* gu, int64_t ld, int32_t rows, int32_t I, void* out, int64_t ldo, void* stream);

/* ------------------------------------------------------------------------------------------------ loss
 * Shifted cross entropy of LlamaForCausalLM.forward modeling.py:600-610: logits bf16 (B, T, V), labels int64 (B, T);
 * position t predicts labels[t+1]; ignore_index -100; writes loss_sum[0] (fp32) and n_valid[0] (int32);
 * both must be zeroed by the caller. */
int32_t mm_ce_loss(const void* logits, const int64_t* labels, int32_t B, int32_t T, int32_t V, float* loss_sum,
                   int32_t* n_valid, void* stream);

/* ------------------------------------------------------------------------------------------------ training step
 * Backward halves of the HBM-bound ops + the optimizer (SURVEY.md §8f rank 1).  The reference trains through autograd of
 * modeling.py driven by llm_trainer.py:184-188 (compute_loss -> backward) with AdamW (train.sh, fp32 master weights in
 * DeepSpeed).  All contractions of the backward pass are mm_gemm_fwd calls (dX: MN-major B; dW: MN-major A and B).
 *
 * mm_rmsnorm_bwd: y = x * rstd * g (LlamaRMSNorm modeling.py:311-319).  dx = rstd*(g*dy) - rstd^3/cols * x * sum(g*dy*x)
 *   (+ dres when given: the residual branch's gradient), dg[c] += sum_r dy*x*rstd in fp32: through dg_partials
 *   ([mm_rmsnorm_bwd_parts(rows)][cols] fp32 workspace: per-CTA column sums reduced in a fixed order — deterministic, and
 *   no grid-size-way atomic contention on `cols` addresses) or, when dg_partials is null, with atomics. */
int32_t mm_rmsnorm_bwd_parts(int32_t rows);
int32_t mm_rmsnorm_bwd(const void* dy, const void* x, const float* rstd, const void* g, const void* dres, void* dx,
                       float* dg, float* dg_partials, int32_t rows, int32_t cols, void* stream);
/* LlamaMLP modeling.py:139-140 on separate gate / up activations: h = silu(gate) * up over n contiguous elements. */
int32_t mm_swiglu_fwd(const void* gate, const void* up, void* h, int64_t n, void* stream);
int32_t mm_swiglu_bwd(const void* dh, const void* gate, const void* up, void* dgate, void* dup, int64_t n, void* stream);
/* Attention backward through the softmax (LlamaAttention modeling.py:197-215; nn.MultiheadAttention): S = q.k^T (pre-scale)
 * and dP = dO.v^T, fp32 [B][H][Tq][ld]; writes P = softmax(scale*S + mask) and dS = scale * P * (dP - sum_j P_j dP_j) as
 * bf16 with the same layout.  Masks as in mm_attn_fwd. */
int32_t mm_attn_softmax_bwd(const float* S, const float* dP, void* P, void* dS, int32_t B, int32_t H, int32_t Tq,
                            int32_t Tk, int64_t ld, float scale, int32_t causal, const int32_t* key_mask, float p_drop,
                            const uint64_t* seed_dev, uint32_t sid, void* stream);
/* Training-mode attention dropout (reference: nn.MultiheadAttention(dropout=0.1), modeling.py:879-909; torch drops the
 * softmax probabilities, functional.py:6640-6645).  The mask is a pure function of (*seed_dev, sid, row, column) through
 * Philox4x32-10 (csrc/philox.cuh): forward and backward kernels regenerate it, nothing is stored; `seed_dev` is a DEVICE
 * 64-bit seed so a captured CUDA graph draws a fresh mask per replay, `sid` separates the dropout sites.  p_drop == 0
 * switches dropout off (seed_dev may be null).  With p_drop > 0, mm_attn_softmax_bwd uses dP <- m . dP and writes Pd = m . P.
 * mm_attn_softmax_fwd: S fp32 [B][H][Tq][ld] -> Pd = dropout(softmax(scale * S + mask)) bf16, same layout. */
int32_t mm_attn_softmax_fwd(const float* S, void* P, int32_t B, int32_t H, int32_t Tq, int32_t Tk, int64_t ld, float scale,
                            int32_t causal, const int32_t* key_mask, float p_drop, const uint64_t* seed_dev, uint32_t sid,
                            void* stream);
/* Dropout of the alignment attention's probabilities (forward): P' (un-normalised fp16, R x ldp) -> Pm (kept entries,
 * unscaled), rs = (1/l)/(1-p), p_sum_real_d = rs * sum_v Pm_v, p_extra_d = m_V * p_extra (column V = the bias_k key). */
int32_t mm_align_dropout_fwd(const void* P_unnorm_f16, void* Pm_f16, int64_t ldp, const float* inv_l, const float* p_extra,
                             float* rs, float* p_sum_real_d, float* p_extra_d, int32_t R, int32_t V, float p_drop,
                             const uint64_t* seed_dev, uint32_t sid, void* stream);
/* The multipliers themselves (fp32: 0 or 1/(1-p)) of a rows x cols block of stream `sid` — for tests / debugging. */
int32_t mm_dropout_mask(float* out, int64_t ld, int32_t rows, int32_t cols, float p_drop, const uint64_t* seed_dev,
                        uint32_t sid, void* stream);
/* Gradient of mm_ce_loss w.r.t. the logits (modeling.py:600-610), times grad_scale (* *grad_scale_dev when given: the
 * upstream gradient of the loss as a device scalar, so the launch is CUDA-graph capturable) / n_valid; may run in place. */
int32_t mm_ce_bwd(const void* logits, const int64_t* labels, void* dlogits, int32_t B, int32_t T, int32_t V,
                  const int32_t* n_valid, float grad_scale, const float* grad_scale_dev, void* stream);
/* Gradient of mm_embed_gather: dtable[ids[i], :] += dx[i, :] (bf16x2 atomics). */
int32_t mm_embed_scatter_add(const void* dx, int64_t ldx, const int64_t* ids, int64_t n, int32_t dim, int32_t vocab,
                             void* dtable, void* stream);
/* out[c] += sum_r x[r, c]  (bias gradients; fp32 atomics) */
int32_t mm_colsum(const void* x, int64_t ldx, int32_t rows, int32_t cols, float* out, void* stream);
/* Fused AdamW step on one parameter tensor: bf16 working copy p, bf16 gradient g (times grad_scale), fp32 master / m / v.
 * The bias corrections use `step`, or the device int *step_dev when given (graph-replayed training steps). */
int32_t mm_adamw(void* p, const void* g, float* master, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                 float eps, float weight_decay, int32_t step, const int32_t* step_dev, float grad_scale, void* stream);

/* Device-resident optimizer state of the scheduled update (one per optimizer; every step-dependent scalar lives here, so
 * a CUDA graph of the step replays with the right values).  Written by mm_grad_norm, read by mm_adamw_sched.
 * Initialise with step = skipped = arrived = 0, clip_coef = 1, finite = 1, apply = 0. */
typedef struct mm_opt_state {
  int32_t step;      /* optimizer steps taken (skipped steps not counted): the bias-correction step of the update */
  int32_t skipped;   /* steps skipped because their gradients were not finite */
  float lr;          /* learning rate of the latest step: base_lr * lambda(step - 1) */
  float clip_coef;   /* gradient multiplier of the latest step: min(1, max_norm / (grad_norm + 1e-6)), 1 without clipping */
  float grad_norm;   /* global L2 norm of the latest step's gradients, before clipping (0 when no pass ran) */
  int32_t finite;    /* 1 when every gradient element of the latest step was finite */
  int32_t apply;     /* 1 when the latest step updates the parameters (0: skipped) */
  int32_t arrived;   /* CTA arrival counter of mm_grad_norm; 0 between launches */
} mm_opt_state;
/* Learning-rate schedules of transformers.optimization (lambda of the 0-based step; num_cycles = 0.5 for cosine). */
#define MM_SCHED_CONSTANT 0
#define MM_SCHED_CONSTANT_WITH_WARMUP 1
#define MM_SCHED_LINEAR 2
#define MM_SCHED_COSINE 3
/* Partial sums of mm_grad_norm: `partials` holds MM_GRAD_NORM_PARTS doubles. */
#define MM_GRAD_NORM_PARTS 1024
/* Global gradient norm + step bookkeeping of the scheduled update.  table: device int64 [n_tensors][2] = (address, numel)
 * of the bf16 gradients to include.  The sum of squares is deterministic (fixed partition: fp32 per thread over runs of at
 * most 64 elements, fp64 across threads and CTAs, summed in a fixed order): bit-identical run to run and rank to rank.
 * The last CTA writes grad_norm, finite, clip_coef (max_norm <= 0: no clipping); then, if the gradients are finite or
 * skip_nonfinite == 0, step += 1, lr = base_lr * lambda(step - 1) (fp64), apply = 1; otherwise skipped += 1, apply = 0.
 * n_tensors == 0 runs the scalar work only (a schedule without clipping or the finiteness check). */
int32_t mm_grad_norm(const int64_t* table, int32_t n_tensors, double* partials, mm_opt_state* state, float max_norm,
                     int32_t skip_nonfinite, float base_lr, int32_t schedule, int32_t warmup_steps, int32_t total_steps,
                     void* stream);
/* mm_adamw with lr, the gradient multiplier (clip_coef) and the bias-correction step read from *state; a step with
 * state->apply == 0 leaves p, master, m and v untouched. */
int32_t mm_adamw_sched(void* p, const void* g, float* master, float* m, float* v, int64_t n, float beta1, float beta2,
                       float eps, float weight_decay, const mm_opt_state* state, void* stream);

/* Backward of the absorbed alignment attention through its (V + 2)-key softmax (reference: autograd of
 * nn.MultiheadAttention, modeling.py:986-987 / 1007-1008 / 1025-1026).  See train_kernels.cu for the formulas. */
int32_t mm_align_softmax_bwd(const float* G, int64_t ldg, const void* P_unnorm_f16, int64_t ldp, const float* inv_l,
                             const float* d_p_sum_real, const float* p_extra, const float* d_p_extra, float gscale,
                             void* P_bf16, void* dS_bf16, int64_t ldo, float* dstats, int32_t R, int32_t V, float p_drop,
                             const uint64_t* seed_dev, uint32_t sid, void* stream);
/* out[h*hd + d] += sum_n w[(h*Nq + n) * w_stride] * x[n, h*hd + d]; x bf16 (x_fp16 == 0) or fp16. */
int32_t mm_head_weighted_colsum(const void* x, int64_t ldx, int32_t x_fp16, const float* w, int64_t w_stride, int32_t Nq,
                                int32_t E, int32_t head_dim, float* out, void* stream);
/* Data gradient of the Conv1d down-sampler (col2im over overlapping token windows): dfeats[b,t,c] = sum over windows l
 * containing t of dwin[b*Lq + l][(t - l*ss)*C + c]; bf16 in / out. */
int32_t mm_window_gather_add(const void* dwin, int32_t B, int32_t N, int32_t C, int32_t Lq, int32_t kk, int32_t ss,
                             void* dfeats, void* stream);
int32_t mm_cast_f16_bf16(const void* x, int64_t ldx, void* y, int64_t ldy, int32_t rows, int32_t cols, void* stream);

/* ------------------------------------------------------------------------------------------------ gradient all-reduce
 * The one collective of the path: the data-parallel gradient all-reduce of the training step (reference: DeepSpeed ZeRO-3
 * reduce-scatter / all-gather, configs/deepspeed_config.json:22-41; north_star: "a single NCCL all-reduce on gradients").
 * NCCL is bound at run time (dlopen); one communicator per process (one process per GPU).  Bootstrap: rank 0 calls
 * mm_nccl_unique_id, ships the 128 bytes to the other ranks (any channel: torch.distributed store, MPI, a file), every
 * rank calls mm_nccl_init.  mm_nccl_allreduce is in place, asynchronous on `stream`; dtype 0 = bf16, 1 = fp32;
 * average != 0 divides by the group size (ncclAvg). */
int32_t mm_nccl_unique_id(void* out128);
int32_t mm_nccl_init(const void* id128, int32_t world, int32_t rank);
int32_t mm_nccl_allreduce(void* buf, int64_t count, int32_t dtype, int32_t average, void* stream);
int32_t mm_nccl_destroy(void);

/* ------------------------------------------------------------------------------------------------ input pipeline
 * Device-side replacement of the per-sample host work in LLMTrainer.get_self_inputs (llm_trainer.py:306-381).
 *
 * mm_image_preprocess: `_transform(224)` of llm_trainer.py:151-158 on ONE decoded 8-bit RGB image (HWC, row stride ld bytes):
 * Pillow's two-pass antialiased bicubic resize with its 22-bit fixed-point coefficients (tables built by the host with
 * Pillow's arithmetic, restricted to the centre-crop window), then ToTensor + Normalize.  row0 / n_rows: source rows the
 * vertical taps of the cropped output need (tmp holds n_rows x out_w x 3 bytes).  out: (3, out_h, out_w) bf16 or fp32;
 * out_u8 (optional, HWC) receives the 8-bit resized + cropped image (bit-exact with PIL). */
typedef struct mm_image_args {
  const void* src;
  int64_t ld;
  int32_t row0, n_rows;
  int32_t out_h, out_w;
  const int32_t* bounds_h; /* [out_w][2] = (xmin, count) */
  const int32_t* kk_h;     /* [out_w][ksize_h] */
  int32_t ksize_h;
  const int32_t* bounds_v; /* [out_h][2] */
  const int32_t* kk_v;     /* [out_h][ksize_v] */
  int32_t ksize_v;
  float mean[3], std[3];
  void* tmp;
  void* out;
  int32_t out_fp32;
  void* out_u8;
} mm_image_args;
int32_t mm_image_preprocess(const mm_image_args* args, void* stream);
/* whisper.pad_or_trim + whisper.log_mel_spectrogram (llm_trainer.py:338-345) of ONE clip: pcm fp32 [n_samples] at 16 kHz ->
 * (80, 3000) bf16 / fp32.  basisT: fp32 [400][2][208] windowed DFT basis (Hann folded in; cos, -sin; bin index
 * contiguous); mel: fp32 [80][201] filter bank; logspec: scratch fp32 [80][3000]; max_scratch: 4 bytes. */
int32_t mm_log_mel(const float* pcm, int32_t n_samples, const float* basisT, const float* mel, float* logspec,
                   void* max_scratch, void* out, int32_t out_fp32, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MACAW_B200_H_ */
