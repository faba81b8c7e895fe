/*
 * modaltune_b200 -- C ABI of the B200 (sm_100a) kernels for the ModalTune-GigaPath fine-tuning hot path.
 *
 * The reference (martellab-sri/ModalTune) is pure Python: it has no FFI layer.  Its only native boundary on this path
 * is `flash_attn_func(q, k, v, dropout, bias, softmax_scale, is_causal) -> (out, lse)`
 * (models/prov_gigapath/gigapath/torchscale/component/flash_attention.py:11-28), everything else is ATen ops reached
 * through nn.Module.forward.  Each entry point below therefore names the reference Python function it replaces; the
 * Python side (modaltune_b200/_lib.py, ops.py) binds them with ctypes and wraps them in torch.autograd.Functions, and
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers to DEVICE memory, sizes as int64_t, no torch types;  `stream` is a cudaStream_t passed as void*.
 *   - dtype codes: MT_F32 = 0 (float), MT_BF16 = 1 (__nv_bfloat16).  Statistics (mean, rstd, lse, delta) are float.
 *   - the caller owns every buffer (outputs and workspaces are pre-allocated by the caller); kernels never allocate.
 *   - return value: 0 on success, otherwise a cudaError_t / negative MT_E* code; mt_last_error() gives the message.
 *   - single host thread per process, one process per GPU.  No CPU fallback exists behind any entry point.
 */
#ifndef MODALTUNE_B200_H
#define MODALTUNE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MT_F32 0
#define MT_BF16 1

#define MT_E_BADARG (-1)
#define MT_E_UNSUPPORTED (-2)

#define MT_MAX_BRANCHES 8

/* Geometry of LongNet dilated attention for one sequence (torchscale/component/dilated_attention.py:82-144).
 * Branch b uses segment length seg_len[b] (already clamped: g = min(sl, n_tokens)) and dilation ratio[b];
 * head h keeps in-segment offsets floor(h*ratio/n_heads) + j*ratio. */
typedef struct {
  int32_t n_tokens;   /* N, cls included                      */
  int32_t n_heads;    /* 16                                   */
  int32_t head_dim;   /* 48                                   */
  int32_t n_branches; /* <= MT_MAX_BRANCHES                   */
  int32_t seg_len[MT_MAX_BRANCHES];
  int32_t ratio[MT_MAX_BRANCHES];
} mt_dilated_geometry;

/* Train-mode stochastic ops of the frozen encoder (torchscale/architecture/encoder.py:149-152,169-170:
 * Dropout(p) then DropPath on each residual branch; feedforward_network.py:142).  A Philox4x32-10 counter RNG keyed by
 * *seed generates the keep mask of element i of the tensor from (seed, stream_id, i): nothing is stored, the backward
 * regenerates the same mask.  seed and path_scale are DEVICE pointers so that a CUDA graph replays fresh masks when
 * the caller redraws them inside the graph.  A NULL mt_dropout* means eval mode (identity). */
typedef struct {
  float p;                 /* drop probability, 0 <= p < 1; kept elements are scaled by 1 / (1 - p)              */
  const int64_t* seed;     /* device pointer to the 64-bit seed of this step                                      */
  int64_t stream_id;       /* distinct per call site (layer, branch) so that masks are independent               */
  const float* path_scale; /* device pointer to the DropPath factor of the branch (0 or 1 / keep), NULL = 1      */
} mt_dropout;

const char* mt_last_error(void);
int mt_version(void);
/* 1 when the running device is sm_100 (tcgen05 / TMA kernels usable), 0 otherwise, <0 on error */
int mt_device_is_sm100(void);

/* ---- A0: PatchEmbed epilogue + positional embedding + cls row -----------------------------------------------------
 * replaces: PatchEmbed.forward bias add (slide_encoder.py:52-56), `x + pos_embed[:, pos]`, cls concat
 * (longvit_adapter.py:232-246) and coords_to_pos (slide_encoder.py:198-211).
 * proj [L, E] = feats @ W^T (GEMM result, dtype `proj_dtype`), bias [E] f32, coords [L,2] f32 (pixels),
 * table [ngrids, E/2] f32 = 1-D sincos factor, cls [E] f32  ->  x [L+1, E] f32 (row 0 = cls).
 * Index semantics are the reference's: pos = floor(c0 / tile_size) * ngrids + floor(c1 / tile_size) + 1 into the flat
 * table (a column index >= ngrids wraps into the next grid row, pos == 0 is the all-zero cls row); an index outside
 * [0, ngrids^2] -- an IndexError / device assert in the reference -- makes the kernel trap (CUDA error on the stream). */
int mt_embed_assemble(const void* proj, int proj_dtype, const float* bias, const float* coords, const float* table,
                      const float* cls, float* x, int64_t n_tiles, int64_t embed, int64_t ngrids, float tile_size,
                      void* stream);

/* ---- A1: LayerNorm ------------------------------------------------------------------------------------------------
 * replaces: nn.LayerNorm calls in EncoderLayer.forward (torchscale/architecture/encoder.py:137-166) and in
 * CrossAttentionLayer.forward_pre (models/vitadapter/adapter_modules.py:217-218).
 * fwd: y = (x - mean) * rstd * gamma + beta [+ add[row % add_rows]].  x [rows, cols] x_dtype, y y_dtype. */
int mt_layernorm_fwd(const void* x, int x_dtype, const float* gamma, const float* beta, const void* add, int add_dtype,
                     int64_t add_rows, void* y, int y_dtype, float* mean, float* rstd, int64_t rows, int64_t cols,
                     float eps, void* stream);
/* bwd: dx = LN'(dy) [+ residual];  optional dgamma/dbeta [cols] f32 (accumulated with atomics into zeroed buffers);
 * dx_bf16 (or NULL): a second copy of dx rounded to bf16, written in the same pass for the GEMM that consumes the
 * gradient next (saves a separate cast pass over [rows, cols]).  `residual` may be `dx` itself (an in-place add, same
 * dtype): every element is read once, by the thread that then writes it. */
int mt_layernorm_bwd(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* gamma, const float* mean,
                     const float* rstd, const void* residual, int res_dtype, void* dx, int dx_dtype, void* dx_bf16,
                     float* dgamma, float* dbeta, int64_t rows, int64_t cols, void* stream);
/* deterministic mt_layernorm_bwd: dgamma / dbeta are not accumulated with atomics but written (no zeroing needed): every
 * block stores its column partials to `workspace` and a second pass adds them in block order, so the same inputs give
 * the same bits in every run.  workspace_floats >= mt_colreduce_workspace_floats(cols) when dgamma is not NULL. */
int mt_layernorm_bwd_ws(const void* dy, int dy_dtype, const void* x, int x_dtype, const float* gamma, const float* mean,
                        const float* rstd, const void* residual, int res_dtype, void* dx, int dx_dtype, void* dx_bf16,
                        float* dgamma, float* dbeta, int64_t rows, int64_t cols, float* workspace,
                        int64_t workspace_floats, void* stream);
/* workspace of the deterministic column reductions (mt_layernorm_bwd_ws, mt_gated_residual_bwd_ws, mt_colsum_ws) */
int64_t mt_colreduce_workspace_floats(int64_t cols);

/* mt_layernorm_bwd (f32 tensors, cols = 768, residual and bf16 twin required) of the pre-attention LayerNorm of layer
 * l + 1 that ALSO does mt_ffn_bwd_prep for layer l: its dx IS layer l's dy and its x IS layer l's output y, so the row means
 * m1, m2 of layer l's ffn_layernorm backward cost one more read (x1_below = the FFN residual input of layer l) instead of a
 * pass of their own.  rowv [rows, 4] = (mean_f, rstd_f, m1, m2) for MT_EPI_GELU_LN_BWD, dx_bf16 = that GEMM's A operand. */
int mt_layernorm_bwd_ffn_prep(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd,
                              const float* residual, float* dx, void* dx_bf16, const float* x1_below, const float* c1,
                              const float* c2, const float* mean_f, const float* rstd_f, float* rowv, int64_t rows,
                              int64_t cols, int64_t ln_cols, void* stream);

/* residual add fused with the next pre-LN (torchscale/architecture/encoder.py:152-166):
 * x_out = x + D(a [+ abias]) (f32 residual stream, a in a_dtype, abias [cols] f32 or NULL = bias of the GEMM that
 * produced a; D = train-mode dropout + DropPath of the branch, identity when drop is NULL), y = LN(x_out).  cols = 768. */
int mt_add_layernorm_fwd(const float* x, const void* a, int a_dtype, const float* abias, const float* gamma,
                         const float* beta, float* x_out, void* y, int y_dtype, float* mean, float* rstd, int64_t rows, int64_t cols,
                         float eps, const mt_dropout* drop, void* stream);

/* ---- A6: GELU(fp32) + LayerNorm(3072) between fc1 and fc2 ---------------------------------------------------------
 * replaces: `activation_fn(x.float()).type_as(x)` + ffn_layernorm (torchscale/component/feedforward_network.py:135-140)
 * h [rows, cols] = fc1 output; hbias [cols] f32 or NULL is added to it first (fc1's bias, so that the GEMM can keep a
 * plain fp32 output).  y = LN(gelu_erf(h + hbias)). */
int mt_gelu_ln_fwd(const void* h, int h_dtype, const float* hbias, const float* gamma, const float* beta, void* y,
                   int y_dtype,
                   float* mean, float* rstd, int64_t rows, int64_t cols, float eps, void* stream);
/* dh = gelu'(h) * LN'(dy) with u = gelu(h) recomputed. */
int mt_gelu_ln_bwd(const void* dy, int dy_dtype, const void* h, int h_dtype, const float* hbias, const float* gamma,
                   const float* mean,
                   const float* rstd, void* dh, int dh_dtype, int64_t rows, int64_t cols, void* stream);

/* ---- A2 / A6: the frozen linear layers of an encoder layer on the tensor cores, epilogues fused ---------------------
 * replaces: q/k/v_proj, out_proj (torchscale/component/multihead_attention.py:44-54), fc1 / GELU / ffn_layernorm / fc2
 * (feedforward_network.py:132-143), the residual adds of EncoderLayer.forward (architecture/encoder.py:152-175) and
 * the dX GEMMs of their backward (all encoder weights are frozen).
 * C[M, N] = A[M, K] . W[N, K]^T with bf16 operands (row strides lda / ldw in elements), fp32 accumulation in TMEM;
 * N must be a multiple of 256 and K of 64.  What happens to the accumulator is the epilogue `mode`:
 *   MT_EPI_PLAIN        out = acc [+ bias] [+ residual]                       (f32 and / or bf16 output)
 *   MT_EPI_GELU_STATS   h = acc + bias (out_f32, optional);  out_bf16 = u = gelu_erf(h);  out_aux_bf16 = gelu'(h) (optional);
 *                       stats[row][slab] = (sum u, sum u^2) of the
 *                       ROUNDED u over each 128-column slab (`stats` is [M, N / 128, 2], every entry written once, no
 *                       atomics: deterministic): fc1 + GELU + the statistics of ffn_layernorm
 *   MT_EPI_LN_RESIDUAL  out = residual + rstd[row] * (acc - mean[row] * col_c1) + col_c2 with mean / rstd from the
 *                       ln_cols / 128 slab partials of `stats` (added in a fixed order) over `ln_cols` columns: fc2 applied to LayerNorm(u) WITHOUT materialising it, for
 *                       W = W2 diag(gamma), col_c1 = W 1, col_c2 = W2 beta + b2, + the residual add.
 *   MT_EPI_GELU_LN_BWD  out = gelu'(h) * rstd * (acc - m1 - uhat * m2), uhat = (gelu(h) - mean) * rstd: the backward of
 *                       GELU + ffn_layernorm applied to the accumulator of fc2's dX GEMM, for W = (W2 diag(gamma))^T
 *                       (acc_j = gamma_j dn_j); h = `residual` (fc1's fp32 output incl. bias), `stats` = [M, 4] rows of
 *                       (mean, rstd, m1, m2) from mt_ffn_bwd_prep.  The [M, 3072] fp32 gradient of the LayerNorm output
 *                       and the separate GELU'-LN' kernel do not exist on this path. */
#define MT_EPI_PLAIN 0
#define MT_EPI_GELU_STATS 3
#define MT_EPI_LN_RESIDUAL 4
#define MT_EPI_GELU_LN_BWD 5
typedef struct {
  int32_t mode;
  int32_t ln_cols;          /* MT_EPI_LN_RESIDUAL: number of columns the statistics were taken over (3072)      */
  float ln_eps;
  int32_t impl;             /* 0 = pick, 1 = one CTA per 128 x 256 tile, 2 = CTA pairs (cta_group::2, 256 x 256)   */
  const float* bias;        /* [N] or NULL                                                                        */
  const float* residual;    /* [M, N] f32 or NULL, row stride ld_residual                                        */
  const float* col_c1;      /* [N]                                                                                */
  const float* col_c2;      /* [N]                                                                                */
  float* stats;             /* [M, cols / 128, 2] slab partials (see the modes)                                   */
  float* ln_mean_out;       /* MT_EPI_LN_RESIDUAL: [M] or NULL, the row mean / rstd derived from stats, written   */
  float* ln_rstd_out;       /*   once per row (what the backward of the folded LayerNorm needs)                    */
  float* out_f32;           /* [M, N] or NULL, row stride ld_out_f32 (0 = N)                                     */
  void* out_bf16;           /* [M, N] or NULL, row stride ld_out_bf16 (0 = N)                                    */
  int64_t ld_out_f32, ld_out_bf16, ld_residual;
  void* out_aux_bf16;       /* MT_EPI_GELU_STATS: [M, N] gelu'(h) in bf16 or NULL (then out_f32 = h is required): with  */
                            /*   it the backward needs neither h nor a second erf / exp per element                    */
  const void* in_u_bf16;    /* MT_EPI_GELU_LN_BWD: gelu(h) and gelu'(h) [M, N] bf16 as written by MT_EPI_GELU_STATS,   */
  const void* in_g_bf16;    /*   used instead of h (`residual` NULL)                                                   */
} mt_linear_epilogue;
int mt_linear_sm100(const void* a, int64_t lda, const void* w, int64_t ldw, int64_t M, int64_t N, int64_t K,
                    const mt_linear_epilogue* epilogue, void* stream);

/* Row means of the LayerNorm(3072) backward, formed BEFORE fc2's dX GEMM from [rows, 768] tensors only (backward of
 * feedforward_network.py:135-143 with ffn_layernorm folded into fc2): with dn = dy W2,
 *   m1 = mean_j(gamma_j dn_j)       = dy . c1 / ln_cols,              c1 = (W2 diag gamma) 1   (what the forward used)
 *   m2 = mean_j(gamma_j dn_j uhat_j) = dy . (y - x1 - c2) / ln_cols,  because fc2's folded forward IS
 *                                      y - x1 - c2 = (W2 diag gamma) uhat.
 * dy [rows, cols] f32 = gradient of the layer output, y = layer output, x1 = the FFN's residual input (f32), c1, c2
 * [cols]; mean, rstd [rows] = the statistics of ffn_layernorm.  Writes rowv [rows, 4] = (mean, rstd, m1, m2) for
 * MT_EPI_GELU_LN_BWD and dy_bf16 [rows, cols] (the A operand of that GEMM; the dots use these ROUNDED values so that
 * m1 is exactly the mean of the accumulator row).  cols = 768. */
int mt_ffn_bwd_prep(const float* dy, const float* y, const float* x1, const float* c1, const float* c2,
                    const float* mean, const float* rstd, float* rowv, void* dy_bf16, int64_t rows, int64_t cols,
                    int64_t ln_cols, void* stream);

/* ---- A3/A4: dilated attention, all branches, per-branch outputs ---------------------------------------------------
 * replaces: DilatedAttention.gathering x3 + attention_ops -> flash_attn_func, 5 times per layer
 * (torchscale/component/dilated_attention.py:82-111,216-252; multihead_attention.py:109-119; flash_attention.py:11-28).
 * qkv [n_alloc, 3*E] (q | k | v, head-major inside each), row stride `qkv_ld` elements, rows >= n_tokens must be zero
 * and n_alloc a multiple of 16 (sm100 path reads them through TMA).
 * o_br : compact per-branch outputs, branch b at element offset sum_{b'<b} N*E/r_b', layout [N][E/r_b]: row p holds the
 *        16/r_b heads that own position p (heads (p%r)*16/r ..), each head_dim wide.           (dtype)
 * lse_br: same compaction, [N][H/r_b] float, natural-log LSE including the zero-slot keys.
 * impl: 0 = SIMT fp32 math (any dtype; also the on-device cross-check of the tensor-core kernels), >= 1 = tcgen05 / TMA /
 * TMEM kernels (bf16 only): 1 = one CTA per work item, 2 (backward only) = persistent CTAs that pull work items from a
 * device counter (identical arithmetic; hands over between items without draining its pipeline; the default backward),
 * 3 (forward only) = one CTA per work item with 48-key score tiles, four CTAs per SM (the default forward),
 * 4 (backward only) = the deterministic backward (MT_DILATED_BWD_DETERMINISTIC below).  A shared-memory window that is not 1024-byte aligned (never expected) makes the tcgen05
 * kernels trap: the failure surfaces as a CUDA error on the stream, never as silently unwritten outputs. */
int mt_dilated_attn_fwd(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, int64_t n_alloc, int dtype,
                        void* o_br, float* lse_br, int impl, void* stream);

/* ---- A5 (+ inner_attn_ln of A2): LSE merge of the branches fused with LayerNorm -----------------------------------
 * replaces: DilatedAttention.scattering (dilated_attention.py:113-144) + inner_attn_ln (:257-258).
 * attn [N,E] (dtype) = sum_b softmax_b(lse_b) o_b, lse [N,H] f32 = log sum_b exp(lse_b); y = LN(attn). */
int mt_dilated_merge_ln_fwd(const mt_dilated_geometry* geom, const void* o_br, const float* lse_br, int dtype,
                            void* attn, float* lse, const float* gamma, const float* beta, float eps, void* y,
                            float* mean, float* rstd, void* stream);
/* backward of LN then of the (detached-weight) merge.  attn is recomputed from o_br / lse_br (never stored):
 * dattn [N,E] (dtype) = LN'(dy), dy in dy_dtype;  delta_br (lse_br compaction, f32) = dattn[p,h,:] . o_b[p,h,:]. */
int mt_dilated_merge_ln_bwd(const mt_dilated_geometry* geom, const void* dy, int dy_dtype, const void* o_br,
                            const float* lse_br,
                            const float* gamma, const float* mean, const float* rstd, int dtype, void* dattn,
                            float* delta_br, void* stream);

/* ---- backward of A3/A4/A5 -----------------------------------------------------------------------------------------
 * replaces: autograd of the five flash_attn_func calls + gather/scatter (no reference source; flash-attn bwd).
 * dS_b = exp(S - LSE) * (dO V^T - delta_b);  dqkv_f32 [n_alloc, 3E] float (rows >= N are scratch) is ZEROED by the call
 * and accumulated with reductions over branches; dattn [n_alloc, E] with zero rows >= N. */
int mt_dilated_attn_bwd(const mt_dilated_geometry* geom, const void* qkv, int64_t qkv_ld, int64_t n_alloc,
                        const void* dattn, const float* lse, const float* delta_br, int dtype, float* dqkv_f32,
                        int impl, void* stream);
/* impl 4 (bf16, tcgen05): the DETERMINISTIC backward -- the same inputs give bitwise the same dqkv in every run.  Every
 * element of dqkv receives at most one non-zero addition per branch, and the branches are added in a fixed order: the
 * branches run one after another on the stream (b = 0 .. n_branches - 1), each as a query-major dQ kernel (one CTA per
 * query tile streams the key tiles of its segment, dQ leaves once) and a key-major dK / dV kernel (impl 1 without
 * its dQ part).  About 3.5x the forward's tensor work instead of 2.5x. */
#define MT_DILATED_BWD_DETERMINISTIC 4

/* ---- A7/A8: Injector / Extractor cross-attention core (12 heads x 16) ---------------------------------------------
 * replaces: the softmax(QK^T/4)V inside nn.MultiheadAttention called from CrossAttentionLayer.forward_pre
 * (models/vitadapter/adapter_modules.py:225-229); the projections around it stay GEMMs.
 * q [Lq, E'] (row stride ldq elements), k, v [Lk, E'] (row stride ldkv: the two halves of one [Lk, 2E'] projection buffer
 * are fine), o [Lq, E'] (row stride ldo; d_o uses the same stride), lse [Lq, heads] f32; E' = heads*head_dim = 192.
 * Any Lq/Lk: few-query/many-key (Extractor) runs split-K over Lk with an LSE combine, many-query/few-key (Injector)
 * keeps K/V in shared memory.  impl: 0 = SIMT fp32 math (exact: the fp32 parity mode; f32 or bf16 tensors),
 * 1 = mma.sync tensor cores with TF32 operands and fp32 accumulation (f32 tensors; bf16 tensors fall back to 0).
 * Backward: dq [Lq, E'] (row stride lddq), dk, dv [Lk, E'] (row stride lddkv) f32, written (not accumulated). */
int mt_cross_attn_fwd(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, int dtype, void* o,
                      int64_t ldo, float* lse, int64_t lq, int64_t lk, int heads, int head_dim, float* workspace,
                      int64_t workspace_floats, int impl, void* stream);
int mt_cross_attn_bwd(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* o,
                      const void* d_o, int64_t ldo, const float* lse, int dtype, float* dq_f32, int64_t lddq,
                      float* dk_f32, float* dv_f32, int64_t lddkv, int64_t lq, int64_t lk, int heads, int head_dim,
                      int impl, void* stream);
int64_t mt_cross_attn_workspace_floats(int64_t lq, int64_t lk, int heads, int head_dim, int dtype, int impl);
/* deterministic mt_cross_attn_bwd (impl 1, f32 tensors): a loop that is split over CTAs stores its partials to
 * `workspace` ([splits][rows][heads * head_dim]) instead of adding them with atomics, and a second pass sums the splits in
 * index order; unsplit loops store as before.  workspace_floats >= mt_cross_attn_bwd_workspace_floats(...) (may be 0). */
int mt_cross_attn_bwd_ws(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, const void* o,
                         const void* d_o, int64_t ldo, const float* lse, int dtype, float* dq_f32, int64_t lddq,
                         float* dk_f32, float* dv_f32, int64_t lddkv, int64_t lq, int64_t lk, int heads, int head_dim,
                         float* workspace, int64_t workspace_floats, int impl, void* stream);
int64_t mt_cross_attn_bwd_workspace_floats(int64_t lq, int64_t lk, int heads, int head_dim, int dtype, int impl);
/* Head-averaged attention probabilities of a mt_cross_attn_fwd call:  p[i, j] = (1/heads) sum_h exp(q_i^h . k_j^h / 4
 * - lse[i, h]), p [Lq, Lk] f32 with row stride ldp >= Lk.
 * replaces: the attn_weights output (need_weights=True, average_attn_weights=True) of the nn.MultiheadAttention calls of
 * SelfAttentionLayer.forward_pre and CrossAttentionLayer.forward_pre (models/vitadapter/adapter_modules.py:72,87,198,225),
 * which a forward hook on `self_attn` / `multihead_attn` receives.
 * q, k, lse and impl as passed to (and lse as returned by) mt_cross_attn_fwd; k may be any column slice with row stride
 * ldk (the k half of the [Lk, 2E'] k|v buffer, or of a wider shared projection).  The scores are recomputed with the
 * forward's arithmetic (impl 1: TF32 operands, q scaled by log2(e)/4 before rounding), so each row sums to 1 up to
 * rounding.  Every element of p is written exactly once (no atomics): the output is bitwise reproducible. */
int mt_cross_attn_probs(const void* q, int64_t ldq, const void* k, int64_t ldk, int dtype, const float* lse, float* p,
                        int64_t ldp, int64_t lq, int64_t lk, int heads, int head_dim, int impl, void* stream);

/* ---- small fused element-wise pieces ------------------------------------------------------------------------------
 * y[r, c] = a[r, c] + gate[c] * (a[r, c] + b[r, c])      Injector tail `query + gamma * attn` (adapter_modules.py:362)
 *           with attn = a + b already containing the inner residual (:231).  gate may be NULL (=1).  f32 a, dtype b. */
int mt_gated_residual(const float* a, const void* b, int b_dtype, const float* gate, float* y, int64_t rows,
                      int64_t cols, void* stream);
/* backward of mt_gated_residual: da = dy * (1 + gate), db = dy * gate (dtype of b), dgate[c] = sum_r dy * (a + b)
 * (dgate is zeroed by the call and accumulated with atomics);  dysum [cols] or NULL: sum_r dy, from which the caller
 * gets the bias gradient of the projection that produced b (gate * dysum) without a reduction pass over db. */
int mt_gated_residual_bwd(const float* dy, const float* a, const void* b, int b_dtype, const float* gate, float* da,
                          void* db, int db_dtype, float* dgate, float* dysum, int64_t rows, int64_t cols, void* stream);
/* deterministic mt_gated_residual_bwd: dgate / dysum from block partials in `workspace` added in block order
 * (workspace_floats >= mt_colreduce_workspace_floats(cols)). */
int mt_gated_residual_bwd_ws(const float* dy, const float* a, const void* b, int b_dtype, const float* gate, float* da,
                             void* db, int db_dtype, float* dgate, float* dysum, int64_t rows, int64_t cols,
                             float* workspace, int64_t workspace_floats, void* stream);
/* y = x + D(a + bias): residual add after fc2 (torchscale/architecture/encoder.py:169-175), bias [cols] f32 or NULL,
 * D = dropout + DropPath of the branch (drop NULL = identity). */
int mt_residual_bias_add(const float* x, const void* a, int a_dtype, const float* bias, float* y, int64_t rows,
                         int64_t cols, const mt_dropout* drop, void* stream);
int mt_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, void* stream);
/* out[c] = sum_r x[r, c]: the bias gradient `dy.sum(0)` of the adapter's projections (autograd of nn.Linear in
 * models/vitadapter/adapter_modules.py:210-234); x [rows, cols] f32 with row stride ld, cols % 4 == 0, <= 4096. */
int mt_colsum(const float* x, int64_t ld, float* out, int64_t rows, int64_t cols, void* stream);
/* deterministic mt_colsum: block partials in `workspace` added in block order (>= mt_colreduce_workspace_floats(cols)) */
int mt_colsum_ws(const float* x, int64_t ld, float* out, int64_t rows, int64_t cols, float* workspace,
                 int64_t workspace_floats, void* stream);
/* backward of D: dst[i] = src[i] * keep_mask(i) / (1 - p) * path_scale, converted to dst_dtype (the gradient that
 * enters the dX GEMM of the branch).  drop must not be NULL. */
int mt_dropout_bwd_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, const mt_dropout* drop,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MODALTUNE_B200_H */
