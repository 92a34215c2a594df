/* xkv_b200 — C ABI of the B200-native xKV hot path (cross-layer SVD KV-cache compression).
 *
 * The reference (LiuTaowen-Tony/xKV) has no native code and no FFI: its hot path is the
 * Python function chain
 *     FakeLayerMergingCache.update            xKV/customized_cache/fake_layer_merge_dynamic_cache.py:127-153
 *       -> grouped_layer_merging              ...:155-208   (torch.cat over the group's layers)
 *       -> fake_svd                           ...:11-29     (transpose/reshape, torch.linalg.svd, matmul back)
 *       -> apply_rotary_pos_emb               ...:142-152   (RoPE on the reconstructed keys)
 *     decode attention over the dense result  xKV/attn_patch/llama.py:51-69 (SDPA)
 * Every entry point below replaces one of those library-call sites with a hand-written
 * sm_100a kernel (or a stream-ordered sequence of them).  The Python host mirror
 * (xkv_b200/customized_cache, xkv_b200/attn_patch) binds them with ctypes; see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - bf16 buffers are `void*` holding __nv_bfloat16, fp32 buffers are `float*`;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued asynchronously on it,
 *     nothing allocates, nothing synchronises (workspace comes from the caller);
 *   - functions return 0 on success, non-zero on error; xkv_last_error() gives the message
 *     of the calling thread's last failure.
 */
#ifndef XKV_B200_H_
#define XKV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define XKV_API __attribute__((visibility("default")))
#else
#define XKV_API
#endif

#define XKV_MAX_GROUP_LAYERS 16
#define XKV_MAX_GEMM_PROBLEMS 16
#define XKV_MAX_BATCH 16
#define XKV_MAX_LAYER_MAPS 64

/* ---- library ------------------------------------------------------------------------ */
XKV_API const char* xkv_last_error(void);
XKV_API int xkv_version(void);
/* number of kernels this library has launched since load (bench.py's `gpu_launches`) */
XKV_API int64_t xkv_launch_count(void);

/* ---- (1) prefill gather: replaces torch.cat(dim=1) + transpose(1,2).reshape ----------
 * cache:170-171 and cache:13-14.  Gathers the G layers' (bs, H, S, D) bf16 tensors (arbitrary
 * batch/head/token strides, unit stride over D) into the token-major matrix
 * X[bs*S][G*H*D] whose column order is (layer, head, dim), exactly the reference's. */
XKV_API int xkv_pack_group(const void* const* layer_ptrs_host, int num_layers, int bs, int heads, int seq,
                   int head_dim, int64_t stride_b, int64_t stride_h, int64_t stride_s, void* X,
                   void* stream);
/* inverse scatter (used by tests / the dense-materialise debug path): X -> per-layer tensors */
XKV_API int xkv_unpack_group(const void* X, int num_layers, int bs, int heads, int seq, int head_dim,
                     int64_t stride_b, int64_t stride_h, int64_t stride_s, void* const* layer_ptrs_host,
                     void* stream);

/* ---- (2) tcgen05 GEMM engine: replaces torch.linalg.svd / torch.matmul call sites -------
 * cache:20,26.  D (+split slabs) = sum_t A[term_a[t]] * B[term_b[t]]^T, bf16 operands, fp32
 * accumulation in TMEM.  Operands are given as up to three bf16 "limbs" (hi, mid, lo) of an
 * fp32 matrix so that products of fp32 matrices reach ~fp32 accuracy on the bf16 tensor path. */
typedef struct xkv_gemm_problem {
  int32_t M, N, K;
  int32_t num_terms;     /* 1..6 */
  int32_t a_mn_major;    /* 0: A stored [M][lda] (K contiguous); 1: A stored [K][lda] (M contiguous) */
  int32_t b_mn_major;    /* 0: B stored [N][ldb] (K contiguous); 1: B stored [K][ldb] (N contiguous) */
  const void* A[3];      /* bf16 limbs */
  const void* B[3];
  int64_t lda, ldb;      /* leading dimensions in elements (multiples of 8) */
  uint8_t term_a[6], term_b[6];
  void* D;               /* fp32 or bf16 output */
  int64_t ldd;
  int32_t out_bf16;        /* 0: fp32 output, 1: bf16 output */
  int32_t out_transposed;  /* 0: D[M][ldd], 1: D[N][ldd] */
  int32_t sym_upper;       /* 1: compute only tiles that intersect the upper triangle (Gram) */
  int32_t split_k;         /* >= 1: split s accumulates k-blocks of its slice into D + s*split_stride */
  int64_t split_stride;    /* elements */
  int32_t accum_phases;    /* > 1: the k range of a CTA is accumulated in this many sequential pieces that are summed in
                            * fp32 outside the tensor core (long reductions: the Gram over 64K tokens); fp32 output only */
  const int32_t* run_if;   /* optional DEVICE flag (NULL = always): the problem is skipped when *run_if == 0 at run time */
  /* Layered operands (the group's K / V read IN PLACE, no gather): with a_layers > 0 operand A is the column-wise
   * concatenation [A_layer[0] | A_layer[1] | ...] of a_layers equally shaped row-major bf16 matrices, each
   * layer_cols wide (a multiple of 64) with leading dimension lda -- exactly torch.cat(dim=1) + transpose(1,2).reshape of
   * the reference (cache:170-171, :13-14) when every layer tensor is a (1, H, S, D) view of token-major memory.  A[] is
   * ignored then and num_terms must be 1.  Likewise b_layers / B_layer.  One launch holds at most
   * XKV_MAX_LAYER_MAPS layer matrices in total. */
  int32_t a_layers, b_layers, layer_cols;
  const void* A_layer[XKV_MAX_GROUP_LAYERS];
  const void* B_layer[XKV_MAX_GROUP_LAYERS];
} xkv_gemm_problem;
XKV_API int xkv_gemm_grouped(const xkv_gemm_problem* problems_host, int num_problems, void* stream);
/* sizeof(xkv_gemm_problem) of this build (bindings check their mirror of the struct against it) */
XKV_API size_t xkv_gemm_problem_size(void);
/* test hook: nonzero (default) lets a launch whose problems all qualify run in CTA pairs (cta_group::2, one 256 x bn
 * tile per pair: gemm_pair_kernel -- the Gram, the projection, the power step, the triangular solve); 0 sends every
 * launch through the single-CTA 128 x 256 tiles (gemm_kernel).  Same results bit for bit. */
XKV_API void xkv_gemm_set_gram_pair(int on);

/* ---- small fp32 helpers of the factorisation ------------------------------------------ */
/* out[i][j] = sum_s slabs[s][i][j]; with symmetrize=1 the strictly-lower triangle is mirrored
 * from the upper one (Gram). rows x cols, ld in elements. */
XKV_API int xkv_reduce_slabs(const float* slabs, int num_slabs, int64_t slab_stride, int rows, int cols, int64_t ld,
                     int symmetrize, float* out, int64_t ld_out, void* stream);
XKV_API int xkv_reduce_slabs_batched(const float* const* slabs_host, float* const* out_host, int batch, int num_slabs,
                                     int64_t slab_stride, int rows, int cols, int64_t ld, int symmetrize,
                                     int64_t ld_out, void* stream);
/* split an fp32 matrix into bf16 limbs: hi = bf16(x), mid = bf16(x-hi), lo = bf16(x-hi-mid).
 * mid / lo may be NULL. */
XKV_API int xkv_split_bf16(const float* x, int rows, int cols, int64_t ld, void* hi, void* mid, void* lo,
                   int64_t ld_out, void* stream);
XKV_API int xkv_split_bf16_batched(const float* const* x_host, void* const* hi_host, void* const* mid_host,
                                   void* const* lo_host, int batch, int rows, int cols, int64_t ld, int64_t ld_out,
                                   void* stream);
/* Gram post-processing in one pass: hi/mid/lo[b] = bf16 limbs of the full symmetric n x n matrix whose upper-triangle
 * tiles are sum_s slabs[b][s] (split-K slabs `slab_stride` elements apart, as xkv_gemm_grouped writes them with
 * sym_upper = 1).  Equivalent to xkv_reduce_slabs(symmetrize = 1) followed by xkv_split_bf16, without the fp32 round trip. */
XKV_API int xkv_symmetrize_split_bf16(const float* const* slabs_host, int batch, int num_slabs, int64_t slab_stride,
                                      int n, int64_t ld, void* const* hi_host, void* const* mid_host,
                                      void* const* lo_host, int64_t ld_out, void* stream);
/* Token-sharded factorisation (SURVEY section 8e): the only data-path collective is the all-reduce of each matrix's
 * n x n fp32 Gram.  The Gram is symmetric, so only its upper triangle travels: row r contributes its columns
 * [32 * (r / 32), n), packed back to back: xkv_gram_packed_elems(n) = n^2 / 2 + 16 n floats.  pack: full (n x n,
 * symmetric or with a valid upper triangle) -> packed; unpack: packed -> full symmetric matrix (lower = mirrored upper). */
XKV_API size_t xkv_gram_packed_elems(int n);
XKV_API int xkv_gram_pack_upper(const float* full, int n, int64_t ld, float* packed, void* stream);
XKV_API int xkv_gram_unpack_upper(const float* packed, int n, float* full, int64_t ld, void* stream);
/* deterministic N(0,1) test matrix rounded to bf16 (counter-based generator) */
XKV_API int xkv_fill_gaussian_bf16(void* out, int rows, int cols, int64_t ld, uint64_t seed, void* stream);
/* Batched row normalisation: every row of Y[b] (rows x cols fp32, each row is a column of the sketch)
 * is scaled to unit 2-norm in place; if hi_host is non-NULL the bf16 limbs of the scaled rows are
 * written too (mid_host / lo_host may be NULL). */
XKV_API int xkv_normalize_rows(float* const* Y_host, void* const* hi_host, void* const* mid_host,
                               void* const* lo_host, int batch, int rows, int cols, int64_t ld, int64_t ld_out,
                               void* stream);
/* Spectrally shifted power steps (G - c I).  xkv_shift_normalize_rows: Y <- Y - c[b] Q (when Q_host != NULL;
 * Y = Q G just computed, Q the previous orthonormal basis), then row-normalise as xkv_normalize_rows; when
 * rdiag_host != NULL the row norms are recorded (rdiag_first) or multiplied into rdiag[b][0..rows).
 * xkv_rdiag_update: rdiag[b][j] /= Linv[b][j][j] after a Cholesky pass, so that rdiag accumulates diag(R) of
 * Y = R^T Q_new, whose trailing entries converge to lambda_l - c.  xkv_ritz_shift_update:
 * c[b] <- shift_scale * (mean of the last tail_rows entries of rdiag[b] + c[b]). */
XKV_API int xkv_shift_normalize_rows(float* const* Y_host, const float* const* Q_host, float* shift_dev,
                                     float* const* rdiag_host, int rdiag_first, void* const* hi_host,
                                     void* const* mid_host, void* const* lo_host, int batch, int rows, int cols,
                                     int64_t ld, int64_t ld_out, void* stream);
XKV_API int xkv_ritz_shift_update(float* const* rdiag_host, int batch, int rows, int tail_rows, float shift_scale,
                                  float* shift_dev, void* stream);
XKV_API int xkv_rdiag_update(float* const* rdiag_host, const float* const* Linv_host, int batch, int rows,
                             int64_t ld_linv, void* stream);
/* Device-side conditional passes.  xkv_pass_flags: flags_dev[b] = 1 when the Cholesky pass that produced Linv[b] met
 * a pivot L_jj^2 < min_pivot (or a NaN), else 0.  xkv_set_launch_predicate(flags_dev): until reset with NULL, the
 * calling thread's batched launches of xkv_shift_normalize_rows, xkv_reduce_slabs_batched,
 * xkv_cholesky_inverse(_limbs) and xkv_rdiag_update skip matrix b when flags_dev[b] == 0 at run time (GEMM problems
 * carry their own xkv_gemm_problem.run_if).  No host synchronisation: the kernels are always enqueued. */
XKV_API int xkv_pass_flags(const float* const* Linv_host, int batch, int rows, int64_t ld_linv, float min_pivot,
                           int32_t* flags_dev, void* stream);
XKV_API void xkv_set_launch_predicate(const int32_t* flags_dev);
/* Batched blocked Cholesky (S + shift*I) = L L^T of l x l fp32 matrices (l % 64 == 0, symmetric, both
 * triangles present, unit diagonal expected) with explicit inverse Linv = L^{-1} (dense l x l, zero above the
 * diagonal).  One launch: a thread-block cluster per matrix (xkv_chol.cu).  S is scratch and is destroyed.
 * Pivots below pivot_floor are clamped, so the factorisation never fails (CholeskyQR is repeated instead; the
 * shift keeps the fp32 Gram of an ill-conditioned sketch positive).  The _limbs variant also writes the bf16
 * limbs hi + mid + lo ~= Linv (row stride ld_limb) that the tensor-core GEMM Q = Linv Y consumes. */
XKV_API int xkv_cholesky_inverse(float* const* S_host, float* const* Linv_host, int batch, int l, int64_t ld,
                                 float shift, float pivot_floor, void* stream);
XKV_API int xkv_cholesky_inverse_limbs(float* const* S_host, float* const* Linv_host, void* const* hi_host,
                                       void* const* mid_host, void* const* lo_host, int batch, int l, int64_t ld,
                                       int64_t ld_limb, float shift, float pivot_floor, void* stream);
/* Shared-memory two-sided Jacobi eigen-solver for the Rayleigh-Ritz windows: `count` symmetric W x W
 * fp32 matrices (W even, <= 160), one CTA each. evals: eigenvalues sorted descending; Wt (optional):
 * eigenvectors as rows, same order. */
XKV_API int xkv_jacobi_eigh(const float* const* T_host, float* const* evals_host, float* const* Wt_host, int count,
                            int W, int64_t ld, int64_t ld_w, int sweeps, void* stream);
/* fp32 (rows x cols) -> bf16 copy `dst` and/or transposed bf16 copy `dstT` (cols x rows) */
XKV_API int xkv_convert_bf16(const float* src, int rows, int cols, int64_t ld, void* dst, int64_t ld_dst, void* dstT,
                             int64_t ld_dstT, void* stream);

/* out[i] = sqrt(max(in[i], 0)) (Ritz values -> singular values) */
XKV_API int xkv_sqrt_clamp(const float* in, float* out, int count, void* stream);

/* ---- (2) the factorisation driver: replaces fake_svd (cache:11-29) for a batch ------------------
 * X[b] (m x n bf16, row stride ldx)  ~=  A[b] (m x rank bf16) * Vt[b] (rank x n bf16); V[b] (n x rank) is
 * Vt transposed (the layout the decode kernel reads). sigma[b] (optional) receives XKV_FACTORIZE_SIGMA_COUNT
 * leading singular-value estimates. The sketch is round_up(rank + 64, 64) columns wide and must fit: 0 < rank <= m and
 * round_up(rank + 64, 64) <= n. Pure host code: enqueues the kernels above on `stream`. stage_events_host (optional):
 * 7 cudaEvent_t recorded at start / after the Gram GEMM / Gram reduce+split / range finder / power iterations /
 * Rayleigh-Ritz / projection.
 * phase 0 (gram_host may be NULL) does everything on one device.  Token-sharded use (rows of X split over GPUs) splits it
 * in three: phase 1 writes each matrix's LOCAL Gram X_p^T X_p (n x n fp32, symmetric) to gram_host[b] and returns; the
 * caller all-reduces those buffers; phase 3 derives Vt / V from the reduced gram_host[b] and stops (X_host / A_host may
 * be NULL), so that the small-matrix stages of different matrices can run on different ranks; phase 4 only projects,
 * A = X V, with the Vt the caller supplies (e.g. received from the rank that ran phase 3). */
#define XKV_FACTORIZE_SIGMA_COUNT 128
XKV_API size_t xkv_factorize_workspace_bytes(int batch, int m, int n, int rank);
/* Same on a layer group's K (or V) tensors IN PLACE: matrix b is the column-wise concatenation of `layers` row-major
 * bf16 matrices layer_ptrs_host[b * layers + i] (m x layer_cols, row stride ld_layer) -- the reference's
 * torch.cat(dim=1) + transpose(1,2).reshape (cache:170-171, :13-14) when every layer tensor is a (1, H, S, D) view of
 * token-major memory (layer_cols = H * D).  The Gram pass and the projection pass read the layer tensors through
 * per-layer tensor maps: no gather kernel, no packed copy (1 GiB per group at config 2).  n = layers * layer_cols. */
XKV_API int xkv_factorize_groups(const void* const* layer_ptrs_host, int batch, int layers, int layer_cols, int m,
                                 int64_t ld_layer, int rank, void* const* A_host, void* const* Vt_host,
                                 void* const* V_host, float* const* sigma_host, void* workspace, size_t workspace_bytes,
                                 void* const* stage_events_host, void* stream);
XKV_API int xkv_factorize_batch(const void* const* X_host, int batch, int m, int n, int64_t ldx, int rank,
                                void* const* A_host, void* const* Vt_host, void* const* V_host,
                                float* const* sigma_host, float* const* gram_host, int phase, void* workspace,
                                size_t workspace_bytes, void* const* stage_events_host, void* stream);

/* ---- (3) decode-time attention over the factored cache: replaces the SDPA call over dense K^/V^ --------
 * llama.py:58-69 with the reconstruction of cache:26-27 and the RoPE of cache:142-148 fused in.
 *   q          (Hq, D) bf16, post-RoPE query of ONE layer, batch 1
 *   A_k, A_v   (S, rk) / (S, rv) bf16 token factors of the layer's group
 *   Vk_layer   (H*D, rk) bf16: rows [layer_in_group*H*D, +H*D) of the group's right factor V_k (n x rk);
 *   Vv_layer   (H*D, rv) likewise for values
 *   cos, sin   (S, D) bf16 RoPE tables of the prefill positions (half-split convention), or NULL when the
 *              keys were compressed post-RoPE / need none (re_apply_rope=False, deepseek_v2.py:226)
 *   k_tail, v_tail  (H, T, D) bf16 dense decode tokens appended after prefill (keys post-RoPE), T may be 0
 *   out        (Hq, D) bf16 = softmax(scale * q [K^;K_tail]^T) [V^;V_tail] with GQA (Hq/H query heads per kv head)
 * Full-rank K^/V^ are never written to HBM. D in {64, 128}; Hq/H <= 8. */
XKV_API size_t xkv_decode_workspace_bytes(int Hq, int S, int T, int rv);
XKV_API int xkv_decode_attention(const void* q, int Hq, int H, int D, const void* A_k, int64_t lda_k, int rk,
                                 const void* Vk_layer, int64_t ldv_k, const void* A_v, int64_t lda_v, int rv,
                                 const void* Vv_layer, int64_t ldv_v, int S, const void* cos, const void* sin,
                                 int64_t ld_cs, const void* k_tail, const void* v_tail, int T, int64_t tail_stride_h,
                                 int64_t tail_stride_t, float scale, void* out, void* workspace,
                                 size_t workspace_bytes, void* stream);
/* Same, and lse_out[hq] (Hq floats, may be NULL) = log sum_t exp(scale * q_hq . k_t) over the S + T tokens of THIS call.
 * Token shards of a long context (SURVEY section 8e; each rank holds the rows of A_k / A_v of its tokens and the RoPE rows
 * of their positions) each call this on their rows and merge flash-decoding style:
 *   out = sum_p exp(lse_p - lse) out_p,  lse = log sum_p exp(lse_p)      (xkv_b200.parallel.merge_token_shards). */
XKV_API int xkv_decode_attention_lse(const void* q, int Hq, int H, int D, const void* A_k, int64_t lda_k, int rk,
                                     const void* Vk_layer, int64_t ldv_k, const void* A_v, int64_t lda_v, int rv,
                                     const void* Vv_layer, int64_t ldv_v, int S, const void* cos, const void* sin,
                                     int64_t ld_cs, const void* k_tail, const void* v_tail, int T, int64_t tail_stride_h,
                                     int64_t tail_stride_t, float scale, void* out, void* workspace,
                                     size_t workspace_bytes, void* stream, float* lse_out);
/* Multi-token step (speculative verification, a continuation chunk): Tq query tokens per q head in one call.
 *   q, out     (Hq*Tq, D) bf16, row hq*Tq + t = query token t of q head hq (HF's query[0] (Hq, Tq, D) made contiguous)
 *   k_tail, v_tail  (H, T, D): the LAST Tq tail tokens are the queries' own (T >= Tq); query token t sees the whole
 *              compressed prefix and tail tokens [0, T - Tq + t] (causal among the new tokens)
 *   lse_out    Hq*Tq floats (may be NULL), one per row
 * Bounds: (Hq/H)*Tq <= 64 and Hq*Tq <= 512 (XKV_ERR otherwise: callers take a dense path).  Workspace:
 * xkv_decode_workspace_bytes(Hq*Tq, S, T, rv).  Four launches whatever Tq is; the prefix keys are rebuilt once per call on
 * the head_dim 128 path (CTA pairs), once per 8 rows of a kv head on the others.  Tq = 1 is xkv_decode_attention_lse. */
XKV_API int xkv_decode_attention_multi(const void* q, int Hq, int Tq, int H, int D, const void* A_k, int64_t lda_k, int rk,
                                       const void* Vk_layer, int64_t ldv_k, const void* A_v, int64_t lda_v, int rv,
                                       const void* Vv_layer, int64_t ldv_v, int S, const void* cos, const void* sin,
                                       int64_t ld_cs, const void* k_tail, const void* v_tail, int T, int64_t tail_stride_h,
                                       int64_t tail_stride_t, float scale, void* out, void* workspace,
                                       size_t workspace_bytes, void* stream, float* lse_out);
/* One-sided group: exactly one of the layer's two slots is factored, the other stayed dense (merge_key or merge_value off,
 * or a rank that does not fit one side).  Each side is given EITHER as factors (A_*, lda_*, r*, V*_layer, ldv_*; the dense
 * pointer NULL) OR as a dense prefix slot (*_dense, *_stride_h, *_stride_t; A_* NULL):
 *   k_dense    rotated prefix keys, element (t, h, d) at k_dense[h * k_stride_h + t * k_stride_t + d] (an (S, H, D) or
 *              (H, S, D) view); cos / sin are not read for a dense key side
 *   v_dense    prefix values, same addressing
 * Both strides multiples of 8 elements, the base 16-byte aligned; q 16-byte aligned when the key side is dense.  Both sides
 * factored or both dense is an error (use xkv_decode_attention_multi, or SDPA).  Everything else -- q / Tq / heads, the
 * tail and its causal rule, scale, out, lse_out, bounds -- as xkv_decode_attention_multi.  Workspace:
 * xkv_decode_half_workspace_bytes(Hq*Tq, S, T, value_width), value_width = rv for factored values, D for dense ones. */
XKV_API size_t xkv_decode_half_workspace_bytes(int rows, int S, int T, int value_width);
XKV_API int xkv_decode_attention_half(const void* q, int Hq, int Tq, int H, int D, const void* A_k, int64_t lda_k, int rk,
                                      const void* Vk_layer, int64_t ldv_k, const void* k_dense, int64_t k_stride_h,
                                      int64_t k_stride_t, const void* A_v, int64_t lda_v, int rv, const void* Vv_layer,
                                      int64_t ldv_v, const void* v_dense, int64_t v_stride_h, int64_t v_stride_t, int S,
                                      const void* cos, const void* sin, int64_t ld_cs, const void* k_tail,
                                      const void* v_tail, int T, int64_t tail_stride_h, int64_t tail_stride_t,
                                      float scale, void* out, void* workspace, size_t workspace_bytes, void* stream,
                                      float* lse_out);
/* test hook: 1 forces the tile-per-CTA scores kernel (otherwise chosen only when one head's slice of the right
 * factor exceeds 128 KiB of shared memory), 0 restores the automatic choice */
XKV_API void xkv_decode_force_tiled(int on);
/* test hook: persistent scores kernel to use where several apply: 0 automatic (head_dim 128: score MMA in CTA pairs,
 * cta_group::2, half a right-factor slice per CTA), 1 FFMA epilogue, 2 score MMA with one independent CTA per kv head,
 * 3 CTA pairs; 4 = automatic scores kernel, but slab reduction and combine as two launches (default: one cluster launch) */
XKV_API void xkv_decode_set_variant(int variant);
/* Absorbed attention over a token factor: replaces, for the MLA latent slot (deepseek_v2.py:217-235: reconstructed
 * latents -> kv_a_layernorm -> kv_b_proj over the WHOLE cache -> attention, every decode step), the part that touches
 * the cache.  The latent of token t is c_t = V_l a_t and both attention products are linear in it, so with the query
 * folded into the rank space by the caller, q_hat[h] = V_l^T (gamma o W_UK[h]^T q_nope[h]) (Hq x r bf16):
 *     s[h][t]  = scale * ( row_scale[t] * (q_hat[h] . A[t]) + bias_q[h] . bias_k[t] )
 *     u_out[h] = sum_t softmax_t(s)[h][t] * row_scale[t] * A[t]         (Hq x r fp32, rank space)
 *     lse_out[h] = log sum_t exp(s[h][t])                               (for merging with the dense decode tail)
 * row_scale (S fp32, may be NULL = 1): 1 / rms of the reconstructed latent (kv_a_layernorm's per-token factor);
 * bias_q (Hq x bias_dim) / bias_k (S x bias_dim, row stride ld_bias_k) bf16, may both be NULL: the RoPE part
 * q_pe . k_pe.  A (S x r bf16, row stride lda) is read twice; the S x kv_lora_rank latents are never rebuilt. */
XKV_API size_t xkv_decode_absorbed_workspace_bytes(int Hq, int S, int r);
XKV_API int xkv_decode_absorbed(const void* q_hat, int Hq, const void* A, int64_t lda, int r, int S,
                                const float* row_scale, const void* bias_q, const void* bias_k, int64_t ld_bias_k,
                                int bias_dim, float scale, float* u_out, float* lse_out, void* workspace,
                                size_t workspace_bytes, void* stream);
/* RoPE on materialised keys x (rows, H, D) bf16 in place, in the reference's bf16 arithmetic
 * (apply_rotary_pos_emb as called at cache:148,152): x*cos + rotate_half(x)*sin, cos/sin (rows, D). */
XKV_API int xkv_rope_bf16(void* x, int64_t ld_row, int rows, int H, int D, const void* cos, const void* sin,
                          int64_t ld_cs, void* stream);

/* ---- (4) append: project new token rows onto a group's right factor -------------------------------
 * a_out (T x r bf16) = x_new (T x n bf16, the group's token-major rows from xkv_pack_group) * V (n x r bf16).
 * An extension: the reference keeps decode tokens uncompressed (cache:131), so this is opt-in. */
XKV_API size_t xkv_append_workspace_bytes(int T, int n, int r);
XKV_API int xkv_append_project(const void* x_new, int64_t ldx, int T, const void* V, int64_t ldv, int n, int r,
                               void* a_out, int64_t lda, void* workspace, size_t workspace_bytes, void* stream);
/* Several projections in ONE launch (a group's K and V factor: the step is a few microseconds of HBM time, so launches
 * dominate otherwise).  workspace_bytes >= the sum of xkv_append_workspace_bytes(T, n, r) over the problems. */
#define XKV_APPEND_MAX_PROBLEMS 4
typedef struct xkv_append_problem {
  const void* x_new;   /* T x n bf16, row stride ldx */
  const void* V;       /* n x r bf16, row stride ldv */
  void* a_out;         /* T x r bf16, row stride lda */
  int64_t ldx, ldv, lda;
  int32_t n, r;
} xkv_append_problem;
XKV_API int xkv_append_project_batch(const xkv_append_problem* problems_host, int count, int T, void* workspace,
                                     size_t workspace_bytes, void* stream);

/* ---- SLERP / MiniCache branch (layer_merge_impl == "slerp"): replaces fake_minicache_merge -----------
 * cache:32-100, called at cache:183-197 on two layers' rows (rows x d bf16, row stride ld). e1 / e2 receive the
 * merged rows of layer 1 / layer 2 (rows whose angle exceeds d_min + (d_max - d_min) * gamma are replaced by the
 * SLERP direction rescaled to each layer's norm; the others are copied, as the reference does). */
XKV_API size_t xkv_slerp_workspace_bytes(int64_t rows);
XKV_API int xkv_slerp_merge(const void* x1, const void* x2, int64_t rows, int d, int64_t ld, float t, float gamma,
                            void* e1, void* e2, int64_t ld_out, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* XKV_B200_H_ */
