// xkv_b200 — stream-ordered driver of the low-rank factorisation (replaces fake_svd,
// fake_layer_merge_dynamic_cache.py:11-29, for a batch of equally-shaped group matrices).
//
//   X (m x n bf16)  ~=  A (m x r bf16) * Vt (r x n bf16),   A = X V
//
// Pure host code: it carves the caller's workspace and enqueues the kernels of xkv_gemm.cu /
// xkv_small.cu on the caller's stream (no allocation, no synchronisation).  The algorithm is
// documented in xkv_b200/factorize.py and DESIGN.md: Gram -> Gaussian range finder -> shifted
// CholeskyQR -> power steps on G -> windowed Rayleigh-Ritz (shared-memory Jacobi) -> A = X V.
#include <cuda_bf16.h>

#include <vector>

#include "xkv_host.h"

namespace xkv {

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int round_up_int(int x, int k) { return (x + k - 1) / k * k; }

struct Bump {
  char* base;
  size_t off, cap;
  bool overflow;
  void* take(size_t bytes) {
    off = align_up(off, 1024);
    void* p = base ? base + off : nullptr;
    off += bytes;
    if (base && off > cap) overflow = true;
    return p;
  }
  float* f32(size_t n) { return static_cast<float*>(take(n * 4)); }
  void* bf16(size_t n) { return take(n * 2); }
};

// The schedule (DESIGN.md section 2, measured choices in section 8): sketch width l = round_up(rank + 64, 64); a Gaussian
// range finder and 4 power steps on G; 2 CholeskyQR passes after the range finder and after the first step, one pass
// plus a device-decided one after the spectrally shifted steps 1-3; then the Rayleigh-Ritz windows.
constexpr int kOversample = 64;
constexpr int kPowerSteps = 4;
constexpr int kGramPieceTokens = 16384;   // tensor-core accumulation length of the Gram (xkv_gemm_problem.accum_phases)
constexpr int kSmallSplitK = 8;
constexpr int kWindow = 128;              // Rayleigh-Ritz window width (shared-memory Jacobi: even, <= 160)
constexpr int kJacobiSweeps = 3;
constexpr float kSpectralShift = 0.5f;    // c = 0.5 x (mean of the last kShiftTail entries of diag(R)) ~ lambda_l / 2
constexpr int kShiftTail = 8;
constexpr float kCholShift[3] = {3e-4f, 1e-6f, 1e-7f};   // diagonal shift of CholeskyQR pass index 0 / 1 / 2
constexpr float kPivotFloor = 1e-12f;
constexpr float kSecondPassMinPivot = 0.05f;
constexpr uint64_t kSeed = 1234;
static_assert(kWindow == XKV_FACTORIZE_SIGMA_COUNT, "the leading window gives the singular values");

struct Plan {
  int B, m, n, sk, skw;
  // rank r and sketch width l; the Rayleigh-Ritz window is rows [l - kWindow, l) of the basis, of which the
  // r - (l - kWindow) rows left of row r are kept
  int r, l;
  // per-matrix buffers; window 0 straddles row r, window 1 is rows [0, kWindow) (the leading singular values)
  void* g_limb[XKV_MAX_BATCH][3];
  float* f_a[XKV_MAX_BATCH];
  float* f_b[XKV_MAX_BATCH];
  void* lh[XKV_MAX_BATCH];
  void* lm[XKV_MAX_BATCH];
  void* ll[XKV_MAX_BATCH];
  float* s_slabs[XKV_MAX_BATCH];
  float* s_mat[XKV_MAX_BATCH];
  float* linv[XKV_MAX_BATCH];
  float* rdiag[XKV_MAX_BATCH];   // running diag(R) of the current power step
  void* linv_l[XKV_MAX_BATCH][3];
  float* yw[XKV_MAX_BATCH][2];
  void* yw_l[XKV_MAX_BATCH][2][3];
  float* t_slabs[XKV_MAX_BATCH][2];
  float* t_mat[XKV_MAX_BATCH][2];
  float* evals[XKV_MAX_BATCH][2];
  float* wt[XKV_MAX_BATCH];
  void* wsel_l[XKV_MAX_BATCH][3];
  // shared
  float* gram_slabs;  // [B][n][n]
  float* shift_dev;   // [B] spectral shifts of the current power step
  int* pass_flags;    // [B] device decision: this matrix needs a second CholeskyQR pass in the current step
  int* redo_flags;    // [B] device decision: the lightly shifted Cholesky of this matrix broke down, redo it heavily shifted
  size_t bytes;
};

static int make_plan(Plan& P, Bump& bump, int B, int m, int n, int rank) {
  XKV_REQUIRE(B >= 1 && B <= XKV_MAX_BATCH, "factorize: batch %d out of range (1..%d)", B, XKV_MAX_BATCH);
  XKV_REQUIRE(n % 8 == 0, "factorize: n=%d must be a multiple of 8", n);
  P.B = B;
  P.m = m;
  P.n = n;
  const int nkb = (n + 63) / 64;
  P.sk = nkb < kSmallSplitK ? nkb : kSmallSplitK;
  P.skw = nkb < 16 ? nkb : 16;
  P.r = rank;
  P.l = round_up_int(rank + kOversample, 64);   // >= 128 = kWindow for every rank >= 1
  XKV_REQUIRE(rank > 0 && rank <= m && P.l <= n, "factorize: rank %d (sketch %d) does not fit a %d x %d matrix", rank, P.l, m,
              n);
  const size_t nn = n, l = P.l, W = kWindow;
  for (int b = 0; b < B; ++b) {
    for (int i = 0; i < 3; ++i) P.g_limb[b][i] = bump.bf16(nn * nn);
    P.f_a[b] = bump.f32(l * nn);
    P.f_b[b] = bump.f32(l * nn);
    P.lh[b] = bump.bf16(l * nn);
    P.lm[b] = bump.bf16(l * nn);
    P.ll[b] = bump.bf16(l * nn);
    P.s_slabs[b] = bump.f32(static_cast<size_t>(P.sk) * l * l);
    P.s_mat[b] = bump.f32(l * l);
    P.linv[b] = bump.f32(l * l);
    P.rdiag[b] = bump.f32(l);
    for (int i = 0; i < 3; ++i) P.linv_l[b][i] = bump.bf16(l * l);
    for (int w = 0; w < 2; ++w) {
      P.yw[b][w] = bump.f32(W * nn);
      for (int i = 0; i < 3; ++i) P.yw_l[b][w][i] = bump.bf16(W * nn);
      P.t_slabs[b][w] = bump.f32(static_cast<size_t>(P.skw) * W * W);
      P.t_mat[b][w] = bump.f32(W * W);
      P.evals[b][w] = bump.f32(W);
    }
    P.wt[b] = bump.f32(W * W);
    for (int i = 0; i < 3; ++i) P.wsel_l[b][i] = bump.bf16(W * W);
  }
  P.gram_slabs = bump.f32(static_cast<size_t>(B) * nn * nn);
  P.shift_dev = bump.f32(XKV_MAX_BATCH);
  P.pass_flags = reinterpret_cast<int*>(bump.f32(XKV_MAX_BATCH));
  P.redo_flags = reinterpret_cast<int*>(bump.f32(XKV_MAX_BATCH));
  P.bytes = align_up(bump.off, 1024);
  return 0;
}

static const uint8_t T6A[6] = {0, 0, 1, 1, 0, 2}, T6B[6] = {0, 1, 0, 1, 2, 0};

static xkv_gemm_problem problem(const void* a0, const void* a1, const void* a2, long long lda, int a_mn,
                                const void* b0, const void* b1, const void* b2, long long ldb, int b_mn, void* D,
                                long long ldd, int M, int N, int K, int nterms) {
  xkv_gemm_problem p;
  std::memset(&p, 0, sizeof(p));
  p.M = M;
  p.N = N;
  p.K = K;
  p.num_terms = nterms;
  p.a_mn_major = a_mn;
  p.b_mn_major = b_mn;
  p.A[0] = a0;
  p.A[1] = a1;
  p.A[2] = a2;
  p.B[0] = b0;
  p.B[1] = b1;
  p.B[2] = b2;
  p.lda = lda;
  p.ldb = ldb;
  for (int t = 0; t < nterms; ++t) {
    p.term_a[t] = T6A[t];
    p.term_b[t] = T6B[t];
  }
  p.D = D;
  p.ldd = ldd;
  p.split_k = 1;
  return p;
}

// D = A B^T (plain output) restated as D^T = B A^T stored transposed: the same memory, the same sequence of limb products
// per k block, hence the same bits -- but the operand with the long dimension supplies M.  The products with M = sketch
// width (576 / 832: 11 % / 8 % of padding in 128-row tiles, 33 % / 23 % in 256-row ones) and N = n = 4096 become
// M = 4096, N = l, which the CTA-pair kernel tiles exactly (xkv_gemm.cu pair_bn).
static xkv_gemm_problem swap_roles(const xkv_gemm_problem& p) {
  xkv_gemm_problem q = p;
  q.M = p.N;
  q.N = p.M;
  q.a_mn_major = p.b_mn_major;
  q.b_mn_major = p.a_mn_major;
  for (int i = 0; i < 3; ++i) {
    q.A[i] = p.B[i];
    q.B[i] = p.A[i];
  }
  q.lda = p.ldb;
  q.ldb = p.lda;
  for (int t = 0; t < 6; ++t) {
    q.term_a[t] = p.term_b[t];
    q.term_b[t] = p.term_a[t];
  }
  q.out_transposed = p.out_transposed ? 0 : 1;
  return q;
}

static int run_gemms(std::vector<xkv_gemm_problem>& ps, void* stream, int per_launch = XKV_MAX_GEMM_PROBLEMS) {
  if (per_launch > XKV_MAX_GEMM_PROBLEMS) per_launch = XKV_MAX_GEMM_PROBLEMS;
  if (per_launch < 1) per_launch = 1;
  for (size_t i = 0; i < ps.size(); i += per_launch) {
    const int cnt = static_cast<int>(ps.size() - i < static_cast<size_t>(per_launch) ? ps.size() - i : per_launch);
    int rc = xkv_gemm_grouped(ps.data() + i, cnt, stream);
    if (rc) return rc;
  }
  ps.clear();
  return 0;
}

#define XKV_TRY(expr)      \
  do {                     \
    int _rc = (expr);      \
    if (_rc) return _rc;   \
  } while (0)

static inline const __nv_bfloat16* row_bf16(const void* base, long long row, long long ld) {
  return static_cast<const __nv_bfloat16*>(base) + row * ld;
}

}  // namespace xkv

using namespace xkv;

extern "C" size_t xkv_factorize_workspace_bytes(int batch, int m, int n, int rank) {
  Plan P;
  Bump bump{nullptr, 0, 0, false};
  if (batch < 1 || batch > XKV_MAX_BATCH || make_plan(P, bump, batch, m, n, rank)) return 0;
  return P.bytes;
}

// X_host: packed matrices (layers == 0) or per-layer pointers [batch][layers] read in place
static int factorize_impl(const void* const* X_host, int layers, int layer_cols, int batch, int m, int n, int64_t ldx,
                          int rank, void* const* A_host, void* const* Vt_host, void* const* V_host,
                          float* const* sigma_host, float* const* gram_host, int phase, void* workspace,
                          size_t workspace_bytes, void* const* stage_events_host, void* stream) {
  XKV_REQUIRE(phase == 0 || phase == 1 || phase == 3 || phase == 4,
              "factorize: phase must be 0 (all), 1 (Gram only), 3 (right factor from Gram) or 4 (projection)");
  XKV_REQUIRE(workspace && Vt_host && (phase == 1 || phase == 4 || V_host) && (phase == 3 || X_host) &&
                  (phase == 1 || phase == 3 || A_host),
              "factorize: null argument");
  XKV_REQUIRE(phase == 0 || phase == 4 || gram_host != nullptr, "factorize: phases 1 / 3 need the per-matrix Gram buffers");
  static thread_local Plan P;
  Bump bump{static_cast<char*>(workspace), 0, workspace_bytes, false};
  XKV_TRY(make_plan(P, bump, batch, m, n, rank));
  XKV_REQUIRE(!bump.overflow && P.bytes <= workspace_bytes, "factorize: workspace too small (%zu < %zu bytes)",
              workspace_bytes, P.bytes);
  XKV_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "factorize: workspace must be 256-byte aligned");
  const int B = batch, W = kWindow, l = P.l, r = P.r;
  const long long nn = n;
  cudaStream_t st = as_stream(stream);
  int ev = 0;
  auto mark = [&]() -> int {
    if (stage_events_host && stage_events_host[ev])
      XKV_CHECK_CUDA(cudaEventRecord(reinterpret_cast<cudaEvent_t>(stage_events_host[ev]), st));
    ++ev;
    return 0;
  };
  std::vector<xkv_gemm_problem> ps;
  xkv_set_launch_predicate(nullptr);   // a call that failed half-way must not leave this thread's launches predicated
  XKV_TRY(mark());  // 0: start

  // ---- 7. projection A = X V (second and last pass over X); phase 4 runs only this, on a right factor the caller supplies ----
  auto project = [&]() -> int {
    for (int b = 0; b < B; ++b) {
      const void* x0 = layers > 0 ? X_host[static_cast<size_t>(b) * layers] : X_host[b];
      xkv_gemm_problem p = problem(x0, nullptr, nullptr, ldx, 0, Vt_host[b], nullptr, nullptr, nn, 0, A_host[b], r, m, r, n, 1);
      if (layers > 0) {
        p.a_layers = layers;
        p.layer_cols = layer_cols;
        for (int i = 0; i < layers; ++i) p.A_layer[i] = X_host[static_cast<size_t>(b) * layers + i];
      }
      p.out_bf16 = 1;
      ps.push_back(p);
    }
    GemmLowPriorityScope low;
    return run_gemms(ps, stream, layers > 0 ? XKV_MAX_LAYER_MAPS / layers : XKV_MAX_GEMM_PROBLEMS);
  };
  if (phase == 4) return project();

  // ---- 1. Gram matrices and their bf16 limbs ----
  // phase 1 stops after the (local) Gram so that token-sharded callers can all-reduce it; phase 3 resumes
  // from the caller's reduced Gram.
  if (phase != 3) {
    for (int b = 0; b < B; ++b) {
      const void* x0 = layers > 0 ? X_host[static_cast<size_t>(b) * layers] : X_host[b];
      xkv_gemm_problem p = problem(x0, nullptr, nullptr, ldx, 1, x0, nullptr, nullptr, ldx, 1,
                                   P.gram_slabs + static_cast<size_t>(b) * nn * nn, nn, n, n, m, 1);
      if (layers > 0) {   // both operands are the group's layer tensors, read in place
        p.a_layers = p.b_layers = layers;
        p.layer_cols = layer_cols;
        for (int i = 0; i < layers; ++i) p.A_layer[i] = p.B_layer[i] = X_host[static_cast<size_t>(b) * layers + i];
      }
      p.sym_upper = 1;
      const int ph = (m + kGramPieceTokens - 1) / kGramPieceTokens;
      p.accum_phases = ph > 64 ? 64 : ph;
      ps.push_back(p);
    }
    XKV_TRY(run_gemms(ps, stream, layers > 0 ? XKV_MAX_LAYER_MAPS / layers : XKV_MAX_GEMM_PROBLEMS));
  }
  XKV_TRY(mark());  // 1: Gram GEMM (the dominant kernel, timed on its own for the roofline)
  if (phase == 0) {
    // upper-triangle tiles -> symmetric bf16 limbs in one pass (no fp32 Gram round trip)
    const float* sl[XKV_MAX_BATCH];
    void *h0[XKV_MAX_BATCH], *h1[XKV_MAX_BATCH], *h2[XKV_MAX_BATCH];
    for (int b = 0; b < B; ++b) {
      sl[b] = P.gram_slabs + static_cast<size_t>(b) * nn * nn;
      h0[b] = P.g_limb[b][0], h1[b] = P.g_limb[b][1], h2[b] = P.g_limb[b][2];
    }
    XKV_TRY(xkv_symmetrize_split_bf16(sl, B, 1, nn * nn, n, nn, h0, h1, h2, nn, stream));
  } else {
    for (int b = 0; b < B; ++b) {
      float* g = gram_host[b];
      XKV_REQUIRE(g != nullptr, "factorize: null Gram buffer %d", b);
      if (phase == 1)
        XKV_TRY(xkv_reduce_slabs(P.gram_slabs + static_cast<size_t>(b) * nn * nn, 1, nn * nn, n, n, nn, 1, g, nn, stream));
      else
        XKV_TRY(xkv_split_bf16(g, n, n, nn, P.g_limb[b][0], P.g_limb[b][1], P.g_limb[b][2], nn, stream));
    }
  }
  XKV_TRY(mark());  // 2: Gram reduce + limb split
  if (phase == 1) return 0;

  float** cur = P.f_a;
  float** nxt = P.f_b;
  auto swap_bufs = [&]() {
    float** t = cur;
    cur = nxt;
    nxt = t;
  };
  // cur <- orth(cur): row-normalised, shifted CholeskyQR in two passes.  The pass index selects the diagonal shift of
  // the Cholesky (kCholShift); every pass with index > 0 redoes a broken-down Cholesky heavily shifted (device decision).
  // Not `shifted` (range finder, first power step): passes 0 and 1, the first one heavily shifted for the raw sketch.
  // `shifted` (power steps 1-3): cur = Q_prev G and nxt still holds Q_prev, so the first pass (index 1) first forms
  // Q_prev (G - c I).  The basis entering such a step is orthonormal and ordered by dominance, so this one pass is enough
  // unless its Cholesky met a pivot below kSecondPassMinPivot: the device decides per matrix (xkv_pass_flags) whether
  // the second pass (index 2) runs; its kernels are always enqueued and exit at once for the matrices that do not need
  // it.  That pass writes its result over `cur` (its operands are the limb copies), so the buffers are where the
  // following stages expect them either way.
  // With `track`, diag(R) of the step is accumulated in P.rdiag (row norms x Cholesky diagonals).
  // `final_call`: nothing orthonormalises the result again (the last power step): the solve keeps all 6 limb terms
  auto cholqr = [&](bool shifted, bool track, bool final_call) -> int {
    const int first = shifted ? 1 : 0;
    for (int pp = first; pp <= first + 1; ++pp) {
      const bool cond = shifted && pp == 2;
      if (cond) {
        XKV_TRY(xkv_pass_flags(P.linv, B, l, l, kSecondPassMinPivot, P.pass_flags, stream));
        xkv_set_launch_predicate(P.pass_flags);
      }
      int rc = [&]() -> int {
        XKV_TRY(xkv_shift_normalize_rows(cur, (pp == first && shifted) ? nxt : nullptr, P.shift_dev,
                                         track ? P.rdiag : nullptr, pp == first, P.lh, P.lm, P.ll, B, l, n, nn, nn, stream));
        // S = Y Y^T with all 6 limb terms: with a few dominant channels the rounding errors of 3 terms add up
        // coherently above the shift and the Cholesky breaks down (DESIGN.md section 2)
        for (int b = 0; b < B; ++b) {
          xkv_gemm_problem p = problem(P.lh[b], P.lm[b], P.ll[b], nn, 0, P.lh[b], P.lm[b], P.ll[b], nn, 0, P.s_slabs[b],
                                       l, l, l, n, 6);
          p.sym_upper = 1;
          p.split_k = P.sk;
          p.split_stride = static_cast<long long>(l) * l;
          p.run_if = cond ? P.pass_flags + b : nullptr;
          ps.push_back(p);
        }
        XKV_TRY(run_gemms(ps, stream));
        XKV_TRY(xkv_reduce_slabs_batched(P.s_slabs, P.s_mat, B, P.sk, static_cast<long long>(l) * l, l, l, l, 1, l, stream));
        {
          void *h0[XKV_MAX_BATCH], *h1[XKV_MAX_BATCH], *h2[XKV_MAX_BATCH];
          for (int b = 0; b < B; ++b) h0[b] = P.linv_l[b][0], h1[b] = P.linv_l[b][1], h2[b] = P.linv_l[b][2];
          const float shift = kCholShift[pp];
          XKV_TRY(xkv_cholesky_inverse_limbs(P.s_mat, P.linv, h0, h1, h2, B, l, l, l, shift, kPivotFloor, stream));
          if (pp > 0) {
            // A pivot below twice the shift means the fp32 Gram of the basis was numerically indefinite (the pass before
            // left it too ill-conditioned: extreme outlier channels).  Such matrices redo the Cholesky with the heavy
            // shift of pass 0 -- the slabs still hold S -- which costs orthogonality (later passes restore it) but never
            // produces the overflow -> NaN cascade of a clamped pivot.
            XKV_TRY(xkv_pass_flags(P.linv, B, l, l, 2.f * shift, P.redo_flags, stream));
            xkv_set_launch_predicate(P.redo_flags);
            int rc2 = xkv_reduce_slabs_batched(P.s_slabs, P.s_mat, B, P.sk, static_cast<long long>(l) * l, l, l, l, 1, l, stream);
            if (!rc2)
              rc2 = xkv_cholesky_inverse_limbs(P.s_mat, P.linv, h0, h1, h2, B, l, l, l, kCholShift[0], kPivotFloor, stream);
            xkv_set_launch_predicate(cond ? P.pass_flags : nullptr);
            if (rc2) return rc2;
          }
        }
        if (track) XKV_TRY(xkv_rdiag_update(P.rdiag, P.linv, B, l, l, stream));
        // Q = Linv Y, computed as Q^T = Y^T Linv^T with the result stored transposed (same memory, same order of products):
        // the long dimension n becomes M, the sketch width l becomes N, which the CTA-pair GEMM tiles without padding
        // (l = 576 as 3 x 192 columns, 832 as 4 x 208).  A basis that is orthonormalised again later needs only the
        // 3 leading limb terms (orthonormal to ~1e-5 instead of ~1e-7; a product cannot break down).
        for (int b = 0; b < B; ++b) {
          xkv_gemm_problem p = swap_roles(problem(P.linv_l[b][0], P.linv_l[b][1], P.linv_l[b][2], l, 0, P.lh[b], P.lm[b],
                                                  P.ll[b], nn, 1, cond ? cur[b] : nxt[b], nn, l, n, l, final_call ? 6 : 3));
          p.run_if = cond ? P.pass_flags + b : nullptr;
          ps.push_back(p);
        }
        XKV_TRY(run_gemms(ps, stream));
        return 0;
      }();
      if (cond) xkv_set_launch_predicate(nullptr);
      if (rc) return rc;
      if (!cond) swap_bufs();
    }
    return 0;
  };
  // cur <- (limbs lh/lm of the current basis) * G
  auto apply_gram = [&](int nterms) -> int {
    for (int b = 0; b < B; ++b)   // as (G Q^T)^T: see swap_roles
      ps.push_back(swap_roles(problem(P.lh[b], P.lm[b], P.ll[b], nn, 0, P.g_limb[b][0], P.g_limb[b][1], P.g_limb[b][2], nn, 0,
                                      nxt[b], nn, l, n, n, nterms)));
    XKV_TRY(run_gemms(ps, stream));
    swap_bufs();
    return 0;
  };

  // ---- 2-3. Gaussian range finder ----
  for (int b = 0; b < B; ++b) XKV_TRY(xkv_fill_gaussian_bf16(P.lh[b], l, n, nn, kSeed + 7919ull * b, stream));
  XKV_TRY(apply_gram(1));
  XKV_TRY(cholqr(false, false, false));
  XKV_TRY(mark());  // 3: range finder

  // ---- 4. power steps (3-term limb products) ----
  // The first step is plain (the range finder's triangular factor says nothing about eigenvalues); from the
  // second step on the shift c = kSpectralShift * lambda_l comes from diag(R) of the step before.
  XKV_CHECK_CUDA(cudaMemsetAsync(P.shift_dev, 0, XKV_MAX_BATCH * sizeof(float), st));
  for (int it = 0; it < kPowerSteps; ++it) {
    XKV_TRY(xkv_split_bf16_batched(cur, P.lh, P.lm, nullptr, B, l, n, nn, nn, stream));
    XKV_TRY(apply_gram(3));
    if (it > 0) XKV_TRY(xkv_ritz_shift_update(P.rdiag, B, l, kShiftTail, kSpectralShift, P.shift_dev, stream));
    const bool last = it == kPowerSteps - 1;
    XKV_TRY(cholqr(it > 0, !last, last));
  }
  XKV_TRY(mark());  // 4: power iterations

  // ---- 5. windowed Rayleigh-Ritz ----
  // window 0: basis rows [r0, l) straddling row r, whose top wl Ritz vectors replace rows [r0, r); window 1: rows
  // [0, W), diagonalised for the leading singular values
  {
    const int r0 = l - W, wl = r - r0;
    auto w0 = [&](int w) { return w == 0 ? r0 : 0; };   // first basis row of window w
    XKV_TRY(xkv_split_bf16_batched(cur, P.lh, P.lm, P.ll, B, l, n, nn, nn, stream));
    for (int b = 0; b < B; ++b)
      for (int w = 0; w < 2; ++w)
        ps.push_back(swap_roles(problem(row_bf16(P.lh[b], w0(w), nn), row_bf16(P.lm[b], w0(w), nn),
                                        row_bf16(P.ll[b], w0(w), nn), nn, 0, P.g_limb[b][0], P.g_limb[b][1], P.g_limb[b][2],
                                        nn, 0, P.yw[b][w], nn, W, n, n, 6)));   // as (G Qw^T)^T: M = n in CTA pairs, N = W
    XKV_TRY(run_gemms(ps, stream));
    {
      // all windows' limbs in launches of up to XKV_MAX_BATCH matrices
      const float* xs[2 * XKV_MAX_BATCH];
      void *h0[2 * XKV_MAX_BATCH], *h1[2 * XKV_MAX_BATCH], *h2[2 * XKV_MAX_BATCH];
      int cntw = 0;
      for (int b = 0; b < B; ++b)
        for (int w = 0; w < 2; ++w) {
          xs[cntw] = P.yw[b][w];
          h0[cntw] = P.yw_l[b][w][0], h1[cntw] = P.yw_l[b][w][1], h2[cntw] = P.yw_l[b][w][2];
          ++cntw;
        }
      for (int lo = 0; lo < cntw; lo += XKV_MAX_BATCH) {
        const int c = cntw - lo < XKV_MAX_BATCH ? cntw - lo : XKV_MAX_BATCH;
        XKV_TRY(xkv_split_bf16_batched(xs + lo, h0 + lo, h1 + lo, h2 + lo, c, W, n, nn, nn, stream));
      }
    }
    for (int b = 0; b < B; ++b)
      for (int w = 0; w < 2; ++w) {
        xkv_gemm_problem p =
            problem(row_bf16(P.lh[b], w0(w), nn), row_bf16(P.lm[b], w0(w), nn), row_bf16(P.ll[b], w0(w), nn), nn, 0,
                    P.yw_l[b][w][0], P.yw_l[b][w][1], P.yw_l[b][w][2], nn, 0, P.t_slabs[b][w], W, W, W, n, 6);
        p.split_k = P.skw;
        p.split_stride = static_cast<long long>(W) * W;
        ps.push_back(p);
      }
    XKV_TRY(run_gemms(ps, stream));
    const float* tptr[2 * XKV_MAX_BATCH];
    const float* sptr[2 * XKV_MAX_BATCH];
    float* toutp[2 * XKV_MAX_BATCH];
    float* eptr[2 * XKV_MAX_BATCH];
    float* wptr[2 * XKV_MAX_BATCH];
    int cnt = 0;
    for (int b = 0; b < B; ++b)
      for (int w = 0; w < 2; ++w) {
        sptr[cnt] = P.t_slabs[b][w];
        toutp[cnt] = P.t_mat[b][w];
        tptr[cnt] = P.t_mat[b][w];
        eptr[cnt] = P.evals[b][w];
        wptr[cnt] = (w == 0) ? P.wt[b] : nullptr;
        ++cnt;
      }
    for (int lo = 0; lo < cnt; lo += XKV_MAX_BATCH) {
      const int c = cnt - lo < XKV_MAX_BATCH ? cnt - lo : XKV_MAX_BATCH;
      XKV_TRY(xkv_reduce_slabs_batched(sptr + lo, toutp + lo, c, P.skw, static_cast<long long>(W) * W, W, W, W, 0, W, stream));
    }
    XKV_TRY(xkv_jacobi_eigh(tptr, eptr, wptr, cnt, W, W, W, kJacobiSweeps, stream));
    // rows [r0, r) of the basis <- top-wl Ritz vectors of the window: Vw = Wsel * Qw
    {
      const float* xs[XKV_MAX_BATCH];
      void *h0[XKV_MAX_BATCH], *h1[XKV_MAX_BATCH], *h2[XKV_MAX_BATCH];
      for (int b = 0; b < B; ++b) {
        xs[b] = P.wt[b];
        h0[b] = P.wsel_l[b][0], h1[b] = P.wsel_l[b][1], h2[b] = P.wsel_l[b][2];
      }
      XKV_TRY(xkv_split_bf16_batched(xs, h0, h1, h2, B, wl, W, W, W, stream));
    }
    for (int b = 0; b < B; ++b)
      ps.push_back(problem(P.wsel_l[b][0], P.wsel_l[b][1], P.wsel_l[b][2], W, 0, row_bf16(P.lh[b], r0, nn),
                           row_bf16(P.lm[b], r0, nn), row_bf16(P.ll[b], r0, nn), nn, 1,
                           cur[b] + static_cast<size_t>(r0) * nn, nn, wl, n, W, 6));
    XKV_TRY(run_gemms(ps, stream));
    if (sigma_host)
      for (int b = 0; b < B; ++b)
        if (sigma_host[b]) XKV_TRY(xkv_sqrt_clamp(P.evals[b][1], sigma_host[b], W, stream));
  }
  XKV_TRY(mark());  // 5: Rayleigh-Ritz

  // ---- 6. right factor in bf16, both layouts ----
  for (int b = 0; b < B; ++b) XKV_TRY(xkv_convert_bf16(cur[b], r, n, nn, Vt_host[b], nn, V_host[b], r, stream));
  if (phase == 3) return 0;   // the caller projects later (phase 4), possibly on another rank's rows
  XKV_TRY(project());
  XKV_TRY(mark());  // 6: projection
  return 0;
}

extern "C" int xkv_factorize_batch(const void* const* X_host, int batch, int m, int n, int64_t ldx, int rank,
                                   void* const* A_host, void* const* Vt_host, void* const* V_host,
                                   float* const* sigma_host, float* const* gram_host, int phase, void* workspace,
                                   size_t workspace_bytes, void* const* stage_events_host, void* stream) {
  return factorize_impl(X_host, 0, 0, batch, m, n, ldx, rank, A_host, Vt_host, V_host, sigma_host, gram_host, phase,
                        workspace, workspace_bytes, stage_events_host, stream);
}

static int check_layers(int layers, int layer_cols, int64_t ld_layer) {
  XKV_REQUIRE(layers >= 1 && layers <= XKV_MAX_GROUP_LAYERS, "factorize: %d layers per group (1..%d)", layers, XKV_MAX_GROUP_LAYERS);
  XKV_REQUIRE(layer_cols > 0 && layer_cols % 64 == 0, "factorize: layer_cols=%d must be a positive multiple of 64", layer_cols);
  XKV_REQUIRE(ld_layer % 8 == 0 && ld_layer >= layer_cols, "factorize: bad layer row stride");
  return 0;
}

extern "C" int xkv_factorize_groups(const void* const* layer_ptrs_host, int batch, int layers, int layer_cols, int m,
                                    int64_t ld_layer, int rank, void* const* A_host,
                                    void* const* Vt_host, void* const* V_host, float* const* sigma_host, void* workspace,
                                    size_t workspace_bytes, void* const* stage_events_host, void* stream) {
  XKV_TRY(check_layers(layers, layer_cols, ld_layer));
  return factorize_impl(layer_ptrs_host, layers, layer_cols, batch, m, layers * layer_cols, ld_layer, rank, A_host,
                        Vt_host, V_host, sigma_host, nullptr, 0, workspace, workspace_bytes, stage_events_host, stream);
}
