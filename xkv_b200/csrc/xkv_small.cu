// xkv_b200 — the small fp32 kernels around the tensor-core GEMMs of the factorisation:
// split-K reduction / Gram symmetrisation, fp32 -> bf16 limb splitting, the Gaussian test matrix,
// row normalisation (the Cholesky of CholeskyQR lives in xkv_chol.cu), the
// shared-memory Jacobi eigen-solver for the Rayleigh-Ritz window, and bf16 conversion/transposition
// of the right factor.  Together with xkv_gemm.cu they replace torch.linalg.svd
// (fake_layer_merge_dynamic_cache.py:20).
#include "xkv_common.cuh"
#include "xkv_host.h"

namespace xkv {

static int sm_count();

// =============================================================================================
// split-K slab reduction (+ symmetrisation of the Gram matrix)
// =============================================================================================
struct ReduceParams {
  const float* slabs[XKV_MAX_BATCH];
  float* out[XKV_MAX_BATCH];
  const int* run_if;   // optional per-matrix device predicate (xkv_set_launch_predicate)
};
template <int SYM>
__global__ void __launch_bounds__(256) reduce_slabs_kernel(const __grid_constant__ ReduceParams rp, int num_slabs,
                                                           long long slab_stride, int rows, int cols, long long ld,
                                                           long long ldo, int tiles_per_row) {
  __shared__ float tile[32][33];
  if (rp.run_if != nullptr && rp.run_if[blockIdx.y] == 0) return;
  const float* __restrict__ slabs = rp.slabs[blockIdx.y];
  float* __restrict__ out = rp.out[blockIdx.y];
  int bi, bj;
  if (SYM) {
    // linear index over tile pairs bi <= bj
    int t = blockIdx.x;
    bi = 0;
    int cnt = tiles_per_row;
    while (t >= cnt) {
      t -= cnt;
      ++bi;
      --cnt;
    }
    bj = bi + t;
  } else {
    bi = blockIdx.x / tiles_per_row;
    bj = blockIdx.x - bi * tiles_per_row;
  }
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int i = bi * 32 + r, j = bj * 32 + tx;
    float acc = 0.f;
    if (i < rows && j < cols) {
      const float* p = slabs + static_cast<long long>(i) * ld + j;
      for (int s = 0; s < num_slabs; ++s) acc += p[static_cast<long long>(s) * slab_stride];
      if (!SYM || j >= i) out[static_cast<long long>(i) * ldo + j] = acc;
    }
    if (SYM) tile[r][tx] = acc;
  }
  if (SYM) {
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
      // mirrored element: out[bj*32 + r][bi*32 + tx] = sum(bi*32 + tx, bj*32 + r)
      const int i = bj * 32 + r, j = bi * 32 + tx;
      if (i < rows && j < cols && i > j) out[static_cast<long long>(i) * ldo + j] = tile[tx][r];
    }
  }
}

// =============================================================================================
// upper-triangle packing of a symmetric fp32 matrix (the payload of the token-sharded Gram all-reduce)
// =============================================================================================
// Row r contributes its columns [r32, n), r32 = 32 * (r / 32): n^2 / 2 + 16 n floats instead of n^2.
__host__ __device__ inline long long packed_row_offset(int r, int n) {
  const long long g = r / 32;
  return 32 * (g * n - 16 * g * (g - 1)) + (r - 32 * g) * (n - 32 * g);
}
__global__ void __launch_bounds__(256) pack_upper_kernel(const float* __restrict__ full, long long ld, int n,
                                                         float* __restrict__ packed) {
  const int r = blockIdx.x;
  const int c0 = (r / 32) * 32;
  const float* src = full + static_cast<long long>(r) * ld + c0;
  float* dst = packed + packed_row_offset(r, n);
  const int w = n - c0;            // multiple of 4 when n is (c0 is a multiple of 32); rows are 16-byte aligned then
  if ((n & 3) == 0 && (ld & 3) == 0) {
    for (int v = threadIdx.x; v < (w >> 2); v += 256)
      reinterpret_cast<float4*>(dst)[v] = reinterpret_cast<const float4*>(src)[v];
  } else {
    for (int c = threadIdx.x; c < w; c += 256) dst[c] = src[c];
  }
}
// full[i][j] = full[j][i] = packed(i, j) for j >= i: 32 x 32 tiles, mirrored through shared memory
__global__ void __launch_bounds__(256) unpack_upper_kernel(const float* __restrict__ packed, int n, float* __restrict__ full,
                                                           long long ld, int tiles_per_row) {
  __shared__ float tile[32][33];
  int t = blockIdx.x, bi = 0, cnt = tiles_per_row;
  while (t >= cnt) {
    t -= cnt;
    ++bi;
    --cnt;
  }
  const int bj = bi + t;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int i = bi * 32 + r, j = bj * 32 + tx;
    float v = 0.f;
    if (i < n && j < n) {
      v = packed[packed_row_offset(i, n) + (j - bi * 32)];
      if (j >= i) full[static_cast<long long>(i) * ld + j] = v;
    }
    tile[r][tx] = v;
  }
  __syncthreads();
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int i = bj * 32 + r, j = bi * 32 + tx;
    if (i < n && j < n && i > j) full[static_cast<long long>(i) * ld + j] = tile[tx][r];
  }
}

// =============================================================================================
// fp32 -> bf16 limbs
// =============================================================================================
__device__ __forceinline__ void split3(float x, __nv_bfloat16& h, __nv_bfloat16& m, __nv_bfloat16& l) {
  h = __float2bfloat16_rn(x);
  const float r1 = x - __bfloat162float(h);
  m = __float2bfloat16_rn(r1);
  const float r2 = r1 - __bfloat162float(m);
  l = __float2bfloat16_rn(r2);
}

struct SplitParams {
  const float* x[XKV_MAX_BATCH];
  __nv_bfloat16* hi[XKV_MAX_BATCH];
  __nv_bfloat16* mid[XKV_MAX_BATCH];
  __nv_bfloat16* lo[XKV_MAX_BATCH];
};
__global__ void __launch_bounds__(256) split_bf16_kernel(const __grid_constant__ SplitParams sp, int rows, int cols,
                                                         long long ld, long long ldo) {
  const float* __restrict__ x = sp.x[blockIdx.y];
  __nv_bfloat16* __restrict__ hi = sp.hi[blockIdx.y];
  __nv_bfloat16* __restrict__ mid = sp.mid[blockIdx.y];
  __nv_bfloat16* __restrict__ lo = sp.lo[blockIdx.y];
  const int cols4 = cols >> 2;  // host guarantees cols % 4 == 0
  const long long total = static_cast<long long>(rows) * cols4;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(idx / cols4);
    const int c = static_cast<int>(idx - static_cast<long long>(r) * cols4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(x + static_cast<long long>(r) * ld + c);
    __nv_bfloat16 h[4], m[4], l[4];
    split3(v.x, h[0], m[0], l[0]);
    split3(v.y, h[1], m[1], l[1]);
    split3(v.z, h[2], m[2], l[2]);
    split3(v.w, h[3], m[3], l[3]);
    const long long o = static_cast<long long>(r) * ldo + c;
    *reinterpret_cast<uint2*>(hi + o) = *reinterpret_cast<uint2*>(h);
    if (mid) *reinterpret_cast<uint2*>(mid + o) = *reinterpret_cast<uint2*>(m);
    if (lo) *reinterpret_cast<uint2*>(lo + o) = *reinterpret_cast<uint2*>(l);
  }
}


// =============================================================================================
// Gram post-processing in one pass: sum the split-K slabs of the upper-triangle tiles, mirror them, and write the
// three bf16 limbs of the full symmetric matrix (replaces reduce_slabs<1> + split_bf16: the fp32 Gram is read once
// and never written back).  One CTA per 32x32 tile pair bi <= bj, batch in blockIdx.y.
// =============================================================================================
struct SymSplitParams {
  const float* slabs[XKV_MAX_BATCH];
  __nv_bfloat16* hi[XKV_MAX_BATCH];
  __nv_bfloat16* mid[XKV_MAX_BATCH];
  __nv_bfloat16* lo[XKV_MAX_BATCH];
};
__global__ void __launch_bounds__(256) sym_split_kernel(const __grid_constant__ SymSplitParams sp, int num_slabs,
                                                        long long slab_stride, int n, long long ld, long long ldo,
                                                        int tiles_per_row) {
  __shared__ float tile[32][33];
  const float* __restrict__ slabs = sp.slabs[blockIdx.y];
  __nv_bfloat16* __restrict__ hi = sp.hi[blockIdx.y];
  __nv_bfloat16* __restrict__ mid = sp.mid[blockIdx.y];
  __nv_bfloat16* __restrict__ lo = sp.lo[blockIdx.y];
  int t = blockIdx.x, bi = 0, cnt = tiles_per_row;
  while (t >= cnt) {
    t -= cnt;
    ++bi;
    --cnt;
  }
  const int bj = bi + t;
  // thread = (row ty / ty + 16, column pair 2 tx, 2 tx + 1): 8-byte loads per slab, 4-byte stores per limb
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const bool pair_ok = ((ld | ldo | slab_stride) & 1) == 0;   // even strides: the column pairs are 8 / 4-byte aligned
  auto store2 = [&](long long o, float a, float b) {
    __nv_bfloat16 h0, m0, l0, h1, m1, l1;
    split3(a, h0, m0, l0);
    split3(b, h1, m1, l1);
    *reinterpret_cast<__nv_bfloat162*>(hi + o) = __halves2bfloat162(h0, h1);
    *reinterpret_cast<__nv_bfloat162*>(mid + o) = __halves2bfloat162(m0, m1);
    *reinterpret_cast<__nv_bfloat162*>(lo + o) = __halves2bfloat162(l0, l1);
  };
  auto store1 = [&](long long o, float a) {
    __nv_bfloat16 h, m, l;
    split3(a, h, m, l);
    hi[o] = h;
    mid[o] = m;
    lo[o] = l;
  };
#pragma unroll
  for (int rr = 0; rr < 2; ++rr) {
    const int r = ty + 16 * rr;
    const int i = bi * 32 + r, j = bj * 32 + 2 * tx;
    float a0 = 0.f, a1 = 0.f;
    if (i < n && j < n) {
      const float* p = slabs + static_cast<long long>(i) * ld + j;
      if (pair_ok && j + 1 < n) {
        for (int s = 0; s < num_slabs; ++s) {
          const float2 v = *reinterpret_cast<const float2*>(p + static_cast<long long>(s) * slab_stride);
          a0 += v.x;
          a1 += v.y;
        }
      } else {
        for (int s = 0; s < num_slabs; ++s) {
          a0 += p[static_cast<long long>(s) * slab_stride];
          if (j + 1 < n) a1 += p[static_cast<long long>(s) * slab_stride + 1];
        }
      }
      const long long o = static_cast<long long>(i) * ldo + j;
      if (pair_ok && j + 1 < n && j >= i) {          // both columns on or above the diagonal
        store2(o, a0, a1);
      } else {
        if (j >= i) store1(o, a0);
        if (j + 1 < n && j + 1 >= i) store1(o + 1, a1);
      }
    }
    tile[r][2 * tx] = a0;
    tile[r][2 * tx + 1] = a1;
  }
  __syncthreads();
#pragma unroll
  for (int rr = 0; rr < 2; ++rr) {
    // mirrored elements (i, j), (i, j + 1) = (bj*32 + r, bi*32 + 2 tx [+ 1]) take the values computed at the transposed places
    const int r = ty + 16 * rr;
    const int i = bj * 32 + r, j = bi * 32 + 2 * tx;
    if (i < n && j < n) {
      const float a0 = tile[2 * tx][r], a1 = tile[2 * tx + 1][r];
      const long long o = static_cast<long long>(i) * ldo + j;
      if (pair_ok && j + 1 < n && i > j + 1) {        // both strictly below the diagonal
        store2(o, a0, a1);
      } else {
        if (i > j) store1(o, a0);
        if (j + 1 < n && i > j + 1) store1(o + 1, a1);
      }
    }
  }
}

// =============================================================================================
// deterministic Gaussian test matrix (counter-based: value depends only on seed and position)
// =============================================================================================
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__global__ void __launch_bounds__(256) fill_gaussian_kernel(__nv_bfloat16* __restrict__ out, int rows, int cols,
                                                            long long ld, uint64_t seed) {
  const int cols2 = cols >> 1;  // host guarantees cols % 2 == 0
  const long long total = static_cast<long long>(rows) * cols2;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(idx / cols2);
    const int c = static_cast<int>(idx - static_cast<long long>(r) * cols2) * 2;
    const uint64_t z = mix64(seed * 0xD1342543DE82EF95ull + static_cast<uint64_t>(idx));
    const float u1 = (static_cast<float>(static_cast<uint32_t>(z >> 40)) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = (static_cast<float>(static_cast<uint32_t>(z) >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float rad = sqrtf(-2.0f * __logf(u1));
    float sn, cs;
    __sincosf(6.283185307179586f * u2, &sn, &cs);
    *reinterpret_cast<uint32_t*>(out + static_cast<long long>(r) * ld + c) = pack_bf16x2(rad * cs, rad * sn);
  }
}

// =============================================================================================
// row normalisation (each row of Yt is a column of Y), optionally emitting bf16 limbs
// =============================================================================================
struct NormParams {
  float* Y[XKV_MAX_BATCH];
  const float* Q[XKV_MAX_BATCH];   // optional: previous orthonormal basis, Y <- Y - c[b] * Q before normalising
  __nv_bfloat16* hi[XKV_MAX_BATCH];
  __nv_bfloat16* mid[XKV_MAX_BATCH];
  __nv_bfloat16* lo[XKV_MAX_BATCH];
  float* rdiag[XKV_MAX_BATCH];     // optional: running diagonal of the triangular factor R of Y = R^T Q_new
  const float* Linv[XKV_MAX_BATCH];
  float* c;                        // per-matrix spectral shift (device), used when Q != null
  int rows, cols, tail, rdiag_first;
  float shift_scale;
  long long ld, ldo, ld_linv;
  const int* run_if;               // optional per-matrix device predicate (xkv_set_launch_predicate)
  int* flags;                      // pass_flag_kernel output
  float inv_min_pivot;
};

// Spectral shift of the power steps.  Orthogonal iteration Y = Q (G - c I) = R^T Q_new makes diag(R) converge
// to the eigenvalues lambda_j - c, so the trailing `tail` entries of diag(R) of the previous step estimate
// lambda_l, the largest unwanted eigenvalue: c_new = shift_scale * (mean_tail diag(R) + c_old).  With
// c = lambda_l / 2 the unwanted spectrum [0, lambda_l] maps to [-c, c] and the convergence ratio of direction i
// drops from lambda_l / lambda_i to (lambda_l / 2) / (lambda_i - lambda_l / 2).  diag(R) is accumulated over
// the CholeskyQR passes: row norm (normalize_rows_kernel) times the Cholesky diagonal 1 / Linv_jj (below).
// Unlike Rayleigh quotients it is insensitive to trailing basis vectors that are still polluted by the
// dominant directions (the Gram-Schmidt step removes those before the norm is taken).
__global__ void __launch_bounds__(256) ritz_shift_kernel(const __grid_constant__ NormParams p) {
  __shared__ float red[8];
  const float* rd = p.rdiag[blockIdx.x];
  float acc = 0.f;
  for (int j = p.rows - p.tail + threadIdx.x; j < p.rows; j += blockDim.x) acc += rd[j];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    p.c[blockIdx.x] = fmaxf(p.shift_scale * (t / static_cast<float>(p.tail) + p.c[blockIdx.x]), 0.f);
  }
}
// rdiag[j] /= Linv[j][j]  (the Cholesky diagonal L_jj = 1 / Linv_jj of the pass that just finished)
__global__ void __launch_bounds__(256) rdiag_update_kernel(const __grid_constant__ NormParams p) {
  if (p.run_if != nullptr && p.run_if[blockIdx.y] == 0) return;
  float* rd = p.rdiag[blockIdx.y];
  const float* li = p.Linv[blockIdx.y];
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < p.rows) rd[j] = rd[j] / li[static_cast<long long>(j) * p.ld_linv + j];
}

// flags[b] = 1 when the Cholesky pass that just finished met a pivot L_jj^2 < min_pivot (S has a unit diagonal, so the
// pivot is the squared sine of the angle between row j and the span of the rows before it): the pass was then
// ill-conditioned, its output is orthonormal only to ~ eps / pivot, and a second pass is worth its cost.  A NaN
// diagonal raises the flag too.
__global__ void __launch_bounds__(256) pass_flag_kernel(const __grid_constant__ NormParams p) {
  if (p.run_if != nullptr && p.run_if[blockIdx.x] == 0) {   // gated by the launch predicate: a skipped matrix raises no flag
    if (threadIdx.x == 0) p.flags[blockIdx.x] = 0;
    return;
  }
  const float* li = p.Linv[blockIdx.x];
  int bad = 0;
  for (int j = threadIdx.x; j < p.rows; j += blockDim.x) {
    const float d = li[static_cast<long long>(j) * p.ld_linv + j];   // 1 / L_jj
    if (!(d * d <= p.inv_min_pivot)) bad = 1;
  }
  bad = __syncthreads_or(bad);
  if (threadIdx.x == 0) p.flags[blockIdx.x] = bad ? 1 : 0;
}

__global__ void __launch_bounds__(256) normalize_rows_kernel(const __grid_constant__ NormParams p) {
  __shared__ float red[8];
  __shared__ float scale_s;
  if (p.run_if != nullptr && p.run_if[blockIdx.y] == 0) return;
  float* row = p.Y[blockIdx.y] + static_cast<long long>(blockIdx.x) * p.ld;
  const int cols4 = p.cols >> 2;
  float acc = 0.f;
  if (p.Q[blockIdx.y] != nullptr) {
    const float* qrow = p.Q[blockIdx.y] + static_cast<long long>(blockIdx.x) * p.ld;
    const float cshift = p.c[blockIdx.y];
    for (int c = threadIdx.x; c < cols4; c += blockDim.x) {
      float4 v = reinterpret_cast<const float4*>(row)[c];
      const float4 q = reinterpret_cast<const float4*>(qrow)[c];
      v.x = fmaf(-cshift, q.x, v.x);
      v.y = fmaf(-cshift, q.y, v.y);
      v.z = fmaf(-cshift, q.z, v.z);
      v.w = fmaf(-cshift, q.w, v.w);
      reinterpret_cast<float4*>(row)[c] = v;   // re-read below by the same thread
      acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
  } else
  for (int c = threadIdx.x; c < cols4; c += blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(row)[c];
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    scale_s = t > 0.f ? rsqrtf(t) : 0.f;
    if (p.rdiag[blockIdx.y] != nullptr) {
      float* rd = p.rdiag[blockIdx.y] + blockIdx.x;
      *rd = (p.rdiag_first ? 1.f : *rd) * sqrtf(t);
    }
  }
  __syncthreads();
  const float sc = scale_s;
  __nv_bfloat16* hi = p.hi[blockIdx.y];
  __nv_bfloat16* mid = p.mid[blockIdx.y];
  __nv_bfloat16* lo = p.lo[blockIdx.y];
  const long long o0 = static_cast<long long>(blockIdx.x) * p.ldo;
  for (int c = threadIdx.x; c < cols4; c += blockDim.x) {
    float4 v = reinterpret_cast<const float4*>(row)[c];
    v.x *= sc;
    v.y *= sc;
    v.z *= sc;
    v.w *= sc;
    reinterpret_cast<float4*>(row)[c] = v;
    if (hi) {
      __nv_bfloat16 h[4], m[4], l[4];
      split3(v.x, h[0], m[0], l[0]);
      split3(v.y, h[1], m[1], l[1]);
      split3(v.z, h[2], m[2], l[2]);
      split3(v.w, h[3], m[3], l[3]);
      *reinterpret_cast<uint2*>(hi + o0 + 4 * c) = *reinterpret_cast<uint2*>(h);
      if (mid) *reinterpret_cast<uint2*>(mid + o0 + 4 * c) = *reinterpret_cast<uint2*>(m);
      if (lo) *reinterpret_cast<uint2*>(lo + o0 + 4 * c) = *reinterpret_cast<uint2*>(l);
    }
  }
}

// =============================================================================================
// Shared-memory two-sided Jacobi eigen-solver for the Rayleigh-Ritz window (W <= 160, W even)
// One CTA per matrix; A and the eigenvector accumulator V both live in shared memory.
// Parallel cyclic ordering (round-robin tournament): W/2 disjoint rotations per round.
// Output: eigenvalues sorted descending, eigenvectors as ROWS of Wt in the same order.
// =============================================================================================
struct JacobiParams {
  const float* T[2 * XKV_MAX_BATCH];  // W x W symmetric inputs (ld)
  float* evals[2 * XKV_MAX_BATCH];    // W
  float* Wt[2 * XKV_MAX_BATCH];       // W x W (ld_w), may be null (values only)
  int W, sweeps;
  float tol;
  long long ld, ld_w;
};
constexpr int JAC_THREADS = 512;

// WT > 0: window width known at compile time (index arithmetic becomes shifts / multiplies); WT == 0: p.W
template <int WT>
__global__ void __launch_bounds__(JAC_THREADS, 1) jacobi_kernel(const __grid_constant__ JacobiParams p) {
  extern __shared__ float jsm[];
  const int W = WT > 0 ? WT : p.W, WP = W + 1, H = W / 2;
  float* A = jsm;                 // W x WP
  float* V = A + W * WP;          // W x WP
  float* cs = V + W * WP;         // 2 * H
  int* pij = reinterpret_cast<int*>(cs + 2 * H);  // 2 * H
  const int tid = threadIdx.x;
  const float* T = p.T[blockIdx.x];
  const bool want_vec = p.Wt[blockIdx.x] != nullptr;
  for (int e = tid; e < W * W; e += JAC_THREADS) {
    const int r = e / W, c = e - r * W;
    // symmetrise on load: use the average of the two triangles
    A[r * WP + c] = 0.5f * (T[static_cast<long long>(r) * p.ld + c] + T[static_cast<long long>(c) * p.ld + r]);
    V[r * WP + c] = (r == c) ? 1.f : 0.f;
  }
  __shared__ unsigned int off_max;   // largest |a_ij| / sqrt(a_ii a_jj) rotated away in the current sweep
  if (tid == 0) off_max = 0u;
  __syncthreads();
  for (int sweep = 0; sweep < p.sweeps; ++sweep) {
    for (int round = 0; round < W - 1; ++round) {
      if (tid < H) {
        const int q = tid;
        int a = (round + q) % (W - 1);
        int b = (q == 0) ? (W - 1) : (round - q + (W - 1)) % (W - 1);
        const int i = min(a, b), j = max(a, b);
        const float aii = A[i * WP + i], ajj = A[j * WP + j], aij = A[i * WP + j];
        float c = 1.f, s = 0.f;
        const float scale = sqrtf(fabsf(aii * ajj));
        if (fabsf(aij) > 1e-12f * scale && aij != 0.f) {
          const float tau = (ajj - aii) / (2.f * aij);
          const float t = (tau >= 0.f ? 1.f : -1.f) / (fabsf(tau) + sqrtf(1.f + tau * tau));
          c = rsqrtf(1.f + t * t);
          s = t * c;
          // non-negative floats order like their bit patterns
          atomicMax(&off_max, __float_as_uint(fminf(fabsf(aij) / fmaxf(scale, 1e-30f), 1e30f)));
        }
        cs[2 * q] = c;
        cs[2 * q + 1] = s;
        pij[2 * q] = i;
        pij[2 * q + 1] = j;
      }
      __syncthreads();
      // column rotations: A <- A J, V <- V J
      for (int e = tid; e < W * H; e += JAC_THREADS) {
        const int x = e / H, q = e - x * H;
        const float c = cs[2 * q], s = cs[2 * q + 1];
        const int i = pij[2 * q], j = pij[2 * q + 1];
        const float ai = A[x * WP + i], aj = A[x * WP + j];
        A[x * WP + i] = c * ai - s * aj;
        A[x * WP + j] = s * ai + c * aj;
        if (want_vec) {
          const float vi = V[x * WP + i], vj = V[x * WP + j];
          V[x * WP + i] = c * vi - s * vj;
          V[x * WP + j] = s * vi + c * vj;
        }
      }
      __syncthreads();
      // row rotations: A <- J^T A
      for (int e = tid; e < W * H; e += JAC_THREADS) {
        const int q = e / W, y = e - q * W;
        const float c = cs[2 * q], s = cs[2 * q + 1];
        const int i = pij[2 * q], j = pij[2 * q + 1];
        const float ai = A[i * WP + y], aj = A[j * WP + y];
        A[i * WP + y] = c * ai - s * aj;
        A[j * WP + y] = s * ai + c * aj;
      }
      __syncthreads();
    }
    // The window of T = Q^T G Q is close to diagonal after the power steps (orthogonal iteration converges to
    // Schur form), so Jacobi converges quadratically from the first sweep: stop as soon as a whole sweep met
    // no off-diagonal element above p.tol (relative); one more sweep would change the vectors by O(tol^2).
    const float swept = __uint_as_float(off_max);
    __syncthreads();
    if (swept < p.tol) break;
    if (tid == 0) off_max = 0u;
    __syncthreads();
  }
  // sort eigenvalues descending by rank counting; emit eigenvectors as rows of Wt
  if (tid < W) {
    const float d = A[tid * WP + tid];
    int rank = 0;
    for (int u = 0; u < W; ++u) {
      const float du = A[u * WP + u];
      rank += (du > d) || (du == d && u < tid);
    }
    pij[tid] = rank;  // W == 2H entries
    p.evals[blockIdx.x][rank] = d;
  }
  __syncthreads();
  if (want_vec) {
    float* Wt = p.Wt[blockIdx.x];
    for (int e = tid; e < W * W; e += JAC_THREADS) {
      const int t = e / W, x = e - t * W;  // eigenvector t (column of V), component x
      Wt[static_cast<long long>(pij[t]) * p.ld_w + x] = V[x * WP + t];
    }
  }
}

// =============================================================================================
// fp32 -> bf16 conversion with optional transposed copy (right factor: Vt (r x n) and V (n x r))
// =============================================================================================
__global__ void __launch_bounds__(256) convert_bf16_kernel(const float* __restrict__ src, int rows, int cols,
                                                           long long ld, __nv_bfloat16* __restrict__ dst, long long ldd,
                                                           __nv_bfloat16* __restrict__ dstT, long long lddT) {
  __shared__ float tile[32][33];
  const int bi = blockIdx.y, bj = blockIdx.x;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int i = bi * 32 + r, j = bj * 32 + tx;
    float v = 0.f;
    if (i < rows && j < cols) {
      v = src[static_cast<long long>(i) * ld + j];
      if (dst) dst[static_cast<long long>(i) * ldd + j] = __float2bfloat16_rn(v);
    }
    tile[r][tx] = v;
  }
  if (dstT) {
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
      const int j = bj * 32 + r, i = bi * 32 + tx;  // dstT[j][i] = src[i][j]
      if (i < rows && j < cols) dstT[static_cast<long long>(j) * lddT + i] = __float2bfloat16_rn(tile[tx][r]);
    }
  }
}

__global__ void sqrt_clamp_kernel(const float* __restrict__ in, float* __restrict__ out, int count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = sqrtf(fmaxf(in[i], 0.f));
}

static int sm_count() { return device_sm_count(); }

const int*& launch_predicate() {
  static thread_local const int* pred = nullptr;
  return pred;
}

}  // namespace xkv

using namespace xkv;

extern "C" void xkv_set_launch_predicate(const int32_t* flags_dev) { launch_predicate() = flags_dev; }

extern "C" int xkv_pass_flags(const float* const* Linv_host, int batch, int rows, int64_t ld_linv, float min_pivot,
                              int32_t* flags_dev, void* stream) {
  XKV_REQUIRE(Linv_host && flags_dev && batch >= 1 && batch <= XKV_MAX_BATCH, "pass_flags: bad arguments");
  XKV_REQUIRE(min_pivot > 0.f, "pass_flags: min_pivot must be positive");
  NormParams p;
  std::memset(&p, 0, sizeof(p));
  for (int b = 0; b < batch; ++b) p.Linv[b] = Linv_host[b];
  p.rows = rows;
  p.ld_linv = ld_linv;
  p.flags = flags_dev;
  p.inv_min_pivot = 1.f / min_pivot;
  p.run_if = launch_predicate();
  pass_flag_kernel<<<batch, 256, 0, as_stream(stream)>>>(p);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_reduce_slabs_batched(const float* const* slabs_host, float* const* out_host, int batch, int num_slabs,
                                        int64_t slab_stride, int rows, int cols, int64_t ld, int symmetrize,
                                        int64_t ld_out, void* stream) {
  XKV_REQUIRE(slabs_host && out_host && batch >= 1 && batch <= XKV_MAX_BATCH, "reduce_slabs: bad batch");
  XKV_REQUIRE(num_slabs >= 1 && rows > 0 && cols > 0, "reduce_slabs: bad arguments");
  ReduceParams rp;
  std::memset(&rp, 0, sizeof(rp));
  for (int b = 0; b < batch; ++b) {
    XKV_REQUIRE(slabs_host[b] && out_host[b], "reduce_slabs: null matrix %d", b);
    rp.slabs[b] = slabs_host[b];
    rp.out[b] = out_host[b];
  }
  rp.run_if = launch_predicate();
  const int tr = (rows + 31) / 32, tc = (cols + 31) / 32;
  if (symmetrize) {
    XKV_REQUIRE(rows == cols, "reduce_slabs: symmetrize needs a square matrix");
    reduce_slabs_kernel<1><<<dim3(tr * (tr + 1) / 2, batch), 256, 0, as_stream(stream)>>>(rp, num_slabs, slab_stride, rows,
                                                                                      cols, ld, ld_out, tr);
  } else {
    reduce_slabs_kernel<0><<<dim3(tr * tc, batch), 256, 0, as_stream(stream)>>>(rp, num_slabs, slab_stride, rows, cols, ld,
                                                                                ld_out, tc);
  }
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_reduce_slabs(const float* slabs, int num_slabs, int64_t slab_stride, int rows, int cols, int64_t ld,
                                int symmetrize, float* out, int64_t ld_out, void* stream) {
  XKV_REQUIRE(slabs && out, "reduce_slabs: bad arguments");
  return xkv_reduce_slabs_batched(&slabs, &out, 1, num_slabs, slab_stride, rows, cols, ld, symmetrize, ld_out, stream);
}

extern "C" size_t xkv_gram_packed_elems(int n) {
  if (n <= 0) return 0;
  return static_cast<size_t>(packed_row_offset(n - 1, n) + (n - ((n - 1) / 32) * 32));
}

extern "C" int xkv_gram_pack_upper(const float* full, int n, int64_t ld, float* packed, void* stream) {
  XKV_REQUIRE(full && packed && n > 0 && ld >= n, "gram pack: bad arguments");
  pack_upper_kernel<<<n, 256, 0, as_stream(stream)>>>(full, ld, n, packed);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_gram_unpack_upper(const float* packed, int n, float* full, int64_t ld, void* stream) {
  XKV_REQUIRE(full && packed && n > 0 && ld >= n, "gram unpack: bad arguments");
  const int tr = (n + 31) / 32;
  unpack_upper_kernel<<<tr * (tr + 1) / 2, 256, 0, as_stream(stream)>>>(packed, n, full, ld, tr);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_symmetrize_split_bf16(const float* const* slabs_host, int batch, int num_slabs, int64_t slab_stride,
                                         int n, int64_t ld, void* const* hi_host, void* const* mid_host,
                                         void* const* lo_host, int64_t ld_out, void* stream) {
  XKV_REQUIRE(slabs_host && hi_host && mid_host && lo_host && batch >= 1 && batch <= XKV_MAX_BATCH,
              "symmetrize_split: bad arguments");
  XKV_REQUIRE(num_slabs >= 1 && n > 0, "symmetrize_split: bad sizes");
  SymSplitParams sp;
  std::memset(&sp, 0, sizeof(sp));
  for (int b = 0; b < batch; ++b) {
    XKV_REQUIRE(slabs_host[b] && hi_host[b] && mid_host[b] && lo_host[b], "symmetrize_split: null matrix %d", b);
    sp.slabs[b] = slabs_host[b];
    sp.hi[b] = static_cast<__nv_bfloat16*>(hi_host[b]);
    sp.mid[b] = static_cast<__nv_bfloat16*>(mid_host[b]);
    sp.lo[b] = static_cast<__nv_bfloat16*>(lo_host[b]);
  }
  const int tr = (n + 31) / 32;
  sym_split_kernel<<<dim3(tr * (tr + 1) / 2, batch), 256, 0, as_stream(stream)>>>(sp, num_slabs, slab_stride, n, ld, ld_out,
                                                                              tr);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_split_bf16_batched(const float* const* x_host, void* const* hi_host, void* const* mid_host,
                                      void* const* lo_host, int batch, int rows, int cols, int64_t ld, int64_t ld_out,
                                      void* stream) {
  XKV_REQUIRE(x_host && hi_host && batch >= 1 && batch <= XKV_MAX_BATCH, "split_bf16: bad batch");
  XKV_REQUIRE(rows > 0 && cols > 0 && cols % 4 == 0 && ld % 4 == 0 && ld_out % 4 == 0,
              "split_bf16: cols/ld must be multiples of 4");
  SplitParams sp;
  std::memset(&sp, 0, sizeof(sp));
  for (int b = 0; b < batch; ++b) {
    XKV_REQUIRE(x_host[b] && hi_host[b], "split_bf16: null matrix %d", b);
    sp.x[b] = x_host[b];
    sp.hi[b] = static_cast<__nv_bfloat16*>(hi_host[b]);
    sp.mid[b] = mid_host ? static_cast<__nv_bfloat16*>(mid_host[b]) : nullptr;
    sp.lo[b] = lo_host ? static_cast<__nv_bfloat16*>(lo_host[b]) : nullptr;
  }
  const long long total = static_cast<long long>(rows) * (cols / 4);
  long long grid = (total + 255) / 256;
  const long long cap = static_cast<long long>(sm_count()) * 16 / batch + 1;
  if (grid > cap) grid = cap;
  split_bf16_kernel<<<dim3(static_cast<int>(grid), batch), 256, 0, as_stream(stream)>>>(sp, rows, cols, ld, ld_out);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_split_bf16(const float* x, int rows, int cols, int64_t ld, void* hi, void* mid, void* lo,
                              int64_t ld_out, void* stream) {
  XKV_REQUIRE(x && hi, "split_bf16: bad arguments");
  return xkv_split_bf16_batched(&x, &hi, mid ? &mid : nullptr, lo ? &lo : nullptr, 1, rows, cols, ld, ld_out, stream);
}

extern "C" int xkv_fill_gaussian_bf16(void* out, int rows, int cols, int64_t ld, uint64_t seed, void* stream) {
  XKV_REQUIRE(out && rows > 0 && cols > 0 && cols % 2 == 0 && ld % 2 == 0, "fill_gaussian: bad arguments");
  const long long total = static_cast<long long>(rows) * (cols / 2);
  long long grid = (total + 255) / 256;
  const long long cap = static_cast<long long>(sm_count()) * 16;
  if (grid > cap) grid = cap;
  fill_gaussian_kernel<<<static_cast<int>(grid), 256, 0, as_stream(stream)>>>(static_cast<__nv_bfloat16*>(out), rows,
                                                                              cols, ld, seed);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_normalize_rows(float* const* Y_host, void* const* hi_host, void* const* mid_host,
                                  void* const* lo_host, int batch, int rows, int cols, int64_t ld, int64_t ld_out,
                                  void* stream) {
  XKV_REQUIRE(Y_host && batch >= 1 && batch <= XKV_MAX_BATCH, "normalize_rows: bad batch");
  XKV_REQUIRE(rows > 0 && cols > 0 && cols % 4 == 0 && ld % 4 == 0 && ld_out % 4 == 0,
              "normalize_rows: cols/ld must be multiples of 4");
  NormParams p;
  std::memset(&p, 0, sizeof(p));
  for (int b = 0; b < batch; ++b) {
    p.Y[b] = Y_host[b];
    p.hi[b] = hi_host ? static_cast<__nv_bfloat16*>(hi_host[b]) : nullptr;
    p.mid[b] = mid_host ? static_cast<__nv_bfloat16*>(mid_host[b]) : nullptr;
    p.lo[b] = lo_host ? static_cast<__nv_bfloat16*>(lo_host[b]) : nullptr;
  }
  p.rows = rows;
  p.cols = cols;
  p.ld = ld;
  p.ldo = ld_out;
  normalize_rows_kernel<<<dim3(rows, batch), 256, 0, as_stream(stream)>>>(p);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_shift_normalize_rows(float* const* Y_host, const float* const* Q_host, float* shift_dev,
                                        float* const* rdiag_host, int rdiag_first, void* const* hi_host,
                                        void* const* mid_host, void* const* lo_host, int batch, int rows, int cols,
                                        int64_t ld, int64_t ld_out, void* stream) {
  XKV_REQUIRE(Y_host && batch >= 1 && batch <= XKV_MAX_BATCH, "shift_normalize_rows: bad batch");
  XKV_REQUIRE(rows > 0 && cols > 0 && cols % 4 == 0 && ld % 4 == 0 && ld_out % 4 == 0,
              "shift_normalize_rows: cols/ld must be multiples of 4");
  XKV_REQUIRE(!Q_host || shift_dev, "shift_normalize_rows: a shifted step needs the device shifts");
  NormParams p;
  std::memset(&p, 0, sizeof(p));
  for (int b = 0; b < batch; ++b) {
    XKV_REQUIRE(Y_host[b] && (!Q_host || Q_host[b]), "shift_normalize_rows: null matrix %d", b);
    p.Y[b] = Y_host[b];
    p.Q[b] = Q_host ? Q_host[b] : nullptr;
    p.rdiag[b] = rdiag_host ? rdiag_host[b] : nullptr;
    p.hi[b] = hi_host ? static_cast<__nv_bfloat16*>(hi_host[b]) : nullptr;
    p.mid[b] = mid_host ? static_cast<__nv_bfloat16*>(mid_host[b]) : nullptr;
    p.lo[b] = lo_host ? static_cast<__nv_bfloat16*>(lo_host[b]) : nullptr;
  }
  p.c = shift_dev;
  p.rows = rows;
  p.cols = cols;
  p.rdiag_first = rdiag_first;
  p.ld = ld;
  p.ldo = ld_out;
  p.run_if = launch_predicate();
  normalize_rows_kernel<<<dim3(rows, batch), 256, 0, as_stream(stream)>>>(p);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_ritz_shift_update(float* const* rdiag_host, int batch, int rows, int tail_rows, float shift_scale,
                                     float* shift_dev, void* stream) {
  XKV_REQUIRE(rdiag_host && shift_dev && batch >= 1 && batch <= XKV_MAX_BATCH, "ritz_shift_update: bad arguments");
  XKV_REQUIRE(tail_rows >= 1 && tail_rows <= rows, "ritz_shift_update: tail_rows out of range");
  NormParams p;
  std::memset(&p, 0, sizeof(p));
  for (int b = 0; b < batch; ++b) p.rdiag[b] = rdiag_host[b];
  p.c = shift_dev;
  p.rows = rows;
  p.tail = tail_rows;
  p.shift_scale = shift_scale;
  ritz_shift_kernel<<<batch, 256, 0, as_stream(stream)>>>(p);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_rdiag_update(float* const* rdiag_host, const float* const* Linv_host, int batch, int rows,
                                int64_t ld_linv, void* stream) {
  XKV_REQUIRE(rdiag_host && Linv_host && batch >= 1 && batch <= XKV_MAX_BATCH, "rdiag_update: bad arguments");
  NormParams p;
  std::memset(&p, 0, sizeof(p));
  for (int b = 0; b < batch; ++b) {
    p.rdiag[b] = rdiag_host[b];
    p.Linv[b] = Linv_host[b];
  }
  p.rows = rows;
  p.ld_linv = ld_linv;
  p.run_if = launch_predicate();
  rdiag_update_kernel<<<dim3((rows + 255) / 256, batch), 256, 0, as_stream(stream)>>>(p);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_jacobi_eigh(const float* const* T_host, float* const* evals_host, float* const* Wt_host, int count,
                               int W, int64_t ld, int64_t ld_w, int sweeps, void* stream) {
  XKV_REQUIRE(T_host && evals_host && count >= 1 && count <= 2 * XKV_MAX_BATCH, "jacobi: bad count");
  XKV_REQUIRE(W >= 2 && W <= 160 && W % 2 == 0, "jacobi: window W=%d must be even and <= 160", W);
  JacobiParams p;
  std::memset(&p, 0, sizeof(p));
  for (int b = 0; b < count; ++b) {
    XKV_REQUIRE(T_host[b] && evals_host[b], "jacobi: null matrix %d", b);
    p.T[b] = T_host[b];
    p.evals[b] = evals_host[b];
    p.Wt[b] = Wt_host ? Wt_host[b] : nullptr;
  }
  p.W = W;
  p.sweeps = sweeps;
  p.tol = 1e-4f;   // a sweep whose largest rotated element is below this leaves off-diagonals of O(tol^2)
  p.ld = ld;
  p.ld_w = ld_w;
  const size_t smem = static_cast<size_t>(2 * W * (W + 1) + 2 * W) * sizeof(float) + 64;
  static PerDevice<bool> configured;
  if (!configured()) {
    XKV_CHECK_CUDA(cudaFuncSetAttribute(jacobi_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    XKV_CHECK_CUDA(cudaFuncSetAttribute(jacobi_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    XKV_CHECK_CUDA(cudaFuncSetAttribute(jacobi_kernel<160>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    configured() = true;
  }
  if (W == 128)
    jacobi_kernel<128><<<count, JAC_THREADS, smem, as_stream(stream)>>>(p);
  else if (W == 160)
    jacobi_kernel<160><<<count, JAC_THREADS, smem, as_stream(stream)>>>(p);
  else
    jacobi_kernel<0><<<count, JAC_THREADS, smem, as_stream(stream)>>>(p);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_convert_bf16(const float* src, int rows, int cols, int64_t ld, void* dst, int64_t ld_dst, void* dstT,
                                int64_t ld_dstT, void* stream) {
  XKV_REQUIRE(src && (dst || dstT) && rows > 0 && cols > 0, "convert_bf16: bad arguments");
  dim3 grid((cols + 31) / 32, (rows + 31) / 32);
  convert_bf16_kernel<<<grid, 256, 0, as_stream(stream)>>>(src, rows, cols, ld, static_cast<__nv_bfloat16*>(dst),
                                                           ld_dst, static_cast<__nv_bfloat16*>(dstT), ld_dstT);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_sqrt_clamp(const float* in, float* out, int count, void* stream) {
  XKV_REQUIRE(in && out && count > 0, "sqrt_clamp: bad arguments");
  sqrt_clamp_kernel<<<(count + 255) / 256, 256, 0, as_stream(stream)>>>(in, out, count);
  XKV_LAUNCHED();
  return 0;
}
