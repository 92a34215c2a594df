// xkv_b200 — blocked Cholesky (S + shift*I) = L L^T with explicit inverse Linv = L^{-1}, ONE launch:
// a thread-block cluster per matrix, cluster barriers instead of kernel boundaries.
//
// This is the serial heart of CholeskyQR (the orthogonalisation after every power step of the
// factorisation that replaces torch.linalg.svd, fake_layer_merge_dynamic_cache.py:20).  The previous
// version spent 2 launches per 64-column panel plus 2 per inverse level (~35 launches, ~0.6 ms for
// l = 576); here the whole thing is one kernel whose CTAs exchange 64x64 tiles through L2.
//
// Layout trick: every block product C = A B reads both operands "k-major" ([k][row] / [k][col]) from shared
// memory.  To get that layout straight from row-major global tiles, the factor is kept TRANSPOSED in the upper
// triangle of S (block (k,i), k < i, holds L[i,k]^T = R[k,i]), and the inverse is kept both plain (lower
// blocks of Linv) and transposed (upper blocks of Linv) until the final phase clears the upper blocks.
//
//   Phase F, step k:  every CTA factors the diagonal block S(k,k) redundantly (register-resident
//                     Gauss-Jordan sweep that yields X = L_kk^{-1} directly)            -> Xt in smem
//                     panel   L[i,k]^T -> S(k,i)      for i > k, dealt round-robin over the cluster
//                     --- cluster barrier ---
//                     update  S(j,i) -= L[j,k] L[i,k]^T   for k < j <= i, dealt round-robin
//                     --- cluster barrier ---
//   Phase I, level s = 1, 2, 4, ...: for each aligned pair of diagonal super-blocks [A 0; B C]
//                     pass 0: T = B A^{-1}             (staged in the free lower blocks of S)
//                     pass 1: Linv[C,A] = -C^{-1} T    (written plain and transposed)
//   Final:            zero the upper blocks of Linv, optionally emit its bf16 limbs (the GEMM operand).
#include <cooperative_groups.h>
#include <cuda_bf16.h>

#include <cstdlib>

#include "xkv_common.cuh"
#include "xkv_host.h"

namespace cg = cooperative_groups;

namespace xkv {

constexpr int CB = 64;             // block size
constexpr int CBK = CB + 4;        // shared-memory row stride of a k-major tile (rows stay 16-byte aligned)
constexpr int CTILE = CB * CBK;
constexpr int CH_THREADS = 256;
constexpr int CH_SMEM_FLOATS = 5 * CTILE + 2 * 128 + 2 * 64;

struct CholFusedParams {
  float* S[XKV_MAX_BATCH];
  float* Linv[XKV_MAX_BATCH];
  __nv_bfloat16* hi[XKV_MAX_BATCH];
  __nv_bfloat16* mid[XKV_MAX_BATCH];
  __nv_bfloat16* lo[XKV_MAX_BATCH];
  int l, nblk;                 // matrix size and its number of CB blocks
  long long ld, ld_limb;
  float pivot_floor, shift;
  const int* run_if;   // optional per-matrix device predicate (xkv_set_launch_predicate): the whole cluster exits
};

__device__ __forceinline__ void split3f(float x, __nv_bfloat16& h, __nv_bfloat16& m, __nv_bfloat16& l) {
  h = __float2bfloat16_rn(x);
  const float r1 = x - __bfloat162float(h);
  m = __float2bfloat16_rn(r1);
  const float r2 = r1 - __bfloat162float(m);
  l = __float2bfloat16_rn(r2);
}

// row-major 64x64 global tile -> smem [k][idx] (stride CBK).  L2 loads: the tile was written by another CTA.
__device__ __forceinline__ void load_tile(float* dst, const float* src, long long ld) {
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int e = threadIdx.x + it * CH_THREADS;
    const int row = e >> 4, c4 = (e & 15) * 4;
    const float4 v = __ldcg(reinterpret_cast<const float4*>(src + static_cast<long long>(row) * ld + c4));
    *reinterpret_cast<float4*>(dst + row * CBK + c4) = v;
  }
}

// acc[i][j] += sum_k Ak[k][tr+i] * Bk[k][tc+j]
__device__ __forceinline__ void tile_mma(float (&acc)[4][4], const float* Ak, const float* Bk) {
  const int tr = (threadIdx.x >> 4) * 4;
  const int tc = (threadIdx.x & 15) * 4;
#pragma unroll 8
  for (int k = 0; k < CB; ++k) {
    const float4 a = *reinterpret_cast<const float4*>(Ak + k * CBK + tr);
    const float4 b = *reinterpret_cast<const float4*>(Bk + k * CBK + tc);
    const float av[4] = {a.x, a.y, a.z, a.w};
    const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
  }
}

// Factor the 64x64 SPD block D (+ shift on the diagonal) and produce X = L^{-1} (lower triangular), with the
// augmented matrix [D | I] (64 x 128) held in registers: thread (cc, par) owns column cc, rows 2u + par.
// Right-looking sweep, one barrier per column j: the owners of row j and of column j publish them, then every
// thread applies  Aug[i][cc] -= D[i][j] * Aug[j][cc] / D[j][j]  to its rows i > j.  Row j of the identity half
// scaled by 1/sqrt(d) is row j of X (forward substitution in right-looking form).  L itself is never needed.
//   Xt[kk][c] = X[c][kk]   (k-major operand for  P = S[i,k] X^T  and for the inverse products)
//   x_plain (optional, global): X row-major with zeros above the diagonal.
// (No __restrict__ on the shared-memory pointers: rowj / lraw are written by OTHER threads between barriers, and
// with restrict the compiler forwards this thread's stale loads across __syncthreads.)
__device__ __forceinline__ void diag_factor(const float* D, long long ld, float shift, float pivot_floor, float* Xt,
                                            float* rowj, float* lraw, float* x_plain) {
  const int cc = threadIdx.x & 127, par = threadIdx.x >> 7;
  float v[32];
  if (cc < CB) {
#pragma unroll
    for (int u = 0; u < 32; ++u) {
      const int i = 2 * u + par;
      v[u] = __ldcg(D + static_cast<long long>(i) * ld + cc) + (i == cc ? shift : 0.f);
    }
  } else {
#pragma unroll
    for (int u = 0; u < 32; ++u) v[u] = (2 * u + par == cc - CB) ? 1.f : 0.f;
  }
#pragma unroll
  for (int j = 0; j < CB; ++j) {
    float* rj = rowj + (j & 1) * 128;
    float* lr = lraw + (j & 1) * 64;
    const int u_first = (j / 2) & ~3;           // first 4-group that still contains a row > j
    if (par == (j & 1)) rj[cc] = v[j >> 1];
    if (cc == j) {
#pragma unroll
      for (int u4 = 0; u4 < 32; u4 += 4)
        if (u4 >= u_first)
          *reinterpret_cast<float4*>(lr + par * 32 + u4) = make_float4(v[u4], v[u4 + 1], v[u4 + 2], v[u4 + 3]);
    }
    __syncthreads();
    if (cc >= j) {                              // finished columns of the D half hold final values
      const float d = fmaxf(rj[j], pivot_floor);
      const float rjp = __fdividef(rj[cc], d);
#pragma unroll
      for (int u4 = 0; u4 < 32; u4 += 4) {
        if (u4 >= u_first) {
          const float4 l4 = *reinterpret_cast<const float4*>(lr + par * 32 + u4);
          const float lv[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int u = u4 + q;
            if (2 * u > j || (2 * u + 1 > j && par == 1)) v[u] = fmaf(-lv[q], rjp, v[u]);
          }
        }
      }
      if (par == (j & 1)) v[j >> 1] *= rsqrtf(d);
    }
  }
  // identity half now holds X: thread (64 + c, par) has X[2u + par][c]
  if (cc >= CB) {
    const int c = cc - CB;
#pragma unroll
    for (int u = 0; u < 32; ++u) Xt[c * CBK + 2 * u + par] = v[u];
    if (x_plain != nullptr) {
#pragma unroll
      for (int u = 0; u < 32; ++u) x_plain[static_cast<long long>(2 * u + par) * ld + c] = v[u];
    }
  }
}

// ---- software pipeline over 64x64x64 block products ------------------------------------------------------
// A CTA's share of a phase is a list of products (A tile, B tile) -> output tile.  The operand tiles of product
// t+1 are in flight (cp.async, L2 -> shared, two buffers) while product t runs on the FFMA pipe: measured on the
// first version, a tile product cost ~4 us of which ~1.4 us was arithmetic, the rest exposed L2 round trips.
struct Prod {
  const float* a;   // row-major global tile, used as Ak[kk][r]
  const float* b;   // row-major global tile, used as Bk[kk][c]; nullptr: the resident Xt tile
  int oi, oj;       // output block
  bool first, last; // first / last product of its output tile
};
__device__ __forceinline__ void prefetch_tile(float* dst, const float* src, long long ld) {
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int e = threadIdx.x + it * CH_THREADS;
    const int row = e >> 4, c4 = (e & 15) * 4;
    const uint32_t d = smem_u32(dst + row * CBK + c4);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + static_cast<long long>(row) * ld + c4)
                 : "memory");
  }
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

enum { EPI_PANEL = 0, EPI_UPDATE = 1, EPI_STORE = 2, EPI_INV = 3 };

// Gen: bool next(Prod&).  Buffers: bufA[2], bufB[2] (CTILE floats each), Xt resident.
template <int EPI, class Gen>
__device__ __forceinline__ void run_products(Gen& gen, float* bufs, const float* Xt, float* S, float* Li, long long ld) {
  const int tid = threadIdx.x, tr = (tid >> 4) * 4, tc = (tid & 15) * 4;
  auto blk = [&](float* base, int bi, int bj) -> float* {
    return base + static_cast<long long>(bi) * CB * ld + static_cast<long long>(bj) * CB;
  };
  Prod cur, nxt;
  bool has = gen.next(cur);
  if (!has) return;
  int st = 0;
  prefetch_tile(bufs + 0 * CTILE, cur.a, ld);
  if (cur.b) prefetch_tile(bufs + 2 * CTILE, cur.b, ld);
  cp_async_commit();
  float acc[4][4];
  while (has) {
    const bool has_n = gen.next(nxt);
    if (has_n) {
      prefetch_tile(bufs + (st ^ 1) * CTILE, nxt.a, ld);
      if (nxt.b) prefetch_tile(bufs + (2 + (st ^ 1)) * CTILE, nxt.b, ld);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    if (cur.first) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    }
    float4 cin[4];
    if (EPI == EPI_UPDATE) {   // the output tile is read-modify-write: fetch it under the arithmetic
      const float* g = blk(S, cur.oi, cur.oj);
#pragma unroll
      for (int a = 0; a < 4; ++a) cin[a] = __ldcg(reinterpret_cast<const float4*>(g + static_cast<long long>(tr + a) * ld + tc));
    }
    tile_mma(acc, bufs + st * CTILE, cur.b ? bufs + (2 + st) * CTILE : Xt);
    if (cur.last) {
      if (EPI == EPI_PANEL) {          // S(oi,oj)[c'][r] = acc[r][c']  (transposed store of L[i,k])
        float* g = blk(S, cur.oi, cur.oj);
#pragma unroll
        for (int b = 0; b < 4; ++b)
          *reinterpret_cast<float4*>(g + static_cast<long long>(tc + b) * ld + tr) =
              make_float4(acc[0][b], acc[1][b], acc[2][b], acc[3][b]);
      } else if (EPI == EPI_UPDATE) {  // S(oi,oj) -= acc
        float* g = blk(S, cur.oi, cur.oj);
#pragma unroll
        for (int a = 0; a < 4; ++a)
          *reinterpret_cast<float4*>(g + static_cast<long long>(tr + a) * ld + tc) =
              make_float4(cin[a].x - acc[a][0], cin[a].y - acc[a][1], cin[a].z - acc[a][2], cin[a].w - acc[a][3]);
      } else if (EPI == EPI_STORE) {   // S(oi,oj) = acc
        float* g = blk(S, cur.oi, cur.oj);
#pragma unroll
        for (int a = 0; a < 4; ++a)
          *reinterpret_cast<float4*>(g + static_cast<long long>(tr + a) * ld + tc) =
              make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
      } else {                         // Linv(oi,oj) = -acc, Linv(oj,oi) = -acc^T
        float* g = blk(Li, cur.oi, cur.oj);
        float* gt = blk(Li, cur.oj, cur.oi);
#pragma unroll
        for (int a = 0; a < 4; ++a)
          *reinterpret_cast<float4*>(g + static_cast<long long>(tr + a) * ld + tc) =
              make_float4(-acc[a][0], -acc[a][1], -acc[a][2], -acc[a][3]);
#pragma unroll
        for (int b = 0; b < 4; ++b)
          *reinterpret_cast<float4*>(gt + static_cast<long long>(tc + b) * ld + tr) =
              make_float4(-acc[0][b], -acc[1][b], -acc[2][b], -acc[3][b]);
      }
    }
    __syncthreads();   // everybody is done with buffer `st` before the prefetch of the next-but-one product refills it
    cur = nxt;
    has = has_n;
    st ^= 1;
  }
}

__global__ void __launch_bounds__(CH_THREADS, 1) chol_cluster_kernel(const __grid_constant__ CholFusedParams p) {
  extern __shared__ __align__(16) float chol_sm[];
  if (p.run_if != nullptr && p.run_if[blockIdx.y] == 0) return;   // uniform over the cluster, before any barrier
  cg::cluster_group cluster = cg::this_cluster();
  const int CL = static_cast<int>(cluster.num_blocks());
  const int c = static_cast<int>(cluster.block_rank());
  float* bufs = chol_sm;               // [A0 | A1 | B0 | B1]
  float* Xt = bufs + 4 * CTILE;
  float* rowj = Xt + CTILE;
  float* lraw = rowj + 2 * 128;
  float* S = p.S[blockIdx.y];
  float* Li = p.Linv[blockIdx.y];
  const long long ld = p.ld;
  const int nblk = p.nblk;
  const int tid = threadIdx.x;
  auto blk = [&](float* base, int bi, int bj) -> float* {
    return base + static_cast<long long>(bi) * CB * ld + static_cast<long long>(bj) * CB;
  };
  auto publish_xt = [&](int k) {   // S(k,k) <- X_k^T: the k-major operand of the inverse products
    float* g = blk(S, k, k);
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int e = tid + it * CH_THREADS;
      const int row = e >> 4, c4 = (e & 15) * 4;
      *reinterpret_cast<float4*>(g + static_cast<long long>(row) * ld + c4) =
          *reinterpret_cast<const float4*>(Xt + row * CBK + c4);
    }
  };

  // ---------------- phase F ----------------
  // Look-ahead: the diagonal factorisation of step k+1 (a serial 64-column sweep, ~8 us) is taken off the
  // critical path.  Its owner updates tile (k+1, k+1) first, factors it and publishes X_{k+1}^T in S(k+1, k+1)
  // while the other CTAs work through the rest of the trailing update; after the barrier everybody just loads it.
  constexpr int kSkipRounds = 3;   // update rounds the look-ahead owner sits out (~ T_diag / T_tile)
  for (int k = 0; k < nblk; ++k) {
    if (k == 0) {
      diag_factor(blk(S, 0, 0), ld, p.shift, p.pivot_floor, Xt, rowj, lraw, c == 0 ? blk(Li, 0, 0) : nullptr);
    } else {
      load_tile(Xt, blk(S, k, k), ld);   // X_k^T, published by the look-ahead owner during step k-1
    }
    __syncthreads();
    {
      // panel: L[i,k] = S[i,k] X_k^T, stored transposed over S(k,i)
      struct PanelGen {
        float* S; long long ld; int k, i, nblk, CL;
        __device__ bool next(Prod& q) {
          if (i >= nblk) return false;
          q.a = S + static_cast<long long>(k) * CB * ld + static_cast<long long>(i) * CB;
          q.b = nullptr;
          q.oi = k; q.oj = i; q.first = q.last = true;
          i += CL;
          return true;
        }
      } gen{S, ld, k, k + 1 + c, nblk, CL};
      run_products<EPI_PANEL>(gen, bufs, Xt, S, Li, ld);
    }
    cluster.sync();
    if (k == 0 && c == 0) publish_xt(0);   // only after the barrier: peers were still reading S(0,0) before it
    const int nt = nblk - k - 1;
    const int ntiles = nt * (nt + 1) / 2;     // tile e = ii (ii + 1) / 2 + jj, 0 <= jj <= ii < nt; e = 0 is (k+1, k+1)
    const int own = (k + 1) % CL;             // look-ahead owner of step k+1
    struct UpdateGen {
      float* S; long long ld; int k, e, e_end, early, others, CL, rel;
      __device__ bool next(Prod& q) {
        for (; e < e_end; ++e) {
          if (e > 0) {
            const int t = e - 1;
            const int who = t < early ? t % others : (t - early) % CL;
            if (who != rel) continue;
          }
          int ii = static_cast<int>((sqrtf(8.f * static_cast<float>(e) + 1.f) - 1.f) * 0.5f);
          while (ii * (ii + 1) / 2 > e) --ii;
          while ((ii + 1) * (ii + 2) / 2 <= e) ++ii;
          const int jj = e - ii * (ii + 1) / 2;
          const int i = k + 1 + ii, j = k + 1 + jj;
          q.a = S + static_cast<long long>(k) * CB * ld + static_cast<long long>(j) * CB;
          q.b = S + static_cast<long long>(k) * CB * ld + static_cast<long long>(i) * CB;
          q.oi = j; q.oj = i; q.first = q.last = true;
          ++e;
          return true;
        }
        return false;
      }
    };
    const int others = CL - 1;
    const int early = others > 0 ? kSkipRounds * others : 0;
    const int rel = (c - own - 1 + 2 * CL) % CL;   // 0 .. CL-2 for the others (ring order), CL-1 for the owner
    if (ntiles > 0 && c == own) {
      UpdateGen g0{S, ld, k, 0, 1, early, others > 0 ? others : 1, CL, rel};
      run_products<EPI_UPDATE>(g0, bufs, Xt, S, Li, ld);
      diag_factor(blk(S, k + 1, k + 1), ld, p.shift, p.pivot_floor, Xt, rowj, lraw, blk(Li, k + 1, k + 1));
      __syncthreads();
      publish_xt(k + 1);
      __syncthreads();
    }
    {
      UpdateGen g1{S, ld, k, 1, ntiles, early, others > 0 ? others : 1, CL, rel};
      run_products<EPI_UPDATE>(g1, bufs, Xt, S, Li, ld);
    }
    cluster.sync();
  }

  // ---------------- phase I ----------------
  for (int s = 1; s < nblk; s <<= 1) {
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
      // pass 0: T(i,j) = sum_{t=j}^{a+s-1} L[i,t] Linv[t,j]      (staged at the lower block S(i,j))
      // pass 1: Linv(i,j) = -sum_{t=a+s}^{i} Linv[i,t] T[t,j]
      struct InvGen {
        float* S; float* Li; long long ld; int nblk, s, pass, CL, c;
        int i, j, t, cnt; bool open;
        __device__ const float* at(const float* base, int bi, int bj) const {
          return base + static_cast<long long>(bi) * CB * ld + static_cast<long long>(bj) * CB;
        }
        __device__ bool next(Prod& q) {
          for (;;) {
            if (i >= nblk) return false;
            const int a = (i / (2 * s)) * 2 * s;
            if (i < a + s) { ++i; j = -1; open = false; continue; }   // row i must lie in the C half of its pair
            if (!open) {
              // advance to the next tile (i, j) of this row that belongs to this CTA
              j = (j < 0) ? a : j + 1;
              bool found = false;
              for (; j < a + s; ++j, ++cnt)
                if ((cnt + i) % CL == c) { found = true; break; }
              if (!found) { ++i; j = -1; continue; }
              ++cnt;
              t = pass == 0 ? j : a + s;
              open = true;
            }
            const int t1 = pass == 0 ? a + s : i + 1;
            q.oi = i; q.oj = j;
            q.first = (t == (pass == 0 ? j : a + s));
            q.last = (t + 1 == t1);
            if (pass == 0) {
              q.a = at(S, t, i);                       // L[i,t]^T
              q.b = at(Li, t, j);                      // Linv[t,j]  (t == j: X_j, zero upper)
            } else {
              q.a = t < i ? at(Li, t, i) : at(S, i, i);   // Linv[i,t]^T  (t == i: X_i^T)
              q.b = at(S, t, j);                       // T[t,j]
            }
            ++t;
            if (q.last) open = false;
            return true;
          }
        }
      } gen{S, Li, ld, nblk, s, pass, CL, c, 0, -1, 0, 0, false};
      if (pass == 0)
        run_products<EPI_STORE>(gen, bufs, Xt, S, Li, ld);
      else
        run_products<EPI_INV>(gen, bufs, Xt, S, Li, ld);
      cluster.sync();
    }
  }

  // ---------------- final: clear the transposed copies, emit bf16 limbs ----------------
  __nv_bfloat16* hi = p.hi[blockIdx.y];
  __nv_bfloat16* mid = p.mid[blockIdx.y];
  __nv_bfloat16* lo = p.lo[blockIdx.y];
  const int l4 = p.l >> 2;
  for (int r = c; r < p.l; r += CL) {
    const int bi = r / CB;
    float* row = Li + static_cast<long long>(r) * ld;
    for (int q = tid; q < l4; q += CH_THREADS) {
      const int col = q * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (col / CB > bi)
        *reinterpret_cast<float4*>(row + col) = v;
      else
        v = __ldcg(reinterpret_cast<const float4*>(row + col));
      if (hi != nullptr) {
        __nv_bfloat16 h[4], m[4], w[4];
        split3f(v.x, h[0], m[0], w[0]);
        split3f(v.y, h[1], m[1], w[1]);
        split3f(v.z, h[2], m[2], w[2]);
        split3f(v.w, h[3], m[3], w[3]);
        const long long o = static_cast<long long>(r) * p.ld_limb + col;
        *reinterpret_cast<uint2*>(hi + o) = *reinterpret_cast<uint2*>(h);
        if (mid != nullptr) *reinterpret_cast<uint2*>(mid + o) = *reinterpret_cast<uint2*>(m);
        if (lo != nullptr) *reinterpret_cast<uint2*>(lo + o) = *reinterpret_cast<uint2*>(w);
      }
    }
  }
}

}  // namespace xkv

using namespace xkv;

extern "C" int xkv_cholesky_inverse_limbs(float* const* S_host, float* const* Linv_host, void* const* hi_host,
                                          void* const* mid_host, void* const* lo_host, int batch, int l, int64_t ld,
                                          int64_t ld_limb, float shift, float pivot_floor, void* stream) {
  XKV_REQUIRE(S_host && Linv_host && batch >= 1 && batch <= XKV_MAX_BATCH, "cholesky: bad batch");
  XKV_REQUIRE(l > 0 && l % CB == 0, "cholesky: l=%d must be a positive multiple of %d", l, CB);
  XKV_REQUIRE(ld % 4 == 0 && ld >= l, "cholesky: ld must be a multiple of 4 and >= l");
  XKV_REQUIRE(!hi_host || (ld_limb % 4 == 0 && ld_limb >= l), "cholesky: ld_limb must be a multiple of 4 and >= l");
  CholFusedParams p;
  std::memset(&p, 0, sizeof(p));
  for (int b = 0; b < batch; ++b) {
    XKV_REQUIRE(S_host[b] && Linv_host[b], "cholesky: null matrix %d", b);
    XKV_REQUIRE((reinterpret_cast<uintptr_t>(S_host[b]) & 15) == 0 && (reinterpret_cast<uintptr_t>(Linv_host[b]) & 15) == 0,
                "cholesky: matrices must be 16-byte aligned");
    p.S[b] = S_host[b];
    p.Linv[b] = Linv_host[b];
    p.hi[b] = hi_host ? static_cast<__nv_bfloat16*>(hi_host[b]) : nullptr;
    p.mid[b] = mid_host ? static_cast<__nv_bfloat16*>(mid_host[b]) : nullptr;
    p.lo[b] = lo_host ? static_cast<__nv_bfloat16*>(lo_host[b]) : nullptr;
  }
  p.l = l;
  p.nblk = l / CB;
  p.ld = ld;
  p.ld_limb = ld_limb;
  p.pivot_floor = pivot_floor;
  p.shift = shift;
  p.run_if = launch_predicate();
  const int smem = CH_SMEM_FLOATS * static_cast<int>(sizeof(float));
  static PerDevice<bool> attr_set;
  if (!attr_set()) {
    XKV_CHECK_CUDA(cudaFuncSetAttribute(chol_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set() = true;
  }
  int CL = p.nblk >= 6 ? 8 : (p.nblk >= 3 ? 4 : (p.nblk == 2 ? 2 : 1));
  cudaLaunchConfig_t cfg;
  std::memset(&cfg, 0, sizeof(cfg));
  cfg.blockDim = dim3(CH_THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = as_stream(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // Wide factors (>= 20 blocks: sketch width 1280 and up, config 4 values) have enough tiles per step for 16 CTAs -- a non-portable cluster
  // size, used only when the device can keep one such cluster per matrix resident at once.
  static PerDevice<int> cl16_state;   // 0: not probed; 1 + resident 16-CTA clusters of this kernel on this device
  int& cl16_probe = cl16_state();
  if (cl16_probe == 0) {
    int cl16_clusters = 0;
    if (cudaFuncSetAttribute(chol_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
      cfg.gridDim = dim3(16, 1, 1);
      attr[0].val.clusterDim.x = 16;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, chol_cluster_kernel, &cfg) == cudaSuccess) cl16_clusters = n;
    }
    (void)cudaGetLastError();
    cl16_probe = 1 + cl16_clusters;
  }
  if (p.nblk >= 20 && cl16_probe - 1 >= batch) CL = 16;
  cfg.gridDim = dim3(CL, batch, 1);
  attr[0].val.clusterDim.x = CL;
  XKV_CHECK_CUDA(cudaLaunchKernelEx(&cfg, chol_cluster_kernel, p));
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_cholesky_inverse(float* const* S_host, float* const* Linv_host, int batch, int l, int64_t ld,
                                    float shift, float pivot_floor, void* stream) {
  return xkv_cholesky_inverse_limbs(S_host, Linv_host, nullptr, nullptr, nullptr, batch, l, ld, 0, shift, pivot_floor,
                                    stream);
}
