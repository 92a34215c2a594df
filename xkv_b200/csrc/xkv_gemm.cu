// xkv_b200 — grouped tcgen05 GEMM engine (sm_100a).
//
// One kernel serves every matrix product of the factorisation (reference call sites:
// torch.linalg.svd / torch.matmul, fake_layer_merge_dynamic_cache.py:20,26):
//   Gram          G  = X^T X          both operands MN-major tiles of X, symmetric tile set, split-K
//   power step    Yt = Qt G           K-major x K-major (G symmetric), multi-limb terms
//   small Grams   S  = Yt Yt^T        K-major x K-major
//   tri-solve     Qt = Linv Yt        K-major x MN-major
//   Ritz vectors  Vt = Wt Qt          K-major x MN-major
//   projection    A  = X V            K-major x K-major, bf16 output
//
// Structure (one 128 x 256 output tile per CTA, 192 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D boxes, 128B swizzle, 4-stage mbarrier ring
//   warp 1      allocates 256 TMEM columns, one lane issues tcgen05.mma (M128 N256 K16, bf16 -> fp32),
//               tcgen05.commit releases smem stages / publishes the accumulator
//   warps 2..5  epilogue: tcgen05.ld (32 lanes x 32 columns) -> registers -> global (fp32 / bf16,
//               optionally transposed)
// Problems are passed by value in __grid_constant__ parameter space (tensor maps included), so a
// launch needs no device-side descriptor memory.
//
// Two kernels share this structure: gemm_kernel (one CTA per 128 x 256 tile: the small-M products -- Gram of the basis,
// Rayleigh-Ritz window, the decode's P A_v) and gemm_pair_kernel (a CTA PAIR per 256 x bn tile, cta_group::2: the Gram,
// the projection, and the power step / triangular solve / window product with their operand roles swapped by the
// factorisation driver so that the long dimension is M).  xkv_gemm_grouped picks per launch (pair_bn); both give the
// same bits.
#include <cstdlib>

#include "xkv_common.cuh"
#include "xkv_host.h"

namespace xkv {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
constexpr int STAGES = 4;
constexpr int A_TILE_BYTES = BM * BK * 2;  // 16 KiB
constexpr int B_TILE_BYTES = BN * BK * 2;  // 32 KiB
constexpr int STAGE_BYTES = A_TILE_BYTES + B_TILE_BYTES;
constexpr int CHUNK_BYTES = 64 * BK * 2;   // one 64-wide MN-major chunk: BK rows x 128 B
constexpr int GEMM_THREADS = 192;
constexpr int TMEM_COLS = 256;
constexpr size_t GEMM_SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;

struct alignas(64) GemmProb {
  CUtensorMap a_map[3];
  CUtensorMap b_map[3];
  void* D;
  long long ldd;
  long long split_stride;
  int M, N, K;
  int nterms;
  int tiles_m, tiles_n, ntiles;
  int split_k, kblocks_per_split, nkb;
  int cta_begin;
  int bn;              // N tile (256; the pair kernel: any multiple of 16 up to 256)
  // pair kernel, limb terms: a ring stage holds every DISTINCT limb tile of a k block once (A slots, then B slots, 16 KiB
  // each) and all the terms' MMAs read from it -- 3 terms load 2 + 2 tiles instead of 3 + 3, 6 terms 3 + 3 instead of 6 + 6
  int na, nb;                        // distinct A / B limbs
  unsigned char la[3], lb[3];        // slot -> limb
  unsigned char sa[3], sb[3];        // limb -> slot
  int pstages;                       // ring depth of this problem: ring bytes / ((na + nb) * 16 KiB)
  int out_bf16, out_transposed, sym_upper;
  unsigned char ta[6], tb[6];
  const int* run_if;   // optional device predicate: the problem's CTAs exit at once when *run_if == 0
  int phases;          // sequential accumulation phases per CTA (two TMEM accumulators), see gemm_kernel
  // layered operands: operand columns [i * layer_cols, (i + 1) * layer_cols) come from GemmParams::layer_maps[begin + i]
  int a_layers, a_layer_begin, b_layers, b_layer_begin, layer_cols;
};
struct GemmParams {
  int nprob;
  int pair_stages;   // gemm_pair_kernel: ring depth (PG_STAGES)
  GemmProb p[XKV_MAX_GEMM_PROBLEMS];
  CUtensorMap layer_maps[XKV_MAX_LAYER_MAPS];
};

// Tensor map and in-layer column of column `col` of a layered operand.  Columns past the last layer map to the last
// layer with an out-of-bounds coordinate (TMA zero-fills), like the tail of an ordinary operand.
__device__ __forceinline__ const CUtensorMap* layer_map(const GemmParams& P, int begin, int layers, int layer_cols, int col,
                                                        int& col_in_layer) {
  int li = col / layer_cols;
  li = li < layers ? li : layers - 1;
  col_in_layer = col - li * layer_cols;
  return &P.layer_maps[begin + li];
}

template <int A_MN, int B_MN>
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_kernel(const __grid_constant__ GemmParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;    // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // ---- locate this CTA's problem / split / tile ----
  int pi = 0;
  while (pi + 1 < P.nprob && static_cast<int>(blockIdx.x) >= P.p[pi + 1].cta_begin) ++pi;
  const GemmProb& pr = P.p[pi];
  if (pr.run_if != nullptr && *pr.run_if == 0) return;   // uniform per CTA, before any barrier / TMEM allocation
  const int local = static_cast<int>(blockIdx.x) - pr.cta_begin;
  const int split = local / pr.ntiles;
  int t = local - split * pr.ntiles;
  int tm, tn;
  if (pr.sym_upper) {
    tm = 0;
    tn = 0;
    for (int i = 0; i < pr.tiles_m; ++i) {
      const int first = (i * BM) / BN;
      const int cnt = pr.tiles_n - first;
      if (t < cnt) {
        tm = i;
        tn = first + t;
        break;
      }
      t -= cnt;
    }
  } else {
    tm = t / pr.tiles_n;
    tn = t - tm * pr.tiles_n;
  }
  const int m0 = tm * BM;
  const int n0 = tn * BN;
  const int kb0 = split * pr.kblocks_per_split;
  const int kb1 = min(kb0 + pr.kblocks_per_split, pr.nkb);
  const int nk = max(kb1 - kb0, 0);
  const int niter = nk * pr.nterms;
  // Accumulation phases: a tensor-core accumulator that runs over tens of thousands of tokens loses the low bits
  // of the small Gram entries (the fp32 adder of the MMA truncates; measured on the 65536-token Gram: 1.2 % excess
  // reconstruction error at the rank boundary, 0.4 % with four phases).  With phases > 1 the k range is cut into
  // `nph` pieces that alternate between two TMEM accumulators; the epilogue warps add each finished piece into the
  // fp32 output (plain load-add-store: a tile is owned by one CTA) while the MMAs of the next piece run.
  const int nph = max(1, min(pr.phases, nk));
  const uint32_t tmem_cols = nph > 1 ? 2 * TMEM_COLS : TMEM_COLS;

  // ---- one-time setup ----
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(&tmem_full_bar[0], 1);
    mbar_init(&tmem_full_bar[1], 1);
    mbar_init(&tmem_empty_bar[0], 4);   // one arrival per epilogue warp
    mbar_init(&tmem_empty_bar[1], 4);
    mbar_fence_init();
    for (int i = 0; i < 3; ++i) {
      tma_prefetch_desc(&pr.a_map[i]);
      tma_prefetch_desc(&pr.b_map[i]);
    }
  }
  if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (whole warp in the loop, one elected lane issues) =====================
    // Layered operands: which layer matrix a 64-column chunk of this CTA's tile comes from is fixed for the whole kernel
    // (MN-major: the chunk's column is m0 / n0 + 64 c) or advances with the k block (K-major): resolved here, outside the
    // loop, so that the issue path has no integer division.
    const CUtensorMap* a_chunk_map[BM / 64];
    int a_chunk_col[BM / 64];
    const CUtensorMap* b_chunk_map[BN / 64];
    int b_chunk_col[BN / 64];
#pragma unroll
    for (int c = 0; c < BM / 64; ++c) {
      a_chunk_col[c] = m0 + 64 * c;
      a_chunk_map[c] = (A_MN && pr.a_layers) ? layer_map(P, pr.a_layer_begin, pr.a_layers, pr.layer_cols, m0 + 64 * c, a_chunk_col[c]) : nullptr;
    }
#pragma unroll
    for (int c = 0; c < BN / 64; ++c) {
      b_chunk_col[c] = n0 + 64 * c;
      b_chunk_map[c] = (B_MN && pr.b_layers) ? layer_map(P, pr.b_layer_begin, pr.b_layers, pr.layer_cols, n0 + 64 * c, b_chunk_col[c]) : nullptr;
    }
    // K-major layered operand: (layer, column inside the layer) of the current k block, advanced incrementally
    int ka_layer = 0, ka_col = 0, kb_layer = 0, kb_col = 0;
    if (!A_MN && pr.a_layers) {
      ka_layer = (kb0 * BK) / pr.layer_cols;
      ka_col = kb0 * BK - ka_layer * pr.layer_cols;
    }
    if (!B_MN && pr.b_layers) {
      kb_layer = (kb0 * BK) / pr.layer_cols;
      kb_col = kb0 * BK - kb_layer * pr.layer_cols;
    }
    // One elected lane runs the whole loop (waits included): no re-election / reconvergence per k block, the loop state
    // stays in uniform registers, and (term, k block) advance without a division.
    if (elect_one()) {
      int s = 0, term = 0, kb = kb0;
      uint32_t ph = 0;
      for (int it = 0; it < niter; ++it) {
        const CUtensorMap* amap = &pr.a_map[pr.ta[term]];
        const CUtensorMap* bmap = &pr.b_map[pr.tb[term]];
        uint8_t* sA = smem + s * STAGE_BYTES;
        uint8_t* sB = sA + A_TILE_BYTES;
        mbar_wait(&empty_bar[s], ph ^ 1u);
        mbar_expect_tx(&full_bar[s], STAGE_BYTES);
        if (A_MN == 0) {
          if (pr.a_layers)
            tma_load_2d(sA, &P.layer_maps[pr.a_layer_begin + min(ka_layer, pr.a_layers - 1)], &full_bar[s],
                        ka_layer < pr.a_layers ? ka_col : pr.layer_cols, m0);
          else
            tma_load_2d(sA, amap, &full_bar[s], kb * BK, m0);
        } else {
#pragma unroll
          for (int c = 0; c < BM / 64; ++c)
            tma_load_2d(sA + c * CHUNK_BYTES, a_chunk_map[c] ? a_chunk_map[c] : amap, &full_bar[s], a_chunk_col[c], kb * BK);
        }
        if (B_MN == 0) {
          if (pr.b_layers)
            tma_load_2d(sB, &P.layer_maps[pr.b_layer_begin + min(kb_layer, pr.b_layers - 1)], &full_bar[s],
                        kb_layer < pr.b_layers ? kb_col : pr.layer_cols, n0);
          else
            tma_load_2d(sB, bmap, &full_bar[s], kb * BK, n0);
        } else {
#pragma unroll
          for (int c = 0; c < BN / 64; ++c)
            tma_load_2d(sB + c * CHUNK_BYTES, b_chunk_map[c] ? b_chunk_map[c] : bmap, &full_bar[s], b_chunk_col[c], kb * BK);
        }
        // layered operands take one term: every iteration is a new k block
        if (!A_MN && pr.a_layers && (ka_col += BK) >= pr.layer_cols) {
          ka_col -= pr.layer_cols;
          ++ka_layer;
        }
        if (!B_MN && pr.b_layers && (kb_col += BK) >= pr.layer_cols) {
          kb_col -= pr.layer_cols;
          ++kb_layer;
        }
        if (++term == pr.nterms) {
          term = 0;
          ++kb;
        }
        if (++s == STAGES) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer: one elected lane runs the whole loop =====================
    // (see decode_scores_mma2_kernel: a warp-converged loop that re-elects a lane and rebuilds the descriptors every k
    // block costs ~300 clk of issue per block; the descriptors advance by 64-bit adds on the start-address field,
    // 16-byte units, no carry below 256 KiB)
    constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, A_MN, B_MN);
    constexpr uint64_t kStageStep = STAGE_BYTES >> 4;
    constexpr uint64_t kAStep = (A_MN ? 2048 : 32) >> 4, kBStep = (B_MN ? 2048 : 32) >> 4;
    if (elect_one()) {
      const uint32_t a_base0 = smem_u32(smem);
      const uint64_t a_desc0 = A_MN ? umma_desc_sw128(a_base0, CHUNK_BYTES, 1024) : umma_desc_sw128(a_base0, 16, 1024);
      const uint64_t b_desc0 = B_MN ? umma_desc_sw128(a_base0 + A_TILE_BYTES, CHUNK_BYTES, 1024)
                                    : umma_desc_sw128(a_base0 + A_TILE_BYTES, 16, 1024);
      uint64_t a_desc = a_desc0, b_desc = b_desc0;
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      for (int phs = 0; phs < nph; ++phs) {
        const uint32_t acc = tmem_base + static_cast<uint32_t>(phs & 1) * TMEM_COLS;
        if (phs >= 2) {   // the epilogue must have drained this accumulator (phase phs - 2)
          mbar_wait(&tmem_empty_bar[phs & 1], static_cast<uint32_t>(((phs >> 1) - 1) & 1));
          tc_fence_after();
        }
        const int it_end = (nph == 1) ? niter : static_cast<int>((static_cast<long long>(nk) * (phs + 1)) / nph) * pr.nterms;
        const int it_begin = it;
        for (; it < it_end; ++it) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          umma_bf16_ss(acc, a_desc, b_desc, idesc, it > it_begin ? 1u : 0u);
          umma_bf16_ss(acc, a_desc + kAStep, b_desc + kBStep, idesc, 1u);
          umma_bf16_ss(acc, a_desc + 2 * kAStep, b_desc + 2 * kBStep, idesc, 1u);
          umma_bf16_ss(acc, a_desc + 3 * kAStep, b_desc + 3 * kBStep, idesc, 1u);
          umma_commit(&empty_bar[s]);  // frees the smem stage once these MMAs have read it
          a_desc += kStageStep;
          b_desc += kStageStep;
          if (++s == STAGES) {
            s = 0;
            ph ^= 1u;
            a_desc = a_desc0;
            b_desc = b_desc0;
          }
        }
        umma_commit(&tmem_full_bar[phs & 1]);  // this phase's accumulator is complete
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue (warps 2..5) =====================
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int row = m0 + q * 32 + lane;
    const bool row_ok = row < pr.M;
    float* outf = reinterpret_cast<float*>(pr.D) + static_cast<long long>(split) * pr.split_stride;
    __nv_bfloat16* outh = reinterpret_cast<__nv_bfloat16*>(pr.D) + static_cast<long long>(split) * pr.split_stride;
    const bool vec_ok = (pr.ldd % 8 == 0) && ((reinterpret_cast<uintptr_t>(pr.D) & 15) == 0) &&
                        ((pr.split_stride % 8) == 0);
#pragma unroll 1
    for (int phs = 0; phs < nph; ++phs) {
    // Later phases add into what this same thread stored one phase ago (phases > 1 implies plain fp32 output).  Those
    // partial sums are fetched one column block ahead, the first block before the accumulator is even complete, so the
    // L2 round trips overlap the MMAs / the arithmetic of the block before.
    float4 pre[8];
    auto prefetch = [&](int c) -> bool {
      const int col0 = n0 + c * 32;
      if (!(phs > 0 && row_ok && vec_ok && c < BN / 32 && col0 + 32 <= pr.N)) return false;
      const float4* src = reinterpret_cast<const float4*>(outf + static_cast<long long>(row) * pr.ldd + col0);
#pragma unroll
      for (int j = 0; j < 8; ++j) pre[j] = src[j];
      return true;
    };
    bool have_pre = prefetch(0);
    mbar_wait(&tmem_full_bar[phs & 1], static_cast<uint32_t>((phs >> 1) & 1));
    tc_fence_after();
    const uint32_t acc = tmem_base + static_cast<uint32_t>(phs & 1) * TMEM_COLS;
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      const int col0 = n0 + c * 32;
      if (col0 >= pr.N) break;  // warp-uniform
      uint32_t v[32];
      __syncwarp();
      if (niter > 0) {
        tmem_ld_32x32(acc + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(c * 32), v);
        float4 cur[8];
        const bool have_cur = have_pre;
#pragma unroll
        for (int j = 0; j < 8; ++j) cur[j] = pre[j];
        have_pre = prefetch(c + 1);
        tmem_ld_wait();
        if (have_cur) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + cur[j].x);
            v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + cur[j].y);
            v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + cur[j].z);
            v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + cur[j].w);
          }
        } else if (phs > 0 && row_ok) {
          const float* src = outf + static_cast<long long>(row) * pr.ldd + col0;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (col0 + j < pr.N) v[j] = __float_as_uint(__uint_as_float(v[j]) + src[j]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0u;
      }
      const bool full = (col0 + 32 <= pr.N);
      if (!pr.out_transposed) {
        if (!row_ok) {
          // rows past M (zero-filled by TMA): nothing to store
        } else if (!pr.out_bf16) {
          float* dst = outf + static_cast<long long>(row) * pr.ldd + col0;
          if (full && vec_ok) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              reinterpret_cast<uint4*>(dst)[j] = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < pr.N) dst[j] = __uint_as_float(v[j]);
          }
        } else {
          __nv_bfloat16* dst = outh + static_cast<long long>(row) * pr.ldd + col0;
          if (full && vec_ok) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 w;
              w.x = pack_bf16x2(__uint_as_float(v[8 * j + 0]), __uint_as_float(v[8 * j + 1]));
              w.y = pack_bf16x2(__uint_as_float(v[8 * j + 2]), __uint_as_float(v[8 * j + 3]));
              w.z = pack_bf16x2(__uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
              w.w = pack_bf16x2(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7]));
              reinterpret_cast<uint4*>(dst)[j] = w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < pr.N) dst[j] = __float2bfloat16_rn(__uint_as_float(v[j]));
          }
        }
      } else {
        // transposed store: for a fixed column the warp's 32 rows are contiguous in memory
        if (!pr.out_bf16) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (row_ok && col0 + j < pr.N)
              outf[static_cast<long long>(col0 + j) * pr.ldd + row] = __uint_as_float(v[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (row_ok && col0 + j < pr.N)
              outh[static_cast<long long>(col0 + j) * pr.ldd + row] = __float2bfloat16_rn(__uint_as_float(v[j]));
        }
      }
    }
    if (phs + 2 < nph) {   // hand the accumulator back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty_bar[phs & 1]);
    }
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
// The same products in CTA PAIRS (cta_group::2, the two SMs of a TPC): a 256 x bn output tile per pair, bn <= 256.
// CTA r of the pair streams ITS 128 rows of A and HALF of the tile's B rows (bn / 2), the even CTA issues one M = 256,
// N = bn tcgen05.mma per K = 16 slice and each CTA receives its 128 rows x bn columns of the tile in its own tensor
// memory.  Why: the single-CTA 128 x 256 tile pulls 48 KiB from L2 per k block (96 B/clk per SM at the MMA rate, and
// 12 KiB of shared-memory operand reads per MMA); the pair pulls <= 32 KiB per CTA (64 B/clk, 8 KiB per MMA) for the same
// flops -- on a power-capped part less operand traffic is a higher tensor clock -- and has room for 6 ring stages
// instead of 4.  Measured on the Gram of the bench step (8 matrices 65536 x 4096, same box): 7.7 -> 6.25 ms.
// A runtime tile width lets the products with a narrow N (the sketch width l = 576 / 832 as N = 3 x 192 / 4 x 208)
// run without padding.  Used for launches whose M is large enough not to pay for the 256-row granularity (pair_bn):
// the Gram, the projection A = X V, and -- with the operand roles swapped by the factorisation driver, output stored
// transposed -- the power step G Q^T and the triangular solve.  MN-major B operands need bn = 256 (64-column chunks).
// Everything else is gemm_kernel: limb terms, layered operands read in place, split-K slabs, accumulation phases.
// Barriers: full[s] lives in the even CTA (both CTAs' loads complete on it); empty[s] and tmem_full[2] exist in each
// CTA and are signalled by multicast commits; tmem_empty[2] lives in the even CTA and counts the epilogue warps of both.
// ---------------------------------------------------------------------------------------------
constexpr int PG_BM = 256;                              // pair tile rows (128 per CTA)
constexpr int PG_STAGES = 6;                            // ring depth (5 / 6 / 7 measured equal, 4 slower: DESIGN.md)
constexpr int PG_MAX_STAGES = 7;
constexpr int PG_A_BYTES = BM * BK * 2;                 // this CTA's 128 rows of A
constexpr int PG_B_BYTES = (BN / 2) * BK * 2;           // this CTA's half of the tile's B rows (bn / 2 <= 128)
constexpr int PG_STAGE_BYTES = PG_A_BYTES + PG_B_BYTES; // 32 KiB
constexpr size_t pg_smem_bytes(int stages) { return static_cast<size_t>(stages) * PG_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/; }

template <int A_MN, int B_MN>
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_pair_kernel(const __grid_constant__ GemmParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + P.pair_stages * PG_STAGE_BYTES);   // behind the launch's ring
  uint64_t* empty_bar = full_bar + PG_MAX_STAGES;
  uint64_t* tmem_full_bar = empty_bar + PG_MAX_STAGES;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;          // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int crank = static_cast<int>(cluster_ctarank());
  const bool leader = crank == 0;

  // ---- locate this pair's problem / split / tile (cta_begin counts CTAs: two per pair tile) ----
  int pi = 0;
  while (pi + 1 < P.nprob && static_cast<int>(blockIdx.x) >= P.p[pi + 1].cta_begin) ++pi;
  const GemmProb& pr = P.p[pi];
  if (pr.run_if != nullptr && *pr.run_if == 0) return;   // uniform over the pair, before any barrier / TMEM allocation
  const int bn = pr.bn;
  const int nstages = pr.pstages;
  const int na = pr.na;
  const uint32_t stage_bytes = static_cast<uint32_t>(pr.na + pr.nb) * PG_A_BYTES;
  const int local = (static_cast<int>(blockIdx.x) - pr.cta_begin) >> 1;
  const int split = local / pr.ntiles;
  int t = local - split * pr.ntiles;
  int tm = 0, tn = 0;
  if (pr.sym_upper) {   // bn = 256: square pair tiles
    for (int i = 0; i < pr.tiles_m; ++i) {
      const int cnt = pr.tiles_n - i;
      if (t < cnt) {
        tm = i;
        tn = i + t;
        break;
      }
      t -= cnt;
    }
  } else {
    tm = t / pr.tiles_n;
    tn = t - tm * pr.tiles_n;
  }
  const int m0 = tm * PG_BM + crank * BM;   // this CTA's rows of the tile
  const int n0 = tn * bn;                   // the tile's columns (all bn land in this CTA's tensor memory)
  const int nb0 = n0 + crank * (bn >> 1);   // the B rows this CTA loads
  const int n_end = min(pr.N, n0 + bn);
  const int kb0 = split * pr.kblocks_per_split;
  const int kb1 = min(kb0 + pr.kblocks_per_split, pr.nkb);
  const int nk = max(kb1 - kb0, 0);
  const int niter = nk * pr.nterms;
  const int nph = max(1, min(pr.phases, nk));
  const uint32_t tmem_cols = nph > 1 ? 2 * TMEM_COLS : TMEM_COLS;
  const uint32_t b_bytes = B_MN ? static_cast<uint32_t>(PG_B_BYTES) : static_cast<uint32_t>(bn >> 1) * (BK * 2);

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < nstages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(&tmem_full_bar[0], 1);
    mbar_init(&tmem_full_bar[1], 1);
    mbar_init(&tmem_empty_bar[0], 8);   // one arrival per epilogue warp of BOTH CTAs
    mbar_init(&tmem_empty_bar[1], 8);
    mbar_fence_init();
    tma_prefetch_desc(&pr.a_map[pr.ta[0]]);
    tma_prefetch_desc(&pr.b_map[pr.tb[0]]);
  }
  if (warp == 1) tmem_alloc_pair(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's loads, commits and arrivals target this CTA's barriers: all initialised first
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (in each CTA; completions are counted on the even CTA's barrier) =====================
    // MN-major operands: two 64-column chunks per CTA, the layer matrix of a chunk is fixed for the whole kernel
    const CUtensorMap* a_chunk_map[2];
    const CUtensorMap* b_chunk_map[2];
    int a_chunk_col[2], b_chunk_col[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      a_chunk_col[c] = m0 + 64 * c;
      a_chunk_map[c] = (A_MN && pr.a_layers) ? layer_map(P, pr.a_layer_begin, pr.a_layers, pr.layer_cols, m0 + 64 * c, a_chunk_col[c]) : nullptr;
      b_chunk_col[c] = nb0 + 64 * c;
      b_chunk_map[c] = (B_MN && pr.b_layers) ? layer_map(P, pr.b_layer_begin, pr.b_layers, pr.layer_cols, nb0 + 64 * c, b_chunk_col[c]) : nullptr;
    }
    // K-major layered operand: (layer, column inside the layer) of the current k block, advanced incrementally
    int ka_layer = 0, ka_col = 0, kb_layer = 0, kb_col = 0;
    if (!A_MN && pr.a_layers) {
      ka_layer = (kb0 * BK) / pr.layer_cols;
      ka_col = kb0 * BK - ka_layer * pr.layer_cols;
    }
    if (!B_MN && pr.b_layers) {
      kb_layer = (kb0 * BK) / pr.layer_cols;
      kb_col = kb0 * BK - kb_layer * pr.layer_cols;
    }
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      const uint32_t full0 = cluster_map_shared(smem_u32(&full_bar[0]), 0);
      const uint32_t tx = 2u * (static_cast<uint32_t>(pr.na) * PG_A_BYTES + static_cast<uint32_t>(pr.nb) * b_bytes);
      for (int kb = kb0; kb < kb1; ++kb) {
        uint8_t* sA = smem + s * stage_bytes;
        uint8_t* sB = sA + na * PG_A_BYTES;
        mbar_wait(&empty_bar[s], ph ^ 1u);
        if (leader) mbar_expect_tx(&full_bar[s], tx);
        const uint32_t fb = full0 + static_cast<uint32_t>(s * 8);
        for (int i = 0; i < pr.na; ++i) {   // every distinct A limb of this k block, once
          const CUtensorMap* amap = &pr.a_map[pr.la[i]];
          uint8_t* dst = sA + i * PG_A_BYTES;
          if (A_MN == 0) {
            if (pr.a_layers)
              tma_load_2d_pair(dst, &P.layer_maps[pr.a_layer_begin + min(ka_layer, pr.a_layers - 1)], fb,
                               ka_layer < pr.a_layers ? ka_col : pr.layer_cols, m0);
            else
              tma_load_2d_pair(dst, amap, fb, kb * BK, m0);
          } else {
#pragma unroll
            for (int c = 0; c < 2; ++c)
              tma_load_2d_pair(dst + c * CHUNK_BYTES, a_chunk_map[c] ? a_chunk_map[c] : amap, fb, a_chunk_col[c], kb * BK);
          }
        }
        for (int i = 0; i < pr.nb; ++i) {
          const CUtensorMap* bmap = &pr.b_map[pr.lb[i]];
          uint8_t* dst = sB + i * PG_B_BYTES;
          if (B_MN == 0) {
            if (pr.b_layers)
              tma_load_2d_pair(dst, &P.layer_maps[pr.b_layer_begin + min(kb_layer, pr.b_layers - 1)], fb,
                               kb_layer < pr.b_layers ? kb_col : pr.layer_cols, nb0);
            else
              tma_load_2d_pair(dst, bmap, fb, kb * BK, nb0);
          } else {
#pragma unroll
            for (int c = 0; c < 2; ++c)
              tma_load_2d_pair(dst + c * CHUNK_BYTES, b_chunk_map[c] ? b_chunk_map[c] : bmap, fb, b_chunk_col[c], kb * BK);
          }
        }
        // layered operands take one term: one tile per k block
        if (!A_MN && pr.a_layers && (ka_col += BK) >= pr.layer_cols) {
          ka_col -= pr.layer_cols;
          ++ka_layer;
        }
        if (!B_MN && pr.b_layers && (kb_col += BK) >= pr.layer_cols) {
          kb_col -= pr.layer_cols;
          ++kb_layer;
        }
        if (++s == nstages) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer: one elected lane of the even CTA =====================
    if (leader) {
      const uint32_t idesc = umma_idesc_bf16(PG_BM, 0, A_MN, B_MN) | (static_cast<uint32_t>(bn >> 3) << 17);
      constexpr uint64_t kAStep = (A_MN ? 2048 : 32) >> 4, kBStep = (B_MN ? 2048 : 32) >> 4;
      constexpr uint64_t kSlot = PG_A_BYTES >> 4;   // one limb slot (A and B slots are the same size)
      if (elect_one()) {
        const uint64_t kStageStep = stage_bytes >> 4;
        const uint32_t base = smem_u32(smem);
        const uint64_t a_desc0 = A_MN ? umma_desc_sw128(base, CHUNK_BYTES, 1024) : umma_desc_sw128(base, 16, 1024);
        const uint64_t b_desc0 = B_MN ? umma_desc_sw128(base + na * PG_A_BYTES, CHUNK_BYTES, 1024)
                                      : umma_desc_sw128(base + na * PG_A_BYTES, 16, 1024);
        uint64_t a_desc = a_desc0, b_desc = b_desc0;
        int s = 0;
        uint32_t ph = 0;
        int kb = 0;   // k blocks done
        for (int phs = 0; phs < nph; ++phs) {
          const uint32_t acc = tmem_base + static_cast<uint32_t>(phs & 1) * TMEM_COLS;
          if (phs >= 2) {   // the epilogues of both CTAs must have drained this accumulator (phase phs - 2)
            mbar_wait_cluster(&tmem_empty_bar[phs & 1], static_cast<uint32_t>(((phs >> 1) - 1) & 1));
            tc_fence_after();
          }
          const int kb_end = (nph == 1) ? nk : static_cast<int>((static_cast<long long>(nk) * (phs + 1)) / nph);
          const int kb_begin = kb;
          for (; kb < kb_end; ++kb) {
            mbar_wait_cluster(&full_bar[s], ph);
            tc_fence_after();
            for (int t = 0; t < pr.nterms; ++t) {   // the terms of this k block in order, each from its limbs' slots
              const uint64_t ad = a_desc + kSlot * pr.sa[pr.ta[t]];
              const uint64_t bd = b_desc + kSlot * pr.sb[pr.tb[t]];
              umma_bf16_ss_pair(acc, ad, bd, idesc, (kb > kb_begin || t > 0) ? 1u : 0u);
              umma_bf16_ss_pair(acc, ad + kAStep, bd + kBStep, idesc, 1u);
              umma_bf16_ss_pair(acc, ad + 2 * kAStep, bd + 2 * kBStep, idesc, 1u);
              umma_bf16_ss_pair(acc, ad + 3 * kAStep, bd + 3 * kBStep, idesc, 1u);
            }
            umma_commit_pair(&empty_bar[s]);   // frees the stage in BOTH CTAs once these MMAs have read it
            a_desc += kStageStep;
            b_desc += kStageStep;
            if (++s == nstages) {
              s = 0;
              ph ^= 1u;
              a_desc = a_desc0;
              b_desc = b_desc0;
            }
          }
          umma_commit_pair(&tmem_full_bar[phs & 1]);   // this phase's accumulator is complete (both CTAs' halves)
        }
      }
      __syncwarp();
    }
  } else {
    // ===================== epilogue (warps 2..5 of each CTA, on its own 128 rows) =====================
    const int q = warp & 3;
    const int row = m0 + q * 32 + lane;
    const bool row_ok = row < pr.M;
    float* outf = reinterpret_cast<float*>(pr.D) + static_cast<long long>(split) * pr.split_stride;
    __nv_bfloat16* outh = reinterpret_cast<__nv_bfloat16*>(pr.D) + static_cast<long long>(split) * pr.split_stride;
    const bool vec_ok = (pr.ldd % 8 == 0) && ((reinterpret_cast<uintptr_t>(pr.D) & 15) == 0) && ((pr.split_stride % 8) == 0);
    const uint32_t tempty0 = cluster_map_shared(smem_u32(&tmem_empty_bar[0]), 0);
    const int ncb = (bn + 31) >> 5;   // 32-column blocks of the tile (the last one may be half used: bn % 16 == 0)
#pragma unroll 1
    for (int phs = 0; phs < nph; ++phs) {
      // later phases add into what this same thread stored one phase ago (phases > 1 implies plain fp32 output); the
      // partial sums are fetched one column block ahead, the first one before the accumulator is complete
      float4 pre[8];
      auto prefetch = [&](int c) -> bool {
        const int col0 = n0 + c * 32;
        if (!(phs > 0 && row_ok && vec_ok && c < ncb && col0 + 32 <= n_end)) return false;
        const float4* src = reinterpret_cast<const float4*>(outf + static_cast<long long>(row) * pr.ldd + col0);
#pragma unroll
        for (int j = 0; j < 8; ++j) pre[j] = src[j];
        return true;
      };
      bool have_pre = prefetch(0);
      mbar_wait(&tmem_full_bar[phs & 1], static_cast<uint32_t>((phs >> 1) & 1));
      tc_fence_after();
      const uint32_t acc = tmem_base + static_cast<uint32_t>(phs & 1) * TMEM_COLS;
#pragma unroll 1
      for (int c = 0; c < ncb; ++c) {
        const int col0 = n0 + c * 32;
        if (col0 >= n_end) break;  // warp-uniform
        uint32_t v[32];
        __syncwarp();
        if (niter > 0) {
          tmem_ld_32x32(acc + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(c * 32), v);
          float4 cur[8];
          const bool have_cur = have_pre;
#pragma unroll
          for (int j = 0; j < 8; ++j) cur[j] = pre[j];
          have_pre = prefetch(c + 1);
          tmem_ld_wait();
          if (have_cur) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + cur[j].x);
              v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + cur[j].y);
              v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + cur[j].z);
              v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + cur[j].w);
            }
          } else if (phs > 0 && row_ok) {
            const float* src = outf + static_cast<long long>(row) * pr.ldd + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < n_end) v[j] = __float_as_uint(__uint_as_float(v[j]) + src[j]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        const bool full = (col0 + 32 <= n_end);
        if (!pr.out_transposed) {
          if (!row_ok) {
            // rows past M (zero-filled by TMA): nothing to store
          } else if (!pr.out_bf16) {
            float* dst = outf + static_cast<long long>(row) * pr.ldd + col0;
            if (full && vec_ok) {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                reinterpret_cast<uint4*>(dst)[j] = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < n_end) dst[j] = __uint_as_float(v[j]);
            }
          } else {
            __nv_bfloat16* dst = outh + static_cast<long long>(row) * pr.ldd + col0;
            if (full && vec_ok) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                uint4 w;
                w.x = pack_bf16x2(__uint_as_float(v[8 * j + 0]), __uint_as_float(v[8 * j + 1]));
                w.y = pack_bf16x2(__uint_as_float(v[8 * j + 2]), __uint_as_float(v[8 * j + 3]));
                w.z = pack_bf16x2(__uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
                w.w = pack_bf16x2(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7]));
                reinterpret_cast<uint4*>(dst)[j] = w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < n_end) dst[j] = __float2bfloat16_rn(__uint_as_float(v[j]));
            }
          }
        } else {
          // transposed store: for a fixed column the warp's 32 rows are contiguous in memory
          if (!pr.out_bf16) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (row_ok && col0 + j < n_end)
                outf[static_cast<long long>(col0 + j) * pr.ldd + row] = __uint_as_float(v[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (row_ok && col0 + j < n_end)
                outh[static_cast<long long>(col0 + j) * pr.ldd + row] = __float2bfloat16_rn(__uint_as_float(v[j]));
          }
        }
      }
      if (phs + 2 < nph) {   // hand the accumulator back to the issuer (in the even CTA)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty0 + static_cast<uint32_t>((phs & 1) * 8));
      }
    }
  }

  // ---- teardown: nobody leaves (or frees tensor memory) while the pair's MMAs, commits or arrivals are pending ----
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static bool g_gram_pair = true;   // xkv_gemm_set_gram_pair

// N tile of the problem in the pair kernel, 0 = the problem stays on single-CTA tiles.  Pairs are used where the 256-row
// tile granularity costs nothing (M large, a multiple of 256, or its last 256 rows more than half used) and the operand
// layouts allow it: the symmetric tile set only in the Gram form (square 256 x 256 tiles), an MN-major B in 64-column
// chunks (bn = 256), a K-major B at any multiple of 16: N is cut into the fewest tiles of at most 256 columns, equally wide.
static int pair_bn(const xkv_gemm_problem& p) {
  if (!g_gram_pair) return 0;
  const int rem = p.M % PG_BM;
  if (!(p.M >= 2048 || rem == 0 || rem > BM)) return 0;
  if (p.sym_upper) return (p.a_mn_major && p.b_mn_major && p.M == p.N) ? BN : 0;
  if (p.b_mn_major) return BN;
  const int ntn = (p.N + BN - 1) / BN;
  const int w = (p.N + ntn - 1) / ntn;
  return (w + 15) & ~15;
}

static int build_problem(const xkv_gemm_problem& in, GemmProb& out, int& cta_cursor, GemmParams& params, int& map_cursor,
                         int pair_n = 0) {
  const bool pair = pair_n > 0;
  const int bn = pair ? pair_n : BN;   // N tile; the pair kernel loads bn / 2 B rows per CTA
  XKV_REQUIRE(in.M > 0 && in.N > 0 && in.K > 0, "gemm: empty problem M=%d N=%d K=%d", in.M, in.N, in.K);
  XKV_REQUIRE(in.num_terms >= 1 && in.num_terms <= 6, "gemm: num_terms=%d out of range", in.num_terms);
  XKV_REQUIRE(in.lda % 8 == 0 && in.ldb % 8 == 0, "gemm: lda/ldb must be multiples of 8 elements");
  XKV_REQUIRE(in.split_k >= 1, "gemm: split_k must be >= 1");
  XKV_REQUIRE(in.D != nullptr, "gemm: null output");
  std::memset(&out, 0, sizeof(out));
  bool used_a[3] = {false, false, false}, used_b[3] = {false, false, false};
  for (int t = 0; t < in.num_terms; ++t) {
    XKV_REQUIRE(in.term_a[t] < 3 && in.term_b[t] < 3, "gemm: limb index out of range");
    used_a[in.term_a[t]] = true;
    used_b[in.term_b[t]] = true;
    out.ta[t] = in.term_a[t];
    out.tb[t] = in.term_b[t];
  }
  // layered operands: one tensor map per layer matrix in the launch's pool; the limb slots alias the first layer
  XKV_REQUIRE(in.a_layers >= 0 && in.a_layers <= XKV_MAX_GROUP_LAYERS && in.b_layers >= 0 && in.b_layers <= XKV_MAX_GROUP_LAYERS,
              "gemm: at most %d layers per operand", XKV_MAX_GROUP_LAYERS);
  if (in.a_layers > 0 || in.b_layers > 0) {
    XKV_REQUIRE(in.num_terms == 1, "gemm: layered operands take one term");
    XKV_REQUIRE(in.layer_cols > 0 && in.layer_cols % 64 == 0, "gemm: layer_cols=%d must be a positive multiple of 64", in.layer_cols);
  }
  for (int side = 0; side < 2; ++side) {
    const int layers = side == 0 ? in.a_layers : in.b_layers;
    if (layers == 0) continue;
    const void* const* ptrs = side == 0 ? in.A_layer : in.B_layer;
    const bool mn = side == 0 ? in.a_mn_major != 0 : in.b_mn_major != 0;
    const long long ld = side == 0 ? in.lda : in.ldb;
    const int other = side == 0 ? in.M : in.N;   // extent of the operand's M / N dimension
    if (side == 1 && in.a_layers == in.b_layers && in.a_mn_major && in.b_mn_major && in.lda == in.ldb &&
        std::memcmp(in.A_layer, in.B_layer, sizeof(void*) * layers) == 0) {
      out.b_layer_begin = out.a_layer_begin;   // X^T X: both operands are the same layer matrices, same boxes
      continue;
    }
    (side == 0 ? out.a_layer_begin : out.b_layer_begin) = map_cursor;
    for (int i = 0; i < layers; ++i) {
      XKV_REQUIRE(ptrs[i] != nullptr && (reinterpret_cast<uintptr_t>(ptrs[i]) & 15) == 0, "gemm: layer %d null or unaligned", i);
      XKV_REQUIRE(map_cursor < XKV_MAX_LAYER_MAPS, "gemm: more than %d layer matrices in one launch", XKV_MAX_LAYER_MAPS);
      int rc;
      if (!mn)   // K-major: rows = M (or N) index, the layer supplies layer_cols of the K columns
        rc = encode_tmap_2d_bf16(&params.layer_maps[map_cursor++], ptrs[i], in.layer_cols, other, ld, BK,
                                 side == 0 ? BM : (pair ? bn / 2 : BN));
      else       // MN-major: rows = K index, the layer supplies layer_cols of the M (or N) columns
        rc = encode_tmap_2d_bf16(&params.layer_maps[map_cursor++], ptrs[i], in.layer_cols, in.K, ld, 64, BK);
      if (rc) return rc;
    }
  }
  out.a_layers = in.a_layers;
  out.b_layers = in.b_layers;
  out.layer_cols = in.layer_cols;
  XKV_REQUIRE(in.a_layers == 0 || (in.a_mn_major ? in.M : in.K) <= in.a_layers * in.layer_cols, "gemm: layered A narrower than the problem");
  XKV_REQUIRE(in.b_layers == 0 || (in.b_mn_major ? in.N : in.K) <= in.b_layers * in.layer_cols, "gemm: layered B narrower than the problem");
  for (int i = 0; i < 3; ++i) {
    // unused limbs alias limb 0 so every tensor map in parameter space is valid to prefetch
    const void* a = in.a_layers > 0 ? in.A_layer[0] : (used_a[i] ? in.A[i] : in.A[in.term_a[0]]);
    const void* b = in.b_layers > 0 ? in.B_layer[0] : (used_b[i] ? in.B[i] : in.B[in.term_b[0]]);
    XKV_REQUIRE(a != nullptr && b != nullptr, "gemm: null operand limb %d", i);
    XKV_REQUIRE((reinterpret_cast<uintptr_t>(a) & 15) == 0 && (reinterpret_cast<uintptr_t>(b) & 15) == 0,
                "gemm: operands must be 16-byte aligned");
    int rc = 0;
    if (in.a_layers > 0)
      out.a_map[i] = params.layer_maps[out.a_layer_begin];   // valid to prefetch; the loads go through the layer maps
    else if (!in.a_mn_major)
      rc = encode_tmap_2d_bf16(&out.a_map[i], a, in.K, in.M, in.lda, BK, BM);
    else
      rc = encode_tmap_2d_bf16(&out.a_map[i], a, in.M, in.K, in.lda, 64, BK);
    if (rc) return rc;
    if (in.b_layers > 0)
      out.b_map[i] = params.layer_maps[out.b_layer_begin];
    else if (!in.b_mn_major)
      rc = encode_tmap_2d_bf16(&out.b_map[i], b, in.K, in.N, in.ldb, BK, pair ? bn / 2 : BN);
    else
      rc = encode_tmap_2d_bf16(&out.b_map[i], b, in.N, in.K, in.ldb, 64, BK);
    if (rc) return rc;
  }
  out.D = in.D;
  out.ldd = in.ldd;
  out.split_stride = in.split_stride;
  out.M = in.M;
  out.N = in.N;
  out.K = in.K;
  out.nterms = in.num_terms;
  const int bm = pair ? PG_BM : BM;   // the pair kernel's tile is 256 x bn, two CTAs
  out.bn = bn;
  out.tiles_m = (in.M + bm - 1) / bm;
  out.tiles_n = (in.N + bn - 1) / bn;
  out.sym_upper = in.sym_upper ? 1 : 0;
  if (out.sym_upper) {
    int cnt = 0;
    for (int i = 0; i < out.tiles_m; ++i) cnt += out.tiles_n - (i * bm) / bn;
    out.ntiles = cnt;
  } else {
    out.ntiles = out.tiles_m * out.tiles_n;
  }
  for (int i = 0; i < 3; ++i) {   // distinct limbs in slot order (pair kernel)
    if (used_a[i]) {
      out.sa[i] = static_cast<unsigned char>(out.na);
      out.la[out.na++] = static_cast<unsigned char>(i);
    }
    if (used_b[i]) {
      out.sb[i] = static_cast<unsigned char>(out.nb);
      out.lb[out.nb++] = static_cast<unsigned char>(i);
    }
  }
  out.nkb = (in.K + BK - 1) / BK;
  out.split_k = in.split_k;
  out.kblocks_per_split = (out.nkb + in.split_k - 1) / in.split_k;
  out.out_bf16 = in.out_bf16 ? 1 : 0;
  out.out_transposed = in.out_transposed ? 1 : 0;
  out.run_if = in.run_if;
  out.phases = in.accum_phases > 1 ? in.accum_phases : 1;
  XKV_REQUIRE(out.phases == 1 || (!in.out_bf16 && !in.out_transposed),
              "gemm: accum_phases > 1 needs a plain fp32 output");
  out.cta_begin = cta_cursor;
  cta_cursor += out.ntiles * out.split_k * (pair ? 2 : 1);
  return 0;
}

bool& gemm_low_priority() {
  static thread_local bool low = false;
  return low;
}

template <int A_MN, int B_MN>
static int launch_pair_variant(GemmParams& params, int grid, cudaStream_t stream) {
  auto kern = gemm_pair_kernel<A_MN, B_MN>;
  static PerDevice<bool> configured;  // per instantiation and device
  if (!configured()) {
    XKV_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(pg_smem_bytes(PG_MAX_STAGES))));
    configured() = true;
  }
  params.pair_stages = PG_STAGES;
  for (int i = 0; i < params.nprob; ++i) {   // each problem cuts the launch's ring into stages of its own size
    const int stage = (params.p[i].na + params.p[i].nb) * PG_A_BYTES;
    const int st = params.pair_stages * PG_STAGE_BYTES / stage;
    params.p[i].pstages = st > PG_MAX_STAGES ? PG_MAX_STAGES : st;
  }
  cudaLaunchConfig_t cfg;
  std::memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid, 1, 1);
  cfg.blockDim = dim3(GEMM_THREADS, 1, 1);
  cfg.dynamicSmemBytes = pg_smem_bytes(params.pair_stages);
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.numAttrs = 1;
  if (gemm_low_priority()) {
    attr[1].id = cudaLaunchAttributePriority;
    attr[1].val.priority = 0;
    cfg.numAttrs = 2;
  }
  cfg.attrs = attr;
  XKV_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, params));
  XKV_LAUNCHED();
  return 0;
}

template <int A_MN, int B_MN>
static int launch_variant(const GemmParams& params, int grid, cudaStream_t stream) {
  auto kern = gemm_kernel<A_MN, B_MN>;
  static PerDevice<bool> configured;  // per instantiation and device
  if (!configured()) {
    XKV_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(GEMM_SMEM_BYTES)));
    configured() = true;
  }
  if (gemm_low_priority()) {   // see xkv_host.h: the projection yields freed SMs to the other chains' small kernels
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(GEMM_THREADS, 1, 1);
    cfg.dynamicSmemBytes = GEMM_SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributePriority;
    attr[0].val.priority = 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    XKV_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, params));
  } else {
    kern<<<grid, GEMM_THREADS, GEMM_SMEM_BYTES, stream>>>(params);
  }
  XKV_LAUNCHED();
  return 0;
}

}  // namespace xkv

extern "C" size_t xkv_gemm_problem_size(void) { return sizeof(xkv_gemm_problem); }
extern "C" void xkv_gemm_set_gram_pair(int on) { xkv::g_gram_pair = on != 0; }

extern "C" int xkv_gemm_grouped(const xkv_gemm_problem* problems, int num_problems, void* stream) {
  using namespace xkv;
  XKV_REQUIRE(problems != nullptr && num_problems >= 1, "gemm: no problems");
  XKV_REQUIRE(num_problems <= XKV_MAX_GEMM_PROBLEMS, "gemm: at most %d problems per launch", XKV_MAX_GEMM_PROBLEMS);
  const int a_mn = problems[0].a_mn_major ? 1 : 0;
  const int b_mn = problems[0].b_mn_major ? 1 : 0;
  static thread_local GemmParams params;  // ~22 KiB, keep it off the stack
  params.nprob = num_problems;
  int cursor = 0, map_cursor = 0;
  bool pair = true;   // one kernel per launch: pairs only when every problem qualifies
  for (int i = 0; i < num_problems; ++i) pair = pair && pair_bn(problems[i]) > 0;
  for (int i = 0; i < num_problems; ++i) {
    XKV_REQUIRE((problems[i].a_mn_major ? 1 : 0) == a_mn && (problems[i].b_mn_major ? 1 : 0) == b_mn,
                "gemm: all problems of one launch must share operand majors");
    int rc = build_problem(problems[i], params.p[i], cursor, params, map_cursor, pair ? pair_bn(problems[i]) : 0);
    if (rc) return rc;
  }
  cudaStream_t st = as_stream(stream);
  if (pair) {
    if (!a_mn && !b_mn) return launch_pair_variant<0, 0>(params, cursor, st);
    if (!a_mn && b_mn) return launch_pair_variant<0, 1>(params, cursor, st);
    if (a_mn && !b_mn) return launch_pair_variant<1, 0>(params, cursor, st);
    return launch_pair_variant<1, 1>(params, cursor, st);
  }
  if (!a_mn && !b_mn) return launch_variant<0, 0>(params, cursor, st);
  if (!a_mn && b_mn) return launch_variant<0, 1>(params, cursor, st);
  if (a_mn && !b_mn) return launch_variant<1, 0>(params, cursor, st);
  return launch_variant<1, 1>(params, cursor, st);
}
