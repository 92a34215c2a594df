// xkv_b200 — decode-time attention over the factored cache (north-star step 3).
//
// The reference stores dense K^ = bf16(U_r S_r V_r^T) (fake_layer_merge_dynamic_cache.py:26-27,176),
// applies RoPE to it (:142-148) and runs SDPA with GQA over [K^ ; decode tokens] (llama.py:51-69).
// Here the factors stay factored:
//
//   scores   K^ tile = A_k[128 tokens, r_k] * Bk_l^T is formed by tcgen05.mma in TMEM, rounded to bf16,
//            rotated (RoPE in the reference's bf16 arithmetic) and contracted with q in the epilogue;
//            only the (Hq x S) fp32 scores go to HBM, the full-rank keys never do.
//   softmax  one pass per q-head: max, exp, row sum; probabilities written once as bf16.
//   values   absorbed form  o = ((P A_v) Bv_l^T) / rowsum : P A_v is a tensor-core GEMM over the token
//            dimension (xkv_gemm.cu, split-K), Bv_l is applied to the (Hq x r_v) result; no V^ tile is
//            ever formed.
//   tail     decode tokens appended after prefill stay dense and exact (reference: mode='decode' skips
//            merging, cache:131); their scores / values join the same softmax.
#include <cooperative_groups.h>

#include "xkv_common.cuh"
#include "xkv_host.h"

namespace cg = cooperative_groups;

namespace xkv {

constexpr int DBM = 128;  // tokens per tile
constexpr int DBN = 256;  // K^ columns per tile (256 / head_dim kv heads)
constexpr int DBK = 64;
constexpr int DSTAGES = 2;  // 2 x 48 KiB stages -> two CTAs per SM: one CTA's epilogue overlaps the other's MMA
constexpr int D_A_BYTES = DBM * DBK * 2;
constexpr int D_B_BYTES = DBN * DBK * 2;
constexpr int D_STAGE_BYTES = D_A_BYTES + D_B_BYTES;
constexpr int D_THREADS = 192;
constexpr int D_TMEM_COLS = 256;
constexpr int D_MAX_QPK = 8;  // q heads per kv head
constexpr size_t D_SMEM_BYTES = DSTAGES * D_STAGE_BYTES + 1024 + 256 + DBN * D_MAX_QPK * sizeof(float);

struct alignas(64) ScoreParams {
  CUtensorMap a_map;  // A_k  (S x r_k), box {64, 128}
  CUtensorMap b_map;  // Bk_l (H*D x r_k), box {64, 256}
  CUtensorMap b_head_map;  // Bk_l, box {64, D}: one kv head (persistent kernel)
  CUtensorMap q_map;       // q (rows x D), box {64, 16}: the q rows of one pass of a kv head (score MMA)
  CUtensorMap b_half_map;  // Bk_l, box {64, 64}: half a kv head's dims (pair kernel)
  CUtensorMap q_half_map;  // q, box {64, nq16 / 2}: the q rows one CTA of a pair supplies to the score MMA
  const __nv_bfloat16* q;    // (rows, D): row r = hq * Tq + t, query token t of q head hq
  const __nv_bfloat16* cos;  // (S, D) or null
  const __nv_bfloat16* sin;
  float* scores;             // (rows, ld_scores)
  long long ld_cs, ld_scores;
  // qpk: q rows per kv head (q heads per kv head x query tokens), contiguous from h * qpk.  The kernels other than the
  // pair kernel take at most D_MAX_QPK of them per CTA: kv head h is worked in npass passes of <= 8 rows (pass_rows).
  int S, rk, H, qpk, tiles_n, nkb, npass;
  int stages;   // ring slots of the score-MMA kernel
  float scale;
};

__device__ __forceinline__ float bf16r(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// first q row and row count of pass p of kv head h (npass == 1, the single-token case: rows h * qpk, qpk of them)
__device__ __forceinline__ int pass_row0(const ScoreParams& P, int h, int p) { return h * P.qpk + p * D_MAX_QPK; }
__device__ __forceinline__ int pass_rows(const ScoreParams& P, int p) { return min(D_MAX_QPK, P.qpk - p * D_MAX_QPK); }

template <int D>
__global__ void __launch_bounds__(D_THREADS, 2) decode_scores_kernel(const __grid_constant__ ScoreParams P) {
  constexpr int HPT = DBN / D;        // kv heads per tile
  constexpr int NCH = D / 32;         // 32-column chunks per head
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + DSTAGES * D_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + DSTAGES;
  uint64_t* tmem_full_bar = empty_bar + DSTAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
  float* q_s = reinterpret_cast<float*>(smem + DSTAGES * D_STAGE_BYTES + 256);  // [HPT * qpk][D]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tm = blockIdx.x / P.tiles_n, tn = blockIdx.x - tm * P.tiles_n;
  const int m0 = tm * DBM, n0 = tn * DBN;
  const int h0 = n0 / D;  // first kv head of this tile
  const int pass = blockIdx.y, nrow = pass_rows(P, pass);

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < DSTAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(tmem_full_bar, 1);
    mbar_fence_init();
    tma_prefetch_desc(&P.a_map);
    tma_prefetch_desc(&P.b_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, D_TMEM_COLS);
  if (warp >= 2) {
    // stage this tile's q rows of this pass as fp32: q_s[(hh * nrow + g) * D + d]
    const int nq = HPT * nrow * D;
    for (int e = threadIdx.x - 64; e < nq; e += 128) {
      const int d = e % D, hg = e / D;
      const int hh = hg / nrow, g = hg - hh * nrow;
      const int h = h0 + hh;
      q_s[e] = (h < P.H) ? __bfloat162float(P.q[static_cast<long long>(pass_row0(P, h, pass) + g) * D + d]) : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // warps 0 / 1: the whole warp runs the loop, one elected lane issues (see elect_one)
  if (warp == 0) {
    int s = 0;
    uint32_t ph = 0;
    for (int kb = 0; kb < P.nkb; ++kb) {
      uint8_t* sA = smem + s * D_STAGE_BYTES;
      mbar_wait(&empty_bar[s], ph ^ 1u);
      if (elect_one()) {
        mbar_expect_tx(&full_bar[s], D_STAGE_BYTES);
        tma_load_2d(sA, &P.a_map, &full_bar[s], kb * DBK, m0);
        tma_load_2d(sA + D_A_BYTES, &P.b_map, &full_bar[s], kb * DBK, n0);
      }
      __syncwarp();
      if (++s == DSTAGES) {
        s = 0;
        ph ^= 1u;
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16(DBM, DBN, 0, 0);
    int s = 0;
    uint32_t ph = 0;
    for (int kb = 0; kb < P.nkb; ++kb) {
      mbar_wait(&full_bar[s], ph);
      tc_fence_after();
      const uint32_t a_base = smem_u32(smem + s * D_STAGE_BYTES);
      const uint32_t b_base = a_base + D_A_BYTES;
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < DBK / 16; ++k)
          umma_bf16_ss(tmem_base, umma_desc_sw128(a_base + k * 32, 16, 1024), umma_desc_sw128(b_base + k * 32, 16, 1024),
                       idesc, (kb > 0 || k > 0) ? 1u : 0u);
        umma_commit(&empty_bar[s]);
      }
      __syncwarp();
      if (++s == DSTAGES) {
        s = 0;
        ph ^= 1u;
      }
    }
    if (elect_one()) umma_commit(tmem_full_bar);
    __syncwarp();
  } else {
    // ============ epilogue: K^ row (this thread's token) -> bf16 -> RoPE -> dot with the q heads ============
    const int qd = warp & 3;
    const int tok = m0 + qd * 32 + lane;
    const bool tok_ok = tok < P.S;
    const bool rope = P.cos != nullptr;
    float acc[HPT][D_MAX_QPK];
#pragma unroll
    for (int hh = 0; hh < HPT; ++hh)
#pragma unroll
      for (int g = 0; g < D_MAX_QPK; ++g) acc[hh][g] = 0.f;
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16);
#pragma unroll 1
    for (int c = 0; c < NCH / 2; ++c) {
      // cos/sin of dims [32c, 32c+32) (identical for the partner dims +D/2 in the half-split convention)
      uint32_t cs[16], sn[16];
      if (rope && tok_ok) {
        const uint4* cp = reinterpret_cast<const uint4*>(P.cos + static_cast<long long>(tok) * P.ld_cs + c * 32);
        const uint4* sp = reinterpret_cast<const uint4*>(P.sin + static_cast<long long>(tok) * P.ld_cs + c * 32);
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const uint4 cv = cp[v], sv = sp[v];
          cs[4 * v] = cv.x, cs[4 * v + 1] = cv.y, cs[4 * v + 2] = cv.z, cs[4 * v + 3] = cv.w;
          sn[4 * v] = sv.x, sn[4 * v + 1] = sv.y, sn[4 * v + 2] = sv.z, sn[4 * v + 3] = sv.w;
        }
      } else {
#pragma unroll
        for (int v = 0; v < 16; ++v) cs[v] = 0x3F803F80u, sn[v] = 0u;  // cos = 1, sin = 0
      }
#pragma unroll
      for (int hh = 0; hh < HPT; ++hh) {
        uint32_t x1[32], x2[32];
        __syncwarp();
        tmem_ld_32x32(lane_addr + static_cast<uint32_t>(hh * D + c * 32), x1);
        tmem_ld_32x32(lane_addr + static_cast<uint32_t>(hh * D + (c + NCH / 2) * 32), x2);
        tmem_ld_wait();
        const float* qh = q_s + (hh * nrow) * D;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float k1 = bf16r(__uint_as_float(x1[j]));
          const float k2 = bf16r(__uint_as_float(x2[j]));
          float o1 = k1, o2 = k2;
          if (rope) {
            const uint32_t cw = cs[j >> 1], sw = sn[j >> 1];
            const float cf = __uint_as_float((j & 1) ? (cw & 0xFFFF0000u) : (cw << 16));
            const float sf = __uint_as_float((j & 1) ? (sw & 0xFFFF0000u) : (sw << 16));
            // HF apply_rotary_pos_emb in bf16: k*cos + rotate_half(k)*sin, every op rounded to bf16
            o1 = bf16r(bf16r(k1 * cf) + bf16r(-k2 * sf));
            o2 = bf16r(bf16r(k2 * cf) + bf16r(k1 * sf));
          }
          const int d1 = c * 32 + j, d2 = d1 + D / 2;
#pragma unroll
          for (int g = 0; g < D_MAX_QPK; ++g)
            if (g < nrow) acc[hh][g] = fmaf(qh[g * D + d1], o1, fmaf(qh[g * D + d2], o2, acc[hh][g]));
        }
      }
    }
    if (tok_ok) {
#pragma unroll
      for (int hh = 0; hh < HPT; ++hh) {
        const int h = h0 + hh;
        if (h < P.H) {
#pragma unroll
          for (int g = 0; g < D_MAX_QPK; ++g)
            if (g < nrow) P.scores[static_cast<long long>(pass_row0(P, h, pass) + g) * P.ld_scores + tok] = acc[hh][g] * P.scale;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, D_TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------
// Persistent variant: one CTA per SM owns ONE kv head, keeps that head's slice of the right factor
// (D x r_k bf16, <= 128 KiB) resident in shared memory for the whole launch and streams A_k token tiles
// through a 4-stage TMA ring.  Four TMEM accumulators (4 x D columns) let the MMAs run up to three tiles ahead of
// the epilogue.  Compared with the tile-per-CTA kernel above it never re-reads the right factor
// (L2 -> SM traffic per layer 786 MB -> 536 MB at config 2) and has no per-tile prologue.
// ---------------------------------------------------------------------------------------------
constexpr int PA_STAGES = 4;
constexpr int P_EPI_WARPS = 16;                   // four warps per TMEM lane quarter: each takes a quarter of the dims
constexpr int P_PARTS = P_EPI_WARPS / 4;
constexpr int P_NACC = 4;                         // TMEM accumulators (4 x 128 columns = all of TMEM at head_dim 128)
constexpr int P_THREADS = 64 + 32 * P_EPI_WARPS;  // TMA warp + MMA warp + epilogue warps
constexpr int PB_MAX_BYTES = 128 * 1024;
constexpr size_t P_SMEM_BYTES = PB_MAX_BYTES + PA_STAGES * D_A_BYTES + 1024 + 256 + 128 * D_MAX_QPK * sizeof(float) +
                                (P_PARTS - 1) * 2 * DBM * D_MAX_QPK * sizeof(float);

template <int D>
__global__ void __launch_bounds__(P_THREADS, 1) decode_scores_persistent_kernel(const __grid_constant__ ScoreParams P) {
  constexpr int B_KB_BYTES = D * DBK * 2;  // one 64-wide K block of the head's right factor
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sB = smem;
  uint8_t* sA = smem + PB_MAX_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sA + PA_STAGES * D_A_BYTES);
  uint64_t* empty_bar = full_bar + PA_STAGES;
  uint64_t* tfull_bar = empty_bar + PA_STAGES;   // [P_NACC]
  uint64_t* tempty_bar = tfull_bar + P_NACC;     // [P_NACC]
  uint64_t* b_bar = tempty_bar + P_NACC;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_bar + 1);
  float* q_s = reinterpret_cast<float*>(sA + PA_STAGES * D_A_BYTES + 256);  // [D][8]: q heads of this kv head, dim-major
  float* part = q_s + 128 * D_MAX_QPK;                                      // [2][128 tokens][8] partial scores

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // CTA -> (kv head h, pass) of one of the H * npass row sets, and the token tiles slot, slot + nslots, ...
  const int nv = P.H * P.npass;
  const int vh = blockIdx.x % nv;
  const int h = vh / P.npass, pass = vh - h * P.npass;
  const int row0 = pass_row0(P, h, pass), nrow = pass_rows(P, pass);
  const int slot = blockIdx.x / nv;
  const int nslots = (gridDim.x - vh + nv - 1) / nv;   // CTAs that share this row set
  const int ntiles = (P.S + DBM - 1) / DBM;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < PA_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < P_NACC; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], P_EPI_WARPS);   // one arrive per epilogue warp
    }
    mbar_init(b_bar, 1);
    mbar_fence_init();
    tma_prefetch_desc(&P.a_map);
    tma_prefetch_desc(&P.b_head_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, P_NACC * D);
  if (warp >= 2) {
    for (int e = threadIdx.x - 64; e < D * D_MAX_QPK; e += 32 * P_EPI_WARPS) {
      const int d = e / D_MAX_QPK, g = e - d * D_MAX_QPK;
      q_s[e] = g < nrow ? __bfloat162float(P.q[static_cast<long long>(row0 + g) * D + d]) : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(b_bar, static_cast<uint32_t>(P.nkb) * B_KB_BYTES);
      for (int kb = 0; kb < P.nkb; ++kb) tma_load_2d(sB + kb * B_KB_BYTES, &P.b_head_map, b_bar, kb * DBK, h * D);
    }
    __syncwarp();
    if (elect_one()) {   // one lane runs the whole loop (see decode_scores_mma2_kernel)
      int s = 0;
      uint32_t ph = 0;
      for (int tile = slot; tile < ntiles; tile += nslots) {
        for (int kb = 0; kb < P.nkb; ++kb) {
          mbar_wait(&empty_bar[s], ph ^ 1u);
          mbar_expect_tx(&full_bar[s], D_A_BYTES);
          tma_load_2d(sA + s * D_A_BYTES, &P.a_map, &full_bar[s], kb * DBK, tile * DBM);
          if (++s == PA_STAGES) {
            s = 0;
            ph ^= 1u;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16(DBM, D, 0, 0);
    constexpr uint64_t kKStep = 32 >> 4, kStageStep = D_A_BYTES >> 4, kBlockStep = B_KB_BYTES >> 4;
    mbar_wait(b_bar, 0);
    if (elect_one()) {   // one lane issues everything, descriptors advance by 64-bit adds (see decode_scores_mma2_kernel)
      const uint64_t a_desc0 = umma_desc_sw128(smem_u32(sA), 16, 1024);
      const uint64_t b_desc0 = umma_desc_sw128(smem_u32(sB), 16, 1024);
      uint64_t a_desc = a_desc0;
      int s = 0, acc = 0;
      uint32_t ph = 0, acc_ph = 0u;   // acc_ph: one phase bit per accumulator
      for (int tile = slot; tile < ntiles; tile += nslots) {
        mbar_wait(&tempty_bar[acc], ((acc_ph >> acc) & 1u) ^ 1u);   // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_addr = tmem_base + static_cast<uint32_t>(acc * D);
        uint64_t b_desc = b_desc0;
        for (int kb = 0; kb < P.nkb; ++kb) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          umma_bf16_ss(d_addr, a_desc, b_desc, idesc, kb > 0 ? 1u : 0u);
          umma_bf16_ss(d_addr, a_desc + kKStep, b_desc + kKStep, idesc, 1u);
          umma_bf16_ss(d_addr, a_desc + 2 * kKStep, b_desc + 2 * kKStep, idesc, 1u);
          umma_bf16_ss(d_addr, a_desc + 3 * kKStep, b_desc + 3 * kKStep, idesc, 1u);
          umma_commit(&empty_bar[s]);
          b_desc += kBlockStep;
          a_desc += kStageStep;
          if (++s == PA_STAGES) {
            s = 0;
            ph ^= 1u;
            a_desc = a_desc0;
          }
        }
        umma_commit(&tfull_bar[acc]);
        acc_ph ^= 1u << acc;
        acc = (acc + 1) % P_NACC;
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue: 16 warps, four per TMEM lane quarter; each thread owns one token and PP rotation pairs
    // (d, d + D/2) of it.  ncu on the 8-warp version: the epilogue, not the MMA or the TMA ring, set the pace
    // (two warps per scheduler cannot hide the LDS / convert / FMA dependency chains), hence more, lighter warps,
    // packed FFMA2 for the q dot products, and the cos/sin words fetched one tile ahead. =====
    constexpr int PP = D / 2 / P_PARTS;   // rotation pairs per thread: 16 (D = 128) or 8 (D = 64)
    constexpr int CW = PP / 2;            // packed bf16x2 words of cos (and of sin) per thread
    const int ew = warp - 2;
    const int qd = warp & 3;              // TMEM lane quarter (hardware: warp id mod 4)
    const int prt = ew >> 2;              // which quarter of the rotation pairs
    const int row = qd * 32 + lane;       // token row inside the tile
    const int d0 = prt * PP;              // first dim of the low half; partners are d0 + D/2 ...
    const bool rope = P.cos != nullptr;
    int acc = 0, pb = 0;            // accumulator in use; parity of the partial-score buffer
    uint32_t acc_ph = 0u;
    uint32_t cs_next[CW], sn_next[CW];
    auto fetch_cs = [&](int tile_idx) {
      const int t = tile_idx * DBM + row;
      if (rope && tile_idx < ntiles && t < P.S) {
        const uint4* cp = reinterpret_cast<const uint4*>(P.cos + static_cast<long long>(t) * P.ld_cs + d0);
        const uint4* sp = reinterpret_cast<const uint4*>(P.sin + static_cast<long long>(t) * P.ld_cs + d0);
#pragma unroll
        for (int v = 0; v < CW / 4; ++v) {
          const uint4 cv = __ldg(cp + v), sv = __ldg(sp + v);
          cs_next[4 * v] = cv.x, cs_next[4 * v + 1] = cv.y, cs_next[4 * v + 2] = cv.z, cs_next[4 * v + 3] = cv.w;
          sn_next[4 * v] = sv.x, sn_next[4 * v + 1] = sv.y, sn_next[4 * v + 2] = sv.z, sn_next[4 * v + 3] = sv.w;
        }
      } else {
#pragma unroll
        for (int v = 0; v < CW; ++v) cs_next[v] = 0x3F803F80u, sn_next[v] = 0u;   // cos = 1, sin = 0
      }
    };
    fetch_cs(slot);
    for (int tile = slot; tile < ntiles; tile += nslots) {
      const int tok = tile * DBM + row;
      const bool tok_ok = tok < P.S;
      float2 sc01 = make_float2(0.f, 0.f), sc23 = sc01, sc45 = sc01, sc67 = sc01;
      uint32_t cs[CW], sn[CW];
#pragma unroll
      for (int v = 0; v < CW; ++v) cs[v] = cs_next[v], sn[v] = sn_next[v];
      fetch_cs(tile + nslots);
      mbar_wait(&tfull_bar[acc], (acc_ph >> acc) & 1u);
      acc_ph ^= 1u << acc;
      tc_fence_after();
      const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + static_cast<uint32_t>(acc * D);
      uint32_t x1[PP], x2[PP];
      __syncwarp();
      tmem_ld_cols<PP>(lane_addr + static_cast<uint32_t>(d0), x1);
      tmem_ld_cols<PP>(lane_addr + static_cast<uint32_t>(D / 2 + d0), x2);
      tmem_ld_wait();
      // accumulator columns of this thread are in registers: hand the buffer back to the MMA warp right away
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
#pragma unroll
      for (int jp = 0; jp < PP / 2; ++jp) {
        // two dims at a time in packed bf16: the reference's RoPE is bf16 arithmetic (each product and the sum
        // rounded to bf16), which is exactly what HMUL2.BF16 / HADD2.BF16 compute
        const __nv_bfloat162 k1 = __floats2bfloat162_rn(__uint_as_float(x1[2 * jp]), __uint_as_float(x1[2 * jp + 1]));
        const __nv_bfloat162 k2 = __floats2bfloat162_rn(__uint_as_float(x2[2 * jp]), __uint_as_float(x2[2 * jp + 1]));
        __nv_bfloat162 o1 = k1, o2 = k2;
        if (rope) {
          const __nv_bfloat162 cw = *reinterpret_cast<const __nv_bfloat162*>(&cs[jp]);
          const __nv_bfloat162 sw = *reinterpret_cast<const __nv_bfloat162*>(&sn[jp]);
          o1 = __hadd2(__hmul2(k1, cw), __hmul2(__hneg2(k2), sw));
          o2 = __hadd2(__hmul2(k2, cw), __hmul2(k1, sw));
        }
        const float o1v[2] = {__low2float(o1), __high2float(o1)};
        const float o2v[2] = {__low2float(o2), __high2float(o2)};
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int d1 = d0 + 2 * jp + u, d2 = d1 + D / 2;
          const float2 a = make_float2(o1v[u], o1v[u]), b = make_float2(o2v[u], o2v[u]);
          const float4 qa = *reinterpret_cast<const float4*>(q_s + d1 * D_MAX_QPK);
          const float4 qb = *reinterpret_cast<const float4*>(q_s + d2 * D_MAX_QPK);
          sc01 = __ffma2_rn(make_float2(qa.x, qa.y), a, __ffma2_rn(make_float2(qb.x, qb.y), b, sc01));
          sc23 = __ffma2_rn(make_float2(qa.z, qa.w), a, __ffma2_rn(make_float2(qb.z, qb.w), b, sc23));
          if (nrow > 4) {
            const float4 qc = *reinterpret_cast<const float4*>(q_s + d1 * D_MAX_QPK + 4);
            const float4 qe = *reinterpret_cast<const float4*>(q_s + d2 * D_MAX_QPK + 4);
            sc45 = __ffma2_rn(make_float2(qc.x, qc.y), a, __ffma2_rn(make_float2(qe.x, qe.y), b, sc45));
            sc67 = __ffma2_rn(make_float2(qc.z, qc.w), a, __ffma2_rn(make_float2(qe.z, qe.w), b, sc67));
          }
        }
      }
      const float sc[D_MAX_QPK] = {sc01.x, sc01.y, sc23.x, sc23.y, sc45.x, sc45.y, sc67.x, sc67.y};
      // combine the partial scores of the four dim quarters through shared memory (double-buffered by accumulator)
      if (prt > 0) {
        float* pt = part + (((prt - 1) * 2 + pb) * DBM + row) * D_MAX_QPK;
        *reinterpret_cast<float4*>(pt) = make_float4(sc[0], sc[1], sc[2], sc[3]);
        if (nrow > 4) *reinterpret_cast<float4*>(pt + 4) = make_float4(sc[4], sc[5], sc[6], sc[7]);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * P_EPI_WARPS) : "memory");   // epilogue warps only
      if (prt == 0 && tok_ok) {
        float tot[D_MAX_QPK];
#pragma unroll
        for (int g = 0; g < D_MAX_QPK; ++g) tot[g] = sc[g];
#pragma unroll
        for (int o = 0; o < P_PARTS - 1; ++o) {
          const float* pt = part + ((o * 2 + pb) * DBM + row) * D_MAX_QPK;
          const float4 lo4 = *reinterpret_cast<const float4*>(pt);
          tot[0] += lo4.x, tot[1] += lo4.y, tot[2] += lo4.z, tot[3] += lo4.w;
          if (nrow > 4) {
            const float4 hi4 = *reinterpret_cast<const float4*>(pt + 4);
            tot[4] += hi4.x, tot[5] += hi4.y, tot[6] += hi4.z, tot[7] += hi4.w;
          }
        }
#pragma unroll
        for (int g = 0; g < D_MAX_QPK; ++g)
          if (g < nrow) P.scores[static_cast<long long>(row0 + g) * P.ld_scores + tok] = tot[g] * P.scale;
      }
      acc = (acc + 1) % P_NACC;
      pb ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, P_NACC * D);
  }
}

// ---------------------------------------------------------------------------------------------
// Persistent variant with the q contraction on the tensor core (head_dim 128, the default):
// the epilogue of the kernel above spends three quarters of its instructions on the q . k^ dot products
// (LDS of q, unpack to fp32, FFMA2, partial sums through shared memory), and the bisect in
// profiles/r01_decode_scores_ncu_full.md shows that those instructions, not the MMAs, set the pace.  Here the
// epilogue only rounds the reconstructed keys to bf16, rotates them (packed bf16, the reference's arithmetic) and
// writes them back to TENSOR MEMORY as packed bf16 (tcgen05.st: lane = token, column c = dims 2c, 2c+1); a second
// tcgen05.mma with the A operand in TMEM (TS form) contracts them with the head's q vectors (a 16 x 128 bf16 tile
// in shared memory, loaded once by TMA):  scores[128 tokens x 16] = K^rot[128 x 128] * Q^T.  Both products are
// exact bf16 x bf16 with fp32 accumulation, as before.  Warp roles: 0 TMA, 1 MMA (reconstruction), 2 MMA (scores),
// 4..11 epilogue (two per TMEM lane quarter: dims [0,32)+[64,96) and [32,64)+[96,128)), 12..15 score read-out.
//   TMEM: 2 x 128 columns reconstruction accumulators | 2 x 64 columns K^rot (bf16x2) | 2 x 32 columns scores.
//
// (A cluster form that shared every A_k tile between the kv heads' CTAs by TMA multicast was built in round 2, measured
// no faster -- 119 -> 120 / 129 / 140 us per layer at cluster size 2 / 4 / 8 -- and removed: profiles/r02_decode_scores_bisect.md.
// The default for head_dim 128 is the CTA-pair kernel below; this one remains for devices that cannot hold a pair.)
// ---------------------------------------------------------------------------------------------
constexpr int R_MAX_STAGES = 12;   // ring slots of 16 KiB: as many as fit beside the head's right-factor slice (5 at r_k = 512, 9 at 256)
constexpr int R_EPI_WARPS = 8;
constexpr int R_OUT_WARPS = 4;
constexpr int R_THREADS = 32 * (4 + R_EPI_WARPS + R_OUT_WARPS);
constexpr int R_QROWS = 16;                 // q rows of the score MMA (N = 16 >= q heads per kv head)
constexpr int R_Q_BYTES = 2 * R_QROWS * 128;  // two 64-dim chunks of 16 rows x 128 B
constexpr int R_TMEM_COLS = 512;
constexpr uint32_t R_COL_A2 = 256, R_COL_D2 = 384;
constexpr size_t R_SMEM_LIMIT = 227 * 1024;
constexpr size_t R_FIXED_BYTES = R_Q_BYTES + 1024 /*align*/ + 512 /*barriers*/;
// shared memory of the score-MMA kernel for a right factor of nkb 64-wide rank blocks: (B slice, ring stages, total bytes)
static inline int r_stages_for(int nkb) {
  const size_t b = static_cast<size_t>(nkb) * 128 * DBK * 2;
  int st = static_cast<int>((R_SMEM_LIMIT - R_FIXED_BYTES - b) / D_A_BYTES);
  return st > R_MAX_STAGES ? R_MAX_STAGES : st;
}

__global__ void __launch_bounds__(R_THREADS, 1) decode_scores_mma2_kernel(const __grid_constant__ ScoreParams P) {
  constexpr int D = 128;
  constexpr int B_KB_BYTES = D * DBK * 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int R_STAGES = P.stages;
  uint8_t* sB = smem;                              // nkb x 16 KiB: this head's right-factor slice
  uint8_t* sA = smem + P.nkb * B_KB_BYTES;
  uint8_t* sQ = sA + R_STAGES * D_A_BYTES;         // 1024-byte aligned (all sizes above are multiples of 1024)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sQ + R_Q_BYTES);
  uint64_t* empty_bar = full_bar + R_MAX_STAGES;
  uint64_t* tfull_bar = empty_bar + R_MAX_STAGES;  // [2] reconstruction accumulator ready
  uint64_t* tempty_bar = tfull_bar + 2;            // [2] ... drained by the epilogue warps
  uint64_t* a2full_bar = tempty_bar + 2;           // [2] rotated keys written to TMEM
  uint64_t* a2empty_bar = a2full_bar + 2;          // [2] ... consumed by the score MMAs
  uint64_t* d2full_bar = a2empty_bar + 2;          // [2] scores ready in TMEM
  uint64_t* d2empty_bar = d2full_bar + 2;          // [2] ... read out
  uint64_t* b_bar = d2empty_bar + 2;
  uint64_t* q_bar = b_bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(q_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // CTA `cid` works on kv head h and on the token tiles slot, slot + nslots, ...
  // (kv head, pass) as in decode_scores_persistent_kernel
  const int cid = static_cast<int>(blockIdx.x);
  const int ncta = static_cast<int>(gridDim.x);
  const int nv = P.H * P.npass;
  const int vh = cid % nv;
  const int h = vh / P.npass, pass = vh - h * P.npass;
  const int row0 = pass_row0(P, h, pass), nrow = pass_rows(P, pass);
  const int slot = cid / nv;
  const int nslots = (ncta - vh + nv - 1) / nv;
  const int ntiles = (P.S + DBM - 1) / DBM;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < R_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], R_EPI_WARPS);
      mbar_init(&a2full_bar[i], R_EPI_WARPS);
      mbar_init(&a2empty_bar[i], 1);
      mbar_init(&d2full_bar[i], 1);
      mbar_init(&d2empty_bar[i], R_OUT_WARPS);
    }
    mbar_init(b_bar, 1);
    mbar_init(q_bar, 1);
    mbar_fence_init();
    tma_prefetch_desc(&P.a_map);
    tma_prefetch_desc(&P.b_head_map);
    tma_prefetch_desc(&P.q_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, R_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // warps 0..2: the whole warp runs the loop (waits included), one elected lane issues -- see elect_one()
  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(q_bar, R_Q_BYTES);
      tma_load_2d(sQ, &P.q_map, q_bar, 0, row0);            // dims 0..63 of q rows [row0, row0 + 16)
      tma_load_2d(sQ + R_Q_BYTES / 2, &P.q_map, q_bar, 64, row0);
      mbar_expect_tx(b_bar, static_cast<uint32_t>(P.nkb) * B_KB_BYTES);
      for (int kb = 0; kb < P.nkb; ++kb) tma_load_2d(sB + kb * B_KB_BYTES, &P.b_head_map, b_bar, kb * DBK, h * D);
    }
    __syncwarp();
    if (elect_one()) {   // the whole producer loop in one lane (see the MMA warp)
      int s = 0;
      uint32_t ph = 0;
      for (int tile = slot; tile < ntiles; tile += nslots) {
        for (int kb = 0; kb < P.nkb; ++kb) {
          mbar_wait(&empty_bar[s], ph ^ 1u);
          mbar_expect_tx(&full_bar[s], D_A_BYTES);
          tma_load_2d(sA + s * D_A_BYTES, &P.a_map, &full_bar[s], kb * DBK, tile * DBM);
          if (++s == R_STAGES) {
            s = 0;
            ph ^= 1u;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // Reconstruction MMAs.  At N = 128 an M128 K16 instruction occupies the tensor pipe for 64 clk, so the issuing
    // thread has 256 clk per rank block for the barrier wait, four MMAs and the commit -- and a warp-converged loop
    // that re-elects a lane, rebuilds eight descriptors (~45 uniform-datapath instructions) and reconverges every rank
    // block does not fit in them: the kernel ran at ~100 clk per MMA, issue-bound (tools/probe_mma_rate.cu: 64.2 clk
    // with a bare loop, 82 with two integer modulos in it, 100 with a commit per block on top).  So ONE elected lane
    // runs the whole loop, and the descriptors advance by 64-bit adds (start address field in 16-byte units: +2 per
    // K = 16 step, + stage / block size per rank block; no carry out of the 14-bit field below 256 KiB).
    constexpr uint32_t idesc = umma_idesc_bf16(DBM, D, 0, 0);
    constexpr uint64_t kKStep = 32 >> 4, kStageStep = D_A_BYTES >> 4, kBlockStep = B_KB_BYTES >> 4;
    mbar_wait(b_bar, 0);
    if (elect_one()) {
      const uint64_t a_desc0 = umma_desc_sw128(smem_u32(sA), 16, 1024);
      const uint64_t b_desc0 = umma_desc_sw128(smem_u32(sB), 16, 1024);
      uint64_t a_desc = a_desc0;
      int s = 0, acc = 0;
      uint32_t ph = 0, acc_ph = 0u;
      for (int tile = slot; tile < ntiles; tile += nslots) {
        mbar_wait(&tempty_bar[acc], ((acc_ph >> acc) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_addr = tmem_base + static_cast<uint32_t>(acc * D);
        uint64_t b_desc = b_desc0;
        for (int kb = 0; kb < P.nkb; ++kb) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          umma_bf16_ss(d_addr, a_desc, b_desc, idesc, kb > 0 ? 1u : 0u);
          umma_bf16_ss(d_addr, a_desc + kKStep, b_desc + kKStep, idesc, 1u);
          umma_bf16_ss(d_addr, a_desc + 2 * kKStep, b_desc + 2 * kKStep, idesc, 1u);
          umma_bf16_ss(d_addr, a_desc + 3 * kKStep, b_desc + 3 * kKStep, idesc, 1u);
          umma_commit(&empty_bar[s]);
          b_desc += kBlockStep;
          a_desc += kStageStep;
          if (++s == R_STAGES) {
            s = 0;
            ph ^= 1u;
            a_desc = a_desc0;
          }
        }
        umma_commit(&tfull_bar[acc]);
        acc_ph ^= 1u << acc;
        acc ^= 1;
      }
    }
    __syncwarp();
  } else if (warp == 2) {
    // scores[128 x 16] = K^rot (TMEM, 64 packed columns) * Q^T (shared memory, K-major)
    constexpr uint32_t idesc2 = umma_idesc_bf16(DBM, R_QROWS, 0, 0);
    mbar_wait(q_bar, 0);
    const uint32_t q_base = smem_u32(sQ);
    if (elect_one()) {
      const uint64_t q_desc0 = umma_desc_sw128(q_base, 16, 1024);
      int b = 0;
      uint32_t bph = 0u;
      for (int tile = slot; tile < ntiles; tile += nslots) {
        mbar_wait(&a2full_bar[b], (bph >> b) & 1u);                 // rotated keys of this tile are in TMEM
        mbar_wait(&d2empty_bar[b], ((bph >> b) & 1u) ^ 1u);         // score buffer read out
        tc_fence_after();
        const uint32_t a2 = tmem_base + R_COL_A2 + static_cast<uint32_t>(b * 64);
        const uint32_t d2 = tmem_base + R_COL_D2 + static_cast<uint32_t>(b * 32);
#pragma unroll
        for (int k = 0; k < D / 16; ++k)
          umma_bf16_ts(d2, a2 + static_cast<uint32_t>(k * 8),
                       q_desc0 + static_cast<uint64_t>(((k >> 2) * (R_Q_BYTES / 2) + (k & 3) * 32) >> 4), idesc2, k > 0 ? 1u : 0u);
        umma_commit(&d2full_bar[b]);
        umma_commit(&a2empty_bar[b]);
        bph ^= 1u << b;
        b ^= 1;
      }
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 4 + R_EPI_WARPS) {
    // ===== epilogue: K^ row -> bf16 -> RoPE (packed bf16) -> back to TMEM as the A operand of the score MMA =====
    const int qd = warp & 3;
    const int half = (warp - 4) >> 2;
    const int row = qd * 32 + lane;
    const int d0 = half * 32;           // this thread rotates the pairs (d, d + 64), d in [d0, d0 + 32)
    const bool rope = P.cos != nullptr;
    int acc = 0;
    uint32_t acc_ph = 0u;
    for (int tile = slot; tile < ntiles; tile += nslots) {
      const int tok = tile * DBM + row;
      // cos/sin words of this token: issued before the wait on the accumulator, consumed after it
      uint32_t cs[16], sn[16];
      if (rope && tok < P.S) {
        const uint4* cp = reinterpret_cast<const uint4*>(P.cos + static_cast<long long>(tok) * P.ld_cs + d0);
        const uint4* sp = reinterpret_cast<const uint4*>(P.sin + static_cast<long long>(tok) * P.ld_cs + d0);
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const uint4 cv = __ldg(cp + v), sv = __ldg(sp + v);
          cs[4 * v] = cv.x, cs[4 * v + 1] = cv.y, cs[4 * v + 2] = cv.z, cs[4 * v + 3] = cv.w;
          sn[4 * v] = sv.x, sn[4 * v + 1] = sv.y, sn[4 * v + 2] = sv.z, sn[4 * v + 3] = sv.w;
        }
      } else {
#pragma unroll
        for (int v = 0; v < 16; ++v) cs[v] = 0x3F803F80u, sn[v] = 0u;   // cos = 1, sin = 0
      }
      mbar_wait(&tfull_bar[acc], (acc_ph >> acc) & 1u);
      tc_fence_after();
      const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(qd * 32) << 16);
      const uint32_t lane_addr = lane_base + static_cast<uint32_t>(acc * D);
      uint32_t lo_w[16], hi_w[16];      // packed bf16x2: dims d0 + 2j, d0 + 2j + 1 and their partners + 64
      {
        // read the accumulator, round to bf16 (the reference's cast of the reconstructed keys) and hand the buffer back
        // to the reconstruction MMAs BEFORE the rotation: the issue loop of the tile after next waits for this arrive
        uint32_t x1[32], x2[32];
        __syncwarp();
        tmem_ld_32x32(lane_addr + static_cast<uint32_t>(d0), x1);
        tmem_ld_32x32(lane_addr + static_cast<uint32_t>(D / 2 + d0), x2);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          lo_w[j] = pack_bf16x2(__uint_as_float(x1[2 * j]), __uint_as_float(x1[2 * j + 1]));
          hi_w[j] = pack_bf16x2(__uint_as_float(x2[2 * j]), __uint_as_float(x2[2 * j + 1]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (rope) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const __nv_bfloat162 k1 = *reinterpret_cast<const __nv_bfloat162*>(&lo_w[j]);
          const __nv_bfloat162 k2 = *reinterpret_cast<const __nv_bfloat162*>(&hi_w[j]);
          const __nv_bfloat162 cw = *reinterpret_cast<const __nv_bfloat162*>(&cs[j]);
          const __nv_bfloat162 sw = *reinterpret_cast<const __nv_bfloat162*>(&sn[j]);
          const __nv_bfloat162 o1 = __hadd2(__hmul2(k1, cw), __hmul2(__hneg2(k2), sw));
          const __nv_bfloat162 o2 = __hadd2(__hmul2(k2, cw), __hmul2(k1, sw));
          lo_w[j] = *reinterpret_cast<const uint32_t*>(&o1);
          hi_w[j] = *reinterpret_cast<const uint32_t*>(&o2);
        }
      }
      // K^rot -> TMEM (column c = dims 2c, 2c+1): wait until the score MMAs of two tiles ago released the buffer
      mbar_wait(&a2empty_bar[acc], ((acc_ph >> acc) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t a2 = lane_base + R_COL_A2 + static_cast<uint32_t>(acc * 64);
      __syncwarp();
      tmem_st_32x16(a2 + static_cast<uint32_t>(d0 / 2), lo_w);
      tmem_st_32x16(a2 + static_cast<uint32_t>(32 + d0 / 2), hi_w);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&a2full_bar[acc]);
      acc_ph ^= 1u << acc;
      acc ^= 1;
    }
  } else if (warp >= 4 + R_EPI_WARPS) {
    // ===== score read-out: one warp per TMEM lane quarter, thread = token =====
    const int qd = warp & 3;
    const int row = qd * 32 + lane;
    int b = 0;
    uint32_t bph = 0u;
    for (int tile = slot; tile < ntiles; tile += nslots) {
      const int tok = tile * DBM + row;
      mbar_wait(&d2full_bar[b], (bph >> b) & 1u);
      tc_fence_after();
      uint32_t v[8];
      __syncwarp();
      tmem_ld_32x8(tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + R_COL_D2 + static_cast<uint32_t>(b * 32), v);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&d2empty_bar[b]);
      if (tok < P.S) {
#pragma unroll
        for (int g = 0; g < D_MAX_QPK; ++g)
          if (g < nrow) P.scores[static_cast<long long>(row0 + g) * P.ld_scores + tok] = __uint_as_float(v[g]) * P.scale;
      }
      bph ^= 1u << b;
      b ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, R_TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------
// Pair form of the score-MMA kernel: a CTA PAIR (cta_group::2, the two SMs of a TPC) owns one kv head and works on 256
// tokens per step.  Each CTA streams ITS 128 tokens of A_k, keeps HALF of the head's right-factor slice (64 dims x
// r_k: 64 KiB at r_k = 512 instead of 128) and receives the K^ tile of its tokens (128 x 128, all dims of the head) in
// its own tensor memory: M = 256, N = 128 tcgen05.mma issued by the even CTA.  Why: with the whole slice resident only
// 5 ring slots of 16 KiB fit beside it, and the kernel's time followed the ring depth (2 / 3 / 4 / 5 slots: 114 / 77 /
// 66 / 61 us per layer): a slot is held from the TMA issue until the MMAs that read it RETIRE, so at most ~2-3 loads
// were in flight against an L2 round trip of ~0.6 us.  Half a slice leaves room for 9 slots (7 are used; 7 at r_k 768,
// 5 at 1024 -- ranks whose whole slice does not fit at all).  The epilogue is the single-CTA kernel's, run by both
// CTAs on their own tokens; the score MMA (M = 256, N = nq16: nq16 / 2 q rows from each CTA) is issued by the even CTA
// once BOTH epilogues have written their rotated keys (remote mbarrier arrivals), commits are multicast to both CTAs.
// Multi-token steps: the qpk = (q heads per kv head) x (query tokens) <= 64 rows of a kv head all go through ONE score MMA
// per tile, N = nq16 = qpk rounded up to 16; the 64 score columns of tensor memory hold 64 / nq16 buffers of nq16 columns
// (4 x 16 up to 16 rows: the single-token layout, 2 x 32, then 1 x 48 or 1 x 64).  The reconstruction, the epilogue and
// the 3 rotated-key buffers do not change with the row count.
// ---------------------------------------------------------------------------------------------
constexpr int PR_B_KB_BYTES = 64 * DBK * 2;        // one rank block of a half slice: 64 dims x 128 B
constexpr int PR_A2 = 3, PR_D2 = 4;         // rotated-key / score buffers in tensor memory (score buffers: at most 4)
constexpr uint32_t PR_COL_A2 = 256, PR_COL_D2 = 256 + PR_A2 * 64;   // 256 accumulator columns, then 3 x 64, then 64 score columns
constexpr int PR_SCORE_COLS = 64;
__host__ __device__ constexpr int pair_nq16(int qpk) { return (qpk + 15) & ~15; }
// q rows of one CTA (nq16 / 2), two 64-dim chunks of 128 B per row: 2 KiB up to 16 rows per kv head
__host__ __device__ constexpr int pair_q_bytes(int qpk) { return pair_nq16(qpk) * 128; }
static inline size_t pair_fixed_bytes(int qpk) { return pair_q_bytes(qpk) + 1024 /*align*/ + 512 /*barriers*/; }
static inline int pair_stages_for(int nkb, int qpk) {
  const size_t b = static_cast<size_t>(nkb) * PR_B_KB_BYTES;
  const size_t fixed = pair_fixed_bytes(qpk);
  if (b + fixed + 3 * D_A_BYTES > R_SMEM_LIMIT) return 0;
  int st = static_cast<int>((R_SMEM_LIMIT - fixed - b) / D_A_BYTES);
  // measured (config 2, one layer): 3 / 5 / 6 / 7 / 8 / 9 slots -> 75.6 / 53.8 / 49.9 / 49.5 / 51.4 / 53.0 us: past 7 the extra
  // loads in flight only add L2 contention
  return st > 7 ? 7 : st;
}

// NQ16: the score MMA's N = q rows per kv head rounded up to 16 (a template parameter so that the single-token form,
// NQ16 = 16, keeps its instruction descriptor, buffer ring and read-out as compile-time constants)
template <int NQ16>
__global__ void __launch_bounds__(R_THREADS, 1) decode_scores_pair_kernel(const __grid_constant__ ScoreParams P) {
  constexpr int D = 128;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int R_STAGES = P.stages;
  uint8_t* sB = smem;                              // nkb x 8 KiB: this CTA's half of the head's right-factor slice
  uint8_t* sA = smem + P.nkb * PR_B_KB_BYTES;
  uint8_t* sQ = sA + R_STAGES * D_A_BYTES;
  constexpr int nq16 = NQ16, q_bytes = NQ16 * 128;
  constexpr int nd2 = PR_SCORE_COLS / NQ16;        // score buffers
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sQ + q_bytes);   // used in the even CTA: both CTAs' loads land
  uint64_t* empty_bar = full_bar + R_MAX_STAGES;   // in each CTA: multicast commit
  uint64_t* tfull_bar = empty_bar + R_MAX_STAGES;  // [2] in each CTA: multicast commit
  uint64_t* tempty_bar = tfull_bar + 2;            // [2] even CTA: the epilogue warps of BOTH CTAs
  // Rotated-key and score buffers: 3 and 4 deep (tensor memory: 256 accumulator columns + 3 x 64 + 4 x 16 = 512).  The score
  // MMA of a tile queues BEHIND the reconstruction MMAs already issued (the pipe is in order), so with two buffers each the
  // recurrences  score MMA(t) -> read-out -> score MMA(t + 2)  and  score MMA(t) -> epilogue store(t + 2)  sat at the tile period.
  uint64_t* a2full_bar = tempty_bar + 2;           // [PR_A2] even CTA: both epilogues
  uint64_t* a2empty_bar = a2full_bar + PR_A2;      // [PR_A2] in each CTA: multicast commit
  uint64_t* d2full_bar = a2empty_bar + PR_A2;      // [PR_D2] in each CTA: multicast commit
  uint64_t* d2empty_bar = d2full_bar + PR_D2;      // [PR_D2] even CTA: both read-outs
  uint64_t* b_bar = d2empty_bar + PR_D2;           // even CTA: both half slices
  uint64_t* q_bar = b_bar + 1;                     // even CTA: both q halves
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(q_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int crank = static_cast<int>(cluster_ctarank());
  const bool leader = crank == 0;
  const int pid = static_cast<int>(blockIdx.x) >> 1;
  const int npairs = static_cast<int>(gridDim.x) >> 1;
  const int h = pid % P.H;
  const int slot = pid / P.H;
  const int nslots = (npairs - h + P.H - 1) / P.H;
  const int ntiles = (P.S + 2 * DBM - 1) / (2 * DBM);   // pair tiles of 256 tokens

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < R_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 2 * R_EPI_WARPS);
    }
    for (int i = 0; i < PR_A2; ++i) {
      mbar_init(&a2full_bar[i], 2 * R_EPI_WARPS);
      mbar_init(&a2empty_bar[i], 1);
    }
    for (int i = 0; i < PR_D2; ++i) {
      mbar_init(&d2full_bar[i], 1);
      mbar_init(&d2empty_bar[i], 2 * R_OUT_WARPS);
    }
    mbar_init(b_bar, 1);
    mbar_init(q_bar, 1);
    mbar_fence_init();
    tma_prefetch_desc(&P.a_map);
    tma_prefetch_desc(&P.b_half_map);
    tma_prefetch_desc(&P.q_half_map);
  }
  if (warp == 1) tmem_alloc_pair(tmem_slot, R_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's loads, commits and arrivals target this CTA's barriers: all initialised first
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      // both CTAs load their halves; every completion is counted on the even CTA's barriers
      const uint32_t qb = cluster_map_shared(smem_u32(q_bar), 0), bb = cluster_map_shared(smem_u32(b_bar), 0);
      if (leader) {
        mbar_expect_tx(q_bar, 2 * q_bytes);
        mbar_expect_tx(b_bar, 2u * static_cast<uint32_t>(P.nkb) * PR_B_KB_BYTES);
      }
      tma_load_2d_pair(sQ, &P.q_half_map, qb, 0, h * P.qpk + crank * (nq16 / 2));
      tma_load_2d_pair(sQ + q_bytes / 2, &P.q_half_map, qb, 64, h * P.qpk + crank * (nq16 / 2));
      for (int kb = 0; kb < P.nkb; ++kb)
        tma_load_2d_pair(sB + kb * PR_B_KB_BYTES, &P.b_half_map, bb, kb * DBK, h * D + crank * 64);
      int s = 0;
      uint32_t ph = 0;
      for (int tile = slot; tile < ntiles; tile += nslots) {
        for (int kb = 0; kb < P.nkb; ++kb) {
          mbar_wait(&empty_bar[s], ph ^ 1u);
          if (leader) mbar_expect_tx(&full_bar[s], 2 * D_A_BYTES);
          tma_load_2d_pair(sA + s * D_A_BYTES, &P.a_map, cluster_map_shared(smem_u32(&full_bar[s]), 0), kb * DBK,
                           (2 * tile + crank) * DBM);
          if (++s == R_STAGES) {
            s = 0;
            ph ^= 1u;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * DBM, D, 0, 0);
      constexpr uint64_t kKStep = 32 >> 4, kStageStep = D_A_BYTES >> 4, kBlockStep = PR_B_KB_BYTES >> 4;
      if (elect_one()) {
        mbar_wait_cluster(b_bar, 0);
        const uint64_t a_desc0 = umma_desc_sw128(smem_u32(sA), 16, 1024);
        const uint64_t b_desc0 = umma_desc_sw128(smem_u32(sB), 16, 1024);
        uint64_t a_desc = a_desc0;
        int s = 0, acc = 0;
        uint32_t ph = 0, acc_ph = 0u;
        for (int tile = slot; tile < ntiles; tile += nslots) {
          mbar_wait_cluster(&tempty_bar[acc], ((acc_ph >> acc) & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t d_addr = tmem_base + static_cast<uint32_t>(acc * D);
          uint64_t b_desc = b_desc0;
          for (int kb = 0; kb < P.nkb; ++kb) {
            mbar_wait_cluster(&full_bar[s], ph);
            tc_fence_after();
            umma_bf16_ss_pair(d_addr, a_desc, b_desc, idesc, kb > 0 ? 1u : 0u);
            umma_bf16_ss_pair(d_addr, a_desc + kKStep, b_desc + kKStep, idesc, 1u);
            umma_bf16_ss_pair(d_addr, a_desc + 2 * kKStep, b_desc + 2 * kKStep, idesc, 1u);
            umma_bf16_ss_pair(d_addr, a_desc + 3 * kKStep, b_desc + 3 * kKStep, idesc, 1u);
            umma_commit_pair(&empty_bar[s]);
            b_desc += kBlockStep;
            a_desc += kStageStep;
            if (++s == R_STAGES) {
              s = 0;
              ph ^= 1u;
              a_desc = a_desc0;
            }
          }
          umma_commit_pair(&tfull_bar[acc]);
          acc_ph ^= 1u << acc;
          acc ^= 1;
        }
      }
      __syncwarp();
    }
  } else if (warp == 2) {
    if (leader) {
      // scores[256 x nq16] = K^rot (each CTA's tensor memory) * Q^T (nq16 / 2 q rows from each CTA's shared memory)
      constexpr uint32_t idesc2 = umma_idesc_bf16(2 * DBM, nq16, 0, 0);
      if (elect_one()) {
        mbar_wait_cluster(q_bar, 0);
        const uint64_t q_desc0 = umma_desc_sw128(smem_u32(sQ), 16, 1024);
        int ba = 0, bd = 0;
        uint32_t pa = 0u, pd = 0u;   // phase bit per buffer
        for (int tile = slot; tile < ntiles; tile += nslots) {
          mbar_wait_cluster(&a2full_bar[ba], (pa >> ba) & 1u);
          mbar_wait_cluster(&d2empty_bar[bd], ((pd >> bd) & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t a2 = tmem_base + PR_COL_A2 + static_cast<uint32_t>(ba * 64);
          const uint32_t d2 = tmem_base + PR_COL_D2 + static_cast<uint32_t>(bd * nq16);
#pragma unroll
          for (int k = 0; k < D / 16; ++k)
            umma_bf16_ts_pair(d2, a2 + static_cast<uint32_t>(k * 8),
                              q_desc0 + static_cast<uint64_t>(((k >> 2) * (q_bytes / 2) + (k & 3) * 32) >> 4), idesc2,
                              k > 0 ? 1u : 0u);
          umma_commit_pair(&d2full_bar[bd]);
          umma_commit_pair(&a2empty_bar[ba]);
          pa ^= 1u << ba;
          pd ^= 1u << bd;
          ba = ba + 1 == PR_A2 ? 0 : ba + 1;
          bd = bd + 1 == nd2 ? 0 : bd + 1;
        }
      }
      __syncwarp();
    }
  } else if (warp >= 4 && warp < 4 + R_EPI_WARPS) {
    // ===== epilogue (as in decode_scores_mma2_kernel): K^ row -> bf16 -> RoPE -> tensor memory, on this CTA's tokens =====
    const int qd = warp & 3;
    const int half = (warp - 4) >> 2;
    const int row = qd * 32 + lane;
    const int d0 = half * 32;
    const bool rope = P.cos != nullptr;
    const uint32_t tempty0 = cluster_map_shared(smem_u32(&tempty_bar[0]), 0);
    const uint32_t a2full0 = cluster_map_shared(smem_u32(&a2full_bar[0]), 0);
    int acc = 0, ba = 0;
    uint32_t acc_ph = 0u, pa = 0u;
    for (int tile = slot; tile < ntiles; tile += nslots) {
      const int tok = (2 * tile + crank) * DBM + row;
      uint32_t cs[16], sn[16];
      if (rope && tok < P.S) {
        const uint4* cp = reinterpret_cast<const uint4*>(P.cos + static_cast<long long>(tok) * P.ld_cs + d0);
        const uint4* sp = reinterpret_cast<const uint4*>(P.sin + static_cast<long long>(tok) * P.ld_cs + d0);
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const uint4 cv = __ldg(cp + v), sv = __ldg(sp + v);
          cs[4 * v] = cv.x, cs[4 * v + 1] = cv.y, cs[4 * v + 2] = cv.z, cs[4 * v + 3] = cv.w;
          sn[4 * v] = sv.x, sn[4 * v + 1] = sv.y, sn[4 * v + 2] = sv.z, sn[4 * v + 3] = sv.w;
        }
      } else {
#pragma unroll
        for (int v = 0; v < 16; ++v) cs[v] = 0x3F803F80u, sn[v] = 0u;   // cos = 1, sin = 0
      }
      mbar_wait(&tfull_bar[acc], (acc_ph >> acc) & 1u);
      tc_fence_after();
      const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(qd * 32) << 16);
      const uint32_t lane_addr = lane_base + static_cast<uint32_t>(acc * D);
      uint32_t lo_w[16], hi_w[16];
      {
        uint32_t x1[32], x2[32];
        __syncwarp();
        tmem_ld_32x32(lane_addr + static_cast<uint32_t>(d0), x1);
        tmem_ld_32x32(lane_addr + static_cast<uint32_t>(D / 2 + d0), x2);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          lo_w[j] = pack_bf16x2(__uint_as_float(x1[2 * j]), __uint_as_float(x1[2 * j + 1]));
          hi_w[j] = pack_bf16x2(__uint_as_float(x2[2 * j]), __uint_as_float(x2[2 * j + 1]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty0 + static_cast<uint32_t>(acc * 8));
      if (rope) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const __nv_bfloat162 k1 = *reinterpret_cast<const __nv_bfloat162*>(&lo_w[j]);
          const __nv_bfloat162 k2 = *reinterpret_cast<const __nv_bfloat162*>(&hi_w[j]);
          const __nv_bfloat162 cw = *reinterpret_cast<const __nv_bfloat162*>(&cs[j]);
          const __nv_bfloat162 sw = *reinterpret_cast<const __nv_bfloat162*>(&sn[j]);
          const __nv_bfloat162 o1 = __hadd2(__hmul2(k1, cw), __hmul2(__hneg2(k2), sw));
          const __nv_bfloat162 o2 = __hadd2(__hmul2(k2, cw), __hmul2(k1, sw));
          lo_w[j] = *reinterpret_cast<const uint32_t*>(&o1);
          hi_w[j] = *reinterpret_cast<const uint32_t*>(&o2);
        }
      }
      mbar_wait(&a2empty_bar[ba], ((pa >> ba) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t a2 = lane_base + PR_COL_A2 + static_cast<uint32_t>(ba * 64);
      __syncwarp();
      tmem_st_32x16(a2 + static_cast<uint32_t>(d0 / 2), lo_w);
      tmem_st_32x16(a2 + static_cast<uint32_t>(32 + d0 / 2), hi_w);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(a2full0 + static_cast<uint32_t>(ba * 8));
      acc_ph ^= 1u << acc;
      acc ^= 1;
      pa ^= 1u << ba;
      ba = ba + 1 == PR_A2 ? 0 : ba + 1;
    }
  } else if (warp >= 4 + R_EPI_WARPS) {
    // ===== score read-out: one warp per TMEM lane quarter, thread = token; the qpk score columns in groups of 8 =====
    const int qd = warp & 3;
    const int row = qd * 32 + lane;
    const uint32_t d2empty0 = cluster_map_shared(smem_u32(&d2empty_bar[0]), 0);
    int b = 0;
    uint32_t bph = 0u;
    for (int tile = slot; tile < ntiles; tile += nslots) {
      const int tok = (2 * tile + crank) * DBM + row;
      mbar_wait(&d2full_bar[b], (bph >> b) & 1u);
      tc_fence_after();
      uint32_t v[NQ16 / 8][8];
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + PR_COL_D2 + static_cast<uint32_t>(b * nq16);
      __syncwarp();
#pragma unroll
      for (int c = 0; c < NQ16 / 8; ++c)
        if (c == 0 || c * 8 < P.qpk) tmem_ld_32x8(taddr + static_cast<uint32_t>(c * 8), v[c]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(d2empty0 + static_cast<uint32_t>(b * 8));
      if (tok < P.S) {
#pragma unroll
        for (int c = 0; c < NQ16 / 8; ++c)
#pragma unroll
          for (int g = 0; g < 8; ++g)
            if (c * 8 + g < P.qpk)
              P.scores[static_cast<long long>(h * P.qpk + c * 8 + g) * P.ld_scores + tok] = __uint_as_float(v[c][g]) * P.scale;
      }
      bph ^= 1u << b;
      b = b + 1 == nd2 ? 0 : b + 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // nobody leaves (or frees tensor memory) while the pair's MMAs, commits or arrivals are pending
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, R_TMEM_COLS);
  }
}

// Softmax over L = S + T scores of one q-head in ONE launch, with chunk-local maxima (flash-decoding style): chunk c of
// the compressed prefix is exactly the token range of split-K slab c of U = P A_v (kps k-blocks of 64 tokens), chunk
// `nchunk_s` is the dense tail.  A CTA takes the maximum m_c of its chunk, writes p = exp(s - m_c) as bf16 (the GEMM
// operand) and the fp32 sum l_c; the slab reduction and the combine kernel rescale by exp(m_c - m).  One pass over
// the scores instead of a max launch and an exp launch, and p keeps full bf16 precision inside every chunk.
// The tail chunk's CTA first scores its tokens (scale * q . k_tail): nobody else reads those scores.
// Rows: row r = hq * Tq + t is query token t of q head hq; qpk counts the rows of one kv head (q heads x Tq).  The last Tq
// tail tokens are the queries' own, so row r sees the tail tokens [0, T - Tq + t] (causal); the tail chunk stops there and
// the later tail tokens get no score and no probability (nothing downstream reads past tail_visible).
constexpr int SM_MAX_CHUNKS = 72;   // >= 64 split-K slabs + the tail chunk

// One (q head, chunk) unit, worked by NT threads (NT = 32: one warp, shuffles only -- the prefix chunks, a few KB each;
// NT = 256: the whole block -- the dense tail chunk, which first has to score its tokens).
__device__ __forceinline__ int tail_visible(int T, int Tq, int row) { return T - Tq + row % Tq + 1; }

template <int NT>
__device__ __forceinline__ void softmax_unit(float* __restrict__ scores, long long ld, int S, int T, int Tq, int kps, int nchunk_s,
                                             const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k_tail,
                                             long long sh, long long st, int qpk, int D, float scale,
                                             __nv_bfloat16* __restrict__ prob, long long ldp, float* __restrict__ chunk_max,
                                             float* __restrict__ chunk_sum, const float* __restrict__ raw_bias,
                                             const float* __restrict__ row_scale, float raw_scale, int hq, int ch, float* red,
                                             float* bcast) {
  // MLA path (raw_scale != 0): the scores buffer holds the RAW products q^ . a_t; the score of token t is
  // (raw * row_scale[t] + raw_bias[t]) * raw_scale, applied on the fly in both passes, and the probability that goes to
  // the GEMM is p * row_scale[t] (the value side of the absorbed form) while the chunk sum stays that of p.
  const bool xf = raw_scale != 0.f;
  float* s = scores + hq * ld;
  const float* rb = raw_bias != nullptr ? raw_bias + hq * ld : nullptr;
  __nv_bfloat16* p = prob + hq * ldp;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tid = NT == 32 ? lane : static_cast<int>(threadIdx.x);
  auto load4 = [&](int i) -> float4 {   // four transformed scores from token i (16-byte aligned)
    float4 x = *reinterpret_cast<const float4*>(s + i);
    if (xf) {
      if (row_scale != nullptr) {
        const float4 r4 = *reinterpret_cast<const float4*>(row_scale + i);
        x.x *= r4.x, x.y *= r4.y, x.z *= r4.z, x.w *= r4.w;
      }
      if (rb != nullptr) {
        const float4 b4 = *reinterpret_cast<const float4*>(rb + i);
        x.x += b4.x, x.y += b4.y, x.z += b4.z, x.w += b4.w;
      }
      x.x *= raw_scale, x.y *= raw_scale, x.z *= raw_scale, x.w *= raw_scale;
    }
    return x;
  };
  auto load1 = [&](int i) -> float {
    float x = s[i];
    if (xf) x = (x * (row_scale != nullptr ? row_scale[i] : 1.f) + (rb != nullptr ? rb[i] : 0.f)) * raw_scale;
    return x;
  };
  int i0, i1;
  if (ch < nchunk_s) {
    i0 = min(S, ch * kps * 64);
    i1 = min(S, (ch + 1) * kps * 64);
  } else {
    const int tv = T > 0 ? tail_visible(T, Tq, hq) : 0;
    i0 = S;
    i1 = S + tv;
    const int h = hq / qpk;
    for (int t = warp; t < tv; t += NT / 32) {
      const __nv_bfloat16* kr = k_tail + h * sh + t * st;
      float acc = 0.f;
      for (int d = lane; d < D; d += 32) acc += __bfloat162float(q[hq * D + d]) * __bfloat162float(kr[d]);
      acc = warp_sum(acc);
      if (lane == 0) s[S + t] = acc * scale;
    }
    if (NT > 32) __syncthreads();
  }
  // ---- chunk maximum (prefix chunks start at multiples of 64 tokens: 16-byte aligned rows) ----
  const bool vec = ch < nchunk_s;
  const int nvec = vec ? max(i1 - i0, 0) >> 2 : 0;
  float m = -INFINITY;
  for (int v = tid; v < nvec; v += NT) {
    const float4 x = load4(i0 + 4 * v);
    m = fmaxf(fmaxf(m, fmaxf(x.x, x.y)), fmaxf(x.z, x.w));
  }
  for (int i = i0 + 4 * nvec + tid; i < i1; i += NT) m = fmaxf(m, load1(i));
  m = warp_max(m);
  if (NT > 32) {
    if (lane == 0) red[warp] = m;
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < NT / 32; ++w) m = fmaxf(m, red[w]);
      *bcast = m;
    }
    __syncthreads();
    m = *bcast;
  }
  if (tid == 0) chunk_max[hq * SM_MAX_CHUNKS + ch] = m;
  // ---- p = exp(s - m_c), l_c = sum p (second pass over a few KB that are in L1 / L2) ----
  float sum = 0.f;
  const bool vs = xf && row_scale != nullptr;   // value-side scale of the absorbed form
  for (int v = tid; v < nvec; v += NT) {
    const float4 x = load4(i0 + 4 * v);
    float e0 = __expf(x.x - m), e1 = __expf(x.y - m), e2 = __expf(x.z - m), e3 = __expf(x.w - m);
    sum += (e0 + e1) + (e2 + e3);
    if (vs) {
      // the probability is rounded to bf16 BEFORE the value-side scale, as the separate scale pass did
      const float4 r4 = *reinterpret_cast<const float4*>(row_scale + i0 + 4 * v);
      e0 = bf16r(e0) * r4.x, e1 = bf16r(e1) * r4.y, e2 = bf16r(e2) * r4.z, e3 = bf16r(e3) * r4.w;
    }
    uint2 w;
    w.x = pack_bf16x2(e0, e1);
    w.y = pack_bf16x2(e2, e3);
    *reinterpret_cast<uint2*>(p + i0 + 4 * v) = w;
  }
  for (int i = i0 + 4 * nvec + tid; i < i1; i += NT) {
    float e = __expf(load1(i) - m);
    sum += e;
    if (vs) e = bf16r(e) * row_scale[i];
    p[i] = __float2bfloat16_rn(e);
  }
  sum = warp_sum(sum);
  if (NT > 32) {
    __syncthreads();
    if (lane == 0) red[warp] = sum;
    __syncthreads();
    if (tid == 0)
      for (int w = 1; w < NT / 32; ++w) sum += red[w];
  }
  if (tid == 0) chunk_sum[hq * SM_MAX_CHUNKS + ch] = sum;
}

// grid: ceil(Hq * nchunk_s / 8) blocks whose eight warps take one prefix (q head, chunk) unit each -- no block barrier, the
// whole unit is one L2 round trip, a shuffle reduction, the exps and another shuffle reduction (the one-block-per-unit form
// with its six block barriers took 7-8 us per layer) -- followed by Hq blocks for the tail chunks.
__global__ void __launch_bounds__(256) softmax_chunk_kernel(float* __restrict__ scores, long long ld, int S, int T, int Tq,
                                                            int kps, int nchunk_s, int Hq, const __nv_bfloat16* __restrict__ q,
                                                            const __nv_bfloat16* __restrict__ k_tail, long long sh,
                                                            long long st, int qpk, int D, float scale,
                                                            __nv_bfloat16* __restrict__ prob, long long ldp,
                                                            float* __restrict__ chunk_max, float* __restrict__ chunk_sum,
                                                            const float* __restrict__ raw_bias, const float* __restrict__ row_scale,
                                                            float raw_scale) {
  __shared__ float red[8];
  __shared__ float bcast;
  const int nprefix_blocks = (Hq * nchunk_s + 7) / 8;
  if (static_cast<int>(blockIdx.x) < nprefix_blocks) {
    const int unit = static_cast<int>(blockIdx.x) * 8 + static_cast<int>(threadIdx.x >> 5);
    if (unit >= Hq * nchunk_s) return;
    softmax_unit<32>(scores, ld, S, T, Tq, kps, nchunk_s, q, k_tail, sh, st, qpk, D, scale, prob, ldp, chunk_max, chunk_sum, raw_bias,
                     row_scale, raw_scale, unit / nchunk_s, unit % nchunk_s, red, &bcast);
  } else {
    softmax_unit<256>(scores, ld, S, T, Tq, kps, nchunk_s, q, k_tail, sh, st, qpk, D, scale, prob, ldp, chunk_max, chunk_sum, raw_bias,
                      row_scale, raw_scale, static_cast<int>(blockIdx.x) - nprefix_blocks, nchunk_s, red, &bcast);
  }
}

// Weights of the chunks in the global softmax of head hq: w_s[c] = exp(m_c - m), m = max_c m_c (0 for an empty chunk,
// m_c = -inf), stats = {m, sum_c w_c l_c}.  Warp 0 does it in parallel (three chunks per lane); ends with a barrier.
__device__ __forceinline__ void head_weights(const float* __restrict__ chunk_max, const float* __restrict__ chunk_sum,
                                             int hq, int nchunks, float* w_s, float* stats) {
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    const float* cm = chunk_max + hq * SM_MAX_CHUNKS;
    float v[3];
    float m = -INFINITY;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int c = lane + 32 * k;
      v[k] = c < nchunks ? cm[c] : -INFINITY;
      m = fmaxf(m, v[k]);
    }
    m = warp_max(m);
    float rs = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int c = lane + 32 * k;
      if (c < nchunks) {
        const float w = __expf(v[k] - m);
        w_s[c] = w;
        rs = fmaf(w, chunk_sum[hq * SM_MAX_CHUNKS + c], rs);
      }
    }
    rs = warp_sum(rs);
    if (lane == 0) {
      stats[0] = m;
      stats[1] = rs;
    }
  }
  __syncthreads();
}

// U[e] = sum over the split-K slabs s of exp(m_s - m) * (P_s A_v)[e]  (P_s is relative to its chunk's maximum m_s).
// The sum over ~50 slabs is a chain of L2 round trips, so it is cut four ways: thread (e, g) adds the slabs g, g + 4, ...
// (all loads independent), shared memory adds the four partial sums.
__global__ void __launch_bounds__(256) reduce_u_kernel(const float* __restrict__ slabs, int nslabs, long long slab_stride,
                                                       int rv, const float* __restrict__ chunk_max,
                                                       const float* __restrict__ chunk_sum, int nchunks,
                                                       float* __restrict__ U, int normalise, float* __restrict__ lse_out) {
  __shared__ float part[4][64];
  __shared__ float w_s[SM_MAX_CHUNKS];
  __shared__ float stats[2];
  const int hq = blockIdx.y;
  const int el = threadIdx.x & 63, g = threadIdx.x >> 6;
  const int j = blockIdx.x * 64 + el;
  const long long e = static_cast<long long>(hq) * rv + j;
  // the slab values do not depend on the weights: they are in flight while warp 0 works the weights out
  float v[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const int sl = g + 4 * k;
    v[k] = (j < rv && sl < nslabs) ? slabs[sl * slab_stride + e] : 0.f;
  }
  head_weights(chunk_max, chunk_sum, hq, nchunks, w_s, stats);
  float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const int sl = g + 4 * k;
    if (sl < nslabs) a[k & 3] = fmaf(w_s[sl], v[k], a[k & 3]);
  }
  part[g][el] = (a[0] + a[1]) + (a[2] + a[3]);
  __syncthreads();
  // normalise: U / (sum of the softmax) and the log-sum-exp, what absorbed_finalize_kernel did in a launch of its own
  if (g == 0 && j < rv) U[e] = ((part[0][el] + part[1][el]) + (part[2][el] + part[3][el])) * (normalise ? 1.f / stats[1] : 1.f);
  if (lse_out != nullptr && blockIdx.x == 0 && threadIdx.x == 0) lse_out[hq] = stats[0] + logf(stats[1]);
}

// o[hq][d] = ( sum_j U[hq][j] * Bv[(h*D + d)][j]  +  sum_t p_tail[hq][t] * v_tail[h][t][d] ) / rowsum[hq]
// (hq: a q row as in softmax_unit, h = hq / qpk its kv head; qpk counts the rows of a kv head)
// grid (rows, D / 8), 8 warps x 1 output dim (a short dependency chain per warp; U is re-read by the D / 8 blocks of a head).
__global__ void __launch_bounds__(256) combine_kernel(const float* __restrict__ slabs, int nslabs, long long slab_stride,
                                                      int rv, const __nv_bfloat16* __restrict__ Bv, long long ldb,
                                                      const __nv_bfloat16* __restrict__ prob, long long ldp, int S, int T,
                                                      int Tq, const __nv_bfloat16* __restrict__ v_tail, long long sh, long long st,
                                                      const float* __restrict__ rowsum, int qpk, int D,
                                                      __nv_bfloat16* __restrict__ out,
                                                      const float* __restrict__ chunk_max, int nchunks,
                                                      float* __restrict__ lse_out) {
  extern __shared__ float u_s[];  // rv floats
  const int hq = blockIdx.x, h = hq / qpk;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int j = threadIdx.x; j < rv; j += blockDim.x) u_s[j] = slabs[static_cast<long long>(hq) * rv + j];
  (void)nslabs;
  (void)slab_stride;
  __syncthreads();
  // global maximum and denominator from the chunk-local ones; the tail chunk is the last one
  __shared__ float w_s[SM_MAX_CHUNKS];
  __shared__ float stats[2];
  head_weights(chunk_max, rowsum, hq, nchunks, w_s, stats);
  const float m = stats[0], rs = stats[1];
  const float inv = 1.f / rs;
  const float w_tail = T > 0 ? w_s[nchunks - 1] : 0.f;
  const int tv = T > 0 ? tail_visible(T, Tq, hq) : 0;   // causal: the tail tokens this row sees
  if (lse_out != nullptr && blockIdx.y == 0 && threadIdx.x == 0) {
    // log-sum-exp of this head's scaled scores over the tokens of THIS call: what a flash-decoding style merge of
    // token shards needs besides the normalised output
    lse_out[hq] = m + logf(rs);
  }
  for (int d = blockIdx.y * 8 + warp; d < min(D, blockIdx.y * 8 + 8); d += 8) {
    const __nv_bfloat16* row = Bv + static_cast<long long>(h * D + d) * ldb;
    float acc = 0.f;
    for (int j = lane * 2; j < rv; j += 64) {
      const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(row + j);
      acc = fmaf(u_s[j], __bfloat162float(b2.x), fmaf(u_s[j + 1], __bfloat162float(b2.y), acc));
    }
    float acc_t = 0.f;
    for (int t = lane; t < tv; t += 32)
      acc_t = fmaf(__bfloat162float(prob[hq * ldp + S + t]), __bfloat162float(v_tail[h * sh + t * st + d]), acc_t);
    acc = warp_sum(fmaf(w_tail, acc_t, acc));
    if (lane == 0) out[hq * D + d] = __float2bfloat16_rn(acc * inv);
  }
}

// Slab reduction and combine in ONE launch: the RC_CL CTAs of a thread-block cluster share a q head.  CTA c sums its
// rv / RC_CL columns of U over the split-K slabs (weighted by exp(m_s - m), fixed order: deterministic), writes them into
// the shared memory of every CTA of the cluster (distributed shared memory), and after one cluster barrier each CTA
// contracts the whole U row with ITS D / RC_CL rows of the layer's value factor.  Replaces reduce_u_kernel +
// combine_kernel (two launches and a round trip of U through L2) on the Llama path.
// DENSE_V: the value slot of the group is dense (one-sided groups, xkv_decode_attention_half): the slabs hold
// U_s = P_s V_h (rv = D columns) and the identity takes the place of Bv_l -- output dim d of a row is U[d] itself.
constexpr int RC_CL = 8;
template <bool DENSE_V>
__global__ void __launch_bounds__(256) reduce_combine_kernel(const float* __restrict__ slabs, int nslabs, long long slab_stride,
                                                             int rv, const __nv_bfloat16* __restrict__ Bv, long long ldb,
                                                             const __nv_bfloat16* __restrict__ prob, long long ldp, int S, int T,
                                                             int Tq, const __nv_bfloat16* __restrict__ v_tail, long long sh, long long st,
                                                             const float* __restrict__ rowsum, int qpk, int D,
                                                             __nv_bfloat16* __restrict__ out,
                                                             const float* __restrict__ chunk_max, int nchunks,
                                                             float* __restrict__ lse_out) {
  extern __shared__ float u_s[];  // rv floats: the whole U row of this head, filled by the cluster
  __shared__ float part[128];
  __shared__ float w_s[SM_MAX_CHUNKS];
  __shared__ float stats[2];
  cg::cluster_group cluster = cg::this_cluster();
  const int cr = static_cast<int>(cluster.block_rank());   // == blockIdx.y
  const int hq = blockIdx.x, h = hq / qpk;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cpc = (rv + RC_CL - 1) / RC_CL;                // columns of U this CTA reduces (<= 128)
  const int el = threadIdx.x & 127, g = threadIdx.x >> 7;
  const int j = cr * cpc + el;
  const bool active = el < cpc && j < rv;
  const long long e = static_cast<long long>(hq) * rv + j;
  float v[32];   // slabs g, g + 2, ...: all loads in flight while warp 0 works the weights out
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    const int sl = g + 2 * k;
    v[k] = (active && sl < nslabs) ? slabs[sl * slab_stride + e] : 0.f;
  }
  head_weights(chunk_max, rowsum, hq, nchunks, w_s, stats);
  float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    const int sl = g + 2 * k;
    if (sl < nslabs) a[k & 3] = fmaf(w_s[sl], v[k], a[k & 3]);
  }
  const float mine = (a[0] + a[1]) + (a[2] + a[3]);
  if (g == 1) part[el] = mine;
  __syncthreads();
  if (g == 0 && active) {
    const float u = mine + part[el];
#pragma unroll
    for (int r = 0; r < RC_CL; ++r) cluster.map_shared_rank(u_s, r)[j] = u;
  }
  cluster.sync();
  const float m = stats[0], rs = stats[1];
  const float inv = 1.f / rs;
  const float w_tail = T > 0 ? w_s[nchunks - 1] : 0.f;
  if (lse_out != nullptr && cr == 0 && threadIdx.x == 0) lse_out[hq] = m + logf(rs);
  const int dpc = (D + RC_CL - 1) / RC_CL;                 // output dims of this CTA
  for (int d = cr * dpc + warp; d < min(D, (cr + 1) * dpc); d += 8) {
    const __nv_bfloat16* row = Bv + static_cast<long long>(h * D + d) * ldb;
    float acc = 0.f;
    if constexpr (DENSE_V) {
      if (lane == 0) acc = u_s[d];
    } else {
      for (int jj = lane * 2; jj < rv; jj += 64) {
        const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(row + jj);
        acc = fmaf(u_s[jj], __bfloat162float(b2.x), fmaf(u_s[jj + 1], __bfloat162float(b2.y), acc));
      }
    }
    const int tv = T > 0 ? tail_visible(T, Tq, hq) : 0;   // causal: the tail tokens this row sees
    float acc_t = 0.f;
    for (int t = lane; t < tv; t += 32)
      acc_t = fmaf(__bfloat162float(prob[hq * ldp + S + t]), __bfloat162float(v_tail[h * sh + t * st + d]), acc_t);
    acc = warp_sum(fmaf(w_tail, acc_t, acc));
    if (lane == 0) out[hq * D + d] = __float2bfloat16_rn(acc * inv);
  }
}

// ---------------------------------------------------------------------------------------------
// One-sided groups (xkv_decode_attention_half): one slot of the layer is factored, the other stayed dense (merge_key /
// merge_value off, or a rank that does not fit one side).  The factored side runs the kernels above; the dense side runs
// one of the two kernels below, feeding the same chunk-local softmax and the same slab reduction + combine.
//
//   dense keys    scores[r][t] = scale * q_r . K[t, h(r)]: a 128-token key tile (already rotated: RoPE was applied once,
//                 when the group was merged) is the A operand of ONE tcgen05.mma per tile, M = 128 tokens, N = nq16 (the
//                 kv head's q rows rounded up to 16, the pair kernel's q tile), K = D.  Every key tile is read once for all
//                 q rows of its head.  Warp roles: 0 TMA, 1 MMA, 2..5 score read-out (the pair kernel's).
//   dense values  U_c^T (D x nq16) = V_h tile^T . P_h^T accumulated in tensor memory over the 64-token blocks of softmax
//                 chunk c: A = the value tile straight from the token-major slot (MN-major, M = D), B = the head's
//                 probability rows (K-major).  One CTA per (kv head, chunk); every value tile is read once.  The fp32 slab
//                 U_c goes to (nchunks, rows, D); reduce_combine_kernel<true> weights, sums and normalises the slabs.
// Both read the dense slot through a 3-D tensor map {D, tokens, heads} (or {D, heads, tokens} when the head stride is
// the smaller one: TMA wants the outer strides of a box in any order but the box layout is the same), so any
// (S, H, D) / (H, S, D) view with strides that are multiples of 8 elements is read in place.
// ---------------------------------------------------------------------------------------------
constexpr int DN_THREADS = 192;     // TMA warp, MMA warp, four read-out warps (one per TMEM lane quarter)
constexpr int DN_MAX_STAGES = 8;
constexpr int DN_NACC = 4;          // score accumulators of nq16 columns (dense-key kernel)
constexpr int DN_VBLK = 64;         // tokens per value block (dense-value kernel)

struct alignas(64) DenseParams {
  CUtensorMap slot_map;   // the dense slot, box {64 dims, tile tokens, 1 head} (dims ordered as slot_tok_dim says)
  CUtensorMap rows_map;   // keys: q (rows x D), box {64, nq16}; values: probabilities (rows x S), box {64 tokens, nq16}
  float* out;             // keys: scores (rows, ld_out); values: slabs (nchunks, rows, D)
  long long ld_out;
  int S, H, qpk, rows, stages;
  int slot_tok_dim;       // 1: the map is {D, S, H}; 2: {D, H, S}
  int kps;                // values: 64-token blocks per softmax chunk
  float scale;
};

__device__ __forceinline__ void load_slot_tile(void* dst, const DenseParams& P, uint64_t* bar, int d0, int t0, int h) {
  if (P.slot_tok_dim == 1)
    tma_load_3d(dst, &P.slot_map, bar, d0, t0, h);
  else
    tma_load_3d(dst, &P.slot_map, bar, d0, h, t0);
}

template <int D, int NQ16>
__global__ void __launch_bounds__(DN_THREADS, 1) decode_dense_scores_kernel(const __grid_constant__ DenseParams P) {
  constexpr int NKC = D / 64;                     // 64-dim chunks of a key tile
  constexpr int TILE_BYTES = NKC * DBM * 128;     // 128 tokens x D
  constexpr int Q_BYTES = NKC * NQ16 * 128;       // the pair kernel's q tile with all nq16 rows in one CTA
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = smem + Q_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sK + P.stages * TILE_BYTES);
  uint64_t* empty_bar = full_bar + DN_MAX_STAGES;
  uint64_t* tfull_bar = empty_bar + DN_MAX_STAGES;   // [DN_NACC]
  uint64_t* tempty_bar = tfull_bar + DN_NACC;        // [DN_NACC]
  uint64_t* q_bar = tempty_bar + DN_NACC;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(q_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // CTA -> kv head h and the token tiles slot, slot + nslots, ... (as decode_scores_mma2_kernel)
  const int h = static_cast<int>(blockIdx.x) % P.H;
  const int slot = static_cast<int>(blockIdx.x) / P.H;
  const int nslots = (static_cast<int>(gridDim.x) - h + P.H - 1) / P.H;
  const int ntiles = (P.S + DBM - 1) / DBM;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < P.stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < DN_NACC; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 4);   // one arrive per read-out warp
    }
    mbar_init(q_bar, 1);
    mbar_fence_init();
    tma_prefetch_desc(&P.slot_map);
    tma_prefetch_desc(&P.rows_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(q_bar, Q_BYTES);
#pragma unroll
      for (int c = 0; c < NKC; ++c) tma_load_2d(sQ + c * NQ16 * 128, &P.rows_map, q_bar, c * 64, h * P.qpk);
      int s = 0;
      uint32_t ph = 0;
      for (int tile = slot; tile < ntiles; tile += nslots) {
        mbar_wait(&empty_bar[s], ph ^ 1u);
        mbar_expect_tx(&full_bar[s], TILE_BYTES);
#pragma unroll
        for (int c = 0; c < NKC; ++c) load_slot_tile(sK + s * TILE_BYTES + c * DBM * 128, P, &full_bar[s], c * 64, tile * DBM, h);
        if (++s == P.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // scores[128 tokens x nq16] = K tile (K-major: 128 B of dims per token row) * Q^T (K-major: 128 B of dims per q row)
    constexpr uint32_t idesc = umma_idesc_bf16(DBM, NQ16, 0, 0);
    if (elect_one()) {
      mbar_wait(q_bar, 0);
      const uint64_t q_desc0 = umma_desc_sw128(smem_u32(sQ), 16, 1024);
      const uint64_t k_desc0 = umma_desc_sw128(smem_u32(sK), 16, 1024);
      int s = 0, acc = 0;
      uint32_t ph = 0, acc_ph = 0u;
      for (int tile = slot; tile < ntiles; tile += nslots) {
        mbar_wait(&tempty_bar[acc], ((acc_ph >> acc) & 1u) ^ 1u);
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint32_t d_addr = tmem_base + static_cast<uint32_t>(acc * NQ16);
        const uint64_t k_desc = k_desc0 + static_cast<uint64_t>((s * TILE_BYTES) >> 4);
#pragma unroll
        for (int k = 0; k < D / 16; ++k)
          umma_bf16_ss(d_addr, k_desc + static_cast<uint64_t>(((k >> 2) * DBM * 128 + (k & 3) * 32) >> 4),
                       q_desc0 + static_cast<uint64_t>(((k >> 2) * NQ16 * 128 + (k & 3) * 32) >> 4), idesc, k > 0 ? 1u : 0u);
        umma_commit(&empty_bar[s]);
        umma_commit(&tfull_bar[acc]);
        acc_ph ^= 1u << acc;
        acc = (acc + 1) % DN_NACC;
        if (++s == P.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
    __syncwarp();
  } else {
    // ===== score read-out (the pair kernel's): thread = token, the qpk score columns in groups of 8 =====
    const int qd = warp & 3;
    const int row = qd * 32 + lane;
    int acc = 0;
    uint32_t acc_ph = 0u;
    for (int tile = slot; tile < ntiles; tile += nslots) {
      const int tok = tile * DBM + row;
      mbar_wait(&tfull_bar[acc], (acc_ph >> acc) & 1u);
      tc_fence_after();
      uint32_t v[NQ16 / 8][8];
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + static_cast<uint32_t>(acc * NQ16);
      __syncwarp();
#pragma unroll
      for (int c = 0; c < NQ16 / 8; ++c)
        if (c == 0 || c * 8 < P.qpk) tmem_ld_32x8(taddr + static_cast<uint32_t>(c * 8), v[c]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (tok < P.S) {
#pragma unroll
        for (int c = 0; c < NQ16 / 8; ++c)
#pragma unroll
          for (int g = 0; g < 8; ++g)
            if (c * 8 + g < P.qpk)
              P.out[static_cast<long long>(h * P.qpk + c * 8 + g) * P.ld_out + tok] = __uint_as_float(v[c][g]) * P.scale;
      }
      acc_ph ^= 1u << acc;
      acc = (acc + 1) % DN_NACC;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

template <int D, int NQ16>
__global__ void __launch_bounds__(DN_THREADS, 1) decode_dense_values_kernel(const __grid_constant__ DenseParams P) {
  constexpr int NKC = D / 64;
  constexpr int CHUNK_BYTES = DN_VBLK * 128;                  // 64 tokens x 64 dims: one MN-major chunk of M
  constexpr int V_BYTES = 2 * CHUNK_BYTES;                    // M = 128 (D = 64: the upper chunk is zero)
  constexpr int STAGE_BYTES = V_BYTES + NQ16 * 128;           // + the head's probability rows of the block
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + P.stages * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + DN_MAX_STAGES;
  uint64_t* tfull_bar = empty_bar + DN_MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = static_cast<int>(blockIdx.x) % P.H;
  const int ch = static_cast<int>(blockIdx.x) / P.H;     // softmax chunk: tokens [ch * kps * 64, (ch + 1) * kps * 64)
  const int t0 = ch * P.kps * DN_VBLK;
  const int t1 = min(P.S, t0 + P.kps * DN_VBLK);
  const int nkb = (t1 - t0 + DN_VBLK - 1) / DN_VBLK;    // >= 1: the host drops empty chunks

  if constexpr (D == 64) {
    // rows 64..127 of the M = 128 product read this chunk: zeros, never loaded (their TMEM lanes are not read out)
    for (int i = threadIdx.x; i < P.stages * CHUNK_BYTES / 16; i += DN_THREADS) {
      const int st = i / (CHUNK_BYTES / 16), o = i - st * (CHUNK_BYTES / 16);
      reinterpret_cast<uint4*>(smem + st * STAGE_BYTES + CHUNK_BYTES)[o] = make_uint4(0u, 0u, 0u, 0u);
    }
    fence_proxy_async_smem();
  }
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < P.stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(tfull_bar, 1);
    mbar_fence_init();
    tma_prefetch_desc(&P.slot_map);
    tma_prefetch_desc(&P.rows_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, 64);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      for (int kb = 0; kb < nkb; ++kb) {
        const int tok = t0 + kb * DN_VBLK;
        uint8_t* st = smem + s * STAGE_BYTES;
        mbar_wait(&empty_bar[s], ph ^ 1u);
        mbar_expect_tx(&full_bar[s], NKC * CHUNK_BYTES + NQ16 * 128);
#pragma unroll
        for (int c = 0; c < NKC; ++c) load_slot_tile(st + c * CHUNK_BYTES, P, &full_bar[s], c * 64, tok, h);
        // tokens past S are zero in both operands (the maps end at S): the tail probabilities beyond the prefix stay out
        tma_load_2d(st + V_BYTES, &P.rows_map, &full_bar[s], tok, h * P.qpk);
        if (++s == P.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // U^T[D x nq16] += V tile^T (MN-major: 128 B of dims per token row, chunks of 64 dims CHUNK_BYTES apart) * P^T
    // (K-major: 128 B of tokens per q row); K = 16 tokens per instruction: +2048 B on A, +32 B on B
    constexpr uint32_t idesc = umma_idesc_bf16(128, NQ16, 1, 0);
    if (elect_one()) {
      const uint64_t a_desc0 = umma_desc_sw128(smem_u32(smem), CHUNK_BYTES, 1024);
      const uint64_t b_desc0 = umma_desc_sw128(smem_u32(smem + V_BYTES), 16, 1024);
      int s = 0;
      uint32_t ph = 0;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint64_t so = static_cast<uint64_t>((s * STAGE_BYTES) >> 4);
#pragma unroll
        for (int k = 0; k < DN_VBLK / 16; ++k)
          umma_bf16_ss(tmem_base, a_desc0 + so + static_cast<uint64_t>((k * 2048) >> 4), b_desc0 + so + static_cast<uint64_t>((k * 32) >> 4),
                       idesc, (kb > 0 || k > 0) ? 1u : 0u);
        umma_commit(&empty_bar[s]);
        if (++s == P.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
      umma_commit(tfull_bar);
    }
    __syncwarp();
  } else {
    // ===== read-out: thread = output dim d (TMEM lane), the qpk q-row columns in groups of 8 =====
    const int qd = warp & 3;
    const int d = qd * 32 + lane;
    if (qd * 32 < D) {
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
      uint32_t v[NQ16 / 8][8];
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16);
      __syncwarp();
#pragma unroll
      for (int c = 0; c < NQ16 / 8; ++c)
        if (c == 0 || c * 8 < P.qpk) tmem_ld_32x8(taddr + static_cast<uint32_t>(c * 8), v[c]);
      tmem_ld_wait();
      float* slab = P.out + (static_cast<long long>(ch) * P.rows + h * P.qpk) * D + d;
#pragma unroll
      for (int c = 0; c < NQ16 / 8; ++c)
#pragma unroll
        for (int g = 0; g < 8; ++g)
          if (c * 8 + g < P.qpk) slab[static_cast<long long>(c * 8 + g) * D] = __uint_as_float(v[c][g]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 64);
  }
}

// ---------------------------------------------------------------------------------------------
// Absorbed attention over the token factor (MLA latents, deepseek_v2.py:217-235): the latent of token t is
// c_t = V_l a_t and both products of the attention are LINEAR in it (kv_b_proj after a per-token RMS scale), so with
// the query folded into the rank space, q^ = V_l^T (gamma o W_UK^T q_nope), the scores are
//     s[h][t] = scale * ( row_scale[t] * (q^[h] . a_t) + bias_q[h] . bias_k[t] )
// (row_scale = 1 / rms of the reconstructed latent, the bias term is the RoPE part q_pe . k_pe) and the values are
//     u[h] = sum_t softmax(s)[h][t] * row_scale[t] * a_t          (rank space; the caller applies V_l, gamma, W_UV).
// Four launches: the raw products q^ A^T (+ the bias GEMM), the chunk-local softmax (which applies row_scale, bias and
// scale to the raw products on the fly and emits p * row_scale), U = P' A, and the slab reduction that also normalises and
// writes the log-sum-exp (round 2, first half: seven launches).  The latents are never reconstructed.
// ---------------------------------------------------------------------------------------------

// RoPE on materialised keys, in the reference's bf16 arithmetic (cache:142-152): x (rows, H, D) in place
__global__ void __launch_bounds__(256) rope_bf16_kernel(__nv_bfloat16* __restrict__ x, long long ld_row, int rows, int H,
                                                        int D, const __nv_bfloat16* __restrict__ cos,
                                                        const __nv_bfloat16* __restrict__ sin, long long ld_cs) {
  const int half = D / 2;
  const long long total = static_cast<long long>(rows) * H * half;
  for (long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int d = static_cast<int>(e % half);
    const long long rh = e / half;
    const int h = static_cast<int>(rh % H);
    const long long row = rh / H;
    __nv_bfloat16* p = x + row * ld_row + h * D;
    const float k1 = __bfloat162float(p[d]), k2 = __bfloat162float(p[d + half]);
    const float c1 = __bfloat162float(cos[row * ld_cs + d]), s1 = __bfloat162float(sin[row * ld_cs + d]);
    const float c2 = __bfloat162float(cos[row * ld_cs + d + half]), s2 = __bfloat162float(sin[row * ld_cs + d + half]);
    p[d] = __float2bfloat16_rn(bf16r(k1 * c1) + bf16r(-k2 * s1));
    p[d + half] = __float2bfloat16_rn(bf16r(k2 * c2) + bf16r(k1 * s2));
  }
}

static inline size_t al(size_t x) { return (x + 1023) / 1024 * 1024; }
// Split-K factor of U = P A_v (M rows): as many K slices as make tiles_m x tiles_n x split CTAs fill the SMs ONCE (a
// 64-way split of 3 column tiles is 192 CTAs = 1.3 waves on 148 SMs: the second wave runs at a third of the machine).
static inline int decode_split_k(int S, int rv, int M) {
  const int nkb = (S + 63) / 64;
  const int tiles_n = (rv + 255) / 256;
  const int tiles_m = (M + 127) / 128;
  const int sms = device_sm_count();
  int split = sms / (tiles_n * tiles_m < 1 ? 1 : tiles_n * tiles_m);
  if (split > nkb) split = nkb;
  if (split > 64) split = 64;
  if (split < 1) split = 1;
  const int per = (nkb + split - 1) / split;   // K blocks per slice, as the GEMM cuts them
  return (nkb + per - 1) / per;                // drop slices that would be empty
}

static bool g_force_tiled_scores = false;  // test hook: exercise the tile-per-CTA scores kernel
static int g_scores_variant = 0;           // test hook: 0 automatic, 1 FFMA epilogue, 2 score MMA in single CTAs, 3 CTA pairs
static bool g_split_reduce_combine = false;   // test hook (variant 4): slab reduction and combine as two launches

// Launch the single-CTA score-MMA kernel (persistent: one CTA per SM, every head at least one).
static int launch_scores_mma2(const ScoreParams& sp, int S, int H, cudaStream_t st) {   // H: row sets (kv heads x passes)
  static PerDevice<bool> configured;
  if (!configured()) {
    XKV_CHECK_CUDA(cudaFuncSetAttribute(decode_scores_mma2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(R_SMEM_LIMIT)));
    configured() = true;
  }
  const size_t smem = R_FIXED_BYTES + static_cast<size_t>(sp.nkb) * 128 * DBK * 2 + static_cast<size_t>(sp.stages) * D_A_BYTES;
  const int ntiles = (S + DBM - 1) / DBM;
  const int sms = device_sm_count();
  int ncta = sms < ntiles * H ? sms : ntiles * H;
  if (ncta < H) ncta = H;
  decode_scores_mma2_kernel<<<ncta, R_THREADS, smem, st>>>(sp);
  return 0;
}

// Launch the pair kernel: one cluster of two CTAs per (kv head, slot).  Returns 0 on success, -1 when the device cannot
// hold such a cluster (the caller falls back to the single-CTA kernels).
static int launch_scores_pair(ScoreParams& sp, int S, int H, cudaStream_t st) {
  static PerDevice<int> state;   // 0: not probed, -1: not launchable, > 0: resident pairs
  int& resident = state();
  sp.stages = pair_stages_for(sp.nkb, sp.qpk);
  if (sp.stages < 3) return -1;
  cudaLaunchConfig_t cfg;
  std::memset(&cfg, 0, sizeof(cfg));
  cfg.blockDim = dim3(R_THREADS, 1, 1);
  cfg.dynamicSmemBytes = pair_fixed_bytes(sp.qpk) + static_cast<size_t>(sp.nkb) * PR_B_KB_BYTES + static_cast<size_t>(sp.stages) * D_A_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (resident == 0) {
    resident = -1;
    const int lim = static_cast<int>(R_SMEM_LIMIT);
    if (cudaFuncSetAttribute(decode_scores_pair_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim) == cudaSuccess &&
        cudaFuncSetAttribute(decode_scores_pair_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim) == cudaSuccess &&
        cudaFuncSetAttribute(decode_scores_pair_kernel<48>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim) == cudaSuccess &&
        cudaFuncSetAttribute(decode_scores_pair_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim) == cudaSuccess) {
      int n = 0;
      cfg.gridDim = dim3(2, 1, 1);
      const size_t launch_smem = cfg.dynamicSmemBytes;
      cfg.dynamicSmemBytes = R_SMEM_LIMIT;   // one CTA per SM whatever the rank (the same for every instantiation)
      if (cudaOccupancyMaxActiveClusters(&n, decode_scores_pair_kernel<16>, &cfg) == cudaSuccess && n >= 1) resident = n;
      cfg.dynamicSmemBytes = launch_smem;
    }
    (void)cudaGetLastError();
  }
  if (resident < 0) return -1;
  const int ptiles = (S + 2 * DBM - 1) / (2 * DBM);
  int npairs = resident < ptiles * H ? resident : ptiles * H;
  if (npairs < H) npairs = H;   // every head needs at least one pair
  cfg.gridDim = dim3(2 * npairs, 1, 1);
  switch (pair_nq16(sp.qpk)) {
    case 16: XKV_CHECK_CUDA(cudaLaunchKernelEx(&cfg, decode_scores_pair_kernel<16>, sp)); break;
    case 32: XKV_CHECK_CUDA(cudaLaunchKernelEx(&cfg, decode_scores_pair_kernel<32>, sp)); break;
    case 48: XKV_CHECK_CUDA(cudaLaunchKernelEx(&cfg, decode_scores_pair_kernel<48>, sp)); break;
    default: XKV_CHECK_CUDA(cudaLaunchKernelEx(&cfg, decode_scores_pair_kernel<64>, sp)); break;
  }
  return 0;
}

// scores[r][t] = scale * q_r . rope(bf16(A_k[t] Bk_l^T)) for the S tokens of the compressed prefix and the `rows` q rows
// (rows / H contiguous rows per kv head): fused reconstruct + RoPE + q.K, one launch (kernel chosen by head_dim, rank and
// the test hooks).  The pair kernel takes all rows of a kv head at once; the others work rows / H > 8 in passes of <= 8
// rows, one CTA set per pass (each pass rebuilds the keys of the whole prefix).
static int launch_scores(const void* q, int rows, int H, int D, const void* A_k, int64_t lda_k, int rk, const void* Vk_layer,
                         int64_t ldv_k, int S, const void* cos, const void* sin, int64_t ld_cs, float scale, float* scores,
                         long long ldl, cudaStream_t st) {
  const int qpk = rows / H;
  const int npass = (qpk + D_MAX_QPK - 1) / D_MAX_QPK;
  int rc;
  static thread_local ScoreParams sp;
  std::memset(&sp, 0, sizeof(sp));
  rc = encode_tmap_2d_bf16(&sp.a_map, A_k, rk, S, lda_k, DBK, DBM);
  if (rc) return rc;
  rc = encode_tmap_2d_bf16(&sp.b_map, Vk_layer, rk, static_cast<uint64_t>(H) * D, ldv_k, DBK, DBN);
  if (rc) return rc;
  rc = encode_tmap_2d_bf16(&sp.b_head_map, Vk_layer, rk, static_cast<uint64_t>(H) * D, ldv_k, DBK, D);
  if (rc) return rc;
  const bool q_tma_ok = D == 128 && (reinterpret_cast<uintptr_t>(q) & 15) == 0;
  if (q_tma_ok) {
    rc = encode_tmap_2d_bf16(&sp.q_map, q, D, rows, D, 64, R_QROWS);
    if (rc) return rc;
    rc = encode_tmap_2d_bf16(&sp.q_half_map, q, D, rows, D, 64, pair_nq16(qpk) / 2);
    if (rc) return rc;
    rc = encode_tmap_2d_bf16(&sp.b_half_map, Vk_layer, rk, static_cast<uint64_t>(H) * D, ldv_k, DBK, 64);
    if (rc) return rc;
  }
  sp.q = static_cast<const __nv_bfloat16*>(q);
  sp.cos = static_cast<const __nv_bfloat16*>(cos);
  sp.sin = static_cast<const __nv_bfloat16*>(sin);
  sp.scores = scores;
  sp.ld_cs = ld_cs;
  sp.ld_scores = ldl;
  sp.S = S;
  sp.rk = rk;
  sp.H = H;
  sp.qpk = qpk;
  sp.npass = 1;
  sp.tiles_n = (H * D + DBN - 1) / DBN;
  sp.nkb = (rk + DBK - 1) / DBK;
  sp.scale = scale;
  sp.stages = r_stages_for(sp.nkb);
  const int grid = ((S + DBM - 1) / DBM) * sp.tiles_n;
  static PerDevice<bool> configured;
  if (!configured()) {
    XKV_CHECK_CUDA(cudaFuncSetAttribute(decode_scores_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(D_SMEM_BYTES)));
    XKV_CHECK_CUDA(cudaFuncSetAttribute(decode_scores_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(D_SMEM_BYTES)));
    XKV_CHECK_CUDA(cudaFuncSetAttribute(decode_scores_persistent_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(P_SMEM_BYTES)));
    XKV_CHECK_CUDA(cudaFuncSetAttribute(decode_scores_persistent_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(P_SMEM_BYTES)));
    configured() = true;
  }
  // CTA pairs (half a slice per CTA, deep ring) when the head layout allows the score MMA: the default for head_dim 128
  if (D == 128 && q_tma_ok && qpk <= PR_SCORE_COLS && !g_force_tiled_scores && (g_scores_variant == 0 || g_scores_variant == 3)) {
    const int prc = launch_scores_pair(sp, S, H, st);
    if (prc > 0) return prc;
    if (prc == 0) {
      XKV_LAUNCHED();
      return 0;
    }
    sp.stages = r_stages_for(sp.nkb);
  }
  sp.npass = npass;
  const int nv = H * npass;   // row sets: (kv head, pass)
  // persistent kernel when one head's slice of the right factor fits in shared memory
  const bool persistent = static_cast<size_t>(sp.nkb) * D * DBK * 2 <= PB_MAX_BYTES && !g_force_tiled_scores;
  if (persistent) {
    const int sms = device_sm_count();
    const int ntiles = (S + DBM - 1) / DBM;
    int pgrid = sms < ntiles * nv ? sms : ntiles * nv;
    if (pgrid < nv) pgrid = nv;   // every row set needs at least one CTA
    if (D == 128 && q_tma_ok && g_scores_variant != 1) {
      rc = launch_scores_mma2(sp, S, nv, st);
      if (rc) return rc;
    } else if (D == 128)
      decode_scores_persistent_kernel<128><<<pgrid, P_THREADS, P_SMEM_BYTES, st>>>(sp);
    else
      decode_scores_persistent_kernel<64><<<pgrid, P_THREADS, P_SMEM_BYTES, st>>>(sp);
  } else if (D == 128) {
    decode_scores_kernel<128><<<dim3(grid, npass), D_THREADS, D_SMEM_BYTES, st>>>(sp);
  } else {
    decode_scores_kernel<64><<<dim3(grid, npass), D_THREADS, D_SMEM_BYTES, st>>>(sp);
  }
  XKV_LAUNCHED();
  return 0;
}

}  // namespace xkv

using namespace xkv;

// Hq: q rows (q heads x query tokens of a multi-token step)
extern "C" size_t xkv_decode_workspace_bytes(int Hq, int S, int T, int rv) {
  const size_t L = static_cast<size_t>(S) + T;
  const size_t ldl = (L + 63) / 64 * 64;
  const int nkb = (S + 63) / 64;
  (void)nkb;
  const int split = 64;   // upper bound of decode_split_k
  const size_t prob_rows = (static_cast<size_t>(Hq) + 127) / 128 * 128;
  size_t b = 0;
  b += al(Hq * ldl * 4);            // scores
  b += al(prob_rows * ldl * 2);     // probabilities (bf16), padded to full 128-row tiles
  b += al(2 * Hq * SM_MAX_CHUNKS * 4);   // per-chunk max / sum of the softmax
  b += al(static_cast<size_t>(split + 1) * Hq * rv * 4);  // split-K slabs of U, then U itself
  return b + 1024;
}

// A dense slot of a one-sided group: (H, S, D) or (S, H, D) view, unit inner stride
struct DenseSlot {
  const void* ptr;
  int64_t stride_h, stride_t;
};

// 3-D tensor map over a dense slot: box {64 dims, `tile` tokens, 1 head}; the token and head dimensions go in the order
// of their strides.  Returns the map's token dimension (1 or 2) through tok_dim.
static int encode_slot_map(CUtensorMap* map, const DenseSlot& slot, int D, int S, int H, int tile, int* tok_dim) {
  const bool tok_first = slot.stride_t <= slot.stride_h;
  const uint64_t dims[3] = {static_cast<uint64_t>(D), static_cast<uint64_t>(tok_first ? S : H), static_cast<uint64_t>(tok_first ? H : S)};
  const uint64_t strides[2] = {static_cast<uint64_t>(tok_first ? slot.stride_t : slot.stride_h),
                               static_cast<uint64_t>(tok_first ? slot.stride_h : slot.stride_t)};
  const uint32_t box[3] = {64u, tok_first ? static_cast<uint32_t>(tile) : 1u, tok_first ? 1u : static_cast<uint32_t>(tile)};
  *tok_dim = tok_first ? 1 : 2;
  return encode_tmap_3d_bf16(map, slot.ptr, dims, strides, box);
}

// Chunks of the dense-value product: about one wave of (kv head, chunk) CTAs, at most 64 (the slab reduction's limit),
// no empty chunk.
static int dense_value_chunks(int S, int H) {
  const int nkb = (S + DN_VBLK - 1) / DN_VBLK;
  int split = device_sm_count() / H;
  if (split > nkb) split = nkb;
  if (split > 64) split = 64;
  if (split < 1) split = 1;
  const int per = (nkb + split - 1) / split;
  return (nkb + per - 1) / per;
}

template <int D, int NQ16>
static int launch_dense_kernel(bool values, const DenseParams& p, int grid, size_t smem, cudaStream_t st) {
  static PerDevice<bool> configured;
  if (!configured()) {
    XKV_CHECK_CUDA(cudaFuncSetAttribute(decode_dense_scores_kernel<D, NQ16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(R_SMEM_LIMIT)));
    XKV_CHECK_CUDA(cudaFuncSetAttribute(decode_dense_values_kernel<D, NQ16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(R_SMEM_LIMIT)));
    configured() = true;
  }
  if (values)
    decode_dense_values_kernel<D, NQ16><<<grid, DN_THREADS, smem, st>>>(p);
  else
    decode_dense_scores_kernel<D, NQ16><<<grid, DN_THREADS, smem, st>>>(p);
  XKV_LAUNCHED();
  return 0;
}

template <int D>
static int launch_dense_d(bool values, const DenseParams& p, int nq16, int grid, size_t smem, cudaStream_t st) {
  switch (nq16) {
    case 16: return launch_dense_kernel<D, 16>(values, p, grid, smem, st);
    case 32: return launch_dense_kernel<D, 32>(values, p, grid, smem, st);
    case 48: return launch_dense_kernel<D, 48>(values, p, grid, smem, st);
    default: return launch_dense_kernel<D, 64>(values, p, grid, smem, st);
  }
}

// scores[r][t] = scale * q_r . K[t, h(r)] over the dense (already rotated) prefix keys: decode_dense_scores_kernel,
// one CTA per (kv head, slot) up to one per SM.
static int launch_dense_scores(const void* q, int rows, int H, int D, const DenseSlot& k, int S, float scale, float* scores,
                               long long ldl, cudaStream_t st) {
  static thread_local DenseParams p;
  std::memset(&p, 0, sizeof(p));
  const int qpk = rows / H, nq16 = pair_nq16(qpk);
  int rc = encode_slot_map(&p.slot_map, k, D, S, H, DBM, &p.slot_tok_dim);
  if (rc) return rc;
  rc = encode_tmap_2d_bf16(&p.rows_map, q, D, rows, D, 64, nq16);
  if (rc) return rc;
  p.out = scores, p.ld_out = ldl, p.S = S, p.H = H, p.qpk = qpk, p.rows = rows, p.scale = scale;
  const size_t tile = static_cast<size_t>(D / 64) * DBM * 128, fixed = static_cast<size_t>(D / 64) * nq16 * 128 + 1024 + 512;
  p.stages = static_cast<int>((R_SMEM_LIMIT - fixed) / tile);
  if (p.stages > DN_MAX_STAGES) p.stages = DN_MAX_STAGES;
  const int ntiles = (S + DBM - 1) / DBM;
  int grid = device_sm_count() < ntiles * H ? device_sm_count() : ntiles * H;
  if (grid < H) grid = H;
  const size_t smem = fixed + p.stages * tile;
  return D == 128 ? launch_dense_d<128>(false, p, nq16, grid, smem, st) : launch_dense_d<64>(false, p, nq16, grid, smem, st);
}

// slabs[c] (rows, D) = P[:, chunk c] V (kv head of the row) over the dense prefix values: decode_dense_values_kernel,
// one CTA per (kv head, chunk)
static int launch_dense_values(const __nv_bfloat16* prob, long long ldp, int rows, int H, int D, const DenseSlot& v, int S,
                               int kps, int nchunks, float* slabs, cudaStream_t st) {
  static thread_local DenseParams p;
  std::memset(&p, 0, sizeof(p));
  const int qpk = rows / H, nq16 = pair_nq16(qpk);
  int rc = encode_slot_map(&p.slot_map, v, D, S, H, DN_VBLK, &p.slot_tok_dim);
  if (rc) return rc;
  rc = encode_tmap_2d_bf16(&p.rows_map, prob, S, rows, ldp, 64, nq16);
  if (rc) return rc;
  p.out = slabs, p.ld_out = D, p.S = S, p.H = H, p.qpk = qpk, p.rows = rows, p.kps = kps;
  const size_t stage = 2 * DN_VBLK * 128 + static_cast<size_t>(nq16) * 128, fixed = 1024 + 512;
  p.stages = static_cast<int>((R_SMEM_LIMIT - fixed) / stage);
  if (p.stages > DN_MAX_STAGES) p.stages = DN_MAX_STAGES;
  const size_t smem = fixed + p.stages * stage;
  return D == 128 ? launch_dense_d<128>(true, p, nq16, H * nchunks, smem, st)
                  : launch_dense_d<64>(true, p, nq16, H * nchunks, smem, st);
}

// The fused chain behind xkv_decode_attention_multi (both sides factored: A_k and A_v given) and
// xkv_decode_attention_half (one side given as a dense slot instead): scores of the prefix, chunk-local softmax with the
// causal tail, the value product per chunk, slab reduction + combine.  Arguments are checked by the callers.
static int decode_chain(const void* q, int Hq, int Tq, int H, int D, const void* A_k, int64_t lda_k, int rk,
                        const void* Vk_layer, int64_t ldv_k, const DenseSlot& k_dense, const void* A_v, int64_t lda_v, int rv,
                        const void* Vv_layer, int64_t ldv_v, const DenseSlot& v_dense, int S, const void* cos,
                        const void* sin, int64_t ld_cs, const void* k_tail, const void* v_tail, int T,
                        int64_t tail_stride_h, int64_t tail_stride_t, float scale, void* out, void* workspace,
                        void* stream, float* lse_out) {
  cudaStream_t st = as_stream(stream);
  const bool dense_k = A_k == nullptr, dense_v = A_v == nullptr;
  const int rows = Hq * Tq;
  const int qpk = rows / H;
  const int vw = dense_v ? D : rv;   // columns of U: the value factor's rank, or head_dim for a dense value slot
  const size_t L = static_cast<size_t>(S) + T;
  const long long ldl = static_cast<long long>((L + 63) / 64 * 64);
  const int nkb_s = (S + 63) / 64;
  (void)nkb_s;
  const int split = dense_v ? dense_value_chunks(S, H) : decode_split_k(S, rv, rows);
  char* w = static_cast<char*>(workspace);
  float* scores = reinterpret_cast<float*>(w);
  w += al(rows * ldl * 4);
  __nv_bfloat16* prob = reinterpret_cast<__nv_bfloat16*>(w);
  w += al((static_cast<size_t>(rows) + 127) / 128 * 128 * ldl * 2);
  float* rowsum = reinterpret_cast<float*>(w);        // per-chunk sums of p
  float* chunk_max = rowsum + rows * SM_MAX_CHUNKS;
  w += al(2 * rows * SM_MAX_CHUNKS * 4);
  float* u_slabs = reinterpret_cast<float*>(w);
  w += al(static_cast<size_t>(split + 1) * rows * vw * 4);

  // ---- scores of the prefix: fused reconstruct + RoPE + q.K, or q.K over the dense rotated keys ----
  int rc = dense_k ? launch_dense_scores(q, rows, H, D, k_dense, S, scale, scores, ldl, st)
                   : launch_scores(q, rows, H, D, A_k, lda_k, rk, Vk_layer, ldv_k, S, cos, sin, ld_cs, scale, scores, ldl, st);
  if (rc) return rc;
  // ---- softmax with chunk-local maxima: chunk c = token range of split-K slab c, last chunk = the dense tail ----
  const int nkb_p = (S + 63) / 64;
  const int kps = (nkb_p + split - 1) / split;          // k-blocks per slab, as xkv_gemm_grouped cuts them
  const int nchunks = split + 1;
  XKV_REQUIRE(nchunks <= SM_MAX_CHUNKS, "decode: too many softmax chunks");
  softmax_chunk_kernel<<<(rows * split + 7) / 8 + rows, 256, 0, st>>>(scores, ldl, S, T, Tq, kps, split, rows, static_cast<const __nv_bfloat16*>(q),
                                                          static_cast<const __nv_bfloat16*>(k_tail), tail_stride_h,
                                                          tail_stride_t, qpk, D, scale, prob, ldl, chunk_max, rowsum, nullptr, nullptr,
                                                          0.f);
  XKV_LAUNCHED();
  if (dense_v) {
    // ---- U_c = P[:, chunk c] V_h per softmax chunk, then o = (sum_c w_c U_c + P_tail V_tail) / rowsum ----
    rc = launch_dense_values(prob, ldl, rows, H, D, v_dense, S, kps, split, u_slabs, st);
    if (rc) return rc;
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(rows, RC_CL, 1);
    cfg.blockDim = dim3(256, 1, 1);
    cfg.dynamicSmemBytes = D * sizeof(float);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 1;
    attr[0].val.clusterDim.y = RC_CL;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    XKV_CHECK_CUDA(cudaLaunchKernelEx(&cfg, reduce_combine_kernel<true>, static_cast<const float*>(u_slabs), split,
                                      static_cast<long long>(rows) * D, D, static_cast<const __nv_bfloat16*>(nullptr),
                                      0LL, static_cast<const __nv_bfloat16*>(prob), ldl, S, T, Tq,
                                      static_cast<const __nv_bfloat16*>(v_tail), static_cast<long long>(tail_stride_h),
                                      static_cast<long long>(tail_stride_t), static_cast<const float*>(rowsum), qpk, D,
                                      static_cast<__nv_bfloat16*>(out), static_cast<const float*>(chunk_max), nchunks, lse_out));
    XKV_LAUNCHED();
    return 0;
  }
  // ---- U = P[:, :S] * A_v  (tokens are the contraction: P K-major, A_v MN-major) ----
  xkv_gemm_problem gp;
  std::memset(&gp, 0, sizeof(gp));
  gp.M = rows;
  gp.N = rv;
  gp.K = S;
  gp.num_terms = 1;
  gp.a_mn_major = 0;
  gp.b_mn_major = 1;
  gp.A[0] = prob;
  gp.B[0] = A_v;
  gp.lda = ldl;
  gp.ldb = lda_v;
  gp.D = u_slabs;
  gp.ldd = rv;
  gp.split_k = split;
  gp.split_stride = static_cast<long long>(rows) * rv;
  rc = xkv_gemm_grouped(&gp, 1, stream);
  if (rc) return rc;
  // ---- o = (U Bv_l^T + P_tail V_tail) / rowsum, U reduced over the split-K slabs by the same launch ----
  if (rv <= 128 * RC_CL && split <= 64 && !g_split_reduce_combine) {
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(rows, RC_CL, 1);
    cfg.blockDim = dim3(256, 1, 1);
    cfg.dynamicSmemBytes = rv * sizeof(float);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 1;
    attr[0].val.clusterDim.y = RC_CL;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    XKV_CHECK_CUDA(cudaLaunchKernelEx(&cfg, reduce_combine_kernel<false>, static_cast<const float*>(u_slabs), split,
                                      static_cast<long long>(rows) * rv, rv, static_cast<const __nv_bfloat16*>(Vv_layer),
                                      static_cast<long long>(ldv_v), static_cast<const __nv_bfloat16*>(prob), ldl, S, T, Tq,
                                      static_cast<const __nv_bfloat16*>(v_tail), static_cast<long long>(tail_stride_h),
                                      static_cast<long long>(tail_stride_t), static_cast<const float*>(rowsum), qpk, D,
                                      static_cast<__nv_bfloat16*>(out), static_cast<const float*>(chunk_max), nchunks, lse_out));
    XKV_LAUNCHED();
    return 0;
  }
  float* U = u_slabs + static_cast<size_t>(split) * rows * rv;
  reduce_u_kernel<<<dim3((rv + 63) / 64, rows), 256, 0, st>>>(u_slabs, split, static_cast<long long>(rows) * rv, rv, chunk_max,
                                                              rowsum, nchunks, U, 0, nullptr);
  XKV_LAUNCHED();
  combine_kernel<<<dim3(rows, (D + 7) / 8), 256, rv * sizeof(float), st>>>(
      U, 1, 0, rv, static_cast<const __nv_bfloat16*>(Vv_layer), ldv_v, prob, ldl, S,
      T, Tq, static_cast<const __nv_bfloat16*>(v_tail), tail_stride_h, tail_stride_t, rowsum, qpk, D,
      static_cast<__nv_bfloat16*>(out), chunk_max, nchunks, lse_out);
  XKV_LAUNCHED();
  return 0;
}

// Multi-token step: q / out (Hq * Tq, D), row hq * Tq + t = query token t of q head hq; the last Tq of the T tail tokens
// are the queries' own and attention among them is causal.  Internally every per-head quantity is per ROW (rows = Hq Tq,
// qpk below = rows per kv head).
extern "C" int xkv_decode_attention_multi(const void* q, int Hq, int Tq, int H, int D, const void* A_k, int64_t lda_k, int rk,
                                          const void* Vk_layer, int64_t ldv_k, const void* A_v, int64_t lda_v, int rv,
                                          const void* Vv_layer, int64_t ldv_v, int S, const void* cos, const void* sin,
                                          int64_t ld_cs, const void* k_tail, const void* v_tail, int T, int64_t tail_stride_h,
                                          int64_t tail_stride_t, float scale, void* out, void* workspace,
                                          size_t workspace_bytes, void* stream, float* lse_out) {
  XKV_REQUIRE(q && A_k && Vk_layer && A_v && Vv_layer && out && workspace, "decode: null argument");
  XKV_REQUIRE(D == 64 || D == 128, "decode: head_dim %d not supported (64 or 128)", D);
  XKV_REQUIRE(Tq >= 1, "decode: Tq=%d query tokens (at least 1)", Tq);
  XKV_REQUIRE(H >= 1 && Hq >= 1 && Hq % H == 0, "decode: unsupported head counts Hq=%d H=%d", Hq, H);
  XKV_REQUIRE((Hq / H) * Tq <= 64 && Hq * Tq <= 512,
              "decode: %d q heads per kv head x %d query tokens (at most 64 rows per kv head) and %d q heads (at most 512 "
              "rows in all) is past the fused kernel's bounds", Hq / H, Tq, Hq);
  XKV_REQUIRE(S >= 1 && T >= 0 && rk >= 1 && rv >= 1 && rv % 2 == 0, "decode: bad sizes");
  // a single query may come without a tail (xkv_decode_attention); several queries attend to their own tokens
  XKV_REQUIRE(Tq == 1 || T >= Tq, "decode: the tail (T=%d) must hold the Tq=%d query tokens", T, Tq);
  XKV_REQUIRE(T == 0 || (k_tail && v_tail), "decode: tail pointers missing");
  XKV_REQUIRE((cos == nullptr) == (sin == nullptr), "decode: cos and sin must both be given or both be null");
  XKV_REQUIRE(cos == nullptr || ld_cs % 8 == 0, "decode: cos/sin row stride must be a multiple of 8");
  XKV_REQUIRE(workspace_bytes >= xkv_decode_workspace_bytes(Hq * Tq, S, T, rv), "decode: workspace too small");
  XKV_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "decode: workspace must be 256-byte aligned");
  const DenseSlot none = {nullptr, 0, 0};
  return decode_chain(q, Hq, Tq, H, D, A_k, lda_k, rk, Vk_layer, ldv_k, none, A_v, lda_v, rv, Vv_layer, ldv_v, none, S, cos,
                      sin, ld_cs, k_tail, v_tail, T, tail_stride_h, tail_stride_t, scale, out, workspace, stream, lse_out);
}

extern "C" size_t xkv_decode_half_workspace_bytes(int rows, int S, int T, int value_width) {
  // the layout of xkv_decode_workspace_bytes; the slabs are value_width (r_v, or head_dim for a dense value slot) wide
  return xkv_decode_workspace_bytes(rows, S, T, value_width);
}

extern "C" int xkv_decode_attention_half(const void* q, int Hq, int Tq, int H, int D, const void* A_k, int64_t lda_k, int rk,
                                         const void* Vk_layer, int64_t ldv_k, const void* k_dense, int64_t k_stride_h,
                                         int64_t k_stride_t, const void* A_v, int64_t lda_v, int rv, const void* Vv_layer,
                                         int64_t ldv_v, const void* v_dense, int64_t v_stride_h, int64_t v_stride_t, int S,
                                         const void* cos, const void* sin, int64_t ld_cs, const void* k_tail,
                                         const void* v_tail, int T, int64_t tail_stride_h, int64_t tail_stride_t,
                                         float scale, void* out, void* workspace, size_t workspace_bytes, void* stream,
                                         float* lse_out) {
  const bool kf = A_k != nullptr, vf = A_v != nullptr;
  XKV_REQUIRE(!(kf && k_dense) && !(vf && v_dense), "decode_half: a side is given both as factors and as a dense slot");
  XKV_REQUIRE((kf || k_dense) && (vf || v_dense), "decode_half: the key and the value side each need factors or a dense slot");
  XKV_REQUIRE(kf != vf,
              "decode_half: exactly one side must be factored (both factored: xkv_decode_attention_multi; both dense: SDPA)");
  XKV_REQUIRE(q && out && workspace && (!kf || Vk_layer) && (!vf || Vv_layer), "decode_half: null argument");
  XKV_REQUIRE(D == 64 || D == 128, "decode_half: head_dim %d not supported (64 or 128)", D);
  XKV_REQUIRE(Tq >= 1, "decode_half: Tq=%d query tokens (at least 1)", Tq);
  XKV_REQUIRE(H >= 1 && Hq >= 1 && Hq % H == 0, "decode_half: unsupported head counts Hq=%d H=%d", Hq, H);
  XKV_REQUIRE((Hq / H) * Tq <= 64 && Hq * Tq <= 512,
              "decode_half: %d q heads per kv head x %d query tokens (at most 64 rows per kv head) and %d q heads (at most "
              "512 rows in all) is past the fused kernel's bounds", Hq / H, Tq, Hq);
  XKV_REQUIRE(S >= 1 && T >= 0 && (!kf || rk >= 1) && (!vf || (rv >= 1 && rv % 2 == 0)), "decode_half: bad sizes");
  XKV_REQUIRE(Tq == 1 || T >= Tq, "decode_half: the tail (T=%d) must hold the Tq=%d query tokens", T, Tq);
  XKV_REQUIRE(T == 0 || (k_tail && v_tail), "decode_half: tail pointers missing");
  XKV_REQUIRE((cos == nullptr) == (sin == nullptr), "decode_half: cos and sin must both be given or both be null");
  XKV_REQUIRE(cos == nullptr || ld_cs % 8 == 0, "decode_half: cos/sin row stride must be a multiple of 8");
  const void* dense = kf ? v_dense : k_dense;
  const int64_t sh = kf ? v_stride_h : k_stride_h, stt = kf ? v_stride_t : k_stride_t;
  // TMA reads the slot in place: 16-byte aligned base, strides of whole 16-byte units (a slot is never copied)
  XKV_REQUIRE((reinterpret_cast<uintptr_t>(dense) & 15) == 0 && sh > 0 && stt > 0 && sh % 8 == 0 && stt % 8 == 0,
              "decode_half: the dense %s slot needs a 16-byte aligned base and head / token strides that are positive "
              "multiples of 8 elements (got %lld / %lld)", kf ? "value" : "key", static_cast<long long>(sh),
              static_cast<long long>(stt));
  XKV_REQUIRE(kf || (reinterpret_cast<uintptr_t>(q) & 15) == 0, "decode_half: q must be 16-byte aligned");
  XKV_REQUIRE(workspace_bytes >= xkv_decode_half_workspace_bytes(Hq * Tq, S, T, vf ? rv : D), "decode_half: workspace too small");
  XKV_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "decode_half: workspace must be 256-byte aligned");
  const DenseSlot ks = {k_dense, k_stride_h, k_stride_t}, vs = {v_dense, v_stride_h, v_stride_t};
  return decode_chain(q, Hq, Tq, H, D, A_k, lda_k, rk, Vk_layer, ldv_k, ks, A_v, lda_v, rv, Vv_layer, ldv_v, vs, S, cos, sin,
                      ld_cs, k_tail, v_tail, T, tail_stride_h, tail_stride_t, scale, out, workspace, stream, lse_out);
}

extern "C" int xkv_decode_attention_lse(const void* q, int Hq, int H, int D, const void* A_k, int64_t lda_k, int rk,
                                        const void* Vk_layer, int64_t ldv_k, const void* A_v, int64_t lda_v, int rv,
                                        const void* Vv_layer, int64_t ldv_v, int S, const void* cos, const void* sin,
                                        int64_t ld_cs, const void* k_tail, const void* v_tail, int T, int64_t tail_stride_h,
                                        int64_t tail_stride_t, float scale, void* out, void* workspace,
                                        size_t workspace_bytes, void* stream, float* lse_out) {
  XKV_REQUIRE(H >= 1 && Hq % H == 0 && Hq / H <= D_MAX_QPK && Hq <= 128, "decode: unsupported head counts Hq=%d H=%d", Hq, H);
  return xkv_decode_attention_multi(q, Hq, 1, H, D, A_k, lda_k, rk, Vk_layer, ldv_k, A_v, lda_v, rv, Vv_layer, ldv_v, S, cos,
                                    sin, ld_cs, k_tail, v_tail, T, tail_stride_h, tail_stride_t, scale, out, workspace,
                                    workspace_bytes, stream, lse_out);
}

extern "C" size_t xkv_decode_absorbed_workspace_bytes(int Hq, int S, int r) {
  const size_t ldl = (static_cast<size_t>(S) + 63) / 64 * 64;
  size_t b = 0;
  b += 2 * al(Hq * ldl * 4);                                // scores, bias scores
  b += al(128 * ldl * 2);                                   // probabilities (bf16)
  b += al(2 * Hq * SM_MAX_CHUNKS * 4);                      // per-chunk max / sum
  b += al(static_cast<size_t>(64 + 1) * Hq * r * 4);        // split-K slabs of U, then U
  return b + 1024;
}

extern "C" int xkv_decode_absorbed(const void* q_hat, int Hq, const void* A, int64_t lda, int r, int S,
                                   const float* row_scale, const void* bias_q, const void* bias_k, int64_t ld_bias_k,
                                   int bias_dim, float scale, float* u_out, float* lse_out, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  XKV_REQUIRE(q_hat && A && u_out && workspace, "absorbed decode: null argument");
  XKV_REQUIRE(Hq >= 1 && Hq <= 128 && S >= 1 && r >= 8 && r % 8 == 0 && lda % 8 == 0, "absorbed decode: bad sizes");
  XKV_REQUIRE((bias_q == nullptr) == (bias_k == nullptr), "absorbed decode: bias_q and bias_k go together");
  XKV_REQUIRE(bias_q == nullptr || (bias_dim >= 8 && bias_dim % 8 == 0 && ld_bias_k % 8 == 0),
              "absorbed decode: the bias width must be a multiple of 8");
  XKV_REQUIRE(workspace_bytes >= xkv_decode_absorbed_workspace_bytes(Hq, S, r), "absorbed decode: workspace too small");
  XKV_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "absorbed decode: workspace must be 256-byte aligned");
  cudaStream_t st = as_stream(stream);
  const long long ldl = static_cast<long long>((static_cast<size_t>(S) + 63) / 64 * 64);
  const int split = decode_split_k(S, r, Hq);
  char* w = static_cast<char*>(workspace);
  float* scores = reinterpret_cast<float*>(w);
  w += al(Hq * ldl * 4);
  float* bias = reinterpret_cast<float*>(w);
  w += al(Hq * ldl * 4);
  __nv_bfloat16* prob = reinterpret_cast<__nv_bfloat16*>(w);
  w += al(128 * ldl * 2);
  float* rowsum = reinterpret_cast<float*>(w);
  float* chunk_max = rowsum + Hq * SM_MAX_CHUNKS;
  w += al(2 * Hq * SM_MAX_CHUNKS * 4);
  float* u_slabs = reinterpret_cast<float*>(w);
  // ---- raw scores: q^ A^T (and the bias term q_pe k_pe^T), tokens along N ----
  xkv_gemm_problem gp[2];
  std::memset(gp, 0, sizeof(gp));
  gp[0].M = Hq, gp[0].N = S, gp[0].K = r, gp[0].num_terms = 1;
  gp[0].A[0] = q_hat, gp[0].B[0] = A, gp[0].lda = r, gp[0].ldb = lda;
  gp[0].D = scores, gp[0].ldd = ldl, gp[0].split_k = 1;
  int np = 1;
  if (bias_q != nullptr) {
    gp[1].M = Hq, gp[1].N = S, gp[1].K = bias_dim, gp[1].num_terms = 1;
    gp[1].A[0] = bias_q, gp[1].B[0] = bias_k, gp[1].lda = bias_dim, gp[1].ldb = ld_bias_k;
    gp[1].D = bias, gp[1].ldd = ldl, gp[1].split_k = 1;
    np = 2;
  }
  int rc = xkv_gemm_grouped(gp, np, stream);
  if (rc) return rc;
  // ---- softmax with chunk-local maxima (chunk c = token range of split-K slab c; no dense tail here); the per-token
  // scale, the bias term and the softmax scale are applied to the raw products on the fly, and the probabilities leave
  // already multiplied by the value-side per-token scale (three elementwise launches folded into this one) ----
  const int nkb_p = (S + 63) / 64;
  const int kps = (nkb_p + split - 1) / split;
  const int nchunks = split + 1;
  XKV_REQUIRE(nchunks <= SM_MAX_CHUNKS, "absorbed decode: too many softmax chunks");
  XKV_REQUIRE(scale != 0.f, "absorbed decode: the softmax scale must not be zero");
  XKV_REQUIRE(row_scale == nullptr || (reinterpret_cast<uintptr_t>(row_scale) & 15) == 0, "absorbed decode: row_scale must be 16-byte aligned");
  softmax_chunk_kernel<<<(Hq * split + 7) / 8 + Hq, 256, 0, st>>>(scores, ldl, S, 0, 1, kps, split, Hq, nullptr, nullptr, 0, 0, 1, 0, scale,
                                                          prob, ldl, chunk_max, rowsum, bias_q != nullptr ? bias : nullptr,
                                                          row_scale, scale);
  XKV_LAUNCHED();
  // ---- U = P' A (tokens are the contraction) ----
  xkv_gemm_problem gu;
  std::memset(&gu, 0, sizeof(gu));
  gu.M = Hq, gu.N = r, gu.K = S, gu.num_terms = 1;
  gu.a_mn_major = 0, gu.b_mn_major = 1;
  gu.A[0] = prob, gu.B[0] = A, gu.lda = ldl, gu.ldb = lda;
  gu.D = u_slabs, gu.ldd = r, gu.split_k = split;
  gu.split_stride = static_cast<long long>(Hq) * r;
  rc = xkv_gemm_grouped(&gu, 1, stream);
  if (rc) return rc;
  // slab reduction, normalisation and log-sum-exp in one launch
  reduce_u_kernel<<<dim3((r + 63) / 64, Hq), 256, 0, st>>>(u_slabs, split, static_cast<long long>(Hq) * r, r, chunk_max, rowsum,
                                                           nchunks, u_out, 1, lse_out);
  XKV_LAUNCHED();
  return 0;
}

extern "C" int xkv_rope_bf16(void* x, int64_t ld_row, int rows, int H, int D, const void* cos, const void* sin,
                             int64_t ld_cs, void* stream) {
  XKV_REQUIRE(x && cos && sin && rows > 0 && H > 0 && D % 2 == 0, "rope: bad arguments");
  const long long total = static_cast<long long>(rows) * H * (D / 2);
  long long grid = (total + 255) / 256;
  if (grid > 148 * 16) grid = 148 * 16;
  rope_bf16_kernel<<<static_cast<int>(grid), 256, 0, as_stream(stream)>>>(
      static_cast<__nv_bfloat16*>(x), ld_row, rows, H, D, static_cast<const __nv_bfloat16*>(cos),
      static_cast<const __nv_bfloat16*>(sin), ld_cs);
  XKV_LAUNCHED();
  return 0;
}

extern "C" void xkv_decode_force_tiled(int on) { g_force_tiled_scores = on != 0; }
/* test hook: which persistent scores kernel to use when several apply (0 automatic) */
extern "C" void xkv_decode_set_variant(int variant) {
  g_split_reduce_combine = variant == 4;
  g_scores_variant = variant == 4 ? 0 : variant;
}

extern "C" int xkv_decode_attention(const void* q, int Hq, int H, int D, const void* A_k, int64_t lda_k, int rk,
                                    const void* Vk_layer, int64_t ldv_k, const void* A_v, int64_t lda_v, int rv,
                                    const void* Vv_layer, int64_t ldv_v, int S, const void* cos, const void* sin,
                                    int64_t ld_cs, const void* k_tail, const void* v_tail, int T, int64_t tail_stride_h,
                                    int64_t tail_stride_t, float scale, void* out, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  return xkv_decode_attention_lse(q, Hq, H, D, A_k, lda_k, rk, Vk_layer, ldv_k, A_v, lda_v, rv, Vv_layer, ldv_v, S, cos, sin,
                                  ld_cs, k_tail, v_tail, T, tail_stride_h, tail_stride_t, scale, out, workspace,
                                  workspace_bytes, stream, nullptr);
}
