// Full-ranking evaluation on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
// (reference: recad/workflow/normal.py:57-93 / 111-160; the score tile is lightgcn.py:115-120's
//  U_b . I^T, never materialised.)
//
// Scores are fp32-accurate: every operand block (a user row, a 64-item tile) is scaled by a power of two 2^k so that
// its largest |x| stays below 2^15, and split into two fp16 terms x 2^k = hi + lo (11 + 11 significant bits,
// tc_common.cuh split_f16).  A tile is three kind::f16 MMAs accumulated in fp32 in TMEM:
//       S' = A_hi B_hi^T + A_lo B_hi^T + A_hi B_lo^T = S 2^(ku + kt)     (|error| ~ 2^-21 |a||b|)
// The epilogue works in that scaled domain: the power-of-two rescale is exact, so per tile the thresholds (top-K
// tau, the target scores) and the item bias are multiplied by f = 2^(ku + kt) once, and a score is scaled back only
// when it enters the top-K list.
//
// One CTA = 128 users (one TMEM lane each) x ALL items, streamed as 64-item tiles.  The user operand never touches
// shared memory: the epilogue threads load their user's row, split it in registers and park hi / lo in TMEM with
// tcgen05.st (packed fp16 pairs); the MMAs read A from TMEM (the ".ts" form).  Two CTAs share an SM:
//   warp 0    : TMA producer   -- item tiles (hi + lo, 16 KB) into a 2- to 4-stage ring
//   warp 1    : MMA issuer     -- one thread issues 12 tcgen05.mma (3 passes x 4 k-steps of 16) per tile into one
//                                 of 3 TMEM accumulators (128 lanes x 64 columns)
//   warps 2-9 : epilogue       -- two warpgroups over the same 128 lanes; warpgroup w takes the tiles 1 + w, 3 + w, ...
//                                 and ranks each in two halves: a tcgen05.ld of 32 scores, then, in registers, the
//                                 train-item mask, the target-rank counters and a threshold-filtered top-K insertion.
//                                 Each warpgroup keeps its own counters and K-best list; they are merged at the end.
// TMEM columns: [acc0 | acc1 | acc2 | A_hi A_lo], 64 each (A_hi and A_lo are 32 columns of packed pairs).
// The producer / MMA / epilogue run concurrently on mbarrier pipelines (smem full/empty, TMEM full/empty).
// The targets' scores come from the SAME arithmetic: a first 16-column MMA over the gathered target rows.
//
// RECAD_TC_DEBUG (profiling aids): 2 = TMA + MMA pipeline only (no TMEM loads, no ranking); 3 = ranking epilogue +
// TMA with one MMA of a tile's 12 (the accumulator still holds a realistic, coarser score tile).
#include <limits.h>
#include <math.h>
#include <stdlib.h>

#include "rank_epilogue.cuh"
#include "tc_common.cuh"

namespace recad {

constexpr int kTcM = 128;        // users per CTA = TMEM lanes
constexpr int kTcN = 64;         // items per tile = TMEM columns per accumulator
constexpr int kTcK = 64;         // padded embedding width: one 128-byte row of fp16
constexpr int kTcAW = kTcK / 2;  // TMEM columns of one packed fp16 user operand (hi or lo)
constexpr int kTcMaxStages = 4;
constexpr int kTcAcc = 3;
constexpr int kTcEpi = 2 * kTcM;                             // epilogue threads: two warpgroups
constexpr int kTcThreads = 64 + kTcEpi;
constexpr int kTcTgtN = 16;
constexpr int kTcMaxT = 8;
constexpr int kTcCols = 256;                                 // TMEM columns per CTA
constexpr int kTcColA = kTcAcc * kTcN;                       // first column of A_hi; A_lo follows at + kTcAW
constexpr uint32_t kOperandBytes = kTcN * 128;               // a 64-row item tile of hi or lo: 8 KB
constexpr uint32_t kStageBytes = 2 * kOperandBytes;          // hi + lo: 16 KB
constexpr int kTcBars = 1 + 2 * kTcMaxStages + 2 * kTcAcc;

struct TcMaps {
  CUtensorMap b_hi, b_lo, t_hi, t_lo;
};
// the target ids travel as a kernel parameter: the ranking loop reads them from the constant bank, not from registers
struct TcTargets {
  int32_t id[kTcMaxT];
};

// The MMAs leave a tile's scores scaled by 2^k, k = ku + kt, and the epilogue scales thresholds and bias into that
// domain.  2^k is one normal fp32 only for |k| <= 126, but k reaches beyond when the user row's and the tile's largest
// |x| multiply to below about 2^-96 (both 1 * 2^-50: k = 128) or above 2^156, so it is carried as two factors:
// 2^k = f f2 with f = 2^ka, ka = k held to [-126, 126], and f2 = 2^(k - ka) held to the same range, inv = 1 / f.
// Every rescale is exact for |k| <= 252 (f2 = 1 for |k| <= 126: the common case costs nothing); beyond, only for
// operands whose every score is below fp32's smallest subnormal or above its largest value.
__device__ __forceinline__ void pow2_pair(int k, float& f, float& inv, float& f2) {
  const int ka = max(-126, min(126, k));
  const int kb = max(-126, min(126, k - ka));
  f = __int_as_float((127 + ka) << 23);
  inv = __int_as_float((127 - ka) << 23);
  f2 = __int_as_float((127 + kb) << 23);
}

// one arrival per warp on an mbarrier counted in warps (its lanes' TMEM loads have completed: tcgen05.wait::ld)
__device__ __forceinline__ void warp_arrive(uint32_t bar, uint32_t count) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

// ---------------------------------------------------------------------------------------------- the kernel
template <int TMAX>
__global__ void __launch_bounds__(kTcThreads, 2)
fullrank_tc_kernel(const __grid_constant__ TcMaps maps, const TcTargets tgt, const float* __restrict__ user_emb, int D, int64_t n_items,
                   const int32_t* __restrict__ kexp, const int64_t* __restrict__ user_ids, int64_t n_eval,
                   const int64_t* __restrict__ train_rowptr, const int32_t* __restrict__ train_col,
                   const int32_t* __restrict__ targets, int T, int K, const float* __restrict__ item_bias,
                   int32_t* __restrict__ topk_idx, float* __restrict__ topk_val, int32_t* __restrict__ target_rank,
                   float* __restrict__ target_score, int stages, int dbg) {
  extern __shared__ unsigned char smem_raw[];
  // 128-byte-swizzled operand tiles need a 1024-byte aligned base (the launch reserves the slack)
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  // [stage s: B_hi B_lo]* | top-K values | top-K ids | warpgroup 1's rank counts | barriers | tmem ptr
  // a row's two K-best lists (one per warpgroup) are adjacent: [0, K) and [K, 2K), odd pitch between rows
  const int KP = (2 * K) | 1;
  float* topv = reinterpret_cast<float*>(smem + (size_t)stages * kStageBytes);
  int32_t* topi = reinterpret_cast<int32_t*>(topv + (size_t)KP * kTcM);
  int32_t* rk_wg1 = topi + (size_t)KP * kTcM;
  uint64_t* bars = reinterpret_cast<uint64_t*>(rk_wg1 + kTcMaxT * kTcM);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kTcBars);
  const uint32_t sB = smem_u32(smem);
  const uint32_t bar0 = smem_u32(bars);
  const uint32_t bar_a_full = bar0;
  auto bar_b_full = [&](int s) { return bar0 + 8 * (1 + s); };
  auto bar_b_empty = [&](int s) { return bar0 + 8 * (1 + kTcMaxStages + s); };
  auto bar_acc_full = [&](int a) { return bar0 + 8 * (1 + 2 * kTcMaxStages + a); };
  auto bar_acc_empty = [&](int a) { return bar0 + 8 * (1 + 2 * kTcMaxStages + kTcAcc + a); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n_tiles = (n_items + kTcN - 1) / kTcN;
  const int64_t row0 = (int64_t)blockIdx.x * kTcM;

  if (threadIdx.x == 0) {
    mbar_init(bar_a_full, kTcM);
    for (int s = 0; s < kTcMaxStages; ++s) { mbar_init(bar_b_full(s), 1); mbar_init(bar_b_empty(s), 1); }
    for (int a = 0; a < kTcAcc; ++a) { mbar_init(bar_acc_full(a), 1); mbar_init(bar_acc_empty(a), kTcEpi / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(kTcCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int s = 0;
      uint32_t use = 0;
      for (int64_t j = 0; j <= n_tiles; ++j) {      // j = 0 is the 16-row target tile, j >= 1 item tile j-1
        mbar_wait_relaxed(bar_b_empty(s), (use & 1) ^ 1);
        const uint32_t dst = sB + s * kStageBytes;
        if (j == 0) {
          mbar_expect_tx(bar_b_full(s), 2 * kTcTgtN * 128);
          tma_load_2d(dst, &maps.t_hi, 0, 0, bar_b_full(s));
          tma_load_2d(dst + kOperandBytes, &maps.t_lo, 0, 0, bar_b_full(s));
        } else {
          mbar_expect_tx(bar_b_full(s), kStageBytes);
          const int r = (int)((j - 1) * kTcN);
          tma_load_2d(dst, &maps.b_hi, 0, r, bar_b_full(s));
          tma_load_2d(dst + kOperandBytes, &maps.b_lo, 0, r, bar_b_full(s));
        }
        if (++s == stages) { s = 0; ++use; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      mbar_wait(bar_a_full, 0);                     // the epilogue threads have parked A_hi / A_lo in TMEM
      int s = 0;
      uint32_t use = 0;
      for (int64_t j = 0; j <= n_tiles; ++j) {
        const int a = (int)(j % kTcAcc);
        mbar_wait(bar_b_full(s), use & 1);
        mbar_wait(bar_acc_empty(a), ((uint32_t)(j / kTcAcc) & 1) ^ 1);
        tc_fence_after();
        const uint32_t idesc = j == 0 ? umma_idesc_f16(kTcM, kTcTgtN) : umma_idesc_f16(kTcM, kTcN);
        const uint32_t d = tmem_base + a * kTcN;
        const uint32_t bst = sB + s * kStageBytes;
        const int n_pass = dbg == 3 && j >= 1 ? 1 : 3;
        uint32_t acc = 0;
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {      // hi*hi, lo*hi, hi*lo
          if (pass >= n_pass) break;
          const uint32_t ta = tmem_base + kTcColA + (pass == 1 ? kTcAW : 0);
          const uint32_t bo = bst + (pass == 2 ? kOperandBytes : 0);
#pragma unroll
          for (int k = 0; k < kTcK / 16; ++k) {    // 16 fp16 = 8 packed TMEM columns = 32 bytes of a swizzled row
            if (n_pass == 1 && k) break;
            tc_mma_f16_ts(d, ta + k * 8, umma_desc(bo + k * 32), idesc, acc);
            acc = 1;
          }
        }
        tc_commit(bar_b_empty(s));      // the smem stage is free once these MMAs have read it
        tc_commit(bar_acc_full(a));     // ... and the accumulator is complete
        if (++s == stages) { s = 0; ++use; }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: thread = (user row, column half)
    const int wg = (warp - 2) >> 2;                  // warpgroup: every other tile
    const int q = warp & 3;                          // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;
    const int64_t g = row0 + r;
    const bool active = g < n_eval;
    const int64_t uid = active ? user_ids[g] : 0;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    // the user operand: row -> scale 2^ku -> registers -> (fp16 hi, fp16 lo) pairs -> TMEM lane r
    const float* urow = user_emb + uid * D;
    int ku;
    {
      float m = 0.f;
      if (active)
        for (int d = 0; d < D; ++d) m = fmaxf(m, fabsf(__ldg(urow + d)));
      ku = f16_scale_exp(m);
    }
    if (wg == 0) {
#pragma unroll 1
      for (int c = 0; c < kTcK / 32; ++c) {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          const int d = c * 32 + 2 * e;
          const float x0 = (active && d < D) ? __ldg(urow + d) : 0.f;
          const float x1 = (active && d + 1 < D) ? __ldg(urow + d + 1) : 0.f;
          uint16_t h0, l0, h1, l1;
          split_f16(x0, ku, h0, l0);
          split_f16(x1, ku, h1, l1);
          hi[e] = (uint32_t)h0 | ((uint32_t)h1 << 16);
          lo[e] = (uint32_t)l0 | ((uint32_t)l1 << 16);
        }
        tmem_st16(lane_addr + kTcColA + c * 16, hi);
        tmem_st16(lane_addr + kTcColA + kTcAW + c * 16, lo);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(bar_a_full);
    }
    float* rowv = topv + (size_t)r * KP;
    int32_t* rowi = topi + (size_t)r * KP;
    float* myv = rowv + wg * K;
    int32_t* myi = rowi + wg * K;
    for (int k = 0; k < K; ++k) { myv[k] = -INFINITY; myi[k] = -1; }
    float tau = -INFINITY;
    int min_pos = 0;
    int64_t cur = 0, end = 0;
    if (active) { cur = train_rowptr[uid]; end = train_rowptr[uid + 1]; }
    RankState<TMAX> rs;
    rank_state_init(rs, T, targets, train_col, cur, end);
#pragma unroll
    for (int t = 0; t < TMAX; ++t) rs.tg[t] = tgt.id[t];

    // j = 0: the targets' scores, same arithmetic as every other score (both warpgroups read them)
    mbar_wait(bar_acc_full(0), 0);
    tc_fence_after();
    {
      uint32_t v[16];
      tmem_ld16(lane_addr, v);
      tmem_ld_wait();
      float f, inv, f2;
      pow2_pair(ku + __ldg(kexp + n_tiles), f, inv, f2);
#pragma unroll
      for (int t = 0; t < TMAX; ++t)
        if (t < T) {
          const float s = __uint_as_float(v[t]);
          rank_state_set_score(rs, t, (item_bias ? fmaf(__ldg(item_bias + rs.tg[t]) * f2, f, s) : s) * inv * pow2_inv(f2));
        }
    }
    tc_fence_before();
    warp_arrive(bar_acc_empty(0), 1);                // all 8 warps read the target tile

    // one 32-score chunk, in registers: bias, -inf for train / padding / idle, rank counters, top-K
    auto chunk = [&](const uint32_t (&v)[32], int base, uint32_t train_mask, float f, float inv, float f2) {
      const int lim = min(32, (int)n_items - base);
      if (lim <= 0) return;                          // warp-uniform
      float s[32];
#pragma unroll
      for (int e = 0; e < 32; ++e) s[e] = __uint_as_float(v[e]);
      if (item_bias) {                               // uniform addresses: one broadcast load per item
#pragma unroll
        for (int e = 0; e < 32; ++e) s[e] = (e < lim) ? fmaf(__ldg(item_bias + base + e) * f2, f, s[e]) : s[e];
      }
      const uint32_t drop = train_mask | (lim < 32 ? ~0u << lim : 0u) | (active ? 0u : ~0u);
      if (drop) {
#pragma unroll
        for (int e = 0; e < 32; ++e) s[e] = ((drop >> e) & 1u) ? -INFINITY : s[e];
      }
      rank_topk_chunk<32, TMAX>(s, base, T, rs, tau, myv, myi, K, 1, 0, min_pos, f, inv, f2);
    };

    // warpgroup w ranks the whole tiles j = 1 + w, 3 + w, ...: the per-tile work (barrier, train mask, scale) is paid
    // once per 64 scores, and the other warpgroup's tile is ranked at the same time
    int next_c = cur < end ? train_col[cur] : INT_MAX;   // the user's next train item, kept in a register
    const int nt = (int)n_tiles;
    int kt_next = 1 + wg <= nt ? __ldg(kexp + wg) : 0;  // the next tile's scale exponent
    for (int j = 1 + wg; j <= nt; j += 2) {
      const int a = j % kTcAcc;
      const int j0 = (j - 1) * kTcN;
      uint32_t m0 = 0u, m1 = 0u;                     // train items of this tile (sorted list, walking pointer)
      while (next_c < j0 + kTcN) {
        const unsigned o = (unsigned)(next_c - j0);  // items of the other warpgroup's tiles are stepped over
        if (o < 32u) m0 |= 1u << o;
        else if (o < 64u) m1 |= 1u << (o - 32);
        ++cur;
        next_c = cur < end ? train_col[cur] : INT_MAX;
      }
      const int kt = kt_next;
      if (j + 2 <= nt) kt_next = __ldg(kexp + j + 1);
      float f, inv, f2;
      pow2_pair(ku + kt, f, inv, f2);
      mbar_wait(bar_acc_full(a), (uint32_t)(j / kTcAcc) & 1);
      tc_fence_after();
      if (dbg == 2) {                                // (profiling aid: TMA + MMA pipeline only)
        tc_fence_before();
        warp_arrive(bar_acc_empty(a), 2);
        continue;
      }
      uint32_t v[32];
      tmem_ld32(lane_addr + a * kTcN, v);
      tmem_ld_wait();
      chunk(v, j0, m0, f, inv, f2);
      tmem_ld32(lane_addr + a * kTcN + 32, v);
      tmem_ld_wait();
      // the tile now lives in registers: hand the accumulator back BEFORE ranking its second half
      tc_fence_before();
      warp_arrive(bar_acc_empty(a), 2);              // the 4 warps of one warpgroup stand for all 8
      chunk(v, j0 + 32, m1, f, inv, f2);
    }
    // merge: warpgroup 1 hands over its counts; its K-best list already sits next to warpgroup 0's
    if (wg == 1) {
#pragma unroll
      for (int t = 0; t < TMAX; ++t)
        if (t < T) rk_wg1[t * kTcM + r] = rs.rk[t];
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kTcEpi) : "memory");
    if (wg == 0 && active) {
      topk_finalize(rowv, rowi, 2 * K, 1, 0);      // (score desc, id asc) over both lists; the first K are the K best
      for (int k = 0; k < K; ++k) { topk_idx[g * K + k] = rowi[k]; topk_val[g * K + k] = rowv[k]; }
#pragma unroll
      for (int t = 0; t < TMAX; ++t)
        if (t < T) {
          target_rank[g * T + t] = ((rs.in_train >> t) & 1u) ? -1 : rs.rk[t] + rk_wg1[t * kTcM + r];
          target_score[g * T + t] = rs.st[t];
        }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTcCols) : "memory");
  }
}

// One block per 64-row tile of [n_tiles + 1, 64]: tiles 0 .. n_tiles-1 are the items (zero padded), tile n_tiles the
// T gathered target rows (zero padded to 16).  Each tile gets its scale exponent kexp[tile] from its largest |x| and is
// written as fp16 hi / lo rows of 64 (128 bytes, one 128B-swizzle row).
constexpr int kSplitThreads = 256;
__global__ void __launch_bounds__(kSplitThreads)
split_f16_tiles_kernel(const float* __restrict__ src, int64_t n_items, int D, const int32_t* __restrict__ targets, int T,
                       uint16_t* __restrict__ b_hi, uint16_t* __restrict__ b_lo, uint16_t* __restrict__ t_hi,
                       uint16_t* __restrict__ t_lo, int32_t* __restrict__ kexp) {
  constexpr int kPer = kTcN * kTcK / kSplitThreads;
  __shared__ float wmax[kSplitThreads / 32];
  const int64_t n_tiles = (n_items + kTcN - 1) / kTcN;
  const int64_t tile = blockIdx.x;
  const bool tgt = tile == n_tiles;
  float x[kPer];
  float m = 0.f;
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int e = threadIdx.x + i * kSplitThreads;
    const int r = e / kTcK, d = e % kTcK;
    const int64_t item = tgt ? (r < T ? (int64_t)targets[r] : -1) : tile * kTcN + r;
    x[i] = (item >= 0 && item < n_items && d < D) ? src[item * D + d] : 0.f;
    m = fmaxf(m, fabsf(x[i]));
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
  __syncthreads();
  m = wmax[0];
#pragma unroll
  for (int w = 1; w < kSplitThreads / 32; ++w) m = fmaxf(m, wmax[w]);
  const int k = f16_scale_exp(m);
  if (threadIdx.x == 0) kexp[tile] = k;
  uint16_t* hi = tgt ? t_hi : b_hi + tile * kTcN * kTcK;
  uint16_t* lo = tgt ? t_lo : b_lo + tile * kTcN * kTcK;
#pragma unroll
  for (int i = 0; i < kPer; ++i) {
    const int e = threadIdx.x + i * kSplitThreads;
    if (tgt && e >= kTcTgtN * kTcK) break;
    split_f16(x[i], k, hi[e], lo[e]);
  }
}

static CUresult encode_tiled(CUtensorMap* m, CUtensorMapDataType dt, void* base, const cuuint64_t* dims,
                             const cuuint64_t* strides, const cuuint32_t* box) {
  typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p ||
        q != cudaDriverEntryPointSuccess)
      return CUDA_ERROR_NOT_FOUND;
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  const cuuint32_t estr[2] = {1, 1};
  return fn(m, dt, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

int make_tensor_map_f16x64(CUtensorMap* m, const void* base, int64_t rows, int box_rows) {
  const cuuint64_t dims[2] = {(cuuint64_t)kTcK, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)kTcK * 2};
  const cuuint32_t box[2] = {(cuuint32_t)kTcK, (cuuint32_t)box_rows};
  const CUresult r = encode_tiled(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, const_cast<void*>(base), dims, strides, box);
  RECAD_REQUIRE(r == CUDA_SUCCESS, RECAD_ERR_CUDA, "cuTensorMapEncodeTiled failed with %d", (int)r);
  return RECAD_OK;
}

int make_tensor_map_f32(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int box_rows) {
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
  const cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
  const CUresult r = encode_tiled(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, const_cast<float*>(base), dims, strides, box);
  RECAD_REQUIRE(r == CUDA_SUCCESS, RECAD_ERR_CUDA, "cuTensorMapEncodeTiled failed with %d", (int)r);
  return RECAD_OK;
}

}  // namespace recad

using namespace recad;

extern "C" {

// scratch, in this order: item hi, item lo (fp16 [ip, 64] each, ip = n_items rounded up to 64), target hi, target lo
// (fp16 [16, 64] each), the scale exponents (int32 [ip / 64 + 1]: one per item tile, the target tile last)
int64_t recad_fullrank_tc_scratch_floats(int64_t n_eval, int64_t n_items) {
  (void)n_eval;   // the user operand is split in registers and lives in TMEM
  const int64_t ip = (n_items + kTcN - 1) / kTcN * kTcN;
  return kTcK * (ip + kTcTgtN) + ip / kTcN + 1 + 64;
}

int recad_fullrank_eval_tc(const float* user_emb, const float* item_emb, int64_t n_items, int32_t D,
                           const int64_t* user_ids, int64_t n_eval, const int64_t* train_rowptr,
                           const int32_t* train_col, const int32_t* targets, int32_t T, int32_t K,
                           const float* item_bias, int32_t* topk_idx, float* topk_val, int32_t* target_rank,
                           float* target_score, float* scratch, int64_t scratch_floats, void* stream) {
  cudaStream_t s = as_stream(stream);
  RECAD_REQUIRE(user_emb && item_emb && user_ids && train_rowptr && topk_idx && topk_val && scratch, RECAD_ERR_ARG,
                "fullrank_tc: null pointer");
  RECAD_REQUIRE(n_eval > 0 && n_items > 0 && n_items < (int64_t(1) << 31) - kTcN, RECAD_ERR_ARG, "fullrank_tc: bad sizes");
  RECAD_REQUIRE(D >= 1 && D <= kTcK, RECAD_ERR_UNSUPPORTED, "fullrank_tc: D = %d > %d (use recad_fullrank_eval)", D, kTcK);
  RECAD_REQUIRE(K >= 1 && K <= 32, RECAD_ERR_UNSUPPORTED, "fullrank_tc: K = %d > 32 (use recad_fullrank_eval)", K);
  RECAD_REQUIRE(T >= 0 && T <= kTcMaxT && (T == 0 || (targets && target_rank && target_score)), RECAD_ERR_ARG,
                "fullrank_tc: 0 <= T <= %d targets", kTcMaxT);
  RECAD_REQUIRE(scratch_floats >= recad_fullrank_tc_scratch_floats(n_eval, n_items), RECAD_ERR_SCRATCH,
                "fullrank_tc: scratch too small");
  RECAD_REQUIRE(((uintptr_t)scratch & 255) == 0, RECAD_ERR_ARG, "fullrank_tc: scratch must be 256-byte aligned");
  const int64_t np = (n_eval + kTcM - 1) / kTcM * kTcM, ip = (n_items + kTcN - 1) / kTcN * kTcN;
  uint16_t* b_hi = reinterpret_cast<uint16_t*>(scratch);
  uint16_t* b_lo = b_hi + ip * kTcK;
  uint16_t* t_hi = b_lo + ip * kTcK;
  uint16_t* t_lo = t_hi + kTcTgtN * kTcK;
  int32_t* kexp = reinterpret_cast<int32_t*>(t_lo + kTcTgtN * kTcK);
  split_f16_tiles_kernel<<<(unsigned)(ip / kTcN + 1), kSplitThreads, 0, s>>>(item_emb, n_items, D, targets, T, b_hi, b_lo,
                                                                             t_hi, t_lo, kexp);
  RECAD_LAUNCH_CHECK();
  TcMaps maps;
  TcTargets tgt;
  int rc;
  for (int t = 0; t < kTcMaxT; ++t) tgt.id[t] = -1;
  if (T) RECAD_CUDA_CHECK(cudaMemcpyAsync(tgt.id, targets, (size_t)T * 4, cudaMemcpyDeviceToHost, s));
  if ((rc = make_tensor_map_f16x64(&maps.b_hi, b_hi, ip, kTcN))) return rc;
  if ((rc = make_tensor_map_f16x64(&maps.b_lo, b_lo, ip, kTcN))) return rc;
  if ((rc = make_tensor_map_f16x64(&maps.t_hi, t_hi, kTcTgtN, kTcTgtN))) return rc;
  if ((rc = make_tensor_map_f16x64(&maps.t_lo, t_lo, kTcTgtN, kTcTgtN))) return rc;
  // two CTAs per SM: the deepest ring (up to 4 stages) with which both still fit (1 KB per CTA is reserved by the driver)
  const size_t fixed = 1024 + (size_t)((2 * K) | 1) * kTcM * 8 + (size_t)kTcMaxT * kTcM * 4 + kTcBars * 8 + 16;
  static const int force_stages = getenv("RECAD_TC_STAGES") ? atoi(getenv("RECAD_TC_STAGES")) : 0;
  int stages = 2;
  while (stages < kTcMaxStages && 2 * (fixed + (stages + 1) * kStageBytes + 1024) <= 228 * 1024) ++stages;
  if (force_stages >= 1 && force_stages <= kTcMaxStages) stages = force_stages;
  const size_t smem_bytes = fixed + (size_t)stages * kStageBytes;
  RECAD_REQUIRE(smem_bytes <= 227 * 1024, RECAD_ERR_UNSUPPORTED, "fullrank_tc: shared memory %zu B", smem_bytes);
  static const int dbg = getenv("RECAD_TC_DEBUG") ? atoi(getenv("RECAD_TC_DEBUG")) : 0;
#define RECAD_TC_LAUNCH(TMAX)                                                                                          \
  {                                                                                                                    \
    auto kern = fullrank_tc_kernel<TMAX>;                                                                              \
    RECAD_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));             \
    RECAD_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout,                        \
                                          cudaSharedmemCarveoutMaxShared));                                            \
    kern<<<(unsigned)(np / kTcM), kTcThreads, smem_bytes, s>>>(                                                        \
        maps, tgt, user_emb, D, n_items, kexp, user_ids, n_eval, train_rowptr, train_col, targets, T, K, item_bias,         \
        topk_idx, topk_val, target_rank, target_score, stages, dbg);                                                   \
  }
  if (T == 0) RECAD_TC_LAUNCH(0)
  else if (T == 1) RECAD_TC_LAUNCH(1)
  else if (T == 2) RECAD_TC_LAUNCH(2)
  else if (T <= 4) RECAD_TC_LAUNCH(4)
  else RECAD_TC_LAUNCH(8)
#undef RECAD_TC_LAUNCH
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

}  // extern "C"
