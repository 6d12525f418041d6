// Per-row ranking state shared by the two full-rank kernels (eval.cu: exact CUDA-core, eval_tc.cu: tcgen05).
// A thread owns one user; it is handed the user's scores for NC consecutive items at a time (registers) and
// must (a) count, per target, the items that outrank it and (b) keep the K best (score desc, id asc).
//
// The per-score cost decides the kernel's speed (2e11 scores on the synthetic workload), so:
//   * masked / out-of-range scores are set to -inf up front (only when the chunk has any), after which no
//     per-score branch is needed: -inf never counts and never enters the list;
//   * the tie rule "outranks iff s > s_t, or s == s_t and id < target" becomes ONE compare per score: for a
//     chunk entirely before the target the threshold is nextafter(s_t, -inf) (s >= s_t  <=>  s > that), for
//     a chunk entirely after it s_t; only the single chunk that contains the target takes the exact path;
//   * the top-K list is touched only when the chunk maximum beats the current K-th best.
// The tensor-core kernel hands over scores in a power-of-two scaled domain, s' = s f (f = 2^k, exact): the thresholds
// are scaled instead of the scores (s' > thr f  <=>  s > thr), and only a score entering the list is scaled back
// (s' inv).  f may need two factors, f f2 (a scale beyond 2^126 is not one fp32): thresholds are multiplied by f, then
// by f2, and a score entering the list by inv, then by 1 / f2 (pow2_inv: exact, f2 is a normal power of two).  The exact kernel
// passes f = inv = f2 = 1.
#pragma once
#include <math.h>
#include <stdint.h>

namespace recad {

template <int TMAX>
struct RankState {
  static constexpr int N = TMAX > 0 ? TMAX : 1;
  float st[N];      // target score
  int tg[N];        // target item id
  int rk[N];        // running count
  unsigned in_train = 0;  // bit t: the target is one of the user's train items (reported rank -1)
};

// The K best of a row are kept UNSORTED in shared memory; `tau` / `min_pos` (registers) are the value and slot
// of the current worst entry (lowest score, ties: highest id).  A candidate v > tau overwrites that slot and the
// list is rescanned for the new worst: K independent loads, no dependent shift chain.  Rare (about K ln(I / K)
// times per user), hence out of line.  Items arrive in ascending id and only a STRICTLY better score replaces,
// so among equal scores the lower ids survive.  topk_finalize() sorts once at the end.
static __device__ __noinline__ float topk_replace(float v, int32_t item, float* __restrict__ topv, int32_t* __restrict__ topi,
                                                  int K, int stride, int slot, int& min_pos) {
  topv[min_pos * stride + slot] = v;
  topi[min_pos * stride + slot] = item;
  float mv = topv[slot];
  int mi = topi[slot], mp = 0;
#pragma unroll 4
  for (int k = 1; k < K; ++k) {
    const float x = topv[k * stride + slot];
    const int xi = topi[k * stride + slot];
    if (x < mv || (x == mv && xi > mi)) { mv = x; mi = xi; mp = k; }
  }
  min_pos = mp;
  return mv;
}

// order the row's list by (score desc, id asc); empty slots (id -1, -inf) end up last
static __device__ __noinline__ void topk_finalize(float* __restrict__ topv, int32_t* __restrict__ topi, int K, int stride, int slot) {
  for (int a = 0; a < K - 1; ++a) {
    float bv = topv[a * stride + slot];
    int bi = topi[a * stride + slot], bp = a;
    for (int k = a + 1; k < K; ++k) {
      const float x = topv[k * stride + slot];
      const int xi = topi[k * stride + slot];
      if (xi >= 0 && (bi < 0 || x > bv || (x == bv && xi < bi))) { bv = x; bi = xi; bp = k; }
    }
    if (bp != a) {
      topv[bp * stride + slot] = topv[a * stride + slot];
      topi[bp * stride + slot] = topi[a * stride + slot];
      topv[a * stride + slot] = bv;
      topi[a * stride + slot] = bi;
    }
  }
}

// 1 / x for a normal power of two x, exact, without a division: the exponent field is negated about the bias
__device__ __forceinline__ float pow2_inv(float x) { return __int_as_float(0x7f000000 - __float_as_int(x)); }

// nextafterf(x, -inf) without its branches: one ulp down for finite x and +inf, -0 / +0 -> -denorm_min, -inf and nan stay
__device__ __forceinline__ float next_down(float x) {
  const int b = __float_as_int(x);
  const int n = x == 0.f ? (int)0x80000001 : (b < 0 ? b + 1 : b - 1);
  return (x == -INFINITY || x != x) ? x : __int_as_float(n);
}

// (a): per target, count the scores of this chunk that outrank it
template <int NC, int TMAX>
__device__ __forceinline__ void rank_count_chunk(const float (&s)[NC], int64_t base, int T, RankState<TMAX>& rs, float f = 1.f,
                                                 float f2 = 1.f) {
#pragma unroll
  for (int t = 0; t < TMAX; ++t) {
    if (t < T) {
      const int tg = rs.tg[t];
      if (base + NC <= tg || base > tg) {          // warp-uniform: targets are the same for every user
        const float st = rs.st[t] * f * f2;        // nextafter(st, -inf) is derived here, not carried in a register
        const float thr = base > tg ? st : next_down(st);
        int c0 = 0, c1 = 0, c2 = 0, c3 = 0;          // four independent chains: one warp per scheduler has
#pragma unroll                                     // nothing else to hide the add latency behind
        for (int e = 0; e < NC; e += 4) {
          c0 += s[e] > thr ? 1 : 0;
          c1 += s[e + 1] > thr ? 1 : 0;
          c2 += s[e + 2] > thr ? 1 : 0;
          c3 += s[e + 3] > thr ? 1 : 0;
        }
        rs.rk[t] += (c0 + c1) + (c2 + c3);
      } else {                                     // the one chunk that holds the target itself
        const float st = rs.st[t] * f * f2;
#pragma unroll
        for (int e = 0; e < NC; ++e) {
          const int item = (int)base + e;
          if (item == tg) continue;
          rs.rk[t] += (item < tg ? s[e] >= st : s[e] > st) ? 1 : 0;
        }
      }
    }
  }
}

template <int NC, int TMAX>
__device__ __forceinline__ void rank_topk_chunk(float (&s)[NC], int64_t base, int T, RankState<TMAX>& rs, float& tau,
                                                float* __restrict__ topv, int32_t* __restrict__ topi, int K, int stride,
                                                int slot, int& min_pos, float f = 1.f, float inv = 1.f, float f2 = 1.f) {
  static_assert(NC % 8 == 0, "chunks are scanned in groups of 8");
  rank_count_chunk<NC, TMAX>(s, base, T, rs, f, f2);
  // group maxima (8 consecutive items each): only a group that beats tau is looked at element by element
  float gm[NC / 8];
#pragma unroll
  for (int q = 0; q < NC / 8; ++q) {
    const float a = fmaxf(fmaxf(s[8 * q], s[8 * q + 1]), fmaxf(s[8 * q + 2], s[8 * q + 3]));
    const float b = fmaxf(fmaxf(s[8 * q + 4], s[8 * q + 5]), fmaxf(s[8 * q + 6], s[8 * q + 7]));
    gm[q] = fmaxf(a, b);
  }
  float cmax = gm[0];
#pragma unroll
  for (int q = 1; q < NC / 8; ++q) cmax = fmaxf(cmax, gm[q]);
  float ts = tau * f * f2;                           // tau in the scores' domain
  if (cmax > ts) {
#pragma unroll
    for (int q = 0; q < NC / 8; ++q) {
      if (gm[q] > ts) {
#pragma unroll
        for (int e = 8 * q; e < 8 * q + 8; ++e)
          if (s[e] > ts) {
            tau = topk_replace(s[e] * inv * pow2_inv(f2), (int32_t)(base + e), topv, topi, K, stride, slot, min_pos);
            ts = tau * f * f2;
          }
      }
    }
  }
}

template <int TMAX>
__device__ __forceinline__ void rank_state_init(RankState<TMAX>& rs, int T, const int32_t* __restrict__ targets,
                                                const int32_t* __restrict__ train_col, int64_t lo0, int64_t hi0) {
#pragma unroll
  for (int t = 0; t < RankState<TMAX>::N; ++t) {
    rs.st[t] = 0.f; rs.tg[t] = -1; rs.rk[t] = 0;
    if (t < T && t < TMAX) {
      rs.tg[t] = targets[t];
      int64_t lo = lo0, hi = hi0;
      while (lo < hi) { int64_t mid = (lo + hi) >> 1; if (train_col[mid] < rs.tg[t]) lo = mid + 1; else hi = mid; }
      if (lo < hi0 && train_col[lo] == rs.tg[t]) rs.in_train |= 1u << t;
    }
  }
}

template <int TMAX>
__device__ __forceinline__ void rank_state_set_score(RankState<TMAX>& rs, int t, float score) {
  rs.st[t] = score;
}

}  // namespace recad
