// LightGCN BPR step: fused gather + dot + softplus + L2-reg + gradient scatter, dense Adam, and the
// per-epoch driver that strings  propagate -> BPR -> Horner backward -> Adam  for every batch on one
// stream with no host synchronisation (reference: recad/model/victim/lightgcn.py:122-172).
#include <math.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "tc_common.cuh"

namespace recad {

int gemm_tc(const float* A_hi, const float* A_lo, int M, int lda, const float* B_hi, const float* B_lo, int N, int ldb, int K,
            float* Cm, int ldc, const float* bias, bool relu, float* out_hi, float* out_lo, int ld_split, cudaStream_t s);
int csr_normalize_coef(const int64_t* rowptr, const int32_t* colidx, const int64_t* tperm, const float* w, const float* d_inv,
                       const float* gv, int64_t n_rows, float* coef, cudaStream_t s);

// ------------------------------------------------------------------------------------------
// BPR forward + backward.  A group of LPR lanes owns one sample; each lane holds VPL float4 columns
// of the six rows (O_u, O_p, O_n, E_u, E_p, E_n).  Gradients leave through 128-bit vector REDs.
// ------------------------------------------------------------------------------------------
// Where a batch's (user, pos, neg) triples come from.
// RowSamples: rows [*, 3] in sampler order, visited through the epoch permutation (single GPU, reference layout).
template <typename IdxT>
struct RowSamples {
  static constexpr bool kSparse = false;     // every sample of the batch is processed
  const IdxT* samples;
  const IdxT* perm;
  // returns 1 = valid sample, 0 = nothing to do, -1 = id out of range
  __device__ __forceinline__ int fetch(int64_t b, int64_t n_users, int64_t n_items, int64_t& u, int64_t& p, int64_t& n) const {
    const int64_t row = perm ? (int64_t)perm[b] : b;      // the epoch shuffle is this indirection
    u = samples[3 * row]; p = samples[3 * row + 1]; n = samples[3 * row + 2];
    return (u < 0 || u >= n_users || p < 0 || p >= n_items || n < 0 || n >= n_items) ? -1 : 1;
  }
};
// ShardSamples: the GLOBAL epoch as the host sampler emits it (user, index of the positive inside the user's row,
// negative; 32 bit each) + the global permutation.  A rank of the user-sharded path walks the whole global batch and
// keeps the samples whose user it owns -- no routing pass, no per-rank copy of the epoch; the positive ITEM comes out
// of the rank's own rows of the interaction matrix (its users' sorted distinct items, implicit.py:339-343).
struct ShardSamples {
  static constexpr bool kSparse = true;      // only the samples of the rank's own users are processed
  const uint32_t* users;
  const uint32_t* rel;
  const uint32_t* negs;
  const int32_t* perm;
  int64_t user_lo, user_hi;        // global ids [lo, hi) live on this rank as local users 0 .. hi - lo
  const int64_t* pos_rowptr;       // [n_users_local + 1]
  const int32_t* pos_col;          // item ids + pos_col_offset
  int32_t pos_col_offset;
  __device__ __forceinline__ int fetch(int64_t b, int64_t n_users, int64_t n_items, int64_t& u, int64_t& p, int64_t& n) const {
    const int64_t row = perm ? (int64_t)perm[b] : b;
    const int64_t gu = users[row];
    if (gu < user_lo || gu >= user_hi) return 0;
    u = gu - user_lo;
    const int64_t lo = pos_rowptr[u], len = pos_rowptr[u + 1] - lo;
    const int64_t r = rel[row];
    n = negs[row];
    if (u >= n_users || r >= len || n >= n_items) return -1;
    p = (int64_t)pos_col[lo + r] - pos_col_offset;
    return (p < 0 || p >= n_items) ? -1 : 1;
  }
};

// ShardRows: the global epoch as (user, pos, neg) rows; a rank keeps its own users' rows (tests, injected datasets).
struct ShardRows {
  static constexpr bool kSparse = true;
  const int64_t* rows;
  const int64_t* perm;
  int64_t user_lo, user_hi;
  __device__ __forceinline__ int fetch(int64_t b, int64_t n_users, int64_t n_items, int64_t& u, int64_t& p, int64_t& n) const {
    const int64_t row = perm ? perm[b] : b;
    const int64_t gu = rows[3 * row];
    if (gu < user_lo || gu >= user_hi) return 0;
    u = gu - user_lo; p = rows[3 * row + 1]; n = rows[3 * row + 2];
    return (u >= n_users || p < 0 || p >= n_items || n < 0 || n >= n_items) ? -1 : 1;
  }
};

template <int LPR, int VPL, typename Src>
__global__ void __launch_bounds__(256)
bpr_kernel(const float* __restrict__ O, const float* __restrict__ E, int64_t n_users, int64_t n_items,
           const Src src, int64_t b0,
           int64_t B, int64_t B_norm, float grad_scale, float* __restrict__ gO, float* __restrict__ cnt,
           double* __restrict__ loss_acc, int nvec, int* __restrict__ bad) {
  constexpr int GPW = 32 / LPR;  // sample groups per warp
  const int lane = threadIdx.x & 31;
  const int l = lane % LPR;
  const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
  const int64_t n_groups = (int64_t)gridDim.x * blockDim.x / LPR;
  const float inv_B = 1.0f / (float)B_norm;   // the GLOBAL batch size: a rank of a sharded run sees only its users' rows
  float sp_sum = 0.f, sq_sum = 0.f;
  const float4* __restrict__ O4 = reinterpret_cast<const float4*>(O);
  const float4* __restrict__ E4 = reinterpret_cast<const float4*>(E);
  auto process = [&](const bool valid, const int64_t u, const int64_t p, const int64_t n) {
    const int64_t ru = u * nvec, rp = (n_users + p) * nvec, rn = (n_users + n) * nvec;
    float4 ou[VPL], op[VPL], on[VPL];
    float dn = 0.f, dp = 0.f, sq = 0.f;
#pragma unroll
    for (int q = 0; q < VPL; ++q) {
      const int c = l + q * LPR;
      if (valid && c < nvec) {
        ou[q] = __ldg(O4 + ru + c); op[q] = __ldg(O4 + rp + c); on[q] = __ldg(O4 + rn + c);
        const float4 eu = __ldg(E4 + ru + c), ep = __ldg(E4 + rp + c), en = __ldg(E4 + rn + c);
        dn += ou[q].x * on[q].x + ou[q].y * on[q].y + ou[q].z * on[q].z + ou[q].w * on[q].w;
        dp += ou[q].x * op[q].x + ou[q].y * op[q].y + ou[q].z * op[q].z + ou[q].w * op[q].w;
        sq += eu.x * eu.x + eu.y * eu.y + eu.z * eu.z + eu.w * eu.w + ep.x * ep.x + ep.y * ep.y + ep.z * ep.z +
              ep.w * ep.w + en.x * en.x + en.y * en.y + en.z * en.z + en.w * en.w;
      } else {
        ou[q] = op[q] = on[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) {
      dn += __shfl_xor_sync(kFull, dn, o);
      dp += __shfl_xor_sync(kFull, dp, o);
    }
    // x = <u, n> - <u, p>;  softplus with torch's threshold 20;  d softplus = z / (z + 1)
    const float x = dn - dp;
    float sp, sig;
    if (x > 20.f) { sp = x; sig = 1.f; }
    else { const float z = expf(x); sp = log1pf(z); sig = z / (z + 1.f); }
    if (valid) {
      if (l == 0) sp_sum += sp;
      sq_sum += sq;
      const float s = sig * inv_B * grad_scale;
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        const int c = l + q * LPR;
        if (c < nvec) {
          const float4 a = ou[q], pp = op[q], nn = on[q];
          red_add4(gO + (ru + c) * 4, make_float4(s * (nn.x - pp.x), s * (nn.y - pp.y), s * (nn.z - pp.z), s * (nn.w - pp.w)));
          red_add4(gO + (rp + c) * 4, make_float4(-s * a.x, -s * a.y, -s * a.z, -s * a.w));
          red_add4(gO + (rn + c) * 4, make_float4(s * a.x, s * a.y, s * a.z, s * a.w));
        }
      }
      if (l == 0) {
        atomicAdd(cnt + u, 1.0f);
        atomicAdd(cnt + n_users + p, 1.0f);
        atomicAdd(cnt + n_users + n, 1.0f);
      }
    }
  };
  if constexpr (!Src::kSparse) {
    // all lanes of a warp iterate the same number of times (the shuffles inside are warp-wide)
    const int64_t iters = (B + n_groups - 1) / n_groups;
    for (int64_t it = 0; it < iters; ++it) {
      const int64_t b = it * n_groups + group;
      const bool valid = b < B;
      int64_t u = 0, p = 0, n = 0;
      if (valid && src.fetch(b0 + b, n_users, n_items, u, p, n) < 0) {
        if (l == 0) atomicOr(bad, 1);
        u = 0; p = 0; n = 0;
      }
      process(valid, u, p, n);
    }
  } else {
    // Sharded source: a warp looks at 32 samples of the GLOBAL batch at a time, one per lane (coalesced index loads = the
    // ownership test), then its GPW lane groups work through the samples the rank keeps, GPW at a time.  The ids of the
    // NEXT 32 samples are fetched before the current ones are processed.
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int grp = lane / LPR;
    auto fetch32 = [&](int64_t c0, int64_t& fu, int64_t& fp, int64_t& fn) -> int {
      int st = 0;
      fu = 0; fp = 0; fn = 0;
      if (c0 + lane < B) {
        st = src.fetch(b0 + c0 + lane, n_users, n_items, fu, fp, fn);
        if (st < 0) {
          atomicOr(bad, 1);
          fu = 0; fp = 0; fn = 0;
          st = 1;
        }
      }
      return st;
    };
    int64_t nu, np_, nn_;
    int nst = fetch32(warp_global * 32, nu, np_, nn_);
    for (int64_t c0 = warp_global * 32; c0 < B; c0 += n_warps * 32) {
      const int64_t mu = nu, mp = np_, mn = nn_;
      const int st = nst;
      nst = fetch32(c0 + n_warps * 32, nu, np_, nn_);
      unsigned todo = __ballot_sync(kFull, st != 0);
      while (todo) {
        unsigned m = todo;                       // lane group `grp` takes the grp-th lowest pending sample
        int from = -1;
#pragma unroll
        for (int k = 0; k < GPW; ++k) {
          const int low = m ? __ffs(m) - 1 : -1;
          if (k == grp) from = low;
          m &= m - 1;
        }
        todo = m;
        const bool valid = from >= 0;
        const int sl = valid ? from : 0;
        process(valid, __shfl_sync(kFull, mu, sl), __shfl_sync(kFull, mp, sl), __shfl_sync(kFull, mn, sl));
      }
    }
  }
  // block reduction of the two loss partials -> one double atomic each per block
  __shared__ double red[2][8];
  double a = warp_sum((double)sp_sum), c = warp_sum((double)sq_sum);
  const int w = threadIdx.x >> 5;
  if (lane == 0) { red[0][w] = a; red[1][w] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ta = 0, tc = 0;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) { ta += red[0][k]; tc += red[1][k]; }
    atomicAdd(loss_acc + 0, ta);
    atomicAdd(loss_acc + 1, tc);
  }
  (void)GPW;
}

// ------------------------------------------------------------------------------------------
// dense Adam (+ optional L2-reg gradient from batch multiplicities, + optional loss fold)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, const float* __restrict__ cnt, float reg_scale,
            float* __restrict__ m, float* __restrict__ v, int64_t n4, int vec_per_row, AdamScalars a, LossFold fold) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 P = reinterpret_cast<float4*>(p)[i];
    float4 G = reinterpret_cast<const float4*>(g)[i];
    float4 M = reinterpret_cast<float4*>(m)[i];
    float4 V = reinterpret_cast<float4*>(v)[i];
    if (cnt) {
      const float r = reg_scale * cnt[i / vec_per_row];
      G.x = fmaf(r, P.x, G.x); G.y = fmaf(r, P.y, G.y); G.z = fmaf(r, P.z, G.z); G.w = fmaf(r, P.w, G.w);
    }
    adam_update(P.x, G.x, M.x, V.x, a);
    adam_update(P.y, G.y, M.y, V.y, a);
    adam_update(P.z, G.z, M.z, V.z, a);
    adam_update(P.w, G.w, M.w, V.w, a);
    reinterpret_cast<float4*>(p)[i] = P;
    reinterpret_cast<float4*>(m)[i] = M;
    reinterpret_cast<float4*>(v)[i] = V;
  }
  if (fold.acc && blockIdx.x == 0 && threadIdx.x == 0) {
    // final_loss of this batch = mean softplus + lambda * 0.5 * sum sq / B  (lightgcn.py:149-165)
    fold.acc[2] += fold.acc[0] * fold.inv_B + fold.half_lambda * fold.acc[1] * fold.inv_B;
    fold.acc[0] = 0.0;
    fold.acc[1] = 0.0;
  }
}

// scalar tail for n % 4 != 0 (bias vectors)
__global__ void adam_tail_kernel(float* p, const float* g, float* m, float* v, int64_t lo, int64_t n, AdamScalars a) {
  int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float G = g[i], M = m[i], V = v[i], P = p[i];
  adam_update(P, G, M, V, a);
  p[i] = P; m[i] = M; v[i] = V;
}

AdamScalars adam_scalars(float lr, float b1, float b2, float eps, int64_t step) {
  // torch.optim.adam._single_tensor_adam: python-double scalars, cast to fp32 at the tensor op
  const double bc1 = 1.0 - pow((double)b1, (double)step);
  const double bc2 = 1.0 - pow((double)b2, (double)step);
  AdamScalars a;
  a.w1 = (float)(1.0 - (double)b1);
  a.b2 = b2;
  a.w2 = (float)(1.0 - (double)b2);
  a.step_size = (float)((double)lr / bc1);
  a.bc2_sqrt = (float)sqrt(bc2);
  a.eps = eps;
  return a;
}

int launch_adam(float* p, const float* g, const float* cnt, float reg_scale, float* m, float* v, int64_t n, int D,
                const AdamScalars& a, const LossFold& fold, cudaStream_t s) {
  const int64_t n4 = n / 4;
  if (n4 > 0) {
    const int64_t want = (n4 + 255) / 256;
    const unsigned grid = (unsigned)std::min<int64_t>(want, (int64_t)sm_count() * 16);
    adam_kernel<<<grid, 256, 0, s>>>(p, g, cnt, reg_scale, m, v, n4, cnt ? D / 4 : 1, a, fold);
    RECAD_LAUNCH_CHECK();
  }
  if (n % 4) {
    adam_tail_kernel<<<1, 32, 0, s>>>(p, g, m, v, n4 * 4, n, a);
    RECAD_LAUNCH_CHECK();
  }
  return RECAD_OK;
}

template <int LPR, int VPL, typename Src>
static int launch_bpr_t(const float* O, const float* E, int64_t U, int64_t I, const Src& src, int64_t b0, int64_t B, int64_t B_work,
                        int64_t B_norm, float gs, float* gO, float* cnt, double* loss, int nvec, int* bad, cudaStream_t s) {
  const int64_t groups_per_block = 256 / LPR;
  const int64_t want = (B_work + groups_per_block - 1) / groups_per_block;       // B_work: samples expected to be valid
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)sm_count() * 32));
  bpr_kernel<LPR, VPL, Src><<<grid, 256, 0, s>>>(O, E, U, I, src, b0, B, B_norm, gs, gO, cnt, loss, nvec, bad);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

template <typename Src>
static int launch_bpr_src(const float* O, const float* E, int64_t U, int64_t I, const Src& src, int64_t b0, int64_t B, int64_t B_work,
                          int64_t B_norm, float gs, float* gO, float* cnt, double* loss, int D, int* bad, cudaStream_t s) {
  const int nvec = D / 4;
  if (nvec <= 8) return launch_bpr_t<8, 1, Src>(O, E, U, I, src, b0, B, B_work, B_norm, gs, gO, cnt, loss, nvec, bad, s);
  if (nvec <= 16) return launch_bpr_t<16, 1, Src>(O, E, U, I, src, b0, B, B_work, B_norm, gs, gO, cnt, loss, nvec, bad, s);
  if (nvec <= 32) return launch_bpr_t<32, 1, Src>(O, E, U, I, src, b0, B, B_work, B_norm, gs, gO, cnt, loss, nvec, bad, s);
  if (nvec <= 64) return launch_bpr_t<32, 2, Src>(O, E, U, I, src, b0, B, B_work, B_norm, gs, gO, cnt, loss, nvec, bad, s);
  if (nvec <= 128) return launch_bpr_t<32, 4, Src>(O, E, U, I, src, b0, B, B_work, B_norm, gs, gO, cnt, loss, nvec, bad, s);
  return launch_bpr_t<32, 8, Src>(O, E, U, I, src, b0, B, B_work, B_norm, gs, gO, cnt, loss, nvec, bad, s);
}

template <typename IdxT>
static int launch_bpr(const float* O, const float* E, int64_t U, int64_t I, const IdxT* samples, const IdxT* perm,
               int64_t B, int64_t B_norm, float gs, float* gO, float* cnt, double* loss, int D, int* bad,
               cudaStream_t s) {
  const RowSamples<IdxT> src{samples, perm};
  return launch_bpr_src(O, E, U, I, src, 0, B, B, B_norm, gs, gO, cnt, loss, D, bad, s);
}

// sharded path (shard.cu): samples b0 .. b0 + B of the global epoch, of which about B / world belong to this rank
int launch_bpr_shard(const float* O, const float* E, int64_t U, int64_t I, const uint32_t* users, const uint32_t* rel,
                     const uint32_t* negs, const int32_t* perm, int64_t b0, int64_t B, int64_t B_norm, int64_t user_lo,
                     const int64_t* pos_rowptr, const int32_t* pos_col, int32_t pos_col_offset, int world, float gs, float* gO,
                     float* cnt, double* loss, int D, cudaStream_t s) {
  const ShardSamples src{users, rel, negs, perm, user_lo, user_lo + U, pos_rowptr, pos_col, pos_col_offset};
  // groups sized for ~4 global samples each: the ownership test is 12 bytes per sample, the work 4.6 kB per kept sample
  const int64_t B_work = std::max<int64_t>(B / std::max(1, std::min(world, 4)), 1);
  return launch_bpr_src(O, E, U, I, src, b0, B, B_work, B_norm, gs, gO, cnt, loss, D, reinterpret_cast<int*>(loss + 3), s);
}

int launch_bpr_shard_rows(const float* O, const float* E, int64_t U, int64_t I, const int64_t* rows, const int64_t* perm, int64_t b0,
                          int64_t B, int64_t B_norm, int64_t user_lo, int world, float gs, float* gO, float* cnt, double* loss, int D,
                          cudaStream_t s) {
  const ShardRows src{rows, perm, user_lo, user_lo + U};
  const int64_t B_work = std::max<int64_t>(B / std::max(1, std::min(world, 4)), 1);
  return launch_bpr_src(O, E, U, I, src, b0, B, B_work, B_norm, gs, gO, cnt, loss, D, reinterpret_cast<int*>(loss + 3), s);
}

// z = a * x + b * y (float4 grid-stride); z may alias x or y
__global__ void __launch_bounds__(256) axpby_kernel(float* z, float a, const float* x, float b, const float* y, int64_t n4) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 X = reinterpret_cast<const float4*>(x)[i], Y = reinterpret_cast<const float4*>(y)[i];
    reinterpret_cast<float4*>(z)[i] = make_float4(a * X.x + b * Y.x, a * X.y + b * Y.y, a * X.z + b * Y.z, a * X.w + b * Y.w);
  }
}

__global__ void dot_scores_kernel(const float* __restrict__ O, int64_t n_users, const int64_t* __restrict__ users,
                                  const int64_t* __restrict__ items, int64_t B, int nvec, float* __restrict__ out) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const float4* __restrict__ O4 = reinterpret_cast<const float4*>(O);
  const int64_t ru = users[b] * nvec, ri = (n_users + items[b]) * nvec;
  float acc = 0.f;
  for (int c = lane; c < nvec; c += 32) {
    const float4 a = __ldg(O4 + ru + c), q = __ldg(O4 + ri + c);
    acc += a.x * q.x + a.y * q.y + a.z * q.z + a.w * q.w;
  }
  acc = warp_sum(acc);
  if (lane == 0) out[b] = acc;
}

// ------------------------------------------------------------------------------------------
// Backward of pair scores s_b = <Xa[ia_b], Xb[ib_b]> (+ ba[ia_b] + bb[ib_b]) for an upstream gradient g, atomic-free.
// One side at a time: key_b = ia_b << bbits | b, stably radix-sorted, groups the samples of a row in ascending sample
// order; the warp of a group's first key is the row's only writer and adds g_b Xb[ib_b] over the group with plain stores.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pair_keys_kernel(const int64_t* __restrict__ ids, int64_t n_rows, int64_t B, int bbits, uint64_t* __restrict__ keys,
                 int* __restrict__ bad) {
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (int64_t)gridDim.x * blockDim.x) {
    int64_t id = ids[b];
    if (id < 0 || id >= n_rows) { atomicOr(bad, 1); id = 0; }
    keys[b] = ((uint64_t)id << bbits) | (uint64_t)b;
  }
}

// one warp per sorted key; the warp of a row's first key writes dX[row] = sum g_b X[other_b] (+ beta_b V[other_b] when kTwo)
// and db[row] = sum g_b; every other warp returns.  kTwo sums in double: a Hessian product's popular rows collect 10^5 and
// more pairs, and a float running sum of that length loses ~sqrt(count) ulps (1e-5 of the row at 10^5 pairs).
// kJoint (with kTwo): X holds interleaved rows [O | dO] of 2 nvec float4s, gathered once per pair, and the row written is
// [sum g_b O + beta_b dO | sum beta_b O] of the same width, both halves summed in double; V and db are not used.
template <bool kTwo, bool kJoint = false>
__global__ void __launch_bounds__(256)
pair_grad_rows_kernel(const uint64_t* __restrict__ keys, int64_t B, int bbits, const float* __restrict__ g,
                      const float* __restrict__ beta, const int64_t* __restrict__ other, int64_t n_other,
                      const float* __restrict__ X, const float* __restrict__ V, int nvec, float* __restrict__ dX,
                      float* __restrict__ db) {
  static_assert(kTwo || !kJoint, "the joint rows need beta");
  const int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (k >= B) return;
  const uint64_t row = keys[k] >> bbits;
  if (k > 0 && (keys[k - 1] >> bbits) == row) return;
  const uint64_t bmask = (1ull << bbits) - 1;
  const float4* __restrict__ X4 = reinterpret_cast<const float4*>(X);
  const float4* __restrict__ V4 = reinterpret_cast<const float4*>(V);
  float4* __restrict__ dX4 = reinterpret_cast<float4*>(dX);
  for (int c0 = 0; c0 < nvec; c0 += 32) {
    const int c = c0 + lane;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    float gsum = 0.f;
    double dx = 0.0, dy = 0.0, dz = 0.0, dw = 0.0, dg = 0.0;       // kTwo accumulators
    double ex = 0.0, ey = 0.0, ez = 0.0, ew = 0.0;                 // kJoint: the second half
    for (int64_t j = k; j < B; ++j) {
      const uint64_t key = keys[j];
      if ((key >> bbits) != row) break;
      const int64_t b = (int64_t)(key & bmask);
      int64_t o = other[b];
      if (o < 0 || o >= n_other) o = 0;            // reported by the other side's key pass
      const float gv = g[b];
      if constexpr (kJoint) {
        if (c < nvec) {
          const double bv = (double)beta[b];
          const float4 x = __ldg(X4 + o * 2 * nvec + c), y = __ldg(X4 + o * 2 * nvec + nvec + c);
          dx = fma((double)gv, (double)x.x, fma(bv, (double)y.x, dx));
          dy = fma((double)gv, (double)x.y, fma(bv, (double)y.y, dy));
          dz = fma((double)gv, (double)x.z, fma(bv, (double)y.z, dz));
          dw = fma((double)gv, (double)x.w, fma(bv, (double)y.w, dw));
          ex = fma(bv, (double)x.x, ex);
          ey = fma(bv, (double)x.y, ey);
          ez = fma(bv, (double)x.z, ez);
          ew = fma(bv, (double)x.w, ew);
        }
      } else if constexpr (kTwo) {
        dg += (double)gv;
        if (c < nvec) {
          const double bv = (double)beta[b];
          const float4 x = __ldg(X4 + o * nvec + c), y = __ldg(V4 + o * nvec + c);
          dx = fma((double)gv, (double)x.x, fma(bv, (double)y.x, dx));
          dy = fma((double)gv, (double)x.y, fma(bv, (double)y.y, dy));
          dz = fma((double)gv, (double)x.z, fma(bv, (double)y.z, dz));
          dw = fma((double)gv, (double)x.w, fma(bv, (double)y.w, dw));
        }
      } else {
        gsum += gv;
        if (c < nvec) {
          const float4 x = __ldg(X4 + o * nvec + c);
          acc.x += gv * x.x; acc.y += gv * x.y; acc.z += gv * x.z; acc.w += gv * x.w;
        }
      }
    }
    if constexpr (kTwo) {
      acc = make_float4((float)dx, (float)dy, (float)dz, (float)dw);
      gsum = (float)dg;
    }
    if constexpr (kJoint) {
      if (c < nvec) {
        dX4[(int64_t)row * 2 * nvec + c] = acc;
        dX4[(int64_t)row * 2 * nvec + nvec + c] = make_float4((float)ex, (float)ey, (float)ez, (float)ew);
      }
    } else {
      if (c < nvec) dX4[(int64_t)row * nvec + c] = acc;
      if (c0 == 0 && lane == 0 && db) db[row] = gsum;
    }
  }
}

// ------------------------------------------------------------------------------------------
// Seeds of the BPR loss's Hessian-vector product.  Per sample b, x = <O_u, O_n> - <O_u, O_p>, dx its derivative along
// dO = P v, l' / l'' softplus's first two derivatives (torch's threshold 20, as bpr_kernel); the (u, n) pair gets
// (a, c) = (l'' dx / B, l' / B) and the (u, p) pair (-a, -c).  dloss[b] = l' dx + lambda (<V_u, E_u> + <V_p, E_p> + <V_n, E_n>).
// kSeedLanes lanes per sample, 128-bit loads, a fixed shuffle order: no atomics on the results.  Rows of O / dO (and E / V)
// are rstride float4s apart: nvec for tables of their own, 2 nvec for the interleaved [O | dO] rows (dO = O + D).
// ------------------------------------------------------------------------------------------
constexpr int kSeedLanes = 16;

__device__ __forceinline__ float dot4(const float4 a, const float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }

__global__ void __launch_bounds__(256)
bpr_hvp_seeds_kernel(const float* __restrict__ O, const float* __restrict__ dO, int64_t n_users, int64_t n_items,
                     const int64_t* __restrict__ samples, int64_t n, float inv_B, int nvec, int rstride,
                     const float* __restrict__ E, const float* __restrict__ V, float lambda, float* __restrict__ alpha,
                     float* __restrict__ beta, float* __restrict__ dloss, int* __restrict__ bad) {
  const int l = threadIdx.x % kSeedLanes;
  const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / kSeedLanes;
  const int64_t n_groups = (int64_t)gridDim.x * blockDim.x / kSeedLanes;
  const int64_t iters = (n + n_groups - 1) / n_groups;       // the same count on every lane: the shuffles are warp-wide
  const float4* __restrict__ O4 = reinterpret_cast<const float4*>(O);
  const float4* __restrict__ dO4 = reinterpret_cast<const float4*>(dO);
  const float4* __restrict__ E4 = reinterpret_cast<const float4*>(E);
  const float4* __restrict__ V4 = reinterpret_cast<const float4*>(V);
  for (int64_t it = 0; it < iters; ++it) {
    const int64_t b = it * n_groups + group;
    const bool valid = b < n;
    int64_t u = 0, p = 0, q = 0;
    if (valid) {
      u = samples[3 * b]; p = samples[3 * b + 1]; q = samples[3 * b + 2];
      if (u < 0 || u >= n_users || p < 0 || p >= n_items || q < 0 || q >= n_items) {
        if (l == 0) atomicOr(bad, 1);
        u = 0; p = 0; q = 0;
      }
    }
    const int64_t ru = u * rstride, rp = (n_users + p) * rstride, rn = (n_users + q) * rstride;
    float dn = 0.f, dp = 0.f, dx = 0.f, reg = 0.f;
    if (valid) {
      for (int c = l; c < nvec; c += kSeedLanes) {
        const float4 ou = __ldg(O4 + ru + c), op = __ldg(O4 + rp + c), on = __ldg(O4 + rn + c);
        const float4 du = __ldg(dO4 + ru + c), dp4 = __ldg(dO4 + rp + c), dn4 = __ldg(dO4 + rn + c);
        dn += dot4(ou, on);
        dp += dot4(ou, op);
        dx += dot4(du, make_float4(on.x - op.x, on.y - op.y, on.z - op.z, on.w - op.w)) +
              dot4(ou, make_float4(dn4.x - dp4.x, dn4.y - dp4.y, dn4.z - dp4.z, dn4.w - dp4.w));
        if (dloss)
          reg += dot4(__ldg(V4 + ru + c), __ldg(E4 + ru + c)) + dot4(__ldg(V4 + rp + c), __ldg(E4 + rp + c)) +
                 dot4(__ldg(V4 + rn + c), __ldg(E4 + rn + c));
      }
    }
#pragma unroll
    for (int o = kSeedLanes / 2; o > 0; o >>= 1) {
      dn += __shfl_xor_sync(kFull, dn, o);
      dp += __shfl_xor_sync(kFull, dp, o);
      dx += __shfl_xor_sync(kFull, dx, o);
      reg += __shfl_xor_sync(kFull, reg, o);
    }
    if (valid && l == 0) {
      const float x = dn - dp;
      float d1, d2;                                 // l'(x), l''(x)
      if (x > 20.f) { d1 = 1.f; d2 = 0.f; }
      else { const float z = expf(x); d1 = z / (z + 1.f); d2 = d1 * (1.f - d1); }
      const float a = d2 * dx * inv_B, c = d1 * inv_B;
      alpha[b] = a; alpha[n + b] = -a;
      beta[b] = c;  beta[n + b] = -c;
      if (dloss) dloss[b] = d1 * dx + lambda * reg;
    }
  }
}

static int64_t align256(int64_t x) { return (x + 255) / 256 * 256; }

static int bit_width(int64_t n) {     // bits needed for the values 0 .. n - 1 (at least 1)
  int b = 1;
  while (b < 63 && ((int64_t)1 << b) < n) ++b;
  return b;
}

enum class PairMode { kBackward, kHvp, kJoint };

// Both sides of the pair pass, one radix sort per side (ids checked into `bad`; the rows no pair reaches are left as they
// are, so the caller zeroes the outputs).  kJoint: Xa / Xb are the interleaved [O | dO] rows of 2D floats of each side and
// outA / outB receive rows of the same width (pair_grad_rows_kernel<true, true>); Va, Vb, dba, dbb are not used.
static int pair_sides(PairMode mode, const float* Xa, const float* Va, int64_t n_a, const float* Xb, const float* Vb,
                      int64_t n_b, int32_t D, const int64_t* ia, const int64_t* ib, int64_t B, const float* alpha,
                      const float* beta, float* outA, float* outB, float* dba, float* dbb, uint64_t* keys, uint64_t* tmp,
                      void* sort_scr, int* bad, cudaStream_t s) {
  const int bbits = bit_width(B);
  const unsigned kgrid = (unsigned)std::min<int64_t>((B + 255) / 256, (int64_t)sm_count() * 16);
  const unsigned wgrid = (unsigned)((B * 32 + 255) / 256);
  for (int side = 0; side < 2; ++side) {
    const int64_t n_rows = side == 0 ? n_a : n_b, n_other = side == 0 ? n_b : n_a;
    const int64_t* ids = side == 0 ? ia : ib;
    pair_keys_kernel<<<kgrid, 256, 0, s>>>(ids, n_rows, B, bbits, keys, bad);
    RECAD_LAUNCH_CHECK();
    int rc = radix_sort_u64(keys, tmp, B, bbits + bit_width(n_rows), sort_scr, s);
    if (rc) return rc;
    const int64_t* other = side == 0 ? ib : ia;
    const float* X = side == 0 ? Xb : Xa;
    float* out = side == 0 ? outA : outB;
    float* db = side == 0 ? dba : dbb;
    if (mode == PairMode::kJoint)
      pair_grad_rows_kernel<true, true><<<wgrid, 256, 0, s>>>(keys, B, bbits, alpha, beta, other, n_other, X, nullptr, D / 4,
                                                               out, nullptr);
    else if (mode == PairMode::kHvp)
      pair_grad_rows_kernel<true><<<wgrid, 256, 0, s>>>(keys, B, bbits, alpha, beta, other, n_other, X, side == 0 ? Vb : Va,
                                                         D / 4, out, db);
    else
      pair_grad_rows_kernel<false><<<wgrid, 256, 0, s>>>(keys, B, bbits, alpha, nullptr, other, n_other, X, nullptr, D / 4,
                                                          out, db);
    RECAD_LAUNCH_CHECK();
  }
  return RECAD_OK;
}

// ------------------------------------------------------------------------------------------
// Per-index sums, atomic-free: key_b = idx_b << bbits | b (idx_b < 0 -> the sentinel n_out, sorted last and not written),
// stably radix-sorted; the thread of a group's first key sums x over the group in ascending b, in double, and is the
// output's only writer.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
index_keys_kernel(const int64_t* __restrict__ idx, int64_t n, int64_t n_out, int bbits, uint64_t* __restrict__ keys,
                  int* __restrict__ bad) {
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < n; b += (int64_t)gridDim.x * blockDim.x) {
    int64_t id = idx[b];
    if (id >= n_out) { atomicOr(bad, 1); id = n_out; }
    if (id < 0) id = n_out;
    keys[b] = ((uint64_t)id << bbits) | (uint64_t)b;
  }
}

__global__ void __launch_bounds__(256)
index_sums_kernel(const uint64_t* __restrict__ keys, int64_t n, int bbits, uint64_t n_out, const float* __restrict__ x,
                  float* __restrict__ out) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint64_t row = keys[k] >> bbits;
  if (row >= n_out || (k > 0 && (keys[k - 1] >> bbits) == row)) return;
  const uint64_t bmask = (1ull << bbits) - 1;
  double acc = 0.0;
  for (int64_t j = k; j < n && (keys[j] >> bbits) == row; ++j) acc += (double)x[keys[j] & bmask];
  out[row] = (float)acc;
}

// Workspace of recad_lightgcn_loss_mixed_values: [N, 2D] float buffers -- the forward layers Y_0 .. Y_{L-1} of [E | S]
// (Y_0 only for L = 0), [O | dO] (L >= 1; it is the Horner's first ping-pong buffer once the pair pass has read it), the
// pair pass's output G, the second ping-pong buffer (L >= 3) -- then the pairs' ids, seeds, sort keys and the id flag.
struct MixedWork {
  float* Y;   // Y_l = Y + l * N * 2D
  float* OO;
  float* G;
  float* X1;
  int64_t *ia, *ib;
  float *alpha, *beta;
  uint64_t *keys, *tmp;
  void* sort_scr;
  int* bad;
};

static int64_t mixed_work(int64_t N, int32_t D, int32_t L, int64_t n, char* base, MixedWork* w) {
  const int64_t rowbuf = N * 2 * (int64_t)D * (int64_t)sizeof(float), B = 2 * n;   // a multiple of 32 bytes
  const int64_t n_y = L > 0 ? L : 1;
  int64_t off = 0;
  auto take = [&](int64_t bytes) { char* p = base ? base + off : nullptr; off += align256(bytes); return p; };
  char* Y = take(n_y * rowbuf);
  char* OO = L > 0 ? take(rowbuf) : Y;
  char* G = take(rowbuf);
  char* X1 = L >= 3 ? take(rowbuf) : nullptr;
  char* ia = take(B * 8);
  char* ib = take(B * 8);
  char* alpha = take(B * 4);
  char* beta = take(B * 4);
  char* keys = take(B * 8);
  char* tmp = take(B * 8);
  char* sort_scr = take(sort_scratch_bytes(B));
  char* bad = take(sizeof(int));
  if (w)
    *w = MixedWork{reinterpret_cast<float*>(Y), reinterpret_cast<float*>(OO), reinterpret_cast<float*>(G),
                   reinterpret_cast<float*>(X1), reinterpret_cast<int64_t*>(ia), reinterpret_cast<int64_t*>(ib),
                   reinterpret_cast<float*>(alpha), reinterpret_cast<float*>(beta), reinterpret_cast<uint64_t*>(keys),
                   reinterpret_cast<uint64_t*>(tmp), sort_scr, reinterpret_cast<int*>(bad)};
  return off;
}

// Edge-value gradient riding on the Horner loop: at step k, before t_k's ping-pong buffer is written again,
// gvals[e] (+)= scale * <t_k[r_e], X[L - 1 - k][c_e]> over the entries of st->graph (A's own entry order; k = 0 writes).
struct HornerValues {
  const float* const* X;   // host array of the L forward layers X_0 = E .. X_{L-1}
  float* gvals;
  float scale;
};

// Operand gather riding on the same loop (recad_lightgcn_candidate_weight_grads): at step k, before t_k's ping-pong buffer is
// written again, the rows of t_k and X[L - 1 - k] (interleaved rows of width W = st->D) land in columns [2kW, 2(k+1)W) of
// the split (3xTF32 hi / lo) GEMM operands, which gemm_tc reads row-major with row stride ld:
//   A row r (r < n_sel, user sel[r]): [t_k | X[L-1-k]][sel[r]] * d_inv[sel[r]] * scale
//   B row i (i < n_items):            [X[L-1-k] | t_k][n_users + i] * d_inv[n_users + i]
// so that <A_r, B_i> summed over k is scale * d_u d_i (g(u, U + i) + g(U + i, u)), g the unscaled SDDMM of the two entries
// of one interaction, stored or not.  Ids of sel outside [0, n_users) read row 0 (the caller reports them).
struct HornerGather {
  const float* const* X;   // host array of the L forward layers, as HornerValues::X
  const int64_t* sel;
  int64_t n_sel, n_users, n_items;
  const float* d_inv;      // [n_users + n_items]
  float scale;
  int ld;
  float *a_hi, *a_lo, *b_hi, *b_lo;
};

// one thread per float4 of one step's 2W-wide column block, the n_sel A rows first, then the n_items B rows
__global__ void __launch_bounds__(256)
gather_split_kernel(const float* __restrict__ t, const float* __restrict__ X, int nvec, const int64_t* __restrict__ sel,
                    int64_t n_sel, int64_t n_users, int64_t n_items, const float* __restrict__ d_inv, float scale, int ld,
                    int col0, float* __restrict__ a_hi, float* __restrict__ a_lo, float* __restrict__ b_hi,
                    float* __restrict__ b_lo) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t row = e / (2 * nvec);
  const int q = (int)(e - row * 2 * nvec);
  if (row >= n_sel + n_items) return;
  const bool a_side = row < n_sel;
  int64_t src;
  float f;
  if (a_side) {
    src = sel[row];
    if (src < 0 || src >= n_users) src = 0;
    f = d_inv[src] * scale;
  } else {
    src = n_users + (row - n_sel);
    f = d_inv[src];
  }
  // A: t first, then X; B: X first, then t
  const bool from_t = (q < nvec) == a_side;
  const float4 x = __ldg(reinterpret_cast<const float4*>(from_t ? t : X) + src * nvec + (q < nvec ? q : q - nvec));
  const float v[4] = {x.x * f, x.y * f, x.z * f, x.w * f};
  float h[4], l[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) split_tf32(v[k], h[k], l[k]);
  const int64_t off = (a_side ? row : row - n_sel) * ld + col0 + 4 * q;
  *reinterpret_cast<float4*>((a_side ? a_hi : b_hi) + off) = make_float4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<float4*>((a_side ? a_lo : b_lo) + off) = make_float4(l[0], l[1], l[2], l[3]);
}

static int horner_gather(const HornerGather* hg, int k, int L, const float* t, int32_t W, void* stream) {
  const int nvec = W / 4;
  const int64_t threads = (hg->n_sel + hg->n_items) * 2 * nvec;
  gather_split_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, as_stream(stream)>>>(
      t, hg->X[L - 1 - k], nvec, hg->sel, hg->n_sel, hg->n_users, hg->n_items, hg->d_inv, hg->scale, hg->ld, 2 * k * W,
      hg->a_hi, hg->a_lo, hg->b_hi, hg->b_lo);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

// Horner: t <- g + A t, L times, so that t = (I + A + ... + A^L) g, over graph_t when set.  The last step is scaled by
// alpha and lands in `out`; out == nullptr: it lands in the X0 / X1 ping-pong buffer of its parity.  *res = the result.
// hv: the SDDMM of each step on its t_k; with out == nullptr as well, the last SpMM (which gvals does not need) is skipped
// and *res is nullptr.  hg (only with hv): the operand gather of each step on its t_k, after the SDDMM.
static int lightgcn_horner(const recad_lightgcn* st, const float* g, float alpha, float* out, const float** res,
                           void* stream, const HornerValues* hv = nullptr, const HornerGather* hg = nullptr) {
  const recad_csr* A = st->graph_t ? st->graph_t : st->graph;
  const int L = st->n_layers;
  const float* t = g;
  for (int k = 0; k < L; ++k) {
    const bool last = k == L - 1;
    if (hv) {
      int rc = recad_csr_sddmm(st->graph, t, hv->X[L - 1 - k], st->D, hv->scale, k > 0, hv->gvals, stream);
      if (rc) return rc;
      if (hg && (rc = horner_gather(hg, k, L, t, st->D, stream))) return rc;
      if (last && !out) {
        *res = nullptr;
        return RECAD_OK;
      }
    }
    float* z = (last && out) ? out : ((k & 1) ? st->X1 : st->X0);
    const int rc = recad_spmm(A, t, nullptr, g, z, last ? alpha : 1.0f, st->D, stream);
    if (rc) return rc;
    t = z;
  }
  *res = t;
  return RECAD_OK;
}

static int check_lightgcn(const recad_lightgcn* st) {
  RECAD_REQUIRE(st && st->graph, RECAD_ERR_ARG, "lightgcn: null state");
  RECAD_REQUIRE(st->n_users > 0 && st->n_items > 0 && st->graph->n_rows == st->n_users + st->n_items, RECAD_ERR_ARG,
                "lightgcn: graph has %lld rows, expected n_users + n_items = %lld", (long long)st->graph->n_rows,
                (long long)(st->n_users + st->n_items));
  RECAD_REQUIRE(st->D >= 4 && st->D % 4 == 0 && st->n_layers >= 0, RECAD_ERR_UNSUPPORTED, "lightgcn: bad D / layers");
  RECAD_REQUIRE(st->E && st->O && (st->n_layers < 2 || (st->X0 && st->X1)) && (st->n_layers < 1 || st->X0),
                RECAD_ERR_ARG, "lightgcn: null buffer");
  return RECAD_OK;
}

// The mixed driver's recurrences up to the Horner pass: Y_0 = [E | S] ([E | 0] when S is null), Y_{l+1} = A Y_l and
// [O | dO] = (1 / (L + 1)) sum_l Y_l (recad_lightgcn_propagate's calls at width 2D), then, for n > 0 rows, the seeds
// (a_b, c_b) from the interleaved rows (and each row's own directional derivative along S into dloss, when given, with the
// regulariser's weight lambda) and
// G = [G_O | G_dO] by the pairs (u, neg), (u, pos); G = 0 for n = 0.  Zeroes w.bad first; ids are flagged there.
static int mixed_recurrence(const recad_lightgcn* st, const recad_csr* A2, const float* S, const int64_t* samples, int64_t n,
                            const MixedWork& w, float* dloss, float lambda, void* stream) {
  cudaStream_t s = as_stream(stream);
  const int32_t D = st->D, D2 = 2 * st->D;
  const int L = st->n_layers;
  const int64_t U = st->n_users, N = st->n_users + st->n_items;
  const size_t row2 = (size_t)D2 * sizeof(float), row1 = (size_t)D * sizeof(float);
  const int64_t stride = N * D2;
  RECAD_CUDA_CHECK(cudaMemcpy2DAsync(w.Y, row2, st->E, row1, row1, N, cudaMemcpyDeviceToDevice, s));
  if (S) RECAD_CUDA_CHECK(cudaMemcpy2DAsync(w.Y + D, row2, S, row1, row1, N, cudaMemcpyDeviceToDevice, s));
  else RECAD_CUDA_CHECK(cudaMemset2DAsync(w.Y + D, row2, 0, row1, N, s));
  for (int k = 0; k < L; ++k) {
    const bool last = k == L - 1;
    const int rc = recad_spmm(A2, w.Y + k * stride, last ? nullptr : w.Y + (k + 1) * stride, k == 0 ? w.Y : w.OO, w.OO,
                              last ? 1.0f / (float)(L + 1) : 1.0f, D2, stream);
    if (rc) return rc;
  }
  RECAD_CUDA_CHECK(cudaMemsetAsync(w.bad, 0, sizeof(int), s));
  if (n == 0) {
    RECAD_CUDA_CHECK(cudaMemsetAsync(w.G, 0, (size_t)stride * sizeof(float), s));
    return RECAD_OK;
  }
  const int64_t want = (n * kSeedLanes + 255) / 256;
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)sm_count() * 32));
  // E / V of the row regulariser's derivative: the two halves of Y_0
  bpr_hvp_seeds_kernel<<<grid, 256, 0, s>>>(w.OO, w.OO + D, U, st->n_items, samples, n, 1.0f / (float)n, D / 4, D2 / 4,
                                            dloss ? w.Y : nullptr, dloss ? w.Y + D : nullptr, lambda,
                                            w.alpha, w.beta, dloss, w.bad);
  RECAD_LAUNCH_CHECK();
  const size_t row3 = 3 * sizeof(int64_t);
  RECAD_CUDA_CHECK(cudaMemcpy2DAsync(w.ia, sizeof(int64_t), samples, row3, sizeof(int64_t), n, cudaMemcpyDeviceToDevice, s));
  RECAD_CUDA_CHECK(cudaMemcpy2DAsync(w.ia + n, sizeof(int64_t), samples, row3, sizeof(int64_t), n, cudaMemcpyDeviceToDevice, s));
  RECAD_CUDA_CHECK(cudaMemcpy2DAsync(w.ib, sizeof(int64_t), samples + 2, row3, sizeof(int64_t), n, cudaMemcpyDeviceToDevice, s));
  RECAD_CUDA_CHECK(cudaMemcpy2DAsync(w.ib + n, sizeof(int64_t), samples + 1, row3, sizeof(int64_t), n, cudaMemcpyDeviceToDevice,
                                     s));
  RECAD_CUDA_CHECK(cudaMemsetAsync(w.G, 0, (size_t)stride * sizeof(float), s));
  return pair_sides(PairMode::kJoint, w.OO, nullptr, U, w.OO + U * D2, nullptr, st->n_items, D, w.ia, w.ib, 2 * n, w.alpha,
                    w.beta, w.G, w.G + U * D2, nullptr, nullptr, w.keys, w.tmp, w.sort_scr, w.bad, s);
}

// The Horner pass of G over A2 at width 2D with the SDDMM hook (gvals = g_v) and, when hg is given, the operand gather.
static int mixed_horner(const recad_lightgcn* st, const recad_csr* A2, const MixedWork& w, float* gvals, HornerGather* hg,
                        void* stream) {
  const int L = st->n_layers;
  const int64_t stride = (st->n_users + st->n_items) * 2 * (int64_t)st->D;
  recad_lightgcn joint = *st;
  joint.graph = A2;
  joint.graph_t = nullptr;
  joint.D = 2 * st->D;
  joint.X0 = w.OO;
  joint.X1 = w.X1;
  std::vector<const float*> layers(L);
  for (int l = 0; l < L; ++l) layers[l] = w.Y + l * stride;
  const HornerValues hv{layers.data(), gvals, 1.0f / (float)(L + 1)};
  if (hg) hg->X = layers.data();
  const float* t = nullptr;
  return lightgcn_horner(&joint, w.G, 1.0f / (float)(L + 1), nullptr, &t, stream, &hv, hg);
}

// ------------------------------------------------------------------------------------------
// Candidate-interaction weight gradients (recad_lightgcn_candidate_weight_grads)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
check_ids_kernel(const int64_t* __restrict__ ids, int64_t n, int64_t n_max, int* __restrict__ bad) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n && (ids[k] < 0 || ids[k] >= n_max)) atomicOr(bad, 1);
}

// G[r, :D] += gO[r] over the interleaved [G_O | G_dO] rows (nvec = D / 4)
__global__ void __launch_bounds__(256)
add_first_half_kernel(float* __restrict__ G, const float* __restrict__ gO, int64_t n_rows, int nvec) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_rows * nvec) return;
  const int64_t row = e / nvec;
  float4* g = reinterpret_cast<float4*>(G) + row * 2 * nvec + (e - row * nvec);
  const float4 a = *g, b = __ldg(reinterpret_cast<const float4*>(gO) + e);
  *g = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}

// kpos[b] = the entry (u_b, n_users + p_b) of row u_b, -1 when it is not stored (or an id is out of range: the seeds kernel
// flags it).  One thread per row of the batch, bisection over the user row's ascending columns: the lookup of
// Graph.entry_index (which interaction_hypergradient uses), O(log deg) whatever the user's degree.
__global__ void __launch_bounds__(256)
positive_entry_kernel(const int64_t* __restrict__ samples, int64_t n, const int64_t* __restrict__ rowptr,
                      const int32_t* __restrict__ colidx, int64_t n_users, int64_t n_items, int64_t* __restrict__ kpos) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  const int64_t u = samples[3 * b], p = samples[3 * b + 1];
  int64_t found = -1;
  if (u >= 0 && u < n_users && p >= 0 && p < n_items) {
    const int32_t col = (int32_t)(n_users + p);
    int64_t lo = rowptr[u], hi = rowptr[u + 1];      // first column >= col in [lo, hi)
    while (lo < hi) {
      const int64_t mid = lo + ((hi - lo) >> 1);
      if (__ldg(colidx + mid) < col) lo = mid + 1;
      else hi = mid;
    }
    if (lo < rowptr[u + 1] && colidx[lo] == col) found = lo;
  }
  kpos[b] = found;
}

// The operands' last columns, hi / lo: A[r, K] = coef[sel[r]], B[i, K] = 1, columns K + 1 .. ld - 1 zero
__global__ void __launch_bounds__(256)
tail_split_kernel(const float* __restrict__ coef, const int64_t* __restrict__ sel, int64_t n_sel, int64_t n_users,
                  int64_t n_items, int K, int ld, float* __restrict__ a_hi, float* __restrict__ a_lo, float* __restrict__ b_hi,
                  float* __restrict__ b_lo) {
  const int w = ld - K;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (n_sel + n_items) * w) return;
  const int64_t row = e / w;
  const int c = K + (int)(e - row * w);
  float h = 0.f, l = 0.f;
  if (row < n_sel) {
    if (c == K) {
      int64_t u = sel[row];
      if (u < 0 || u >= n_users) u = 0;
      split_tf32(coef[u], h, l);
    }
    a_hi[row * ld + c] = h;
    a_lo[row * ld + c] = l;
  } else {
    b_hi[(row - n_sel) * ld + c] = c == K ? 1.f : 0.f;
    b_lo[(row - n_sel) * ld + c] = 0.f;
  }
}

// out[r, i] += es[k] / (n mult[k]) at the stored entries k = (sel[r], n_users + i) of the selected user rows: one warp per r,
// one writer per (r, i) (a row's columns are distinct; a repeated id has rows of its own)
__global__ void __launch_bounds__(256)
sample_part_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, const float* __restrict__ mult,
                   const float* __restrict__ es, float nf, const int64_t* __restrict__ sel, int64_t n_sel, int64_t n_users,
                   int64_t n_items, float* __restrict__ out) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n_sel) return;
  const int64_t u = sel[r];
  if (u < 0 || u >= n_users) return;
  for (int64_t e = rowptr[u] + lane; e < rowptr[u + 1]; e += 32) {
    const float v = es[e];
    const int64_t i = (int64_t)colidx[e] - n_users;
    if (v != 0.f && i >= 0 && i < n_items) out[r * n_items + i] += __fdiv_rn(v, __fmul_rn(nf, mult[e]));
  }
}

// Workspace of recad_lightgcn_candidate_weight_grads: the mixed driver's (MixedWork), then g_v [nnz], coef [N], the rows'
// directional derivatives and positive entries [n], the per-entry sums [nnz] and, for L >= 1, the split operands
// A [n_sel, ld] and B [n_items, ld] (hi and lo each), ld = 4 L D + 4.
struct CandWork {
  MixedWork m;
  float *gvals, *coef, *dloss;
  int64_t* kpos;
  float* es;
  float *a_hi, *a_lo, *b_hi, *b_lo;
};

static int64_t cand_ld(int32_t D, int32_t L) { return L > 0 ? 4 * (int64_t)L * D + 4 : 0; }

static int64_t cand_work(int64_t U, int64_t I, int32_t D, int32_t L, int64_t n, int64_t nnz, int64_t n_sel, char* base,
                         CandWork* w) {
  int64_t off = mixed_work(U + I, D, L, n, base, w ? &w->m : nullptr);
  auto take = [&](int64_t bytes) { char* p = base ? base + off : nullptr; off += align256(bytes); return p; };
  const int64_t ld = cand_ld(D, L);
  char* gvals = take(nnz * 4);
  char* coef = take((U + I) * 4);
  char* dloss = take(n * 4);
  char* kpos = take(n * 8);
  char* es = take(nnz * 4);
  char* a_hi = take(n_sel * ld * 4);
  char* a_lo = take(n_sel * ld * 4);
  char* b_hi = take(I * ld * 4);
  char* b_lo = take(I * ld * 4);
  if (w) {
    w->gvals = reinterpret_cast<float*>(gvals);
    w->coef = reinterpret_cast<float*>(coef);
    w->dloss = reinterpret_cast<float*>(dloss);
    w->kpos = reinterpret_cast<int64_t*>(kpos);
    w->es = reinterpret_cast<float*>(es);
    w->a_hi = reinterpret_cast<float*>(a_hi);
    w->a_lo = reinterpret_cast<float*>(a_lo);
    w->b_hi = reinterpret_cast<float*>(b_hi);
    w->b_lo = reinterpret_cast<float*>(b_lo);
  }
  return off;
}

}  // namespace recad

using namespace recad;

extern "C" {

int recad_bpr_fwd_bwd(const float* O, const float* E, int64_t n_users, int64_t n_items, const int64_t* samples,
                      const int64_t* perm, int64_t B, int64_t B_norm, float grad_scale, float* gO, float* cnt,
                      double* loss_acc, int32_t D, void* stream) {
  RECAD_REQUIRE(O && E && samples && gO && cnt && loss_acc, RECAD_ERR_ARG, "bpr: null pointer");
  RECAD_REQUIRE(B >= 0 && B_norm >= B && B_norm > 0 && D >= 4 && D % 4 == 0 && D <= 1024, RECAD_ERR_UNSUPPORTED, "bpr: bad B or D");
  if (B == 0) return RECAD_OK;
  // loss_acc[3] doubles as the out-of-range flag (stays 0.0 when all ids are valid)
  return launch_bpr<int64_t>(O, E, n_users, n_items, samples, perm, B, B_norm, grad_scale, gO, cnt, loss_acc, D,
                             reinterpret_cast<int*>(loss_acc + 3), as_stream(stream));
}

int recad_adam(float* p, const float* g, const float* cnt, float reg_scale, float* m, float* v, int64_t n, int32_t D,
               float lr, float b1, float b2, float eps, int64_t step, void* stream) {
  RECAD_REQUIRE(p && g && m && v && n > 0 && step >= 1, RECAD_ERR_ARG, "adam: bad argument");
  RECAD_REQUIRE(!cnt || (D >= 4 && D % 4 == 0 && n % D == 0), RECAD_ERR_ARG, "adam: cnt needs n %% D == 0, D %% 4 == 0");
  LossFold none{nullptr, 0.0, 0.0};
  return launch_adam(p, g, cnt, reg_scale, m, v, n, D, adam_scalars(lr, b1, b2, eps, step), none, as_stream(stream));
}

int recad_lightgcn_propagate(const recad_lightgcn* st, void* stream) {
  int rc = check_lightgcn(st);
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  const int64_t N = st->n_users + st->n_items;
  const int L = st->n_layers;
  if (L == 0) {
    RECAD_CUDA_CHECK(cudaMemcpyAsync(st->O, st->E, N * st->D * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return RECAD_OK;
  }
  const float* x = st->E;
  for (int k = 0; k < L; ++k) {
    const bool last = k == L - 1;
    float* y = last ? nullptr : ((k & 1) ? st->X1 : st->X0);
    rc = recad_spmm(st->graph, x, y, k == 0 ? st->E : st->O, st->O, last ? 1.0f / (float)(L + 1) : 1.0f, st->D, stream);
    if (rc) return rc;
    x = y;
  }
  return RECAD_OK;
}

}  // extern "C"

template <typename IdxT>
static int lightgcn_train_epoch_t(const recad_lightgcn* st, const IdxT* samples, const IdxT* perm,
                                  int64_t n_samples, int64_t batch, int64_t step0, void* stream) {
  int rc = check_lightgcn(st);
  if (rc) return rc;
  RECAD_REQUIRE(st->m && st->v && st->g && st->cnt && st->loss_acc && st->X0 && st->X1, RECAD_ERR_ARG,
                "lightgcn_train_epoch: null training buffer");
  RECAD_REQUIRE(samples && n_samples > 0 && batch > 0 && step0 >= 0, RECAD_ERR_ARG, "lightgcn_train_epoch: bad samples");
  cudaStream_t s = as_stream(stream);
  const int64_t N = st->n_users + st->n_items;
  const int L = st->n_layers, D = st->D;
  RECAD_CUDA_CHECK(cudaMemsetAsync(st->loss_acc, 0, 4 * sizeof(double), s));
  int64_t step = step0;
  for (int64_t b0 = 0; b0 < n_samples; b0 += batch) {
    const int64_t B = min(batch, n_samples - b0);
    ++step;
    rc = recad_lightgcn_propagate(st, stream);
    if (rc) return rc;
    RECAD_CUDA_CHECK(cudaMemsetAsync(st->g, 0, N * D * sizeof(float), s));
    RECAD_CUDA_CHECK(cudaMemsetAsync(st->cnt, 0, N * sizeof(float), s));
    rc = launch_bpr(st->O, st->E, st->n_users, st->n_items, perm ? samples : samples + 3 * b0, perm ? perm + b0 : (const IdxT*)nullptr, B, B,
                    1.0f / (float)(L + 1), st->g, st->cnt, st->loss_acc, D, reinterpret_cast<int*>(st->loss_acc + 3), s);
    if (rc) return rc;
    // g already carries the 1 / (L + 1) of the layer mean (BPR's grad_scale)
    const float* t = nullptr;
    rc = lightgcn_horner(st, st->g, 1.0f, nullptr, &t, stream);
    if (rc) return rc;
    LossFold fold{st->loss_acc, 1.0 / (double)B, 0.5 * (double)st->lambda};
    rc = launch_adam(st->E, t, st->cnt, st->lambda / (float)B, st->m, st->v, N * D, D,
                     adam_scalars(st->lr, st->beta1, st->beta2, st->eps, step), fold, s);
    if (rc) return rc;
  }
  return RECAD_OK;
}

extern "C" {

int recad_lightgcn_train_epoch(const recad_lightgcn* st, const int64_t* samples, const int64_t* perm,
                               int64_t n_samples, int64_t batch, int64_t step0, void* stream) {
  return lightgcn_train_epoch_t<int64_t>(st, samples, perm, n_samples, batch, step0, stream);
}

int recad_lightgcn_train_epoch_i32(const recad_lightgcn* st, const int32_t* samples, const int32_t* perm,
                                   int64_t n_samples, int64_t batch, int64_t step0, void* stream) {
  return lightgcn_train_epoch_t<int32_t>(st, samples, perm, n_samples, batch, step0, stream);
}

int recad_bpr_fwd_bwd_i32(const float* O, const float* E, int64_t n_users, int64_t n_items, const int32_t* samples,
                          const int32_t* perm, int64_t B, int64_t B_norm, float grad_scale, float* gO, float* cnt,
                          double* loss_acc, int32_t D, void* stream) {
  RECAD_REQUIRE(O && E && samples && gO && cnt && loss_acc, RECAD_ERR_ARG, "bpr: null pointer");
  RECAD_REQUIRE(B >= 0 && B_norm >= B && B_norm > 0 && D >= 4 && D % 4 == 0 && D <= 1024, RECAD_ERR_UNSUPPORTED, "bpr: bad B or D");
  if (B == 0) return RECAD_OK;
  return launch_bpr<int32_t>(O, E, n_users, n_items, samples, perm, B, B_norm, grad_scale, gO, cnt, loss_acc, D,
                             reinterpret_cast<int*>(loss_acc + 3), as_stream(stream));
}

}  // extern "C"

// rows[k] = (users[k], allpos_col[allpos_rowptr[users[k]] + rel[k]], negs[k])
__global__ void __launch_bounds__(256)
samples_expand_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, const uint32_t* __restrict__ users,
                      const uint32_t* __restrict__ rel, const uint32_t* __restrict__ negs, int64_t n, int32_t* __restrict__ rows) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t u = users[k];
    rows[3 * k] = (int32_t)u;
    rows[3 * k + 1] = col[rowptr[u] + rel[k]];
    rows[3 * k + 2] = (int32_t)negs[k];
  }
}

extern "C" {

int recad_samples_expand(const int64_t* allpos_rowptr, const int32_t* allpos_col, const uint32_t* users, const uint32_t* rel,
                         const uint32_t* negs, int64_t n, int32_t* rows, void* stream) {
  RECAD_REQUIRE(n >= 0 && (n == 0 || (allpos_rowptr && allpos_col && users && rel && negs && rows)), RECAD_ERR_ARG,
                "samples_expand: bad argument");
  if (n == 0) return RECAD_OK;
  const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 16);
  samples_expand_kernel<<<grid, 256, 0, as_stream(stream)>>>(allpos_rowptr, allpos_col, users, rel, negs, n, rows);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

int recad_axpby(float* z, float a, const float* x, float b, const float* y, int64_t n, void* stream) {
  RECAD_REQUIRE(z && x && y && n > 0 && n % 4 == 0, RECAD_ERR_ARG, "axpby: n must be a positive multiple of 4");
  const int64_t n4 = n / 4;
  const unsigned grid = (unsigned)std::min<int64_t>((n4 + 255) / 256, (int64_t)sm_count() * 16);
  axpby_kernel<<<grid, 256, 0, as_stream(stream)>>>(z, a, x, b, y, n4);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

int recad_dot_scores(const float* O, int64_t n_users, const int64_t* users, const int64_t* items, int64_t B, int32_t D,
                     float* scores, void* stream) {
  RECAD_REQUIRE(O && users && items && scores && B > 0 && D >= 4 && D % 4 == 0, RECAD_ERR_ARG, "dot_scores: bad argument");
  const int64_t threads = B * 32;
  dot_scores_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, as_stream(stream)>>>(O, n_users, users, items, B, D / 4, scores);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

int64_t recad_pair_scores_backward_scratch_bytes(int64_t B) {
  if (B < 0) return -1;
  return 2 * align256(B * 8) + align256(sort_scratch_bytes(B)) + 256;
}

int recad_pair_scores_backward(const float* Xa, int64_t n_a, const float* Xb, int64_t n_b, int32_t D, const int64_t* ia,
                               const int64_t* ib, int64_t B, const float* g, float* dXa, float* dXb, float* dba, float* dbb,
                               void* scratch, int64_t scratch_bytes, void* stream) {
  return recad_pair_scores_hvp(Xa, nullptr, n_a, Xb, nullptr, n_b, D, ia, ib, B, g, nullptr, dXa, dXb, dba, dbb, scratch,
                               scratch_bytes, stream);
}

int recad_pair_scores_hvp(const float* Xa, const float* Va, int64_t n_a, const float* Xb, const float* Vb, int64_t n_b,
                          int32_t D, const int64_t* ia, const int64_t* ib, int64_t B, const float* alpha, const float* beta,
                          float* outA, float* outB, float* dba, float* dbb, void* scratch, int64_t scratch_bytes, void* stream) {
  RECAD_REQUIRE(Xa && Xb && outA && outB && n_a > 0 && n_b > 0 && B >= 0 && (B == 0 || (ia && ib && alpha && scratch)),
                RECAD_ERR_ARG, "pair_scores: bad argument");
  RECAD_REQUIRE(!beta || (Va && Vb), RECAD_ERR_ARG, "pair_scores_hvp: beta needs Va and Vb");
  RECAD_REQUIRE(D >= 4 && D % 4 == 0 && D <= 1024, RECAD_ERR_UNSUPPORTED, "pair_scores: D must be a multiple of 4 in [4, 1024]");
  RECAD_REQUIRE(n_a < ((int64_t)1 << 31) && n_b < ((int64_t)1 << 31) && B < ((int64_t)1 << 32) - 1, RECAD_ERR_OVERFLOW,
                "pair_scores: tables below 2^31 rows and B below 2^32 - 1");
  RECAD_REQUIRE(B == 0 || scratch_bytes >= recad_pair_scores_backward_scratch_bytes(B), RECAD_ERR_SCRATCH,
                "pair_scores: scratch too small");
  cudaStream_t s = as_stream(stream);
  RECAD_CUDA_CHECK(cudaMemsetAsync(outA, 0, n_a * D * sizeof(float), s));
  RECAD_CUDA_CHECK(cudaMemsetAsync(outB, 0, n_b * D * sizeof(float), s));
  if (dba) RECAD_CUDA_CHECK(cudaMemsetAsync(dba, 0, n_a * sizeof(float), s));
  if (dbb) RECAD_CUDA_CHECK(cudaMemsetAsync(dbb, 0, n_b * sizeof(float), s));
  if (B == 0) return RECAD_OK;
  char* p = static_cast<char*>(scratch);
  uint64_t* keys = reinterpret_cast<uint64_t*>(p);    p += align256(B * 8);
  uint64_t* tmp = reinterpret_cast<uint64_t*>(p);     p += align256(B * 8);
  void* sort_scr = p;                                 p += align256(sort_scratch_bytes(B));
  int* bad = reinterpret_cast<int*>(p);
  RECAD_CUDA_CHECK(cudaMemsetAsync(bad, 0, sizeof(int), s));
  const int rc = pair_sides(beta ? PairMode::kHvp : PairMode::kBackward, Xa, Va, n_a, Xb, Vb, n_b, D, ia, ib, B, alpha, beta,
                            outA, outB, dba, dbb, keys, tmp, sort_scr, bad, s);
  if (rc) return rc;
  int h_bad = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(!h_bad, RECAD_ERR_ARG, "pair_scores: an id is out of range");
  return RECAD_OK;
}

int recad_bpr_hvp_seeds(const float* O, const float* dO, int64_t n_users, int64_t n_items, const int64_t* samples, int64_t n,
                        int64_t B_norm, int32_t D, const float* E, const float* V, float lambda, float* alpha, float* beta,
                        float* dloss, int32_t* bad, void* stream) {
  RECAD_REQUIRE(O && dO && samples && alpha && beta && bad && n_users > 0 && n_items > 0 && n > 0 && B_norm > 0,
                RECAD_ERR_ARG, "bpr_hvp_seeds: bad argument");
  RECAD_REQUIRE(!dloss || (E && V), RECAD_ERR_ARG, "bpr_hvp_seeds: dloss needs E and V");
  RECAD_REQUIRE(D >= 4 && D % 4 == 0 && D <= 1024, RECAD_ERR_UNSUPPORTED, "bpr_hvp_seeds: D must be a multiple of 4 in [4, 1024]");
  cudaStream_t s = as_stream(stream);
  RECAD_CUDA_CHECK(cudaMemsetAsync(bad, 0, sizeof(int32_t), s));
  const int64_t want = (n * kSeedLanes + 255) / 256;
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)sm_count() * 32));
  bpr_hvp_seeds_kernel<<<grid, 256, 0, s>>>(O, dO, n_users, n_items, samples, n, 1.0f / (float)B_norm, D / 4, D / 4, E, V,
                                            lambda, alpha, beta, dloss, bad);
  RECAD_LAUNCH_CHECK();
  int32_t h_bad = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&h_bad, bad, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(!h_bad, RECAD_ERR_ARG, "bpr_hvp_seeds: an id is out of range");
  return RECAD_OK;
}

int recad_lightgcn_backward(const recad_lightgcn* st, const float* gO, float* gE, void* stream) {
  RECAD_REQUIRE(st && st->graph && gO && gE && gO != gE, RECAD_ERR_ARG, "lightgcn_backward: bad argument");
  RECAD_REQUIRE(st->n_users > 0 && st->n_items > 0 && st->graph->n_rows == st->n_users + st->n_items &&
                    (!st->graph_t || st->graph_t->n_rows == st->graph->n_rows),
                RECAD_ERR_ARG, "lightgcn_backward: graph shape");
  RECAD_REQUIRE(st->D >= 4 && st->D % 4 == 0 && st->n_layers >= 0, RECAD_ERR_UNSUPPORTED, "lightgcn_backward: bad D / layers");
  RECAD_REQUIRE((st->n_layers < 2 || st->X0) && (st->n_layers < 3 || st->X1), RECAD_ERR_ARG,
                "lightgcn_backward: null work buffer");
  const int64_t N = st->n_users + st->n_items;
  if (st->n_layers == 0) {
    RECAD_CUDA_CHECK(cudaMemcpyAsync(gE, gO, N * st->D * sizeof(float), cudaMemcpyDeviceToDevice, as_stream(stream)));
    return RECAD_OK;
  }
  const float* t = nullptr;
  return lightgcn_horner(st, gO, 1.0f / (float)(st->n_layers + 1), gE, &t, stream);
}

int recad_lightgcn_backward_values(const recad_lightgcn* st, const float* gO, const float* const* X, float* gE, float* gvals,
                                   void* stream) {
  RECAD_REQUIRE(st && st->graph && gO && gvals && gO != gE, RECAD_ERR_ARG, "lightgcn_backward_values: bad argument");
  RECAD_REQUIRE(st->n_users > 0 && st->n_items > 0 && st->graph->n_rows == st->n_users + st->n_items &&
                    st->graph->n_cols == st->graph->n_rows &&
                    (!st->graph_t || (st->graph_t->n_rows == st->graph->n_rows && st->graph_t->nnz == st->graph->nnz)),
                RECAD_ERR_ARG, "lightgcn_backward_values: graph shape");
  RECAD_REQUIRE(st->D >= 4 && st->D % 4 == 0 && st->n_layers >= 0, RECAD_ERR_UNSUPPORTED,
                "lightgcn_backward_values: bad D / layers");
  const int L = st->n_layers;
  RECAD_REQUIRE((L < 2 || st->X0) && (L < 3 || st->X1), RECAD_ERR_ARG, "lightgcn_backward_values: null work buffer");
  RECAD_REQUIRE(L == 0 || X, RECAD_ERR_ARG, "lightgcn_backward_values: null layer array");
  for (int l = 0; l < L; ++l) RECAD_REQUIRE(X[l], RECAD_ERR_ARG, "lightgcn_backward_values: layer %d is null", l);
  cudaStream_t s = as_stream(stream);
  const int64_t N = st->n_users + st->n_items;
  if (L == 0) {
    if (st->graph->nnz) RECAD_CUDA_CHECK(cudaMemsetAsync(gvals, 0, st->graph->nnz * sizeof(float), s));
    if (gE) RECAD_CUDA_CHECK(cudaMemcpyAsync(gE, gO, N * st->D * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return RECAD_OK;
  }
  const HornerValues hv{X, gvals, 1.0f / (float)(L + 1)};
  const float* t = nullptr;
  return lightgcn_horner(st, gO, 1.0f / (float)(L + 1), gE, &t, stream, &hv);
}

int64_t recad_lightgcn_loss_mixed_values_work_bytes(int64_t n_rows, int32_t D, int32_t n_layers, int64_t n) {
  if (n_rows <= 0 || D < 4 || n_layers < 0 || n <= 0) return -1;
  return mixed_work(n_rows, D, n_layers, n, nullptr, nullptr);
}

int recad_lightgcn_loss_mixed_values(const recad_lightgcn* st, const recad_csr* A2, const float* S, const int64_t* samples,
                                     int64_t n, float* gvals, void* work, int64_t work_bytes, void* stream) {
  int rc = check_lightgcn(st);
  if (rc) return rc;
  RECAD_REQUIRE(A2 && S && samples && gvals && work && n > 0, RECAD_ERR_ARG, "lightgcn_loss_mixed_values: bad argument");
  const recad_csr* A = st->graph;
  RECAD_REQUIRE(!st->graph_t && A->n_cols == A->n_rows && A2->n_rows == A->n_rows && A2->n_cols == A->n_cols &&
                    A2->nnz == A->nnz,
                RECAD_ERR_ARG, "lightgcn_loss_mixed_values: A2 must be the state's own (symmetric) graph at width 2D");
  const int32_t D = st->D, D2 = 2 * st->D;
  const int L = st->n_layers;
  RECAD_REQUIRE(D2 <= 1024, RECAD_ERR_UNSUPPORTED, "lightgcn_loss_mixed_values: D = %d above 512", D);
  RECAD_REQUIRE(n < ((int64_t)1 << 31) - 1, RECAD_ERR_OVERFLOW, "lightgcn_loss_mixed_values: n below 2^31 - 1");
  const int64_t N = st->n_users + st->n_items;
  RECAD_REQUIRE(work_bytes >= mixed_work(N, D, L, n, nullptr, nullptr), RECAD_ERR_SCRATCH,
                "lightgcn_loss_mixed_values: work too small");
  MixedWork w;
  mixed_work(N, D, L, n, static_cast<char*>(work), &w);
  cudaStream_t s = as_stream(stream);
  rc = mixed_recurrence(st, A2, S, samples, n, w, nullptr, 0.0f, stream);
  if (rc) return rc;
  int h_bad = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&h_bad, w.bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(!h_bad, RECAD_ERR_ARG, "lightgcn_loss_mixed_values: an id is out of range");
  if (L == 0) {
    if (A->nnz) RECAD_CUDA_CHECK(cudaMemsetAsync(gvals, 0, A->nnz * sizeof(float), s));
    return RECAD_OK;
  }
  // g_v = (1 / (L + 1)) sum_j <t_j[r], Y_{L-1-j}[c]> over the 2D columns, t_j the Horner iterates of G over A
  return mixed_horner(st, A2, w, gvals, nullptr, stream);
}

int64_t recad_lightgcn_candidate_weight_grads_work_bytes(int64_t n_users, int64_t n_items, int32_t D, int32_t n_layers,
                                                         int64_t n, int64_t nnz, int64_t n_sel) {
  if (n_users <= 0 || n_items <= 0 || D < 4 || n_layers < 0 || n < 0 || nnz < 0 || n_sel < 0) return -1;
  return cand_work(n_users, n_items, D, n_layers, n, nnz, n_sel, nullptr, nullptr);
}

int recad_lightgcn_candidate_weight_grads(const recad_lightgcn* st, const recad_csr* A2, const float* mult,
                                          const int64_t* tperm, const float* d_inv, const float* gO, const float* S,
                                          const int64_t* samples, int64_t n, float lambda, const int64_t* users, int64_t n_sel,
                                          float* out, void* work, int64_t work_bytes, void* stream) {
  int rc = check_lightgcn(st);
  if (rc) return rc;
  RECAD_REQUIRE(A2 && mult && tperm && d_inv && users && out && work && n_sel > 0 && n >= 0 && (n == 0 || (S && samples)),
                RECAD_ERR_ARG, "lightgcn_candidate_weight_grads: bad argument");
  const recad_csr* A = st->graph;
  RECAD_REQUIRE(!st->graph_t && A->n_cols == A->n_rows && A2->n_rows == A->n_rows && A2->n_cols == A->n_cols &&
                    A2->nnz == A->nnz,
                RECAD_ERR_ARG, "lightgcn_candidate_weight_grads: A2 must be the state's own (symmetric) graph at width 2D");
  const int32_t D = st->D;
  const int L = st->n_layers;
  RECAD_REQUIRE(D <= 512, RECAD_ERR_UNSUPPORTED, "lightgcn_candidate_weight_grads: D = %d above 512", D);
  const int64_t U = st->n_users, I = st->n_items, N = U + I, nnz = A->nnz, ld = cand_ld(D, L);
  RECAD_REQUIRE(n < ((int64_t)1 << 31) - 1 && n_sel < ((int64_t)1 << 31) && I < ((int64_t)1 << 31) && ld < ((int64_t)1 << 31),
                RECAD_ERR_OVERFLOW, "lightgcn_candidate_weight_grads: n, users, items and 4 L D below 2^31");
  RECAD_REQUIRE(work_bytes >= cand_work(U, I, D, L, n, nnz, n_sel, nullptr, nullptr), RECAD_ERR_SCRATCH,
                "lightgcn_candidate_weight_grads: work too small");
  CandWork w;
  cand_work(U, I, D, L, n, nnz, n_sel, static_cast<char*>(work), &w);
  cudaStream_t s = as_stream(stream);
  rc = mixed_recurrence(st, A2, S, samples, n, w.m, w.dloss, lambda, stream);
  if (rc) return rc;
  check_ids_kernel<<<(unsigned)((n_sel + 255) / 256), 256, 0, s>>>(users, n_sel, U, w.m.bad);
  RECAD_LAUNCH_CHECK();
  // G = the mixed seed + [gO | 0]: one Horner pass carries the objective's and the loss's parts together
  if (gO) {
    add_first_half_kernel<<<(unsigned)((N * (D / 4) + 255) / 256), 256, 0, s>>>(w.m.G, gO, N, D / 4);
    RECAD_LAUNCH_CHECK();
  }
  // per-entry sums of the rows' directional derivatives over the rows whose positive pair is that stored entry
  if (n > 0) {
    positive_entry_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(samples, n, A->rowptr, A->colidx, U, I, w.kpos);
    RECAD_LAUNCH_CHECK();
    RECAD_CUDA_CHECK(cudaMemsetAsync(w.es, 0, nnz * sizeof(float), s));
    const int bbits = bit_width(n);
    const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 16);
    index_keys_kernel<<<grid, 256, 0, s>>>(w.kpos, n, nnz, bbits, w.m.keys, w.m.bad);
    RECAD_LAUNCH_CHECK();
    rc = radix_sort_u64(w.m.keys, w.m.tmp, n, bbits + bit_width(nnz + 1), w.m.sort_scr, s);
    if (rc) return rc;
    index_sums_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(w.m.keys, n, bbits, (uint64_t)nnz, w.dloss, w.es);
    RECAD_LAUNCH_CHECK();
  }
  if (L == 0) {
    RECAD_CUDA_CHECK(cudaMemsetAsync(out, 0, (size_t)n_sel * I * sizeof(float), s));
  } else {
    // g_v at the stored entries and, gathered at every step, the operands of <a_u, b_i>
    HornerGather hg{nullptr, users, n_sel, U, I, d_inv, 1.0f / (float)(L + 1), (int)ld, w.a_hi, w.a_lo, w.b_hi, w.b_lo};
    rc = mixed_horner(st, A2, w.m, w.gvals, &hg, stream);
    if (rc) return rc;
    // the row-sum term coef_r = -0.5 d_r^3 P_r of the normalisation backward, then column K = [coef_u] x [1]
    rc = csr_normalize_coef(A->rowptr, A->colidx, tperm, mult, d_inv, w.gvals, N, w.coef, s);
    if (rc) return rc;
    const int K = (int)(4 * (int64_t)L * D);
    tail_split_kernel<<<(unsigned)(((n_sel + I) * (ld - K) + 255) / 256), 256, 0, s>>>(w.coef, users, n_sel, U, I, K, (int)ld,
                                                                                         w.a_hi, w.a_lo, w.b_hi, w.b_lo);
    RECAD_LAUNCH_CHECK();
    rc = gemm_tc(w.a_hi, w.a_lo, (int)n_sel, (int)ld, w.b_hi, w.b_lo, (int)I, (int)ld, K + 1, out, (int)I, w.coef + U, false,
                 nullptr, nullptr, 0, s);
    if (rc) return rc;
  }
  if (n > 0) {
    sample_part_kernel<<<(unsigned)((n_sel * 32 + 255) / 256), 256, 0, s>>>(A->rowptr, A->colidx, mult, w.es, (float)n, users,
                                                                            n_sel, U, I, out);
    RECAD_LAUNCH_CHECK();
  }
  int h_bad = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&h_bad, w.m.bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(!h_bad, RECAD_ERR_ARG, "lightgcn_candidate_weight_grads: a user or sample id is out of range");
  return RECAD_OK;
}

int recad_index_sums(const int64_t* idx, const float* x, int64_t n, int64_t n_out, float* out, void* scratch,
                     int64_t scratch_bytes, void* stream) {
  RECAD_REQUIRE(idx && x && out && scratch && n > 0 && n_out > 0, RECAD_ERR_ARG, "index_sums: bad argument");
  RECAD_REQUIRE(n < ((int64_t)1 << 32) - 1 && n_out < ((int64_t)1 << 31), RECAD_ERR_OVERFLOW,
                "index_sums: n below 2^32 - 1 and n_out below 2^31");
  RECAD_REQUIRE(scratch_bytes >= recad_pair_scores_backward_scratch_bytes(n), RECAD_ERR_SCRATCH, "index_sums: scratch too small");
  cudaStream_t s = as_stream(stream);
  char* p = static_cast<char*>(scratch);
  uint64_t* keys = reinterpret_cast<uint64_t*>(p);    p += align256(n * 8);
  uint64_t* tmp = reinterpret_cast<uint64_t*>(p);     p += align256(n * 8);
  void* sort_scr = p;                                 p += align256(sort_scratch_bytes(n));
  int* bad = reinterpret_cast<int*>(p);
  RECAD_CUDA_CHECK(cudaMemsetAsync(bad, 0, sizeof(int), s));
  RECAD_CUDA_CHECK(cudaMemsetAsync(out, 0, n_out * sizeof(float), s));
  const int bbits = bit_width(n);
  const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 16);
  index_keys_kernel<<<grid, 256, 0, s>>>(idx, n, n_out, bbits, keys, bad);
  RECAD_LAUNCH_CHECK();
  const int rc = radix_sort_u64(keys, tmp, n, bbits + bit_width(n_out + 1), sort_scr, s);
  if (rc) return rc;
  index_sums_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(keys, n, bbits, (uint64_t)n_out, x, out);
  RECAD_LAUNCH_CHECK();
  int h_bad = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(!h_bad, RECAD_ERR_ARG, "index_sums: an index is out of range");
  return RECAD_OK;
}

}  // extern "C"
