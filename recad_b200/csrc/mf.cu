// Biased matrix factorisation, pointwise BCE step (reference: recad/model/victim/mf.py:40-69).
//   pred = <Ue[u], Ie[i]> + Ub[u] + Ib[i] + mean        (mean = the constant `factor_num`, mf.py:26)
//   loss = BCEWithLogits(pred, label) (mean over the batch); dense Adam on the four tables.
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace recad {

// A group of LPR lanes owns one (user, item, label) row.  kTrain: also scatter the gradients.
template <int LPR, int VPL, bool kTrain>
__global__ void __launch_bounds__(256)
mf_kernel(const float* __restrict__ Ue, const float* __restrict__ Ub, const float* __restrict__ Ie,
          const float* __restrict__ Ib, float mean, int64_t n_users, int64_t n_items,
          const int64_t* __restrict__ users, const int64_t* __restrict__ items, const int64_t* __restrict__ samples,
          const int64_t* __restrict__ perm, int64_t B, float inv_B, int nvec, float* __restrict__ pred, float* __restrict__ gUe, float* __restrict__ gUb,
          float* __restrict__ gIe, float* __restrict__ gIb, double* __restrict__ loss_acc, int* __restrict__ bad) {
  const int lane = threadIdx.x & 31, l = lane % LPR;
  const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
  const int64_t n_groups = (int64_t)gridDim.x * blockDim.x / LPR;
  const int64_t iters = (B + n_groups - 1) / n_groups;
  const float4* __restrict__ U4 = reinterpret_cast<const float4*>(Ue);
  const float4* __restrict__ I4 = reinterpret_cast<const float4*>(Ie);
  float loss_sum = 0.f;
  for (int64_t it = 0; it < iters; ++it) {
    const int64_t b = it * n_groups + group;
    const bool valid = b < B;
    int64_t u = 0, i = 0, label = 0;
    if (valid) {
      if (kTrain) {   // (user, item, label) rows, visited through the epoch permutation
        const int64_t row = perm ? perm[b] : b;
        u = samples[3 * row]; i = samples[3 * row + 1]; label = samples[3 * row + 2];
      } else {
        u = users[b]; i = items[b];
      }
      if (u < 0 || u >= n_users || i < 0 || i >= n_items) {
        if (l == 0 && bad) atomicOr(bad, 1);
        u = 0; i = 0;
      }
    }
    float4 a[VPL], q[VPL];
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      const int c = l + k * LPR;
      if (valid && c < nvec) {
        a[k] = __ldg(U4 + u * nvec + c);
        q[k] = __ldg(I4 + i * nvec + c);
        dot += a[k].x * q[k].x + a[k].y * q[k].y + a[k].z * q[k].z + a[k].w * q[k].w;
      } else {
        a[k] = q[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) dot += __shfl_xor_sync(kFull, dot, o);
    if (!valid) continue;  // no warp-wide operation below this point inside the loop
    const float x = dot + __ldg(Ub + u) + __ldg(Ib + i) + mean;
    if (!kTrain) {
      if (l == 0) pred[b] = x;
      continue;
    }
    const float y = (float)label;
    // BCEWithLogits: (1 - y) x - log_sigmoid(x),  log_sigmoid(x) = min(x, 0) - log1p(exp(-|x|))
    if (l == 0) loss_sum += (1.f - y) * x - (fminf(x, 0.f) - log1pf(expf(-fabsf(x))));
    const float g = (1.f / (1.f + expf(-x)) - y) * inv_B;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      const int c = l + k * LPR;
      if (c < nvec) {
        red_add4(gUe + (u * nvec + c) * 4, make_float4(g * q[k].x, g * q[k].y, g * q[k].z, g * q[k].w));
        red_add4(gIe + (i * nvec + c) * 4, make_float4(g * a[k].x, g * a[k].y, g * a[k].z, g * a[k].w));
      }
    }
    if (l == 0) {
      atomicAdd(gUb + u, g);
      atomicAdd(gIb + i, g);
    }
  }
  if (kTrain) {
    __shared__ double red[8];
    double t = warp_sum((double)loss_sum);
    if (lane == 0) red[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
      double tot = 0;
      for (int k = 0; k < (int)(blockDim.x >> 5); ++k) tot += red[k];
      atomicAdd(loss_acc, tot);
    }
  }
}

template <bool kTrain>
static int launch_mf(const recad_mf* st, const int64_t* users, const int64_t* items, const int64_t* samples,
                     const int64_t* perm, int64_t B, int64_t B_norm, float* pred, cudaStream_t s) {
  const int nvec = st->D / 4;
  const float inv_B = 1.0f / (float)B_norm;     // mean over the (global) batch
  int* bad = st->loss_acc ? reinterpret_cast<int*>(st->loss_acc + 3) : nullptr;
#define RECAD_MF_LAUNCH(LPR, VPL)                                                                              \
  {                                                                                                            \
    const int64_t gpb = 256 / LPR;                                                                             \
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((B + gpb - 1) / gpb, (int64_t)sm_count() * 32)); \
    mf_kernel<LPR, VPL, kTrain><<<grid, 256, 0, s>>>(st->Ue, st->Ub, st->Ie, st->Ib, st->mean, st->n_users,     \
                                                     st->n_items, users, items, samples, perm, B, inv_B, nvec, pred, st->gUe, \
                                                     st->gUb, st->gIe, st->gIb, st->loss_acc, bad);            \
  }
  if (nvec <= 8) RECAD_MF_LAUNCH(8, 1)
  else if (nvec <= 16) RECAD_MF_LAUNCH(16, 1)
  else if (nvec <= 32) RECAD_MF_LAUNCH(32, 1)
  else if (nvec <= 64) RECAD_MF_LAUNCH(32, 2)
  else if (nvec <= 128) RECAD_MF_LAUNCH(32, 4)
  else RECAD_MF_LAUNCH(32, 8)
#undef RECAD_MF_LAUNCH
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

static int check_mf(const recad_mf* st, bool train) {
  RECAD_REQUIRE(st && st->Ue && st->Ub && st->Ie && st->Ib, RECAD_ERR_ARG, "mf: null parameter table");
  RECAD_REQUIRE(st->n_users > 0 && st->n_items > 0 && st->D >= 4 && st->D % 4 == 0 && st->D <= 1024,
                RECAD_ERR_UNSUPPORTED, "mf: embedding_size must be a multiple of 4 in [4, 1024]");
  if (train)
    RECAD_REQUIRE(st->mUe && st->mUb && st->mIe && st->mIb && st->vUe && st->vUb && st->vIe && st->vIb && st->gUe &&
                      st->gUb && st->gIe && st->gIb && st->loss_acc,
                  RECAD_ERR_ARG, "mf: null training buffer");
  return RECAD_OK;
}

// Seeds of the BCE loss's Hessian-vector product (recad_mf_hvp_seeds), 16 lanes per row.  Along the direction (dUe, dUb,
// dIe, dIb): dy = <dUe_u, Ie_i> + <Ue_u, dIe_i> + dUb_u + dIb_i, l' = sigmoid(y) - label, l'' = sigmoid (1 - sigmoid);
// alpha[b] = l'' dy / B, beta[b] = l' / B, dloss[b] = l' dy.
__global__ void __launch_bounds__(256)
mf_hvp_seeds_kernel(const float* __restrict__ Ue, const float* __restrict__ Ub, const float* __restrict__ Ie,
                    const float* __restrict__ Ib, float mean, int64_t n_users, int64_t n_items,
                    const int64_t* __restrict__ samples, int64_t n, float inv_B, int nvec, const float* __restrict__ dUe,
                    const float* __restrict__ dUb, const float* __restrict__ dIe, const float* __restrict__ dIb,
                    float* __restrict__ alpha, float* __restrict__ beta, float* __restrict__ dloss, int* __restrict__ bad) {
  constexpr int LPR = 16;
  const int l = threadIdx.x % LPR;
  const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
  const int64_t n_groups = (int64_t)gridDim.x * blockDim.x / LPR;
  const int64_t iters = (n + n_groups - 1) / n_groups;       // the same count on every lane: the shuffles are warp-wide
  const float4* __restrict__ U4 = reinterpret_cast<const float4*>(Ue);
  const float4* __restrict__ I4 = reinterpret_cast<const float4*>(Ie);
  const float4* __restrict__ dU4 = reinterpret_cast<const float4*>(dUe);
  const float4* __restrict__ dI4 = reinterpret_cast<const float4*>(dIe);
  for (int64_t it = 0; it < iters; ++it) {
    const int64_t b = it * n_groups + group;
    const bool valid = b < n;
    int64_t u = 0, i = 0, label = 0;
    if (valid) {
      u = samples[3 * b]; i = samples[3 * b + 1]; label = samples[3 * b + 2];
      if (u < 0 || u >= n_users || i < 0 || i >= n_items) {
        if (l == 0) atomicOr(bad, 1);
        u = 0; i = 0;
      }
    }
    float dot = 0.f, dy = 0.f;
    if (valid) {
      for (int c = l; c < nvec; c += LPR) {
        const float4 a = __ldg(U4 + u * nvec + c), q = __ldg(I4 + i * nvec + c);
        const float4 da = __ldg(dU4 + u * nvec + c), dq = __ldg(dI4 + i * nvec + c);
        dot += a.x * q.x + a.y * q.y + a.z * q.z + a.w * q.w;
        dy += da.x * q.x + da.y * q.y + da.z * q.z + da.w * q.w + a.x * dq.x + a.y * dq.y + a.z * dq.z + a.w * dq.w;
      }
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) {
      dot += __shfl_xor_sync(kFull, dot, o);
      dy += __shfl_xor_sync(kFull, dy, o);
    }
    if (valid && l == 0) {
      const float x = dot + __ldg(Ub + u) + __ldg(Ib + i) + mean;
      const float sig = 1.f / (1.f + expf(-x));
      const float d1 = sig - (float)label, d2 = sig * (1.f - sig);
      const float t = dy + __ldg(dUb + u) + __ldg(dIb + i);
      alpha[b] = d2 * t * inv_B;
      beta[b] = d1 * inv_B;
      if (dloss) dloss[b] = d1 * t;
    }
  }
}

}  // namespace recad

using namespace recad;

extern "C" {

int recad_mf_forward(const recad_mf* st, const int64_t* users, const int64_t* items, int64_t B, float* pred,
                     void* stream) {
  int rc = check_mf(st, false);
  if (rc) return rc;
  RECAD_REQUIRE(users && items && pred && B > 0, RECAD_ERR_ARG, "mf_forward: bad argument");
  return launch_mf<false>(st, users, items, nullptr, nullptr, B, B, pred, as_stream(stream));
}

int recad_mf_train_epoch(const recad_mf* st, const int64_t* samples, const int64_t* perm, int64_t n_samples,
                         int64_t batch, int64_t step0, void* stream) {
  int rc = check_mf(st, true);
  if (rc) return rc;
  RECAD_REQUIRE(samples && n_samples > 0 && batch > 0 && step0 >= 0, RECAD_ERR_ARG, "mf_train_epoch: bad samples");
  cudaStream_t s = as_stream(stream);
  const int64_t U = st->n_users, I = st->n_items, D = st->D;
  // order Ue, Ie, Ub, Ib: both embedding tables stay 16-byte aligned when laid out back to back
  const int64_t sz[4] = {U * D, I * D, U, I};
  float* P[4] = {st->Ue, st->Ie, st->Ub, st->Ib};
  float* M[4] = {st->mUe, st->mIe, st->mUb, st->mIb};
  float* V[4] = {st->vUe, st->vIe, st->vUb, st->vIb};
  float* G[4] = {st->gUe, st->gIe, st->gUb, st->gIb};
  // the four tables laid out back to back (what recad_b200.victim.mf allocates): one memset and
  // one Adam launch per step instead of four
  bool flat = true;
  for (int k = 0; k < 3; ++k)
    flat = flat && P[k + 1] == P[k] + sz[k] && M[k + 1] == M[k] + sz[k] && V[k + 1] == V[k] + sz[k] &&
           G[k + 1] == G[k] + sz[k];
  const int64_t total = sz[0] + sz[1] + sz[2] + sz[3];
  RECAD_CUDA_CHECK(cudaMemsetAsync(st->loss_acc, 0, 4 * sizeof(double), s));
  int64_t step = step0;
  for (int64_t b0 = 0; b0 < n_samples; b0 += batch) {
    const int64_t B = min(batch, n_samples - b0);
    ++step;
    if (flat) {
      RECAD_CUDA_CHECK(cudaMemsetAsync(G[0], 0, total * sizeof(float), s));
    } else {
      for (int k = 0; k < 4; ++k) RECAD_CUDA_CHECK(cudaMemsetAsync(G[k], 0, sz[k] * sizeof(float), s));
    }
    rc = launch_mf<true>(st, nullptr, nullptr, perm ? samples : samples + 3 * b0, perm ? perm + b0 : nullptr, B, B, nullptr, s);
    if (rc) return rc;
    const AdamScalars a = adam_scalars(st->lr, st->beta1, st->beta2, st->eps, step);
    // fold: epoch_sum += batch_sum / B   (half_lambda = 0: no regulariser in MF)
    LossFold fold{st->loss_acc, 1.0 / (double)B, 0.0};
    LossFold none{nullptr, 0.0, 0.0};
    if (flat) {
      rc = launch_adam(P[0], G[0], nullptr, 0.f, M[0], V[0], total, 1, a, fold, s);
      if (rc) return rc;
    } else {
      for (int k = 0; k < 4; ++k) {
        rc = launch_adam(P[k], G[k], nullptr, 0.f, M[k], V[k], sz[k], 1, a, k == 0 ? fold : none, s);
        if (rc) return rc;
      }
    }
  }
  return RECAD_OK;
}

int recad_mf_grad(const recad_mf* st, const int64_t* samples, const int64_t* perm, int64_t B, int64_t B_norm,
                  void* stream) {
  int rc = check_mf(st, true);
  if (rc) return rc;
  RECAD_REQUIRE(samples && B >= 0 && B_norm >= B && B_norm > 0, RECAD_ERR_ARG, "mf_grad: bad batch");
  cudaStream_t s = as_stream(stream);
  const int64_t sz[4] = {st->n_users * st->D, st->n_items * st->D, st->n_users, st->n_items};
  float* G[4] = {st->gUe, st->gIe, st->gUb, st->gIb};
  for (int k = 0; k < 4; ++k) RECAD_CUDA_CHECK(cudaMemsetAsync(G[k], 0, sz[k] * sizeof(float), s));
  if (B == 0) return RECAD_OK;     // a rank may own no row of a short last batch: its gradient is zero
  return launch_mf<true>(st, nullptr, nullptr, samples, perm, B, B_norm, nullptr, s);
}

int recad_mf_hvp_seeds(const recad_mf* st, const float* dUe, const float* dUb, const float* dIe, const float* dIb,
                       const int64_t* samples, int64_t n, int64_t B_norm, float* alpha, float* beta, float* dloss, int32_t* bad,
                       void* stream) {
  int rc = check_mf(st, false);
  if (rc) return rc;
  RECAD_REQUIRE(dUe && dUb && dIe && dIb && samples && alpha && beta && bad && n > 0 && B_norm > 0, RECAD_ERR_ARG,
                "mf_hvp_seeds: bad argument");
  cudaStream_t s = as_stream(stream);
  RECAD_CUDA_CHECK(cudaMemsetAsync(bad, 0, sizeof(int32_t), s));
  const int64_t want = (n * 16 + 255) / 256;
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)sm_count() * 32));
  mf_hvp_seeds_kernel<<<grid, 256, 0, s>>>(st->Ue, st->Ub, st->Ie, st->Ib, st->mean, st->n_users, st->n_items, samples, n,
                                           1.0f / (float)B_norm, st->D / 4, dUe, dUb, dIe, dIb, alpha, beta, dloss, bad);
  RECAD_LAUNCH_CHECK();
  int32_t h_bad = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&h_bad, bad, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(!h_bad, RECAD_ERR_ARG, "mf_hvp_seeds: an id is out of range");
  return RECAD_OK;
}

}  // extern "C"
