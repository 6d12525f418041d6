// Device-resident construction of the symmetric-normalised bipartite adjacency
// (reference: recad/dataset/implicit.py:206-213, 243-298, 320-326), its in-place
// extension with injected fake users (implicit.py:482-494) and the SpMM work plan.
//
// Structure is pure integer work (bit-exact by construction): directed keys
// (row << b | col) for both directions -> stable radix sort -> run-length
// de-duplication (multiplicity = what scipy's csr_matrix sums, implicit.py:206-209)
// -> row pointers.  Values are two fp32 products of a host-supplied d_inv.
#include "common.cuh"

namespace recad {

static int ceil_log2(int64_t n) {
  int b = 1;
  while ((int64_t(1) << b) < n) ++b;
  return b;
}

static int64_t align256(int64_t x) { return (x + 255) / 256 * 256; }

__global__ void make_keys_kernel(const int64_t* __restrict__ users, const int64_t* __restrict__ items, int64_t n,
                                 int64_t U, int64_t I, int bits, uint64_t* __restrict__ keys, int* __restrict__ bad) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  int64_t u = users[e], i = items[e];
  if (u < 0 || u >= U || i < 0 || i >= I) {
    atomicOr(bad, 1);
    u = 0;
    i = 0;
  }
  uint64_t r0 = (uint64_t)u, c0 = (uint64_t)(U + i);
  keys[2 * e] = (r0 << bits) | c0;
  keys[2 * e + 1] = (c0 << bits) | r0;
}

__global__ void head_flags_kernel(const uint64_t* __restrict__ keys, int64_t n, uint32_t* __restrict__ flags) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  flags[j] = (j == 0 || keys[j] != keys[j - 1]) ? 1u : 0u;
}

// One thread per sorted key.  Heads write the compacted entry, its multiplicity (run length) and
// the row pointers of every row that starts at (or is skipped before) this entry.
__global__ void compact_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ pos, int64_t n,
                               int bits, int64_t n_rows, const unsigned long long* __restrict__ nnz_dev,
                               int64_t* __restrict__ rowptr, int32_t* __restrict__ colidx,
                               float* __restrict__ mult) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const uint64_t k = keys[j];
  const bool head = (j == 0) || (k != keys[j - 1]);
  const int64_t row = (int64_t)(k >> bits);
  if (head) {
    const int64_t idx = pos[j];
    int64_t run = 1;
    while (j + run < n && keys[j + run] == k) ++run;
    colidx[idx] = (int32_t)(k & ((uint64_t(1) << bits) - 1));
    mult[idx] = (float)run;
    const int64_t prev_row = (j == 0) ? -1 : (int64_t)(keys[j - 1] >> bits);
    for (int64_t r = prev_row + 1; r <= row; ++r) rowptr[r] = idx;
  }
  if (j == n - 1) {
    const int64_t nnz = (int64_t)*nnz_dev;
    for (int64_t r = row + 1; r <= n_rows; ++r) rowptr[r] = nnz;
  }
}

// degree[r] = sum of multiplicities of row r (the fp32 rowsum of implicit.py:269, exact as an
// integer below 2^24).  One warp per row, fixed order.
__global__ void row_degree_kernel(const int64_t* __restrict__ rowptr, const float* __restrict__ mult,
                                  int64_t n_rows, int32_t* __restrict__ degree) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t lo = rowptr[row], hi = rowptr[row + 1];
  int acc = 0;
  for (int64_t e = lo + lane; e < hi; e += 32) acc += (int)mult[e];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
  if (lane == 0) degree[row] = acc;
}

__device__ __forceinline__ int64_t find_row(const int64_t* __restrict__ rowptr, int64_t n_rows, int64_t e) {
  // largest r with rowptr[r] <= e
  int64_t lo = 0, hi = n_rows;
  while (hi - lo > 1) {
    int64_t mid = (lo + hi) >> 1;
    if (rowptr[mid] <= e) lo = mid; else hi = mid;
  }
  return lo;
}

constexpr int kNormPerThread = 8;
__global__ void normalize_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                 const float* __restrict__ mult, const float* __restrict__ d_inv, int64_t n_rows,
                                 int64_t nnz, float* __restrict__ vals) {
  const int64_t e0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * kNormPerThread;
  if (e0 >= nnz) return;
  int64_t row = find_row(rowptr, n_rows, e0);
  int64_t row_end = rowptr[row + 1];
  float dr = d_inv[row];
  for (int k = 0; k < kNormPerThread; ++k) {
    const int64_t e = e0 + k;
    if (e >= nnz) break;
    while (e >= row_end) {
      ++row;
      row_end = rowptr[row + 1];
      dr = d_inv[row];
    }
    // (d_r * a) * d_c, two roundings: scipy's D.dot(A).dot(D) (implicit.py:273-276)
    vals[e] = __fmul_rn(__fmul_rn(dr, mult[e]), d_inv[colidx[e]]);
  }
}

// ------------------------------------------------------------------------------------------
// weights -> values chain: vals_k = d_r w_k d_c, d_r = (s_r + 1e-14)^(-1/2), s_r = sum of row r's weights
// ------------------------------------------------------------------------------------------
// s_r: one warp per row, fixed order, double accumulator rounded to fp32 once
__global__ void __launch_bounds__(256)
row_sums_kernel(const int64_t* __restrict__ rowptr, const float* __restrict__ w, int64_t n_rows, float* __restrict__ sums) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t lo = rowptr[row], hi = rowptr[row + 1];
  double acc = 0.0;
  for (int64_t e = lo + lane; e < hi; e += 32) acc += (double)w[e];
  acc = warp_sum(acc);
  if (lane == 0) sums[row] = (float)acc;
}

// pass 1 of the backward, one warp per row: coef_r = -0.5 d_r^3 P_r with
// P_r = sum over row r's entries k of (gv_k w_k + gv_{T k} w_{T k}) d_{c(k)} -- row r's own entries carry d_r as their row
// factor, their transposes (the entries of column r) as their column factor
__global__ void __launch_bounds__(256)
norm_bwd_rows_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, const int64_t* __restrict__ tperm,
                     const float* __restrict__ w, const float* __restrict__ d_inv, const float* __restrict__ gv, int64_t n_rows,
                     float* __restrict__ coef) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t lo = rowptr[row], hi = rowptr[row + 1];
  double acc = 0.0;
  for (int64_t e = lo + lane; e < hi; e += 32) {
    const int64_t t = tperm[e];
    acc += ((double)gv[e] * (double)w[e] + (double)gv[t] * (double)w[t]) * (double)d_inv[colidx[e]];
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    const double d = d_inv[row];
    coef[row] = (float)(-0.5 * d * d * d * acc);
  }
}

// pass 2, per entry: gw_k = gv_k d_r d_c + coef_r
__global__ void __launch_bounds__(256)
norm_bwd_entries_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, const float* __restrict__ d_inv,
                        const float* __restrict__ gv, const float* __restrict__ coef, int64_t n_rows, int64_t nnz,
                        float* __restrict__ gw) {
  const int64_t e0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * kNormPerThread;
  if (e0 >= nnz) return;
  int64_t row = find_row(rowptr, n_rows, e0);
  int64_t row_end = rowptr[row + 1];
  float dr = d_inv[row], cr = coef[row];
  for (int k = 0; k < kNormPerThread; ++k) {
    const int64_t e = e0 + k;
    if (e >= nnz) break;
    while (e >= row_end) {
      ++row;
      row_end = rowptr[row + 1];
      dr = d_inv[row];
      cr = coef[row];
    }
    gw[e] = fmaf(gv[e] * dr, d_inv[colidx[e]], cr);
  }
}

// ------------------------------------------------------------------------------------------
// in-place fake-user injection
// ------------------------------------------------------------------------------------------
__global__ void count_fake_items_kernel(const int32_t* __restrict__ fake_items, int64_t n, int64_t I,
                                        uint32_t* __restrict__ cnt_item, int* __restrict__ bad) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  int32_t i = fake_items[k];
  if (i < 0 || i >= I) { atomicOr(bad, 1); return; }
  atomicAdd(&cnt_item[i], 1u);
}

__global__ void append_lens_kernel(const int64_t* __restrict__ rowptr, const int64_t* __restrict__ fake_rowptr,
                                   const uint32_t* __restrict__ cnt_item, int64_t U, int64_t I, int64_t F,
                                   uint32_t* __restrict__ lens) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t Nn = U + F + I;
  if (r >= Nn) return;
  uint32_t len;
  if (r < U) len = (uint32_t)(rowptr[r + 1] - rowptr[r]);
  else if (r < U + F) len = (uint32_t)(fake_rowptr[r - U + 1] - fake_rowptr[r - U]);
  else { int64_t i = r - U - F; len = (uint32_t)(rowptr[U + i + 1] - rowptr[U + i]) + cnt_item[i]; }
  lens[r] = len;
}

__global__ void widen_rowptr_kernel(const uint32_t* __restrict__ off, int64_t n, const unsigned long long* total,
                                    int64_t* __restrict__ rowptr) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n) rowptr[r] = off[r];
  if (r == n) rowptr[n] = (int64_t)*total;
}

__global__ void append_copy_old_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                       const float* __restrict__ mult, int64_t U, int64_t I, int64_t F,
                                       const int64_t* __restrict__ new_rowptr, int32_t* __restrict__ new_colidx,
                                       float* __restrict__ new_mult) {
  const int64_t nnz = rowptr[U + I];
  const int64_t e0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * kNormPerThread;
  if (e0 >= nnz) return;
  int64_t row = find_row(rowptr, U + I, e0);
  for (int k = 0; k < kNormPerThread; ++k) {
    const int64_t e = e0 + k;
    if (e >= nnz) break;
    while (e >= rowptr[row + 1]) ++row;
    const bool user_row = row < U;
    const int64_t nrow = user_row ? row : row + F;
    const int64_t p = new_rowptr[nrow] + (e - rowptr[row]);
    new_colidx[p] = user_row ? colidx[e] + (int32_t)F : colidx[e];  // item columns shift by F
    new_mult[p] = mult[e];
  }
}

__global__ void append_fake_rows_kernel(const int64_t* __restrict__ fake_rowptr, const int32_t* __restrict__ fake_items,
                                        int64_t U, int64_t F, const int64_t* __restrict__ new_rowptr,
                                        int32_t* __restrict__ new_colidx, float* __restrict__ new_mult,
                                        uint64_t* __restrict__ item_keys) {
  const int64_t n = fake_rowptr[F];
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  int64_t f = find_row(fake_rowptr, F, k);
  const int64_t p = new_rowptr[U + f] + (k - fake_rowptr[f]);
  new_colidx[p] = (int32_t)(U + F) + fake_items[k];
  new_mult[p] = 1.0f;
  item_keys[k] = ((uint64_t)(uint32_t)fake_items[k] << 32) | (uint64_t)f;  // sort -> (item, fake user)
}

__global__ void append_item_tails_kernel(const uint64_t* __restrict__ item_keys, int64_t n,
                                         const int64_t* __restrict__ rowptr, int64_t U, int64_t F,
                                         const int64_t* __restrict__ new_rowptr, int32_t* __restrict__ new_colidx,
                                         float* __restrict__ new_mult) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint64_t key = item_keys[k];
  const int64_t i = (int64_t)(key >> 32), f = (int64_t)(key & 0xffffffffu);
  int64_t rank = 0;
  while (k - rank - 1 >= 0 && (int64_t)(item_keys[k - rank - 1] >> 32) == i) ++rank;
  const int64_t old_len = rowptr[U + i + 1] - rowptr[U + i];
  const int64_t p = new_rowptr[U + F + i] + old_len + rank;
  new_colidx[p] = (int32_t)(U + f);
  new_mult[p] = 1.0f;
}

// pass 1 of the normalisation backward on its own: coef [n_rows] from gv [nnz]; no host synchronisation.  Also the row term
// of an interaction that is not stored yet (recad_lightgcn_candidate_weight_grads)
int csr_normalize_coef(const int64_t* rowptr, const int32_t* colidx, const int64_t* tperm, const float* w, const float* d_inv,
                       const float* gv, int64_t n_rows, float* coef, cudaStream_t s) {
  const int T = 256;
  norm_bwd_rows_kernel<<<(unsigned)((n_rows * 32 + T - 1) / T), T, 0, s>>>(rowptr, colidx, tperm, w, d_inv, gv, n_rows, coef);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

}  // namespace recad

using namespace recad;

extern "C" {

int64_t recad_csr_build_scratch_bytes(int64_t n_edges, int64_t n_users, int64_t n_items) {
  const int64_t n = 2 * n_edges;
  return 2 * align256(n * 8) + align256(n * 4) + sort_scratch_bytes(n) + scan_scratch_bytes(n) + 1024;
}

int recad_csr_build_structure(const int64_t* users, const int64_t* items, int64_t n_edges, int64_t n_users,
                              int64_t n_items, int64_t* rowptr, int32_t* colidx, float* mult, int32_t* degree,
                              int64_t* nnz_out, void* scratch, int64_t scratch_bytes, void* stream) {
  cudaStream_t s = as_stream(stream);
  RECAD_REQUIRE(n_edges >= 0 && n_users > 0 && n_items > 0, RECAD_ERR_ARG, "csr_build: bad sizes");
  RECAD_REQUIRE(rowptr && degree && nnz_out, RECAD_ERR_ARG, "csr_build: null output");
  const int64_t N = n_users + n_items;
  RECAD_REQUIRE(N < (int64_t(1) << 31), RECAD_ERR_OVERFLOW, "csr_build: N = %lld exceeds int32 columns", (long long)N);
  RECAD_REQUIRE(2 * n_edges < (int64_t)0xffffffffLL, RECAD_ERR_OVERFLOW, "csr_build: too many edges");
  RECAD_REQUIRE(scratch_bytes >= recad_csr_build_scratch_bytes(n_edges, n_users, n_items), RECAD_ERR_SCRATCH,
                "csr_build: scratch too small");
  const int64_t n = 2 * n_edges;
  if (n == 0) {
    RECAD_CUDA_CHECK(cudaMemsetAsync(rowptr, 0, (N + 1) * sizeof(int64_t), s));
    RECAD_CUDA_CHECK(cudaMemsetAsync(degree, 0, N * sizeof(int32_t), s));
    RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
    *nnz_out = 0;
    return RECAD_OK;
  }
  RECAD_REQUIRE(users && items && colidx && mult && scratch, RECAD_ERR_ARG, "csr_build: null pointer");
  char* p = reinterpret_cast<char*>(scratch);
  uint64_t* keys = reinterpret_cast<uint64_t*>(p); p += align256(n * 8);
  uint64_t* tmp = reinterpret_cast<uint64_t*>(p);  p += align256(n * 8);
  uint32_t* pos = reinterpret_cast<uint32_t*>(p);  p += align256(n * 4);
  unsigned long long* total = reinterpret_cast<unsigned long long*>(p);
  int* bad = reinterpret_cast<int*>(p + 8);        p += 256;
  void* sort_scr = p;                               p += sort_scratch_bytes(n);
  void* scan_scr = p;
  const int bits = ceil_log2(N);
  RECAD_CUDA_CHECK(cudaMemsetAsync(total, 0, 256, s));
  const int T = 256;
  make_keys_kernel<<<(unsigned)((n_edges + T - 1) / T), T, 0, s>>>(users, items, n_edges, n_users, n_items, bits, keys, bad);
  RECAD_LAUNCH_CHECK();
  int rc = radix_sort_u64(keys, tmp, n, 2 * bits, sort_scr, s);
  if (rc) return rc;
  uint32_t* flags = reinterpret_cast<uint32_t*>(tmp);  // the ping-pong buffer is free again
  head_flags_kernel<<<(unsigned)((n + T - 1) / T), T, 0, s>>>(keys, n, flags);
  RECAD_LAUNCH_CHECK();
  rc = exclusive_scan_u32(flags, pos, n, total, scan_scr, s);
  if (rc) return rc;
  compact_kernel<<<(unsigned)((n + T - 1) / T), T, 0, s>>>(keys, pos, n, bits, N, total, rowptr, colidx, mult);
  RECAD_LAUNCH_CHECK();
  row_degree_kernel<<<(unsigned)((N * 32 + T - 1) / T), T, 0, s>>>(rowptr, mult, N, degree);
  RECAD_LAUNCH_CHECK();
  unsigned long long h_total = 0;
  int h_bad = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&h_total, total, 8, cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(!h_bad, RECAD_ERR_ARG, "csr_build: user or item id out of range [0,%lld) x [0,%lld)",
                (long long)n_users, (long long)n_items);
  *nnz_out = (int64_t)h_total;
  return RECAD_OK;
}

int recad_csr_normalize(const int64_t* rowptr, const int32_t* colidx, const float* mult, const float* d_inv,
                        int64_t n_rows, float* vals, void* stream) {
  cudaStream_t s = as_stream(stream);
  RECAD_REQUIRE(rowptr && d_inv && n_rows > 0, RECAD_ERR_ARG, "csr_normalize: bad argument");
  int64_t nnz = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&nnz, rowptr + n_rows, 8, cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  if (nnz == 0) return RECAD_OK;
  RECAD_REQUIRE(colidx && mult && vals, RECAD_ERR_ARG, "csr_normalize: null pointer");
  const int T = 256;
  const int64_t threads = (nnz + kNormPerThread - 1) / kNormPerThread;
  normalize_kernel<<<(unsigned)((threads + T - 1) / T), T, 0, s>>>(rowptr, colidx, mult, d_inv, n_rows, nnz, vals);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

// rowptr[n_rows] must be nnz (one 8-byte device->host copy, synchronises the stream)
static int check_nnz(const int64_t* rowptr, int64_t n_rows, int64_t nnz, cudaStream_t s, const char* who) {
  int64_t have = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&have, rowptr + n_rows, 8, cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(have == nnz, RECAD_ERR_ARG, "%s: the row pointer ends at %lld, not at nnz = %lld", who, (long long)have,
                (long long)nnz);
  return RECAD_OK;
}

int recad_csr_row_sums(const int64_t* rowptr, const float* w, int64_t n_rows, int64_t nnz, float* sums, void* stream) {
  cudaStream_t s = as_stream(stream);
  RECAD_REQUIRE(rowptr && sums && n_rows > 0 && nnz >= 0 && (nnz == 0 || w), RECAD_ERR_ARG, "csr_row_sums: bad argument");
  int rc = check_nnz(rowptr, n_rows, nnz, s, "csr_row_sums");
  if (rc) return rc;
  const int T = 256;
  row_sums_kernel<<<(unsigned)((n_rows * 32 + T - 1) / T), T, 0, s>>>(rowptr, w, n_rows, sums);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

int recad_csr_normalize_backward(const int64_t* rowptr, const int32_t* colidx, const int64_t* tperm, const float* w,
                                 const float* d_inv, const float* gv, int64_t n_rows, int64_t nnz, float* coef, float* gw,
                                 void* stream) {
  cudaStream_t s = as_stream(stream);
  RECAD_REQUIRE(rowptr && d_inv && coef && n_rows > 0 && nnz >= 0, RECAD_ERR_ARG, "csr_normalize_backward: bad argument");
  RECAD_REQUIRE(nnz == 0 || (colidx && tperm && w && gv && gw), RECAD_ERR_ARG, "csr_normalize_backward: null pointer");
  int rc = check_nnz(rowptr, n_rows, nnz, s, "csr_normalize_backward");
  if (rc) return rc;
  if (nnz == 0) return RECAD_OK;
  rc = csr_normalize_coef(rowptr, colidx, tperm, w, d_inv, gv, n_rows, coef, s);
  if (rc) return rc;
  const int T = 256;
  const int64_t threads = (nnz + kNormPerThread - 1) / kNormPerThread;
  norm_bwd_entries_kernel<<<(unsigned)((threads + T - 1) / T), T, 0, s>>>(rowptr, colidx, d_inv, gv, coef, n_rows, nnz, gw);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

int64_t recad_csr_append_scratch_bytes(int64_t n_users, int64_t n_items, int64_t n_fake, int64_t n_fake_edges) {
  const int64_t Nn = n_users + n_items + n_fake;
  return align256(n_items * 4) + 2 * align256((Nn + 1) * 4) + 2 * align256(n_fake_edges * 8 + 8) +
         sort_scratch_bytes(n_fake_edges) + scan_scratch_bytes(Nn + 1) + 1024;
}

int recad_csr_append_users(const int64_t* rowptr, const int32_t* colidx, const float* mult, int64_t U, int64_t I,
                           int64_t F, const int64_t* fake_rowptr, const int32_t* fake_items, int64_t n_fake_edges,
                           int64_t* new_rowptr, int32_t* new_colidx, float* new_mult, int32_t* new_degree,
                           void* scratch, int64_t scratch_bytes, void* stream) {
  cudaStream_t s = as_stream(stream);
  RECAD_REQUIRE(U > 0 && I > 0 && F >= 0 && n_fake_edges >= 0, RECAD_ERR_ARG, "csr_append: bad sizes");
  RECAD_REQUIRE(rowptr && fake_rowptr && new_rowptr && new_degree && scratch, RECAD_ERR_ARG, "csr_append: null pointer");
  RECAD_REQUIRE(scratch_bytes >= recad_csr_append_scratch_bytes(U, I, F, n_fake_edges), RECAD_ERR_SCRATCH,
                "csr_append: scratch too small");
  const int64_t Nn = U + F + I;
  RECAD_REQUIRE(Nn < (int64_t(1) << 31), RECAD_ERR_OVERFLOW, "csr_append: N exceeds int32 columns");
  int64_t nnz_old = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&nnz_old, rowptr + U + I, 8, cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(nnz_old + 2 * n_fake_edges < (int64_t)0xffffffffLL, RECAD_ERR_OVERFLOW, "csr_append: nnz overflow");
  char* p = reinterpret_cast<char*>(scratch);
  uint32_t* cnt_item = reinterpret_cast<uint32_t*>(p); p += align256(I * 4);
  uint32_t* lens = reinterpret_cast<uint32_t*>(p);     p += align256((Nn + 1) * 4);
  uint32_t* offs = reinterpret_cast<uint32_t*>(p);     p += align256((Nn + 1) * 4);
  uint64_t* ikeys = reinterpret_cast<uint64_t*>(p);    p += align256(n_fake_edges * 8 + 8);
  uint64_t* itmp = reinterpret_cast<uint64_t*>(p);     p += align256(n_fake_edges * 8 + 8);
  unsigned long long* total = reinterpret_cast<unsigned long long*>(p);
  int* bad = reinterpret_cast<int*>(p + 8);            p += 256;
  void* sort_scr = p;                                   p += sort_scratch_bytes(n_fake_edges);
  void* scan_scr = p;
  const int T = 256;
  RECAD_CUDA_CHECK(cudaMemsetAsync(cnt_item, 0, I * 4, s));
  RECAD_CUDA_CHECK(cudaMemsetAsync(total, 0, 256, s));
  if (n_fake_edges > 0) {
    RECAD_REQUIRE(fake_items, RECAD_ERR_ARG, "csr_append: null fake_items");
    count_fake_items_kernel<<<(unsigned)((n_fake_edges + T - 1) / T), T, 0, s>>>(fake_items, n_fake_edges, I, cnt_item, bad);
    RECAD_LAUNCH_CHECK();
  }
  append_lens_kernel<<<(unsigned)((Nn + T - 1) / T), T, 0, s>>>(rowptr, fake_rowptr, cnt_item, U, I, F, lens);
  RECAD_LAUNCH_CHECK();
  int rc = exclusive_scan_u32(lens, offs, Nn, total, scan_scr, s);
  if (rc) return rc;
  widen_rowptr_kernel<<<(unsigned)((Nn + 1 + T - 1) / T), T, 0, s>>>(offs, Nn, total, new_rowptr);
  RECAD_LAUNCH_CHECK();
  if (nnz_old > 0) {
    const int64_t threads = (nnz_old + kNormPerThread - 1) / kNormPerThread;
    append_copy_old_kernel<<<(unsigned)((threads + T - 1) / T), T, 0, s>>>(rowptr, colidx, mult, U, I, F, new_rowptr,
                                                                          new_colidx, new_mult);
    RECAD_LAUNCH_CHECK();
  }
  if (n_fake_edges > 0) {
    append_fake_rows_kernel<<<(unsigned)((n_fake_edges + T - 1) / T), T, 0, s>>>(fake_rowptr, fake_items, U, F, new_rowptr,
                                                                                new_colidx, new_mult, ikeys);
    RECAD_LAUNCH_CHECK();
    rc = radix_sort_u64(ikeys, itmp, n_fake_edges, 64, sort_scr, s);
    if (rc) return rc;
    append_item_tails_kernel<<<(unsigned)((n_fake_edges + T - 1) / T), T, 0, s>>>(ikeys, n_fake_edges, rowptr, U, F,
                                                                                 new_rowptr, new_colidx, new_mult);
    RECAD_LAUNCH_CHECK();
  }
  row_degree_kernel<<<(unsigned)((Nn * 32 + T - 1) / T), T, 0, s>>>(new_rowptr, new_mult, Nn, new_degree);
  RECAD_LAUNCH_CHECK();
  int h_bad = 0;
  RECAD_CUDA_CHECK(cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, s));
  RECAD_CUDA_CHECK(cudaStreamSynchronize(s));
  RECAD_REQUIRE(!h_bad, RECAD_ERR_ARG, "csr_append: fake item id out of range");
  return RECAD_OK;
}

}  // extern "C"
