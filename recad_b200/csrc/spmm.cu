// CSR SpMM fused with the LightGCN layer mean:  Y = A X,  Z = alpha * (C + A X).
// (reference: recad/model/victim/lightgcn.py:99-111 `torch.sparse.mm` + stack + mean; the autograd backward of the
// same lines is this kernel again because A_hat is symmetric.)
//
// The product is a gather: per stored entry 8 bytes of (col, val) are streamed and one D*4-byte row of X is fetched.
// On B200 the rows come out of L2 (the item table fits, the user table is made to fit block by block), so the bound
// is L2 -> SM delivery, and the kernel is organised around not wasting any of it:
//   * work unit = one warp per SEGMENT (at most 1024 entries of one row) taken from a PACKED plan: one 16-byte entry
//     {first entry (64 bit), row, (slot + 1) << 11 | count}, loaded one segment ahead, so a segment starts with its
//     bounds in registers instead of a plan -> row pointer -> entries chain of dependent loads;
//   * the matrix is streamed as interleaved (col, val) pairs (`cv`, 8 bytes): the lanes that gather neighbour k load
//     pair k themselves (a broadcast load out of L1) -- no shuffles, which were a third of the L1 data-pipe
//     wavefronts of the first version (profiles/ncu_spmm_r01.md); the pairs of the next round are requested before
//     the gathers of the current round are consumed;
//   * a row of X is covered by D/4 lanes with 128-bit loads, UNR independent gathers in flight per lane;
//   * the plan orders segments longest-first inside each group (no straggler warps at the tail) and may cut the item
//     rows at L2-sized blocks of the user table, processed block by block (recad_b200.ops.PackedPlan);
//   * a row with several segments is finished by whichever of its warps arrives LAST: partial sums are parked in
//     `partials`, a per-row counter elects the last arriver, and it adds the partials in slot order -- deterministic,
//     no second kernel, no second pass.
// The sharded path's epilogue stores a finished row into the owner's NVLink-mapped staging block instead (kScatter).
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"

namespace recad {

constexpr int kSpmmWarps = 8;  // warps per CTA

// Peer-memory epilogue of the sharded path (recad_spmm_scatter): row i of the product is not stored in a local
// Y but sent to the rank that OWNS item i -- dst[i / slice] is that rank's staging block for this sender, mapped
// into this process over NVLink (torch symmetric memory), so the partial sums travel while the SpMM still runs.
constexpr int kMaxPeers = 16;
struct RowScatter {
  float* dst[kMaxPeers];
  int32_t slice;
};

struct SpmmArgs {
  const int4* seg_meta;
  int64_t n_seg;
  const int2* cv;
  const int2* row_mseg;   // per row: (first partial slot, number of segments); only read for multi-segment rows
  int* row_cnt;           // per row arrival counter, zero between launches
  float* partials;
  const float* X;
  float* Y;
  const float* C;
  float* Z;
  float alpha;
};

__device__ __forceinline__ void fma4(float4& a, float w, const float4& x) {
  a.x = fmaf(w, x.x, a.x); a.y = fmaf(w, x.y, a.y); a.z = fmaf(w, x.z, a.z); a.w = fmaf(w, x.w, a.w);
}
__device__ __forceinline__ void add4(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }

template <bool kScatter>
__device__ __forceinline__ void store_row(const SpmmArgs& a, const RowScatter& sc, int64_t row, int nvec, int c, float4 y) {  // Z may alias C
  if (kScatter) {
    const int owner = (int)(row / sc.slice);
    reinterpret_cast<float4*>(sc.dst[owner])[(row - (int64_t)owner * sc.slice) * nvec + c] = y;
    return;
  }
  const int64_t o = row * nvec + c;
  if (a.Y) reinterpret_cast<float4*>(a.Y)[o] = y;
  if (a.Z) {
    float4 cv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a.C) cv = reinterpret_cast<const float4*>(a.C)[o];
    reinterpret_cast<float4*>(a.Z)[o] = make_float4(a.alpha * (cv.x + y.x), a.alpha * (cv.y + y.y), a.alpha * (cv.z + y.z),
                                                    a.alpha * (cv.w + y.w));
  }
}

// after a partial sum was stored: true in every lane of the warp that arrived last for `row`
__device__ __forceinline__ bool last_arriver(const SpmmArgs& a, int row, int lane, int2& ms) {
  __threadfence();
  __syncwarp();
  int last = 0;
  if (lane == 0) {
    ms = __ldg(a.row_mseg + row);
    const int old = atomicAdd(a.row_cnt + row, 1);
    last = old == ms.y - 1;
    if (last) a.row_cnt[row] = 0;                 // ready for the next launch
  }
  last = __shfl_sync(kFull, last, 0);
  if (last) {
    ms.x = __shfl_sync(kFull, ms.x, 0);
    ms.y = __shfl_sync(kFull, ms.y, 0);
    __threadfence();
  }
  return last != 0;
}

template <int D, int UNR, int MINB, bool kScatter>
__global__ void __launch_bounds__(kSpmmWarps * 32, MINB)
spmm_kernel(const __grid_constant__ SpmmArgs a, const __grid_constant__ RowScatter sc) {
  constexpr int LPR = D / 4;               // lanes per row (float4 each)
  constexpr int NPL = 32 / LPR;            // neighbour rows per warp-wide load
  constexpr int R = NPL * UNR;             // entries per round
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPR, l = lane % LPR;
  const int64_t n_warps = (int64_t)gridDim.x * kSpmmWarps;
  int64_t seg = (int64_t)blockIdx.x * kSpmmWarps + (threadIdx.x >> 5);
  if (seg >= a.n_seg) return;
  const float4* __restrict__ X4 = reinterpret_cast<const float4*>(a.X);
  int4 meta = __ldg(a.seg_meta + seg);
  while (true) {
    const int64_t next = seg + n_warps;
    int4 meta_n = make_int4(0, 0, 0, 0);
    if (next < a.n_seg) meta_n = __ldg(a.seg_meta + next);      // one segment ahead
    const int64_t lo = (int64_t)(uint32_t)meta.x | ((int64_t)meta.y << 32);
    const int row = meta.z;
    const int cnt = meta.w & 2047;
    const int slot = (int)((uint32_t)meta.w >> 11) - 1;
    const int2* __restrict__ p = a.cv + lo + sub;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int2 nx[UNR];
#pragma unroll
    for (int u = 0; u < UNR; ++u) nx[u] = (u * NPL + sub < cnt) ? __ldg(p + u * NPL) : make_int2(0, 0);
    for (int j = 0; j < cnt; j += R) {
      float4 x[UNR];
      float w[UNR];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        w[u] = __int_as_float(nx[u].y);
        x[u] = (j + u * NPL + sub < cnt) ? __ldg(X4 + ((uint32_t)nx[u].x * (uint32_t)LPR + (uint32_t)l))   // float4 units; < 2^32 checked on the host
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u)                               // pairs of the next round, under the gathers
        nx[u] = (j + R + u * NPL + sub < cnt) ? __ldg(p + j + R + u * NPL) : make_int2(0, 0);
#pragma unroll
      for (int u = 0; u < UNR; ++u) fma4(acc, w[u], x[u]);
    }
#pragma unroll
    for (int o = 16; o >= LPR; o >>= 1) {
      acc.x += __shfl_xor_sync(kFull, acc.x, o); acc.y += __shfl_xor_sync(kFull, acc.y, o);
      acc.z += __shfl_xor_sync(kFull, acc.z, o); acc.w += __shfl_xor_sync(kFull, acc.w, o);
    }
    if (slot < 0) {
      if (sub == 0) store_row<kScatter>(a, sc, row, LPR, l, acc);
    } else {
      if (sub == 0) reinterpret_cast<float4*>(a.partials)[(int64_t)slot * LPR + l] = acc;
      int2 ms;
      if (last_arriver(a, row, lane, ms)) {
        // partial slots of the row in slot order (fixed association => deterministic), 4 loads in flight per lane
        const float4* __restrict__ P4 = reinterpret_cast<const float4*>(a.partials);
        const int s1 = ms.x + ms.y;
        float4 a4[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) a4[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        int s = ms.x + sub;
        for (; s + 3 * NPL < s1; s += 4 * NPL) {
#pragma unroll
          for (int q = 0; q < 4; ++q) add4(a4[q], __ldcg(P4 + (int64_t)(s + q * NPL) * LPR + l));
        }
        for (; s < s1; s += NPL) add4(a4[0], __ldcg(P4 + (int64_t)s * LPR + l));
        float4 t = make_float4((a4[0].x + a4[1].x) + (a4[2].x + a4[3].x), (a4[0].y + a4[1].y) + (a4[2].y + a4[3].y),
                               (a4[0].z + a4[1].z) + (a4[2].z + a4[3].z), (a4[0].w + a4[1].w) + (a4[2].w + a4[3].w));
#pragma unroll
        for (int o = 16; o >= LPR; o >>= 1) {
          t.x += __shfl_xor_sync(kFull, t.x, o); t.y += __shfl_xor_sync(kFull, t.y, o);
          t.z += __shfl_xor_sync(kFull, t.z, o); t.w += __shfl_xor_sync(kFull, t.w, o);
        }
        if (sub == 0) store_row<kScatter>(a, sc, row, LPR, l, t);
      }
    }
    if (next >= a.n_seg) break;
    seg = next;
    meta = meta_n;
  }
}

// any D that is a multiple of 4 (<= 1024): a lane owns float4 columns lane, lane + 32, ...
constexpr int kGenericMaxVec = 8;
__global__ void __launch_bounds__(kSpmmWarps * 32)
spmm_generic_kernel(const __grid_constant__ SpmmArgs a, int D) {
  const int lane = threadIdx.x & 31;
  const int nvec = D / 4;
  const int64_t n_warps = (int64_t)gridDim.x * kSpmmWarps;
  const float4* __restrict__ X4 = reinterpret_cast<const float4*>(a.X);
  const RowScatter none{};
  for (int64_t seg = (int64_t)blockIdx.x * kSpmmWarps + (threadIdx.x >> 5); seg < a.n_seg; seg += n_warps) {
    const int4 meta = __ldg(a.seg_meta + seg);
    const int64_t lo = (int64_t)(uint32_t)meta.x | ((int64_t)meta.y << 32);
    const int row = meta.z, cnt = meta.w & 2047, slot = (int)((uint32_t)meta.w >> 11) - 1;
    float4 acc[kGenericMaxVec];
#pragma unroll
    for (int q = 0; q < kGenericMaxVec; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < cnt; ++k) {
      const int2 e = __ldg(a.cv + lo + k);
      const float w = __int_as_float(e.y);
#pragma unroll
      for (int q = 0; q < kGenericMaxVec; ++q) {
        const int c = lane + q * 32;
        if (c < nvec) fma4(acc[q], w, __ldg(X4 + (int64_t)e.x * nvec + c));
      }
    }
    if (slot < 0) {
#pragma unroll
      for (int q = 0; q < kGenericMaxVec; ++q)
        if (lane + q * 32 < nvec) store_row<false>(a, none, row, nvec, lane + q * 32, acc[q]);
      continue;
    }
#pragma unroll
    for (int q = 0; q < kGenericMaxVec; ++q)
      if (lane + q * 32 < nvec) reinterpret_cast<float4*>(a.partials)[(int64_t)slot * nvec + lane + q * 32] = acc[q];
    int2 ms;
    if (last_arriver(a, row, lane, ms)) {
      const float4* __restrict__ P4 = reinterpret_cast<const float4*>(a.partials);
#pragma unroll
      for (int q = 0; q < kGenericMaxVec; ++q) {
        const int c = lane + q * 32;
        if (c >= nvec) continue;
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int s = ms.x; s < ms.x + ms.y; ++s) add4(t, __ldcg(P4 + (int64_t)s * nvec + c));
        store_row<false>(a, none, row, nvec, c, t);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- SDDMM
// out[k] (+)= alpha * <G[r_k], X[c_k]> for every stored entry k = (r_k, c_k): the gradient of an SpMM with respect to
// the matrix's values.  The same packed plan drives it (one warp per segment, its entry loaded one segment ahead); G[row]
// sits in registers for the whole segment, the X rows are gathered with D/4 lanes of 128-bit loads, UNR in flight, and
// each dot product is reduced over its LPR lanes with shuffles in a fixed order.  Every entry has exactly one writer, so
// the kernel needs no atomics, partial slots or arrival counters even for multi-segment or column-blocked rows, and
// gives the same bits on every run.  It reads colidx (4 bytes) instead of the (col, val) pairs: the value is not needed.
struct SddmmArgs {
  const int4* seg_meta;
  int64_t n_seg;
  const int32_t* colidx;
  const float* G;
  const float* X;
  float* out;
  float alpha;
  int accumulate;
};

template <int D, int UNR>
__global__ void __launch_bounds__(kSpmmWarps * 32, 4)
sddmm_kernel(const __grid_constant__ SddmmArgs a) {
  constexpr int LPR = D / 4;               // lanes per row (float4 each)
  constexpr int NPL = 32 / LPR;            // entries per warp-wide gather
  constexpr int R = NPL * UNR;             // entries per round
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPR, l = lane % LPR;
  const int64_t n_warps = (int64_t)gridDim.x * kSpmmWarps;
  int64_t seg = (int64_t)blockIdx.x * kSpmmWarps + (threadIdx.x >> 5);
  if (seg >= a.n_seg) return;
  const float4* __restrict__ X4 = reinterpret_cast<const float4*>(a.X);
  const float4* __restrict__ G4 = reinterpret_cast<const float4*>(a.G);
  int4 meta = __ldg(a.seg_meta + seg);
  while (true) {
    const int64_t next = seg + n_warps;
    int4 meta_n = make_int4(0, 0, 0, 0);
    if (next < a.n_seg) meta_n = __ldg(a.seg_meta + next);      // one segment ahead
    const int64_t lo = (int64_t)(uint32_t)meta.x | ((int64_t)meta.y << 32);
    const int cnt = meta.w & 2047;
    const float4 g = cnt ? __ldg(G4 + (int64_t)meta.z * LPR + l) : make_float4(0.f, 0.f, 0.f, 0.f);
    const int32_t* __restrict__ p = a.colidx + lo + sub;
    int nc[UNR];
#pragma unroll
    for (int u = 0; u < UNR; ++u) nc[u] = (u * NPL + sub < cnt) ? __ldg(p + u * NPL) : 0;
    for (int j = 0; j < cnt; j += R) {
      float4 x[UNR];
#pragma unroll
      for (int u = 0; u < UNR; ++u)
        x[u] = (j + u * NPL + sub < cnt) ? __ldg(X4 + ((uint32_t)nc[u] * (uint32_t)LPR + (uint32_t)l))   // < 2^32 checked on the host
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < UNR; ++u)                               // columns of the next round, under the gathers
        nc[u] = (j + R + u * NPL + sub < cnt) ? __ldg(p + j + R + u * NPL) : 0;
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        float d = g.x * x[u].x + g.y * x[u].y + g.z * x[u].z + g.w * x[u].w;
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) d += __shfl_xor_sync(kFull, d, o);
        const int64_t e = lo + j + u * NPL + sub;
        if (l == 0 && j + u * NPL + sub < cnt) a.out[e] = a.accumulate ? fmaf(a.alpha, d, a.out[e]) : a.alpha * d;
      }
    }
    if (next >= a.n_seg) break;
    seg = next;
    meta = meta_n;
  }
}

// any D that is a multiple of 4 (<= 1024): a lane owns float4 columns lane, lane + 32, ...; one entry at a time
__global__ void __launch_bounds__(kSpmmWarps * 32)
sddmm_generic_kernel(const __grid_constant__ SddmmArgs a, int D) {
  const int lane = threadIdx.x & 31;
  const int nvec = D / 4;
  const int64_t n_warps = (int64_t)gridDim.x * kSpmmWarps;
  const float4* __restrict__ X4 = reinterpret_cast<const float4*>(a.X);
  const float4* __restrict__ G4 = reinterpret_cast<const float4*>(a.G);
  for (int64_t seg = (int64_t)blockIdx.x * kSpmmWarps + (threadIdx.x >> 5); seg < a.n_seg; seg += n_warps) {
    const int4 meta = __ldg(a.seg_meta + seg);
    const int64_t lo = (int64_t)(uint32_t)meta.x | ((int64_t)meta.y << 32);
    const int row = meta.z, cnt = meta.w & 2047;
    if (!cnt) continue;
    float4 g[kGenericMaxVec];
#pragma unroll
    for (int q = 0; q < kGenericMaxVec; ++q)
      g[q] = (lane + q * 32 < nvec) ? __ldg(G4 + (int64_t)row * nvec + lane + q * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < cnt; ++k) {
      const int64_t c = __ldg(a.colidx + lo + k);
      float d = 0.f;
#pragma unroll
      for (int q = 0; q < kGenericMaxVec; ++q) {
        if (lane + q * 32 < nvec) {
          const float4 x = __ldg(X4 + c * nvec + lane + q * 32);
          d += g[q].x * x.x + g[q].y * x.y + g[q].z * x.z + g[q].w * x.w;
        }
      }
      d = warp_sum(d);
      if (lane == 0) a.out[lo + k] = a.accumulate ? fmaf(a.alpha, d, a.out[lo + k]) : a.alpha * d;
    }
  }
}

template <int D>
static int launch_sddmm(const SddmmArgs& a, cudaStream_t s) {
  auto kern = sddmm_kernel<D, 4>;
  static int per_sm = 0;
  if (!per_sm) RECAD_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSpmmWarps * 32, 0));
  const int64_t grid = std::min<int64_t>((a.n_seg + kSpmmWarps - 1) / kSpmmWarps, (int64_t)sm_count() * std::max(per_sm, 1));
  kern<<<(unsigned)grid, kSpmmWarps * 32, 0, s>>>(a);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

__global__ void pack_cv_kernel(const int32_t* __restrict__ col, const float* __restrict__ val, int64_t nnz, int2* __restrict__ cv) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (int64_t)gridDim.x * blockDim.x)
    cv[e] = make_int2(col[e], __float_as_int(val[e]));
}

// measured on B200 (profiles/spmm2_sweep_r02.jsonl): 4 gathers in flight per lane, up to 64 registers (4 CTAs / SM)
template <int D, bool kScatter>
static int launch_spmm(const SpmmArgs& a, const RowScatter& sc, cudaStream_t s) {
  auto kern = spmm_kernel<D, 4, 4, kScatter>;
  static int per_sm = 0;
  if (!per_sm) RECAD_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSpmmWarps * 32, 0));
  // persistent launch: the grid is the resident-CTA capacity of the chip and every warp strides over the segment list
  const int64_t grid = std::min<int64_t>((a.n_seg + kSpmmWarps - 1) / kSpmmWarps, (int64_t)sm_count() * std::max(per_sm, 1));
  kern<<<(unsigned)grid, kSpmmWarps * 32, 0, s>>>(a, sc);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

static int check_csr(const recad_csr* A, const char* who) {
  RECAD_REQUIRE(A, RECAD_ERR_ARG, "%s: null matrix", who);
  RECAD_REQUIRE(A->n_rows > 0 && A->n_seg >= A->n_rows && A->seg_meta, RECAD_ERR_ARG, "%s: matrix has no plan (ops.PackedPlan)", who);
  RECAD_REQUIRE(A->nnz == 0 || A->cv, RECAD_ERR_ARG, "%s: null (col, val) pairs (recad_spmm_pack_cv)", who);
  RECAD_REQUIRE(A->n_mrow == 0 || (A->row_mseg && A->row_cnt && A->partials), RECAD_ERR_ARG, "%s: null multi-segment plan", who);
  return RECAD_OK;
}

static SpmmArgs make_args(const recad_csr* A, const float* X, float* Y, const float* C, float* Z, float alpha) {
  SpmmArgs a;
  a.seg_meta = reinterpret_cast<const int4*>(A->seg_meta);
  a.n_seg = A->n_seg;
  a.cv = reinterpret_cast<const int2*>(A->cv);
  a.row_mseg = reinterpret_cast<const int2*>(A->row_mseg);
  a.row_cnt = A->row_cnt;
  a.partials = A->partials;
  a.X = X; a.Y = Y; a.C = C; a.Z = Z; a.alpha = alpha;
  return a;
}

}  // namespace recad

using namespace recad;

extern "C" int recad_spmm_pack_cv(const int32_t* colidx, const float* vals, int64_t nnz, void* cv, void* stream) {
  RECAD_REQUIRE(nnz == 0 || (colidx && vals && cv), RECAD_ERR_ARG, "spmm_pack_cv: null pointer");
  if (nnz == 0) return RECAD_OK;
  const unsigned grid = (unsigned)std::min<int64_t>((nnz + 255) / 256, (int64_t)sm_count() * 16);
  pack_cv_kernel<<<grid, 256, 0, as_stream(stream)>>>(colidx, vals, nnz, reinterpret_cast<int2*>(cv));
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

extern "C" int recad_spmm(const recad_csr* A, const float* X, float* Y, const float* C, float* Z, float alpha,
                          int32_t D, void* stream) {
  cudaStream_t s = as_stream(stream);
  int rc = check_csr(A, "spmm");
  if (rc) return rc;
  RECAD_REQUIRE(X, RECAD_ERR_ARG, "spmm: null X");
  RECAD_REQUIRE(Y || Z, RECAD_ERR_ARG, "spmm: neither Y nor Z requested");
  RECAD_REQUIRE(D >= 4 && D % 4 == 0 && D <= 4 * 32 * kGenericMaxVec, RECAD_ERR_UNSUPPORTED,
                "spmm: D = %d must be a multiple of 4 in [4, %d]", D, 4 * 32 * kGenericMaxVec);
  RECAD_REQUIRE(A->n_cols > 0 && A->n_cols * (int64_t)(D / 4) < ((int64_t)1 << 32), RECAD_ERR_OVERFLOW,
                "spmm: %lld columns x D = %d exceed the 32-bit gather offset", (long long)A->n_cols, D);
  RECAD_REQUIRE((((uintptr_t)X | (uintptr_t)Y | (uintptr_t)C | (uintptr_t)Z | (uintptr_t)A->partials) & 15) == 0,
                RECAD_ERR_ARG, "spmm: buffers must be 16-byte aligned");
  const SpmmArgs a = make_args(A, X, Y, C, Z, alpha);
  const RowScatter none{};
  switch (D) {
    case 8: return launch_spmm<8, false>(a, none, s);        // narrow tables (a column shard of D = 64 over 8 ranks, see DESIGN 6)
    case 16: return launch_spmm<16, false>(a, none, s);
    case 32: return launch_spmm<32, false>(a, none, s);
    case 64: return launch_spmm<64, false>(a, none, s);
    case 128: return launch_spmm<128, false>(a, none, s);
    default: break;
  }
  const int64_t grid = std::min<int64_t>((A->n_seg + kSpmmWarps - 1) / kSpmmWarps, (int64_t)sm_count() * 8);
  spmm_generic_kernel<<<(unsigned)grid, kSpmmWarps * 32, 0, s>>>(a, D);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

extern "C" int recad_csr_sddmm(const recad_csr* A, const float* G, const float* X, int32_t D, float alpha, int32_t accumulate,
                               float* out, void* stream) {
  cudaStream_t s = as_stream(stream);
  RECAD_REQUIRE(A, RECAD_ERR_ARG, "csr_sddmm: null matrix");
  RECAD_REQUIRE(A->n_rows > 0 && A->n_seg >= A->n_rows && A->seg_meta, RECAD_ERR_ARG, "csr_sddmm: matrix has no plan (ops.PackedPlan)");
  RECAD_REQUIRE(G && X && (A->nnz == 0 || (A->colidx && out)), RECAD_ERR_ARG, "csr_sddmm: null pointer");
  RECAD_REQUIRE(D >= 4 && D % 4 == 0 && D <= 4 * 32 * kGenericMaxVec, RECAD_ERR_UNSUPPORTED,
                "csr_sddmm: D = %d must be a multiple of 4 in [4, %d]", D, 4 * 32 * kGenericMaxVec);
  RECAD_REQUIRE(A->n_cols > 0 && A->n_cols * (int64_t)(D / 4) < ((int64_t)1 << 32), RECAD_ERR_OVERFLOW,
                "csr_sddmm: %lld columns x D = %d exceed the 32-bit gather offset", (long long)A->n_cols, D);
  RECAD_REQUIRE((((uintptr_t)G | (uintptr_t)X) & 15) == 0, RECAD_ERR_ARG, "csr_sddmm: G and X must be 16-byte aligned");
  if (A->nnz == 0) return RECAD_OK;
  SddmmArgs a;
  a.seg_meta = reinterpret_cast<const int4*>(A->seg_meta);
  a.n_seg = A->n_seg;
  a.colidx = A->colidx;
  a.G = G; a.X = X; a.out = out; a.alpha = alpha; a.accumulate = accumulate != 0;
  switch (D) {
    case 4: return launch_sddmm<4>(a, s);
    case 8: return launch_sddmm<8>(a, s);
    case 16: return launch_sddmm<16>(a, s);
    case 32: return launch_sddmm<32>(a, s);
    case 64: return launch_sddmm<64>(a, s);
    case 128: return launch_sddmm<128>(a, s);
    default: break;
  }
  const int64_t grid = std::min<int64_t>((A->n_seg + kSpmmWarps - 1) / kSpmmWarps, (int64_t)sm_count() * 8);
  sddmm_generic_kernel<<<(unsigned)grid, kSpmmWarps * 32, 0, s>>>(a, D);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}

// ---------------------------------------------------------------------------------------------- peer-memory path
namespace recad {

struct PeerOut {
  float* out[kMaxPeers];
};

// out[r][e] = sum_s stage[s * stride + e] for every peer r: the owner adds the partial rows its peers sent (fixed
// rank order => every replica receives the same bits) and stores the sum straight into each peer's table
// kMulticast: out[0] is an NVSwitch multicast address -- ONE multimem.st is replicated into every rank's buffer by
// the switch instead of world separate peer stores
template <bool kMulticast>
__global__ void __launch_bounds__(256)
peer_reduce_bcast_kernel(const float4* stage, int n_src, int64_t stride4, int64_t n4, const __grid_constant__ PeerOut po,
                         int n_out) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n4; e += (int64_t)gridDim.x * blockDim.x) {
    float4 a = __ldcg(stage + e);                 // written by peers over NVLink: read at L2, never through L1 / nc
    for (int s = 1; s < n_src; ++s) {
      const float4 p = __ldcg(stage + s * stride4 + e);
      a.x += p.x; a.y += p.y; a.z += p.z; a.w += p.w;
    }
    if (kMulticast) {
      asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(reinterpret_cast<float4*>(po.out[0]) + e),
                   "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w)
                   : "memory");
    } else {
      for (int r = 0; r < n_out; ++r) reinterpret_cast<float4*>(po.out[r])[e] = a;
    }
  }
}

}  // namespace recad

extern "C" int recad_spmm_scatter(const recad_csr* A, const float* X, float* const* dst, int32_t n_dst, int64_t slice_rows,
                                  int32_t D, void* stream) {
  cudaStream_t s = as_stream(stream);
  int rc = check_csr(A, "spmm_scatter");
  if (rc) return rc;
  RECAD_REQUIRE(X && dst, RECAD_ERR_ARG, "spmm_scatter: null argument");
  RECAD_REQUIRE(n_dst >= 1 && n_dst <= kMaxPeers && slice_rows > 0 && slice_rows < ((int64_t)1 << 31) &&
                    slice_rows * n_dst >= A->n_rows,
                RECAD_ERR_ARG, "spmm_scatter: %d destinations of %lld rows do not cover %lld rows", n_dst,
                (long long)slice_rows, (long long)A->n_rows);
  RECAD_REQUIRE(A->n_cols > 0 && A->n_cols * (int64_t)(D / 4) < ((int64_t)1 << 32), RECAD_ERR_OVERFLOW,
                "spmm_scatter: gather offset overflow");
  RowScatter sc{};
  sc.slice = (int32_t)slice_rows;
  for (int r = 0; r < n_dst; ++r) {
    RECAD_REQUIRE(dst[r] && ((uintptr_t)dst[r] & 15) == 0, RECAD_ERR_ARG, "spmm_scatter: destination %d null or misaligned", r);
    sc.dst[r] = dst[r];
  }
  RECAD_REQUIRE((((uintptr_t)X | (uintptr_t)A->partials) & 15) == 0, RECAD_ERR_ARG, "spmm_scatter: buffers must be 16-byte aligned");
  const SpmmArgs a = make_args(A, X, nullptr, nullptr, nullptr, 1.f);
  switch (D) {
    case 32: return launch_spmm<32, true>(a, sc, s);
    case 64: return launch_spmm<64, true>(a, sc, s);
    case 128: return launch_spmm<128, true>(a, sc, s);
    default: break;
  }
  RECAD_REQUIRE(false, RECAD_ERR_UNSUPPORTED, "spmm_scatter: D = %d (supported: 32, 64, 128)", D);
  return RECAD_OK;
}

extern "C" int recad_peer_reduce_bcast(const float* stage, int32_t n_src, int64_t src_stride, int64_t n_floats,
                                       float* const* out, int32_t n_out, int32_t multicast, void* stream) {
  RECAD_REQUIRE(stage && out && n_src >= 1 && n_out >= 1 && n_out <= kMaxPeers && n_floats >= 0 && src_stride >= n_floats,
                RECAD_ERR_ARG, "peer_reduce_bcast: bad argument");
  RECAD_REQUIRE(n_floats % 4 == 0 && src_stride % 4 == 0 && ((uintptr_t)stage & 15) == 0, RECAD_ERR_ARG,
                "peer_reduce_bcast: sizes must be multiples of 4 floats, 16-byte aligned");
  if (n_floats == 0) return RECAD_OK;
  PeerOut po{};
  for (int r = 0; r < n_out; ++r) {
    RECAD_REQUIRE(out[r] && ((uintptr_t)out[r] & 15) == 0, RECAD_ERR_ARG, "peer_reduce_bcast: output %d null or misaligned", r);
    po.out[r] = out[r];
  }
  const int64_t n4 = n_floats / 4;
  const unsigned grid = (unsigned)std::min<int64_t>((n4 + 255) / 256, (int64_t)sm_count() * 8);
  RECAD_REQUIRE(!multicast || n_out == 1, RECAD_ERR_ARG, "peer_reduce_bcast: a multicast store has ONE output address");
  if (multicast)
    peer_reduce_bcast_kernel<true><<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const float4*>(stage), n_src, src_stride / 4,
                                                                        n4, po, n_out);
  else
    peer_reduce_bcast_kernel<false><<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const float4*>(stage), n_src, src_stride / 4,
                                                                         n4, po, n_out);
  RECAD_LAUNCH_CHECK();
  return RECAD_OK;
}
