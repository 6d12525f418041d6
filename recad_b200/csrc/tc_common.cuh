// tcgen05 / TMEM / TMA / mbarrier PTX wrappers shared by the tensor-core kernels (eval_tc.cu, gemm_tc.cu).
// sm_100a only.  Descriptor bit layouts follow cute::UMMA::SmemDescriptor / InstrDescriptor.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <math.h>
#include <stdint.h>

#include "common.cuh"

namespace recad {

// ---------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
// for a waiter that is not on the critical path (a producer running stages ahead): back off between polls so the
// spin does not take issue slots from the warps doing the work
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
  uint32_t done;
  for (;;) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(64);
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// kind::f16: A packed in TMEM (lane = row, two fp16 k elements per 32-bit column, the lower k in the low half), B from
// shared memory, K = 16 per instruction
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// K-major, 128-byte swizzle, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor, version 1 = Blackwell)
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3ffff) >> 4);       // start address
  d |= (uint64_t)1 << 16;                             // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                   // stride byte offset
  d |= (uint64_t)1 << 46;                             // descriptor version
  d |= (uint64_t)2 << 61;                             // SWIZZLE_128B
  return d;
}
// cute::UMMA::InstrDescriptor: D = F32, A = B = TF32, both K-major, dense
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// cute::UMMA::InstrDescriptor: D = F32, A = B = F16 (format 0), both K-major, dense
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }


// x -> (tf32(x), tf32(x - tf32(x))): the two operands of the 3xTF32 scheme
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  uint32_t hb, lb;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(x));
  hi = __uint_as_float(hb);
  const float rem = x - hi;   // exact in fp32
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(rem));
  lo = __uint_as_float(lb);
}

// Two-term fp16 split of a power-of-two scaled operand.  A block (a 64-item tile, a user row) whose largest |x| is m is
// scaled by 2^k, k = f16_scale_exp(m), so that every scaled value is below 2^15 and fits fp16's 5-bit exponent; then
//   hi = fp16_rn(x 2^k),  lo = fp16_rn(x 2^k - hi)          (the subtraction is exact in fp32; 11 + 11 significant bits)
// Scaling is exact, so hi + lo carries x 2^k to ~2^-22 relative, except for elements below fp16's normal range
// (2^-14 after scaling, i.e. 2^-29 of the block's maximum), which keep an absolute accuracy of 2^-25.
__host__ __device__ inline int f16_scale_exp(float m) {
  if (!(m > 0.f) || m > 3.4028235e38f) return 0;   // all-zero block (or inf / nan): unscaled
  int e;
  frexpf(m, &e);                                      // m = f 2^e, f in [0.5, 1)  =>  m 2^(15 - e) < 2^15
  return 15 - e;
}
// x 2^k for |k| <= 252 in two exact power-of-two products (2^k alone may not be a finite fp32)
__device__ __forceinline__ float scale_pow2(float x, int k) {
  const int a = k / 2, b = k - a;
  return (x * __int_as_float((127 + a) << 23)) * __int_as_float((127 + b) << 23);
}
__device__ __forceinline__ void split_f16(float x, int k, uint16_t& hi, uint16_t& lo) {
  const float xs = scale_pow2(x, k);
  const __half h = __float2half_rn(xs);
  hi = __half_as_ushort(h);
  lo = __half_as_ushort(__float2half_rn(xs - __half2float(h)));
}

// 2-D fp32 tensor map [rows, cols] (cols contiguous, cols % 4 == 0), box = [box_rows, 32 cols] with 128-byte swizzle
int make_tensor_map_f32(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int box_rows);
// 2-D fp16 tensor map [rows, 64] (128-byte rows), box = [box_rows, 64] with 128-byte swizzle
int make_tensor_map_f16x64(CUtensorMap* m, const void* base, int64_t rows, int box_rows);

}  // namespace recad
