// 3xTF32 on the tensor cores (mma.sync m16n8k8), shared by the fp32 GEMM kernels (pcc_dense.cu, pcc_head.cu):
// x = hi + lo with hi = tf32(x), lo = tf32(x - hi) and a b ~ a_lo b_hi + a_hi b_lo + a_hi b_hi — error ~2^-21 relative
// per product, fp32 accumulation: the fp32 parity path (rtol 1e-4 against the reference) keeps its accuracy at several
// times the FFMA rate.
#pragma once
#include <stdint.h>

namespace pcc {

// hi = x truncated to TF32 (top 19 bits), lo = x - hi (exact in fp32; the tensor core reads its top 19 bits).
// `cvt.rna.tf32.f32` is emulated with ~6 ALU instructions on this part — the rounding conversion made the split
// 13 instructions per operand element and the kernels ALU bound (profiles/notes_r1.md); truncation costs 2 and
// leaves a relative error of ~2^-20 per product.
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

}  // namespace pcc
