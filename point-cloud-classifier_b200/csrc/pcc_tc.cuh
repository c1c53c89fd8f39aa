// Blackwell (sm_100a) primitives used by the fused kernels: mbarrier, bulk async copies
// (TMA engine, 1-D), tcgen05 MMA / TMEM.  Inline PTX only; no CUTLASS dependency.
//
// Canonical operand image used everywhere ("tile blob"): a [R rows x K] bf16 operand is
// stored as [K/8][R][8] — 8 consecutive K values of one row are 16 contiguous bytes, rows
// are 16 B apart, K-chunks are R*16 B apart.  That is the UMMA SWIZZLE_NONE canonical
// layout (8x8 core matrices of 128 contiguous bytes) and it can be described
//   * as a K-major  operand [R x K]  : SBO = 128 B (8-row groups), LBO = R*16 B (K chunks)
//   * as an MN-major operand [K x R]^T (MN = K-index of the blob, contraction over rows):
//                                      SBO = R*16 B (MN chunks),   LBO = 128 B (8-row groups)
// so one image serves forward, dgrad and wgrad.  A whole blob is contiguous, so it moves
// with a single cp.async.bulk — no tensor map needed.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace pcc {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// one arrival per warp: every lane has issued its smem writes + proxy fence; lane 0 arrives after the warp converged
__device__ __forceinline__ void mbar_arrive_warp(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase completes (or the hint
// expires) instead of spinning — a bare try_wait loop was measured to burn ~25 % of the SM's issue slots in
// the forward kernel (profiles/notes_r1.md)
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ------------------------------------------------------------------ thread-block clusters / CTA pairs
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the mbarrier at the same shared-memory offset in CTA `cta` of the cluster.  Default (release.cta)
// semantics, as CUTLASS' ClusterBarrier::arrive(cta_id) uses for the same hand-overs: the data handed over is read
// by the tensor core (async proxy, ordered by the fence.proxy.async that precedes the arrive), not by the waiting
// thread; a release at cluster scope here cost ~500 cycles per arrival (profiles/notes_r1.md)
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(bar)), "r"(cta));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(ra) : "memory");
}
__device__ __forceinline__ void mbar_arrive_warp_remote(uint64_t* bar, uint32_t cta) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive_remote(bar, cta);
}
// wait with acquire at cluster scope (arrivals come from the peer CTA); traps instead of hanging the GPU if the
// phase never completes (a protocol bug must fail loudly, not dead-lock a persistent kernel)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  const long long t0 = clock64();
  for (;;) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (ok) return;
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_out) {  // one full warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_out)), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS) : "memory");
}
// D[tmem, both CTAs] (+)= A * B with M = 256 split over the pair (128 rows from each CTA's smem) and B's N split
// likewise; issued by ONE thread of the leader CTA, descriptors are CTA-local offsets valid in both CTAs
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all MMAs issued so far complete -> one arrive on `bar` (same offset) in both CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// generic-proxy smem writes -> visible to the async proxy (tensor core / bulk copy reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------ bulk copies (TMA engine, 1-D)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk stores have finished READING their smem source
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all but the most recently committed bulk store have finished reading their smem source
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ------------------------------------------------------------------ TMEM
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_out) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_out)), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t base) {  // the same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive columns -> 32 registers per thread (thread i = lane base + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

// registers -> TMEM, 32 lanes x 32 consecutive columns
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 16 consecutive columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// ------------------------------------------------------------------ UMMA descriptors
// shared-memory matrix descriptor, SWIZZLE_NONE, version 1 (Blackwell)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version
  return d;
}
// SWIZZLE_128B variants.  Operand image: [C/64 slabs][R rows][64 elements], each row of a slab is 128
// bytes whose eight 16-byte chunks are XOR-permuted with (row & 7) (Swizzle<3,4,3>); slabs must be
// 1024-byte aligned.  byte offset of element (row, col):
__host__ __device__ __forceinline__ uint32_t sw128_off(uint32_t row, uint32_t col, uint32_t R) {
  return (col >> 6) * (R * 128u) + row * 128u + ((((col & 63u) >> 3) ^ (row & 7u)) << 4) + ((col & 7u) << 1);
}
// Activation and gradient tiles are 128-row images: one 64-column slab is 16 KB.
constexpr uint32_t kActSlab = 128u * 128u;
// byte offset of the 16-byte chunk holding columns [col0, col0+8) of row r in a 128-row SW128 image
__device__ __forceinline__ uint32_t act_chunk_off(int r, int col0) {
  return (uint32_t)(col0 >> 6) * kActSlab + (uint32_t)r * 128u + ((uint32_t)(((col0 & 63) >> 3) ^ (r & 7)) << 4);
}
// K-major view [R x K]: start = slab base + 32 B per UMMA K step inside the slab; SBO = 1024 (8-row groups)
__device__ __forceinline__ uint64_t make_smem_desc_sw128_k(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;                 // LBO (unused for swizzled K-major): 1
  d |= (uint64_t)(1024u >> 4) << 32;      // SBO
  d |= (uint64_t)1 << 46;                 // version
  d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
  return d;
}
// MN-major view of the same image (MN = column index, contraction over rows): LBO = slab stride
// (64-column groups), SBO = 1024 (8-row groups); K step of 16 rows = +2048 B
__device__ __forceinline__ uint64_t make_smem_desc_sw128_mn(uint32_t saddr, uint32_t slab_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((slab_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)(1024u >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// instruction descriptor, kind::f16: bf16 x bf16 -> fp32; a_mn / b_mn = 1 for MN-major operands
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) /*C=f32*/ | (1u << 7) /*A=bf16*/ | (1u << 10) /*B=bf16*/ | ((uint32_t)a_mn << 15) |
         ((uint32_t)b_mn << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]   (single thread issues)
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread complete -> one arrive on `bar`
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
// relu fused into the conversion (F2FP.RELU): lo/hi = max(x, 0) rounded to bf16
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// packed fp32 pairs (FFMA2: two fp32 FMAs per issue slot)
__device__ __forceinline__ uint64_t f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f32x2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t fmul2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t splat2(float v) { return f32x2(v, v); }
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }
__device__ __forceinline__ uint64_t bf16x2_to_f32x2(uint32_t u) { return f32x2(bf16_lo(u), bf16_hi(u)); }

}  // namespace tc
}  // namespace pcc
