// Shared definitions of the fused bf16 GraphNet path (pcc_gnn*.cu): the neighbour stage of
// /root/reference/models/graph_net.py:65-104 (GraphConv -> act -> BatchNorm1d, twice; fc1 -> act -> bn3 ->
// global_mean_pool) with tcgen05 / TMEM GEMMs.
//
// Data flow (C = hidden_dim = 128, M nodes, train mode):
//   conv1  (CUDA cores, K = 2F <= 16) : x[M,F] -> agg1[M,F] fp32, z1[M,C] fp32, partial sums of act(z1), act(z1)^2
//   bn fin : partials -> scale s = gamma*invstd, shift t = beta - mean*s (+ running statistics)
//   apply  : h1 = bf16( act(z1)*s1 + t1 )                                     [M,C] bf16 (stays in L2: 67 MB)
//   conv2  (ONE tcgen05 kernel)       : CSR gather-reduce of h1 rows -> bf16 A image [agg2 | h1] in shared memory
//                                       -> [128 x 2C] x [2C x C] MMA -> z2 fp32 + BatchNorm partial sums; agg2 kept (bf16)
//   apply  : h2 = bf16( act(z2)*s2 + t2 )
//   fc1    (ONE tcgen05 kernel)       : z3 = h2 Wfc1^T + b; a3 = act(z3); BatchNorm partial sums + per-graph sums of a3
//                                       (mean pooling commutes with the BatchNorm affine); z3 never reaches HBM
// and the mirrored backward (pcc_gnn_bwd.cu).  Activations between kernels: fp32 pre-activations z (needed by act'
// and the BatchNorm backward), bf16 normalised activations h (the GEMM / gather operands).
#pragma once
#include "pcc_act_bf16.cuh"
#include "pcc_common.cuh"
#include "pcc_tc.cuh"

namespace pcc {
namespace gnn {
using namespace tc;

constexpr int kC = 128;              // hidden width of the fused path
constexpr int kFc = 256;             // fc1 width (hard-coded in the reference, graph_net.py:61)
constexpr int kTile = 128;           // nodes per tile (= UMMA M)

// Sum over the 32 lanes of a warp of 32 per-lane values, transposed: afterwards v[0] of lane l holds the sum over
// all lanes of their v[l] (31 shuffles instead of 160).
template <int HALF>
__device__ __forceinline__ void tr_step(float* v, int lane) {
  const bool up = (lane & HALF) != 0;
#pragma unroll
  for (int i = 0; i < HALF; ++i) {
    const float send = up ? v[i] : v[i + HALF];
    const float keep = up ? v[i + HALF] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, HALF);
  }
}
__device__ __forceinline__ float warp_transpose_sum32(float (&v)[32], int lane) {
  tr_step<16>(v, lane);
  tr_step<8>(v, lane);
  tr_step<4>(v, lane);
  tr_step<2>(v, lane);
  tr_step<1>(v, lane);
  return v[0];
}

// 16 values per lane: afterwards lanes l and l ^ 16 hold the sum over all 32 lanes of their v[l & 15]
__device__ __forceinline__ float warp_transpose_sum16(float (&v)[16], int lane) {
  tr_step<8>(v, lane);
  tr_step<4>(v, lane);
  tr_step<2>(v, lane);
  tr_step<1>(v, lane);
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 16);
}

__device__ __forceinline__ float2 bf2_to_f2(uint32_t u) { return make_float2(bf16_lo(u), bf16_hi(u)); }

// ---- reduction of the landed rows of a gather slot (conv forward, aggregation backward): lane owns 4 channels = 8
// bytes of every 256-byte row.  Both gather kernels are issue bound (ncu: 60-65 % issue-slot utilisation, half of the
// samples in this loop), so the loop is written for instruction count: packed f32x2 adds (3 instructions per bf16
// pair: two unpacks, one add), two independent chains, and no weight broadcast when the graph is unweighted.
template <int ROWB>
__device__ __forceinline__ void slot_reduce(const uint8_t* slot, int cnt, int lane, bool weighted, float cw, float (&acc)[4]) {
  uint64_t a01 = f32x2(acc[0], acc[1]), a23 = f32x2(acc[2], acc[3]);
  const uint8_t* p = slot + lane * 8;
  if (!weighted) {
    uint64_t b01 = 0ull, b23 = 0ull;
    int u = 0;
#pragma unroll 1
    for (; u + 4 <= cnt; u += 4) {
      const uint2 v0 = *reinterpret_cast<const uint2*>(p + u * ROWB);
      const uint2 v1 = *reinterpret_cast<const uint2*>(p + (u + 1) * ROWB);
      const uint2 v2 = *reinterpret_cast<const uint2*>(p + (u + 2) * ROWB);
      const uint2 v3 = *reinterpret_cast<const uint2*>(p + (u + 3) * ROWB);
      a01 = fadd2(a01, bf16x2_to_f32x2(v0.x)); a23 = fadd2(a23, bf16x2_to_f32x2(v0.y));
      b01 = fadd2(b01, bf16x2_to_f32x2(v1.x)); b23 = fadd2(b23, bf16x2_to_f32x2(v1.y));
      a01 = fadd2(a01, bf16x2_to_f32x2(v2.x)); a23 = fadd2(a23, bf16x2_to_f32x2(v2.y));
      b01 = fadd2(b01, bf16x2_to_f32x2(v3.x)); b23 = fadd2(b23, bf16x2_to_f32x2(v3.y));
    }
#pragma unroll 1
    for (; u < cnt; ++u) {
      const uint2 v0 = *reinterpret_cast<const uint2*>(p + u * ROWB);
      a01 = fadd2(a01, bf16x2_to_f32x2(v0.x)); a23 = fadd2(a23, bf16x2_to_f32x2(v0.y));
    }
    a01 = fadd2(a01, b01); a23 = fadd2(a23, b23);
  } else {
#pragma unroll 2
    for (int u = 0; u < cnt; ++u) {
      const uint2 v = *reinterpret_cast<const uint2*>(p + u * ROWB);
      const float wu = __shfl_sync(0xffffffffu, cw, u);
      const uint64_t w2 = f32x2(wu, wu);
      a01 = ffma2(w2, bf16x2_to_f32x2(v.x), a01); a23 = ffma2(w2, bf16x2_to_f32x2(v.y), a23);
    }
  }
  f32x2_unpack(a01, acc[0], acc[1]);
  f32x2_unpack(a23, acc[2], acc[3]);
}

// bounded mbarrier wait: a protocol bug traps instead of hanging the GPU.  The clock is read once per 1024 failed
// polls only: with a clock read in every iteration the wait loops were 15 % of ALL instructions the conv forward kernel
// executed (ncu, profiles/r2/ncu_gnn_r2e.txt) — issue slots taken from the warps that had work.
__device__ __forceinline__ void mbar_wait_b(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  for (;;) {
#pragma unroll 1
    for (int i = 0; i < 1024; ++i)
      if (mbar_try_wait(bar, parity)) return;
    if (clock64() - t0 > 20000000000ll) __trap();
  }
}

// Coalesced row stores / loads for "thread = row" epilogues.  A lane that writes 32 consecutive words of its own row
// straight to global memory makes every store instruction touch 32 different 128-byte lines (32 L1 wavefronts per
// instruction — the epilogues of the first version were bound by exactly that).  Staged through a per-warp 4 KB shared
// tile ([32 rows][8 chunks of 16 B], chunk index XOR-ed with row & 7), 8 lanes cover one row's 128 bytes and an
// instruction touches 4 lines.  Both sides of the tile are bank-conflict free.
constexpr int kStageWords = 32 * 32;
__device__ __forceinline__ uint4* stage_chunk(uint32_t* stage, int r, int c) {
  return reinterpret_cast<uint4*>(stage + r * 32 + ((c ^ (r & 7)) << 2));
}
// the lane's 32 words of row `lane` -> tile
__device__ __forceinline__ void stage_put_row(uint32_t* stage, const uint32_t (&v)[32], int lane) {
#pragma unroll
  for (int j = 0; j < 8; ++j) *stage_chunk(stage, lane, j) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
__device__ __forceinline__ void stage_get_row(uint32_t* stage, uint32_t (&v)[32], int lane) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint4 t = *stage_chunk(stage, lane, j);
    v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
  }
}
// v[32]: the lane's 32 words of row `lane`; gdst: row 0 of the warp, first column of the chunk; ld in words
__device__ __forceinline__ void warp_store_rows32(uint32_t* stage, const uint32_t (&v)[32], uint32_t* gdst, size_t ld,
                                                  int rows_valid, int lane) {
  stage_put_row(stage, v, lane);
  __syncwarp();
  const int rsub = lane >> 3, c = lane & 7;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = 4 * i + rsub;
    const uint4 t = *stage_chunk(stage, r, c);
    if (r < rows_valid) *reinterpret_cast<uint4*>(gdst + (size_t)r * ld + 4 * c) = t;
  }
  __syncwarp();
}
// 16-word rows (2 KB tile) for kernels without 4 KB of shared memory per epilogue warp: 4 lanes per row, 8 lines per
// instruction
constexpr int kStage16Words = 32 * 16;
__device__ __forceinline__ uint4* stage16_chunk(uint32_t* stage, int r, int c) {
  return reinterpret_cast<uint4*>(stage + r * 16 + ((c ^ ((r >> 1) & 3)) << 2));
}
__device__ __forceinline__ void warp_store_rows16(uint32_t* stage, const uint32_t (&v)[16], uint32_t* gdst, size_t ld,
                                                  int rows_valid, int lane) {
#pragma unroll
  for (int j = 0; j < 4; ++j) *stage16_chunk(stage, lane, j) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  __syncwarp();
  const int rsub = lane >> 2, c = lane & 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = 8 * i + rsub;
    const uint4 t = *stage16_chunk(stage, r, c);
    if (r < rows_valid) *reinterpret_cast<uint4*>(gdst + (size_t)r * ld + 4 * c) = t;
  }
  __syncwarp();
}
// the mirror, in two steps so that the global loads can be issued early: (1) coalesced loads into registers
// (pre[i] = 16 bytes of row 4i + lane/8), (2) through the tile to the lane that owns the row
__device__ __forceinline__ void warp_prefetch_rows32(uint4 (&pre)[8], const uint32_t* gsrc, size_t ld, int rows_valid, int lane) {
  const int rsub = lane >> 3, c = lane & 7;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = 4 * i + rsub;
    pre[i] = make_uint4(0u, 0u, 0u, 0u);
    if (r < rows_valid) pre[i] = __ldg(reinterpret_cast<const uint4*>(gsrc + (size_t)r * ld + 4 * c));
  }
}
__device__ __forceinline__ void warp_deliver_rows32(uint32_t* stage, const uint4 (&pre)[8], uint32_t (&v)[32], int lane) {
  const int rsub = lane >> 3, c = lane & 7;
#pragma unroll
  for (int i = 0; i < 8; ++i) *stage_chunk(stage, 4 * i + rsub, c) = pre[i];
  __syncwarp();
  stage_get_row(stage, v, lane);
  __syncwarp();
}

struct GnnGraph {
  const int64_t* rowptr;   // [M+1] CSR by target (forward) or by source (backward)
  const int32_t* col;      // [E] neighbour node per CSR slot
  const float* w;          // [E] edge weight per CSR slot, or null
  int mean;                // forward: divide the aggregate by the in-degree
};

}  // namespace gnn
}  // namespace pcc
