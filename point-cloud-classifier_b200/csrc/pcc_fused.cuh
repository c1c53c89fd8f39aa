// Shared definitions of the fused tcgen05 DeepSets kernels (forward, backward chain, wgrad).
#pragma once
#include "pcc_act_bf16.cuh"
#include "pcc_common.cuh"
#include "pcc_tc.cuh"

namespace pcc {
using namespace tc;

constexpr int kMaxLayers = 6;
constexpr int kTileM = 128;
constexpr int kK0 = 16;         // layer-0 K padded to one UMMA K step
constexpr int kEpiWarps = 8;    // epilogue warps: TMEM lane quarter = warp & 3, column group = warp >> 2
constexpr int kProdWarp = 8;    // bulk-copy (TMA engine) producer
constexpr int kMmaWarp = 9;     // TMEM allocator + tcgen05.mma issuer
constexpr int kThreads = 320;
constexpr int kEpiThreads = kEpiWarps * 32;

// Operand images.  H x H layers and all activation / gradient tiles use the SWIZZLE_128B image
// [C/64 slabs][R rows][64 elements] (pcc_tc.cuh); layer 0 (K = 16) keeps the un-swizzled
// [2][R][8] image.  A slab of a weight image is R = H rows x 128 B and is the unit streamed
// through the smem ring; an activation tile is R = 128 rows.
__host__ __device__ constexpr uint32_t w_slab_bytes(int H) { return (uint32_t)H * 128u; }

struct PhiParams {
  const float* x;
  const int64_t* offsets;
  int64_t n, B, num_tiles;
  int d, L, pooling, res_mask;
  const uint8_t* wpack;          // packed bf16 weight blobs, all layers
  const float* w0tab;            // layer-0 table [H][4Q] fp32: {b_0, bf16-rounded W_0 row, 0 ...} (forward)
  uint32_t w_off[kMaxLayers];    // byte offset of layer l inside wpack
  const float* bias[kMaxLayers];
  void* pool_acc;                // float[B*H] (sum/mean) or uint64[B*H] (max)
  long long* trace;              // optional (debug): CTA 0 event timestamps, see trace_ev in pcc_fused_phi.cu
  const int32_t* tile_first;     // [num_tiles] first set intersecting each 128-row tile (seg_prep_kernel)
  const int32_t* tile_last;      // [num_tiles] last set intersecting the tile (poolh mode)
  int poolh;                     // sum / mean pooling commuted with the final Linear: pool the last HIDDEN activations
};

// Segment lookups hoisted out of the persistent kernels (a dependent binary search on the epilogue's
// critical path costs ~2k cycles per tile): tile_first[t] = first set b with offsets[b+1] > 128 t;
// row_set[r] = set of row r (-1 past the last set), row_scale[r] = pooled-gradient scale of that set.
static __global__ void seg_prep_kernel(const int64_t* __restrict__ offsets, int64_t n, int64_t B, int64_t num_tiles,
                                       int pooling, int32_t* __restrict__ tile_first, int32_t* __restrict__ row_set,
                                       float* __restrict__ row_scale) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (tile_first && i < num_tiles) {
    const int64_t r0 = i * kTileM;
    int64_t lo = 0, hi = B;
    while (lo < hi) {
      int64_t mid = (lo + hi) >> 1;
      if (__ldg(offsets + mid + 1) <= r0) lo = mid + 1; else hi = mid;
    }
    tile_first[i] = (int32_t)lo;
  }
  if (row_set && i < n) {
    int64_t lo = 0, hi = B;
    while (lo < hi) {
      int64_t mid = (lo + hi) >> 1;
      if (__ldg(offsets + mid + 1) <= i) lo = mid + 1; else hi = mid;
    }
    int32_t set = -1;
    float scale = 0.f;
    if (lo < B && __ldg(offsets + lo) <= i) {
      set = (int32_t)lo;
      const float cnt = (float)(__ldg(offsets + lo + 1) - __ldg(offsets + lo));
      scale = pooling == PCC_POOL_SUM ? rsqrtf(cnt) : (pooling == PCC_POOL_MEAN ? 1.f / cnt : 1.f);
    }
    row_set[i] = set;
    row_scale[i] = scale;
  }
}

// ------------------------------------------------------------------ weight packing
// W_l fp32 [H, K_l] (nn.Linear layout) -> bf16 operand image: layer 0 un-swizzled [2][H][8] (K padded
// to 16), layers >= 1 SWIZZLE_128B [H/64 slabs][H rows][64]
struct PackParams {
  const float* w[kMaxLayers];
  const float* b0;              // layer-0 bias (for the forward's fp32 layer-0 table)
  uint32_t w0tab_off;           // byte offset of that table inside wpack
  int q4;                       // float4 per table row: 4 q4 - 1 >= d
  uint8_t* wpack;
  uint32_t w_off[kMaxLayers];
  uint32_t wt_off[kMaxLayers];  // transposed images (layers >= 1), used when gridDim.z == 2
  int d, H, L;
};
// blockIdx.z == 0: blob of W_l   (rows = out features, K index = in features)   -> forward / recompute
// blockIdx.z == 1: blob of W_l^T (rows = in features,  K index = out features)  -> dgrad, layers >= 1
static __global__ void pack_weights_kernel(PackParams p) {
  const int l = blockIdx.y;
  if (l >= p.L) return;
  const bool tr = blockIdx.z == 1;
  if (tr && l == 0) return;
  const int K = (l == 0) ? p.d : p.H;   // in features of W_l
  const int Kp = (l == 0) ? kK0 : p.H;
  const int total = (Kp / 8) * p.H;     // one thread per 16-byte chunk
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.wpack + (tr ? p.wt_off[l] : p.w_off[l]));
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int kc = i / p.H, row = i % p.H;
    uint32_t pk[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k0 = kc * 8 + 2 * j;
      float a, b;
      if (!tr) {
        a = (k0 < K) ? __ldg(p.w[l] + (int64_t)row * K + k0) : 0.f;
        b = (k0 + 1 < K) ? __ldg(p.w[l] + (int64_t)row * K + k0 + 1) : 0.f;
      } else {  // element (row = in, k = out) = W[out][in]
        a = __ldg(p.w[l] + (int64_t)k0 * K + row);
        b = __ldg(p.w[l] + (int64_t)(k0 + 1) * K + row);
      }
      pk[j] = pack_bf16x2(a, b);
    }
    // chunk kc (8 K values) of row `row`
    const uint32_t off = (l == 0) ? (uint32_t)i * 16u
                                  : (uint32_t)(kc >> 3) * w_slab_bytes(p.H) + (uint32_t)row * 128u +
                                        ((uint32_t)((kc & 7) ^ (row & 7)) << 4);
    *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(dst) + off) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
}

// byte offsets of the weight images inside the packed buffer (same for forward and backward)
struct PackLayout {
  uint32_t w_off[kMaxLayers], wt_off[kMaxLayers];
  uint32_t w0tab_off;  // [H][16] fp32 (sized for the widest table, q4 = 4)
  int64_t total;
};
inline PackLayout pack_layout(int L, int H) {
  PackLayout w{};
  int64_t o = 0;
  auto take = [&](int64_t bytes) { int64_t at = o; o = (o + bytes + 1023) / 1024 * 1024; return at; };
  for (int l = 0; l < L; ++l) w.w_off[l] = (uint32_t)take((int64_t)((l == 0) ? kK0 : H) * H * 2);
  for (int l = 1; l < L; ++l) w.wt_off[l] = (uint32_t)take((int64_t)H * H * 2);
  w.w0tab_off = (uint32_t)take((int64_t)H * 16 * 4);
  w.total = o;
  return w;
}

static __global__ void zero_u64_kernel(unsigned long long* p, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0ull;
}

// ------------------------------------------------------------------ helpers
__device__ __forceinline__ uint32_t pack_bf16x2_pair(uint64_t v) {
  float lo, hi;
  f32x2_unpack(v, lo, hi);
  return pack_bf16x2(lo, hi);
}

__device__ __forceinline__ uint32_t float_ordered(float v) {
  uint32_t b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float ordered_float(uint32_t o) {
  uint32_t b = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
  return __uint_as_float(b);
}

int check_phi_desc(const pcc_phi_desc* d, const char* where);
void* debug_trace_buffer();  // device buffer set through pcc_debug_set_trace, or null
int64_t phi_bwd_workspace_bytes(const pcc_phi_desc* d, int64_t n, int64_t B);

}  // namespace pcc
