// Fused bf16 GraphNet path, backward kernels (autograd of /root/reference/models/graph_net.py:73-92), see pcc_gnn.cuh.
//
// One block  z = A W^T + b,  a = act(z),  h = BN(a) = a s + t  (s = gamma invstd, t = beta - mean s,  xhat = (a - mean) invstd):
//   dgamma = sum dh xhat,  dbeta = sum dh,  dz = s (dh - dbeta/M - xhat dgamma/M) act'(z)
// so every backward kernel needs the two column sums (dbeta, dgamma) of ITS incoming gradient before it can form dz: the
// kernel that PRODUCES a gradient tensor also accumulates those two sums (per-CTA partials, reduced by
// gnn_bn_bwd_finalize), and the consumer folds the BatchNorm / activation backward into its operand prologue.
//   fc1 bwd  (tcgen05): recompute z3 = h2 Wfc1^T per tile, dz3 (bn3 + mean-pool backward are per-graph / per-channel
//                       terms), dh2 = dz3 Wfc1, dWfc1 += dz3^T h2 in TMEM, sums for bn2
//   conv bwd (tcgen05): dz2 in the prologue, [dagg2 | droot] = dz2 [W_rel | W_root], dW += dz2^T [agg2 | h1] in TMEM
//   agg bwd  (CUDA cores): dh1 = droot + A^T dagg2 (CSR by source, bf16 rows), sums for bn1
//   conv1 bwd (CUDA cores): dz1, dW_rel1 / dW_root1 / db1 (K = 2F)
// The [M,128] gradient tensors between these kernels (dh2, dagg2, droot -> dh1) are bf16; the BatchNorm sums are taken
// from the fp32 values before the store.
#include "pcc_gnn.cuh"

namespace pcc {
namespace gnn {

int gnn_resident_blocks(const void* kern, int threads, int smem_bytes, int64_t want);   // pcc_gnn.cu

// bnb arrays: [5][Cn] = {mean, invstd, scale, c1 = dbeta/M, c2 = dgamma/M}
struct BnBack {
  const float* mean;
  const float* invstd;
  const float* scale;
  const float* c1;
  const float* c2;
};

// partial sums [nblk][2][Cn] (sum dh, sum dh xhat) -> c1, c2, dgamma, dbeta
__global__ void __launch_bounds__(256) gnn_bn_bwd_finalize_kernel(const float* __restrict__ partials, int nblk, int Cn, int64_t rows,
                                           float* __restrict__ c1, float* __restrict__ c2, float* __restrict__ dgamma,
                                           float* __restrict__ dbeta) {
  __shared__ double red[8][2][32];
  const int cl = threadIdx.x & 31, gq = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  double s1 = 0.0, s2 = 0.0;
  if (c < Cn) {
    int b = gq;
    for (; b + 24 < nblk; b += 32) {
      const float a0 = __ldg(partials + (size_t)b * 2 * Cn + c), a1 = __ldg(partials + (size_t)(b + 8) * 2 * Cn + c);
      const float a2 = __ldg(partials + (size_t)(b + 16) * 2 * Cn + c), a3 = __ldg(partials + (size_t)(b + 24) * 2 * Cn + c);
      const float q0 = __ldg(partials + (size_t)b * 2 * Cn + Cn + c), q1 = __ldg(partials + (size_t)(b + 8) * 2 * Cn + Cn + c);
      const float q2 = __ldg(partials + (size_t)(b + 16) * 2 * Cn + Cn + c), q3 = __ldg(partials + (size_t)(b + 24) * 2 * Cn + Cn + c);
      s1 += ((double)a0 + (double)a1) + ((double)a2 + (double)a3);
      s2 += ((double)q0 + (double)q1) + ((double)q2 + (double)q3);
    }
    for (; b < nblk; b += 8) {
      s1 += (double)__ldg(partials + (size_t)b * 2 * Cn + c);
      s2 += (double)__ldg(partials + (size_t)b * 2 * Cn + Cn + c);
    }
  }
  red[gq][0][cl] = s1;
  red[gq][1][cl] = s2;
  __syncthreads();
  if (gq != 0 || c >= Cn) return;
#pragma unroll
  for (int j = 1; j < 8; ++j) { s1 += red[j][0][cl]; s2 += red[j][1][cl]; }
  dbeta[c] = (float)s1;
  dgamma[c] = (float)s2;
  c1[c] = (float)(s1 / (double)rows);
  c2[c] = (float)(s2 / (double)rows);
}

// out[i] = sum_b part[b*count + i]
__global__ void gnn_reduce_kernel(const float* __restrict__ part, int nblk, int64_t count, float* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= count) return;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;   // fixed summation order, four loads in flight
  int b = 0;
  for (; b + 3 < nblk; b += 4) {
    s0 += __ldg(part + (size_t)b * count + i); s1 += __ldg(part + (size_t)(b + 1) * count + i);
    s2 += __ldg(part + (size_t)(b + 2) * count + i); s3 += __ldg(part + (size_t)(b + 3) * count + i);
  }
  for (; b < nblk; ++b) s0 += __ldg(part + (size_t)b * count + i);
  out[i] = (s0 + s1) + (s2 + s3);
}

// ====================================================================== fc1 backward
constexpr int kFbLoadWarps = 4, kFbEpiWarp0 = 4, kFbEpiWarps = 16, kFbMmaWarp = 20, kFbThreads = 21 * 32;
constexpr uint32_t kHImgB = kC * kTile * 2;        // 32 KB
constexpr uint32_t kFcWImgB = kFc * kC * 2;        // 64 KB
constexpr uint32_t kDzImg = kFc * kTile * 2;       // 64 KB: [128 rows][256 cols]

struct Fc1BwdParams {
  const __nv_bfloat16* h_in;   // h2 [M,C]
  const uint8_t* wimg;         // [256][C]
  const float* bias;           // fc1 bias [256]
  const int64_t* membership;
  const float* gs;             // [B,256]: alpha_c G[b,c] / n_b
  const float* kap;            // [256]
  const float* lam;            // [256]
  const float* mu3;            // [256]
  const float* r3;             // [256]
  const float* z_prev;         // z2 [M,C]
  const float* mu_prev;        // bn2 mean [C]
  const float* r_prev;         // bn2 invstd [C]
  __nv_bfloat16* dh_out;       // dh2 [M,C] bf16 (a GEMM-operand-like gradient: conv_bwd rounds dz to bf16 right after)
  float* stat_part;            // [grid][2][C]
  float* dw_part;              // [grid][256][C]
  float* db_part;              // [grid][256]
  int64_t M, num_tiles;
};

template <int ACT>
__global__ void __launch_bounds__(kFbThreads, 1) gnn_fc1_bwd_kernel(const Fc1BwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* Himg = smem;                                  // 2 x 32 KB
  uint8_t* Wimg = smem + 2 * kHImgB;                     // 64 KB
  uint8_t* Dimg = smem + 2 * kHImgB + kFcWImgB;          // 64 KB
  float* cst = reinterpret_cast<float*>(smem + 2 * kHImgB + kFcWImgB + kDzImg);   // bias, kap, lam, mu3, r3 [5][256]; mu2, r2 [2][128]
  float* scratch = cst + 5 * kFc + 2 * kC;                                        // [4][2][C] stats, [4][256] db
  uint64_t* bars = reinterpret_cast<uint64_t*>(scratch + 4 * 2 * kC + 4 * kFc);
  uint64_t* full = bars;           // [2]
  uint64_t* empty = bars + 2;      // [2]
  uint64_t* z_full = bars + 4;
  uint64_t* z_free = bars + 5;     // 8 warps
  uint64_t* dz_ready = bars + 6;   // 8 warps
  uint64_t* dh_full = bars + 7;
  uint64_t* dh_free = bars + 8;    // 8 warps
  uint64_t* wbar = bars + 9;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&full[i], kFbLoadWarps); mbar_init(&empty[i], 1); }
    mbar_init(z_full, 1); mbar_init(z_free, kFbEpiWarps); mbar_init(dz_ready, kFbEpiWarps); mbar_init(dh_full, 1); mbar_init(dh_free, kFbEpiWarps);
    mbar_init(wbar, 1);
    fence_mbar_init();
    mbar_arrive_expect_tx(wbar, kFcWImgB);
    for (int s = 0; s < 4; ++s) bulk_g2s(Wimg + s * (kFcWImgB / 4), p.wimg + (size_t)s * (kFcWImgB / 4), kFcWImgB / 4, wbar);
  }
  // folded constants: da3 = gs - kap - lam (a - mu3) r3 = gs - K1 - K2 a  with K2 = lam r3, K1 = kap - K2 mu3;
  //                   xhat2 = (a - mu2) r2 = a r2 + M2               with M2 = -mu2 r2        (stored: b, -K1, -K2, M2, r2)
  for (int i = threadIdx.x; i < kFc; i += kFbThreads) {
    const float k2 = __ldg(p.lam + i) * __ldg(p.r3 + i);
    cst[i] = __ldg(p.bias + i); cst[kFc + i] = k2 * __ldg(p.mu3 + i) - __ldg(p.kap + i); cst[2 * kFc + i] = -k2;
  }
  for (int i = threadIdx.x; i < kC; i += kFbThreads) {
    const float r = __ldg(p.r_prev + i);
    cst[5 * kFc + i] = -__ldg(p.mu_prev + i) * r; cst[5 * kFc + kC + i] = r;
  }
  if (warp == kFbMmaWarp) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  constexpr uint32_t T_Z = 0, T_DH = 128, T_DW = 256;
  const int64_t my_tiles = (p.num_tiles > (int64_t)blockIdx.x) ? (p.num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (warp < kFbLoadWarps) {
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1, k = it >> 1;
      if (k >= 1) mbar_wait_b(&empty[buf], (uint32_t)((k - 1) & 1));
      // same tile loader as the forward kernel (pcc_gnn.cu)
      for (int c = warp * 32 + lane; c < kTile * (kC / 8); c += kFbLoadWarps * 32) {
        const int r = c >> 4, kc = c & 15;
        const int64_t node = tile * kTile + r;
        const uint4 v = node < p.M ? __ldg(reinterpret_cast<const uint4*>(p.h_in + (size_t)node * kC) + kc) : make_uint4(0u, 0u, 0u, 0u);
        *reinterpret_cast<uint4*>(Himg + buf * kHImgB + act_chunk_off(r, kc * 8)) = v;
      }
      fence_proxy_async();
      mbar_arrive_warp(&full[buf]);
    }
  } else if (warp == kFbMmaWarp) {
    if (lane == 0) {
      constexpr uint32_t IDESC_Z = make_idesc_bf16(128, 128, 0, 0);     // z3 half: [128 rows] x [128 out]
      constexpr uint32_t IDESC_DH = make_idesc_bf16(128, kC, 0, 1);     // dh2: dZ (K-major) x W viewed [in x out]
      constexpr uint32_t IDESC_DW = make_idesc_bf16(128, kC, 1, 1);     // dW half: dZ^T x h2
      mbar_wait_b(wbar, 0);
      const uint32_t h_base = smem_u32(Himg), w_base = smem_u32(Wimg), d_base = smem_u32(Dimg);
      int it = 0;
      uint32_t use = 0;
      for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1, k = it >> 1;
        mbar_wait_b(&full[buf], (uint32_t)(k & 1));
        for (int half = 0; half < 2; ++half, ++use) {
          if (use >= 1) mbar_wait_b(z_free, (use - 1) & 1);
          tc_fence_after();
#pragma unroll
          for (int s = 0; s < kC / 64; ++s)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma_bf16(tmem + T_Z, make_smem_desc_sw128_k(h_base + buf * kHImgB + s * kActSlab + ks * 32),
                        make_smem_desc_sw128_k(w_base + s * (kFc * 128) + half * (128 * 128) + ks * 32), IDESC_Z, (s | ks) != 0);
          umma_commit(z_full);
        }
        mbar_wait_b(dz_ready, (uint32_t)(it & 1));
        if (it >= 1) mbar_wait_b(dh_free, (uint32_t)((it - 1) & 1));
        tc_fence_after();
        // dh2[rows, in] = sum_out dZ[rows, out] W[out, in]
#pragma unroll
        for (int ks = 0; ks < kFc / 16; ++ks)
          umma_bf16(tmem + T_DH, make_smem_desc_sw128_k(d_base + (ks >> 2) * kActSlab + (ks & 3) * 32),
                    make_smem_desc_sw128_mn(w_base + ks * 2048, kFc * 128), IDESC_DH, ks != 0);
        // dW[out, in] += sum_rows dZ[rows, out] h2[rows, in]   (two halves of 128 output features)
#pragma unroll
        for (int o = 0; o < 2; ++o)
#pragma unroll
          for (int ks = 0; ks < kTile / 16; ++ks)
            umma_bf16(tmem + T_DW + o * kC, make_smem_desc_sw128_mn(d_base + o * (2 * kActSlab) + ks * 2048, kActSlab),
                      make_smem_desc_sw128_mn(h_base + buf * kHImgB + ks * 2048, kActSlab), IDESC_DW, (it | ks) != 0);
        umma_commit(&empty[buf]);
        umma_commit(dh_full);
      }
    }
  } else {
    // ===================== epilogue warps 4-19: lane quarter q, 32-column group cg of every 128-column phase
    const int q = warp & 3, cg = (warp - kFbEpiWarp0) >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
    const float* b3 = cst; const float* nK1 = cst + kFc; const float* nK2 = cst + 2 * kFc;   // -K1, -K2
    const float* M2 = cst + 5 * kFc; const float* r2 = cst + 5 * kFc + kC;
    float st2[2][2], db3[2][2];
#pragma unroll
    for (int c = 0; c < 2; ++c) { st2[c][0] = st2[c][1] = 0.f; db3[0][c] = db3[1][c] = 0.f; }
    const int row = q * 32 + lane;
    uint32_t* stage = reinterpret_cast<uint32_t*>(Dimg + cg * kActSlab + q * 32 * 128);   // 4 KB: rows of this quarter, slab cg
    int it = 0;
    uint32_t use = 0;
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int64_t node = tile * kTile + row;
      const bool valid = node < p.M;
      const int64_t gph = valid ? __ldg(p.membership + node) : 0;
      const float* gsr = p.gs + gph * kFc;
#pragma unroll
      for (int half = 0; half < 2; ++half, ++use) {
        // this thread's 32 columns of the per-graph gradient term: issued before the wait for the accumulator
        float gq[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 t4 = __ldg(reinterpret_cast<const float4*>(gsr + half * 128 + cg * 32) + j);
          gq[4 * j] = t4.x; gq[4 * j + 1] = t4.y; gq[4 * j + 2] = t4.z; gq[4 * j + 3] = t4.w;
        }
        mbar_wait_b(z_full, use & 1);
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const int col0 = half * 128 + cg * 32 + c * 16;
          uint32_t v[16];
          tmem_ld16(lane_base + T_Z + cg * 32 + c * 16, v);
          tmem_wait_ld();
          float dz[16];
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            const int col = col0 + j;
            const uint64_t z = fadd2(f32x2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), *reinterpret_cast<const uint64_t*>(b3 + col));
            uint64_t a, g;
            act_and_grad2<ACT>(z, a, g);
            const uint64_t da = ffma2(*reinterpret_cast<const uint64_t*>(nK2 + col), a,
                                      fadd2(f32x2(gq[c * 16 + j], gq[c * 16 + j + 1]), *reinterpret_cast<const uint64_t*>(nK1 + col)));
            f32x2_unpack(fmul2(da, g), dz[j], dz[j + 1]);
            if (!valid) dz[j] = dz[j + 1] = 0.f;
          }
          *reinterpret_cast<uint4*>(Dimg + act_chunk_off(row, col0)) =
              make_uint4(pack_bf16x2(dz[0], dz[1]), pack_bf16x2(dz[2], dz[3]), pack_bf16x2(dz[4], dz[5]), pack_bf16x2(dz[6], dz[7]));
          *reinterpret_cast<uint4*>(Dimg + act_chunk_off(row, col0 + 8)) =
              make_uint4(pack_bf16x2(dz[8], dz[9]), pack_bf16x2(dz[10], dz[11]), pack_bf16x2(dz[12], dz[13]), pack_bf16x2(dz[14], dz[15]));
          db3[half][c] += warp_transpose_sum16(dz, lane);   // (bf16 rounding of dz not applied to the bias gradient)
        }
        tc_fence_before();
        mbar_arrive_warp(z_free);
      }
      fence_proxy_async();
      mbar_arrive_warp(dz_ready);
      // ---- dh2 of the tile: TMEM -> HBM (fp32) + the two column sums the bn2 backward needs.  The z2 values are
      //      fetched coalesced (8 lanes per row) while the dh / dW MMAs run and handed to the row's lane through the
      //      warp's staging tile; dh2 leaves the same way.  The tile lives in the dZ image, which is idle between the
      //      MMAs of this tile (dh_full) and the next tile's dz stores; the warps of a lane quarter write each other's
      //      staging bytes then, hence the quarter barrier at the end.
      const int64_t node0 = tile * kTile + q * 32;
      const int rows_valid = (int)((p.M - node0) < 32 ? (p.M - node0 < 0 ? 0 : p.M - node0) : 32);
      uint4 pre[8];
      warp_prefetch_rows32(pre, reinterpret_cast<const uint32_t*>(p.z_prev) + (size_t)node0 * kC + cg * 32, kC, rows_valid, lane);
      mbar_wait_b(dh_full, (uint32_t)(it & 1));
      tc_fence_after();
      uint32_t zp[32], out[32];
      warp_deliver_rows32(stage, pre, zp, lane);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int col0 = cg * 32 + c * 16;
        uint32_t v[16];
        tmem_ld16(lane_base + T_DH + col0, v);
        tmem_wait_ld();
        float s1[16], s2[16];
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const uint64_t dh = valid ? f32x2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])) : 0ull;
          const uint64_t a = act2<ACT>(f32x2(__uint_as_float(zp[c * 16 + j]), __uint_as_float(zp[c * 16 + j + 1])));
          const uint64_t xh = ffma2(a, *reinterpret_cast<const uint64_t*>(r2 + col0 + j), *reinterpret_cast<const uint64_t*>(M2 + col0 + j));
          f32x2_unpack(dh, s1[j], s1[j + 1]);
          f32x2_unpack(fmul2(dh, xh), s2[j], s2[j + 1]);
          out[c * 16 + j] = __float_as_uint(s1[j]);
          out[c * 16 + j + 1] = __float_as_uint(s1[j + 1]);
        }
        st2[c][0] += warp_transpose_sum16(s1, lane);
        st2[c][1] += warp_transpose_sum16(s2, lane);
      }
      {
        uint32_t w16[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) w16[j] = pack_bf16x2(__uint_as_float(out[2 * j]), __uint_as_float(out[2 * j + 1]));
        warp_store_rows16(stage, w16, reinterpret_cast<uint32_t*>(p.dh_out) + (size_t)node0 * (kC / 2) + cg * 16, kC / 2, rows_valid, lane);
      }
      asm volatile("bar.sync %0, 128;" ::"r"(3 + q) : "memory");
      tc_fence_before();
      mbar_arrive_warp(dh_free);
    }
    // ---- per-CTA partials: bn2 sums, fc1 bias gradient, fc1 weight gradient (TMEM)
    float* sstat = scratch;                 // [4 q][2][C]
    float* sdb = scratch + 4 * 2 * kC;      // [4 q][256]
    if (lane < 16) {
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        sstat[(q * 2 + 0) * kC + cg * 32 + c * 16 + lane] = st2[c][0];
        sstat[(q * 2 + 1) * kC + cg * 32 + c * 16 + lane] = st2[c][1];
        sdb[q * kFc + 0 * 128 + cg * 32 + c * 16 + lane] = db3[0][c];
        sdb[q * kFc + 1 * 128 + cg * 32 + c * 16 + lane] = db3[1][c];
      }
    }
    asm volatile("bar.sync 2, 512;" ::: "memory");
    const int t = threadIdx.x - kFbEpiWarp0 * 32;   // 0..511
    if (t < 2 * kC)
      p.stat_part[(size_t)blockIdx.x * 2 * kC + t] = sstat[(0 * 2 + t / kC) * kC + t % kC] + sstat[(1 * 2 + t / kC) * kC + t % kC] +
                                                     sstat[(2 * 2 + t / kC) * kC + t % kC] + sstat[(3 * 2 + t / kC) * kC + t % kC];
    else if (t < 2 * kC + kFc)
      p.db_part[(size_t)blockIdx.x * kFc + (t - 2 * kC)] = sdb[t - 2 * kC] + sdb[kFc + t - 2 * kC] + sdb[2 * kFc + t - 2 * kC] + sdb[3 * kFc + t - 2 * kC];
    // dW partial [256 out][C in]: TMEM lane = out feature inside its half, column = in feature
    for (int o = 0; o < 2; ++o) {
      float* dst = p.dw_part + ((size_t)blockIdx.x * kFc + o * 128 + row) * kC + cg * 32;
      if (my_tiles > 0) {
        // the last dh_full commit covered every MMA issued before it, the dW ones included
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t v[16];
          tmem_ld16(lane_base + T_DW + o * kC + cg * 32 + c * 16, v);
          tmem_wait_ld();
#pragma unroll
          for (int j = 0; j < 4; ++j)
            reinterpret_cast<float4*>(dst + c * 16)[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                                     __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        }
      } else {
        for (int j = 0; j < 32; ++j) dst[j] = 0.f;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kFbMmaWarp) tmem_dealloc<512>(tmem);
}

// ====================================================================== backward of (mean pool -> BatchNorm affine), graph-sized
// y = P * s + t with P = per-graph mean of a (graph_net.py:89-92 / :96).  From G = dL/dy [B, Cn]:
//   sumG[c] = sum_b G, sumGx[c] = sum_b G xhat(P)      -> dbeta = sumG, dgamma = sumGx,
//   gs[b, c] = G * f / n_b,  kap[c] = f * sumG / M,  lam[c] = f * sumGx / M      (f = s[c], or 1 when use_scale = 0)
// are everything the node-level backward kernels need (da = gs[graph] - kap - lam xhat).  One CTA per 32 columns (32 row
// slices per column, reduced through shared memory in a fixed order).  An empty graph's y is the constant 0 (no node feeds
// it): gs = 0 and it adds nothing to sumG / sumGx.
__global__ void __launch_bounds__(1024) gnn_pool_bwd_prep_kernel(const float* __restrict__ G, const float* __restrict__ P,
                                                                const float* __restrict__ mu, const float* __restrict__ rinv,
                                                                const float* __restrict__ s, const int64_t* __restrict__ counts,
                                                                int64_t B, int Cn, int64_t M, int use_scale, float* __restrict__ gs,
                                                                float* __restrict__ kap, float* __restrict__ lam,
                                                                float* __restrict__ dgamma, float* __restrict__ dbeta) {
  __shared__ float red[2][32][33];
  const int cl = threadIdx.x & 31, sl = threadIdx.x >> 5;   // column of the block's 32, row slice of 32
  const int c = blockIdx.x * 32 + cl;
  float a0 = 0.f, a1 = 0.f;
  if (c < Cn) {
    const float f = use_scale ? s[c] : 1.f, m = mu[c], r = rinv[c];
    for (int64_t b = sl; b < B; b += 32) {
      // the loads of n, G and P issue together (a select, no branch on n): the kernel is latency-bound
      const int64_t n = counts[b];
      const float graw = G[b * Cn + c];
      const float g = n > 0 ? graw : 0.f;
      gs[b * Cn + c] = g * f / (float)(n > 0 ? n : 1);
      a0 += g;
      a1 += g * ((P[b * Cn + c] - m) * r);
    }
  }
  red[0][sl][cl] = a0;
  red[1][sl][cl] = a1;
  __syncthreads();
  if (sl == 0 && c < Cn) {
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) { t0 += red[0][k][cl]; t1 += red[1][k][cl]; }
    const float f = use_scale ? s[c] : 1.f;
    dbeta[c] = t0;
    dgamma[c] = t1;
    kap[c] = f * t0 / (float)M;
    lam[c] = f * t1 / (float)M;
  }
}

// ====================================================================== conv2 backward
// 8 prologue warps (16 rows of every tile each, register-pipelined loads) + 4 epilogue warps (the first one also issues
// the MMAs): 384 threads, so that a prologue thread can hold two batches of 4 rows (96 registers of operands) in flight
constexpr int kCbLoadWarps = 8, kCbMmaWarp = 8, kCbThreads = 12 * 32;
constexpr int kCbBatch = 4, kCbBatches = kTile / kCbLoadWarps / kCbBatch;   // 4 batches of 4 rows per warp and tile
constexpr uint32_t kDz2Img = kC * kTile * 2;          // 32 KB: [128 rows][C cols]
constexpr uint32_t kAinImg = 2 * kC * kTile * 2;      // 64 KB: [128 rows][2C cols]
constexpr uint32_t kCwImg = 2 * kC * kC * 2;          // 64 KB

struct ConvBwdParams {
  const int64_t* membership;   // with dh_graph: graph of every node
  const float* dh_graph;       // optional [B,C] fp32: dL/dh is the same row for every node of a graph (global_mean_pool follows
                               // the block).  Kept in fp32: a rounding error shared by all nodes of a graph does not average out.
  const __nv_bfloat16* dh;     // dL/dh of this block's output [M,C] bf16
  const float* z;              // pre-activation of this block [M,C]
  BnBack bn;                   // [C] arrays
  const __nv_bfloat16* agg;    // [M,C] kept aggregate (A operand, left half)
  const __nv_bfloat16* h_in;   // [M,C] block input (A operand, right half)
  const uint8_t* wimg;         // [C][2C] image
  __nv_bfloat16* dagg_out;     // [M,C] bf16
  __nv_bfloat16* droot_out;    // [M,C] bf16
  float* dw_part;              // [grid][C][2C]
  float* db_part;              // [grid][C]
  int64_t M, num_tiles;
};

template <int ACT>
__global__ void __launch_bounds__(kCbThreads, 1) gnn_conv_bwd_kernel(const ConvBwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* Dimg = smem;                            // 32 KB
  uint8_t* Aimg = smem + kDz2Img;                  // 64 KB
  uint8_t* Wimg = smem + kDz2Img + kAinImg;        // 64 KB
  float* cst = reinterpret_cast<float*>(smem + kDz2Img + kAinImg + kCwImg);   // [5][C]
  float* scratch = cst + 5 * kC;                                              // [kCbLoadWarps][C] db
  uint64_t* bars = reinterpret_cast<uint64_t*>(scratch + kCbLoadWarps * kC);
  uint64_t* full = bars;        // prologue warps
  uint64_t* empty = bars + 1;   // MMA commit
  uint64_t* dx_full = bars + 2;
  uint64_t* dx_free = bars + 3; // 4 warps
  uint64_t* wbar = bars + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
  uint32_t* stage_all = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(bars) + 128);   // [4 warps] 4 KB staging tiles
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(full, kCbLoadWarps); mbar_init(empty, 1); mbar_init(dx_full, 1); mbar_init(dx_free, 4); mbar_init(wbar, 1);
    fence_mbar_init();
    mbar_arrive_expect_tx(wbar, kCwImg);
    for (int s = 0; s < 4; ++s) bulk_g2s(Wimg + s * (kCwImg / 4), p.wimg + (size_t)s * (kCwImg / 4), kCwImg / 4, wbar);
  }
  for (int i = threadIdx.x; i < kC; i += kCbThreads) {
    cst[i] = __ldg(p.bn.mean + i); cst[kC + i] = __ldg(p.bn.invstd + i); cst[2 * kC + i] = __ldg(p.bn.scale + i);
    cst[3 * kC + i] = __ldg(p.bn.c1 + i); cst[4 * kC + i] = __ldg(p.bn.c2 + i);
  }
  if (warp == kCbMmaWarp) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  constexpr uint32_t T_DX = 0, T_DW = 256;
  const int64_t my_tiles = (p.num_tiles > (int64_t)blockIdx.x) ? (p.num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (warp < kCbLoadWarps) {
    // ===================== prologue warps: dz = s (dh - c1 - xhat c2) act'(z) -> bf16 image; [agg | h_in] image
    const int col = 4 * lane;
    const float4 mu = *reinterpret_cast<const float4*>(cst + col), rs = *reinterpret_cast<const float4*>(cst + kC + col);
    const float4 sc = *reinterpret_cast<const float4*>(cst + 2 * kC + col), c1 = *reinterpret_cast<const float4*>(cst + 3 * kC + col);
    const float4 c2 = *reinterpret_cast<const float4*>(cst + 4 * kC + col);
    float db[4] = {0.f, 0.f, 0.f, 0.f};
    // The loop is bound by load latency, not by bytes or instructions (ncu of the first version: 13 % issue utilisation,
    // half of the samples on the first use of a loaded value, and no load in flight while the warps waited for the MMAs to
    // release the images).  So the operands of a batch of 4 rows are loaded into registers one batch AHEAD of their use,
    // across the wait for the images: batch 0 of the next tile is in flight while this tile's MMAs run.
    struct Rows { float4 z[kCbBatch]; uint2 g[kCbBatch], ag[kCbBatch], hr[kCbBatch]; };
    auto load_batch = [&](int64_t tile, int b, Rows& R) {
#pragma unroll
      for (int j = 0; j < kCbBatch; ++j) {
        const int r = warp + kCbLoadWarps * (b * kCbBatch + j);
        const int64_t node = tile * kTile + r;
        R.z[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        R.g[j] = R.ag[j] = R.hr[j] = make_uint2(0u, 0u);
        if (node < p.M) {
          if (p.dh_graph) R.g[j].x = (uint32_t)__ldg(p.membership + node);   // the row itself is read at use (L1-resident table)
          else R.g[j] = __ldg(reinterpret_cast<const uint2*>(p.dh + (size_t)node * kC) + lane);
          R.z[j] = __ldg(reinterpret_cast<const float4*>(p.z + (size_t)node * kC) + lane);
          R.ag[j] = __ldg(reinterpret_cast<const uint2*>(p.agg + (size_t)node * kC) + lane);
          R.hr[j] = __ldg(reinterpret_cast<const uint2*>(p.h_in + (size_t)node * kC) + lane);
        }
      }
    };
    auto process_batch = [&](int64_t tile, int b, const Rows& R) {
#pragma unroll
      for (int j = 0; j < kCbBatch; ++j) {
        const int r = warp + kCbLoadWarps * (b * kCbBatch + j);
        const int64_t node = tile * kTile + r;
        float dz[4] = {0.f, 0.f, 0.f, 0.f};
        if (node < p.M) {
          const float4 z = R.z[j];
          const float4 g = p.dh_graph ? __ldg(reinterpret_cast<const float4*>(p.dh_graph + (size_t)R.g[j].x * kC) + lane)
                                      : make_float4(bf16_lo(R.g[j].x), bf16_hi(R.g[j].x), bf16_lo(R.g[j].y), bf16_hi(R.g[j].y));
          float a;
          a = actf<ACT>(z.x); dz[0] = sc.x * (g.x - c1.x - (a - mu.x) * rs.x * c2.x) * actg<ACT>(z.x, a);
          a = actf<ACT>(z.y); dz[1] = sc.y * (g.y - c1.y - (a - mu.y) * rs.y * c2.y) * actg<ACT>(z.y, a);
          a = actf<ACT>(z.z); dz[2] = sc.z * (g.z - c1.z - (a - mu.z) * rs.z * c2.z) * actg<ACT>(z.z, a);
          a = actf<ACT>(z.w); dz[3] = sc.w * (g.w - c1.w - (a - mu.w) * rs.w * c2.w) * actg<ACT>(z.w, a);
        }
        db[0] += dz[0]; db[1] += dz[1]; db[2] += dz[2]; db[3] += dz[3];
        *reinterpret_cast<uint2*>(Dimg + act_chunk_off(r, col) + ((col & 7) << 1)) =
            make_uint2(pack_bf16x2(dz[0], dz[1]), pack_bf16x2(dz[2], dz[3]));
        *reinterpret_cast<uint2*>(Aimg + act_chunk_off(r, col) + ((col & 7) << 1)) = R.ag[j];
        *reinterpret_cast<uint2*>(Aimg + act_chunk_off(r, kC + col) + ((col & 7) << 1)) = R.hr[j];
      }
    };
    static_assert(kCbBatches == 4, "the pipeline below is written for 4 batches per tile");
    Rows RA, RB;
    if ((int64_t)blockIdx.x < p.num_tiles) load_batch(blockIdx.x, 0, RA);
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      if (it >= 1) mbar_wait_b(empty, (uint32_t)((it - 1) & 1));
      load_batch(tile, 1, RB); process_batch(tile, 0, RA);
      load_batch(tile, 2, RA); process_batch(tile, 1, RB);
      load_batch(tile, 3, RB); process_batch(tile, 2, RA);
      if (tile + gridDim.x < p.num_tiles) load_batch(tile + gridDim.x, 0, RA);
      process_batch(tile, 3, RB);
      fence_proxy_async();
      mbar_arrive_warp(full);
    }
    *reinterpret_cast<float4*>(scratch + warp * kC + col) = make_float4(db[0], db[1], db[2], db[3]);
    asm volatile("bar.sync 3, %0;" ::"n"(kCbLoadWarps * 32) : "memory");
    for (int i = threadIdx.x; i < kC; i += kCbLoadWarps * 32) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kCbLoadWarps; ++w) s += scratch[w * kC + i];
      p.db_part[(size_t)blockIdx.x * kC + i] = s;
    }
  } else {
    // ===================== epilogue warps 8-11: dX accumulator -> dagg (bf16) | droot (bf16)
    const int q = warp & 3;
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
    const int row = q * 32 + lane;
    uint32_t* stage = stage_all + q * kStageWords;
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int64_t node0 = tile * kTile + q * 32;
      const int rows_valid = (int)((p.M - node0) < 32 ? (p.M - node0 < 0 ? 0 : p.M - node0) : 32);
      if (warp == kCbMmaWarp) {
        // The dX accumulator is single-buffered, so the MMAs of a tile can only start after the epilogue of the previous
        // one: the first epilogue warp issues them itself (a dedicated issuer warp would only push the CTA over 12 warps
        // and the prologue threads under the registers their load pipeline needs).
        if (lane == 0) {
          constexpr uint32_t IDESC_DX = make_idesc_bf16(128, 2 * kC, 0, 1);   // [128 rows] x [2C in]: dZ (K-major) x W viewed [in x out]
          constexpr uint32_t IDESC_DW = make_idesc_bf16(128, 2 * kC, 1, 1);   // [C out] x [2C in]: dZ^T x [agg | h]
          const uint32_t d_base = smem_u32(Dimg), a_base = smem_u32(Aimg), w_base = smem_u32(Wimg);
          if (it == 0) mbar_wait_b(wbar, 0);
          mbar_wait_b(full, (uint32_t)(it & 1));
          if (it >= 1) mbar_wait_b(dx_free, (uint32_t)((it - 1) & 1));
          tc_fence_after();
#pragma unroll
          for (int ks = 0; ks < kC / 16; ++ks)
            umma_bf16(tmem + T_DX, make_smem_desc_sw128_k(d_base + (ks >> 2) * kActSlab + (ks & 3) * 32),
                      make_smem_desc_sw128_mn(w_base + ks * 2048, kC * 128), IDESC_DX, ks != 0);
#pragma unroll
          for (int ks = 0; ks < kTile / 16; ++ks)
            umma_bf16(tmem + T_DW, make_smem_desc_sw128_mn(d_base + ks * 2048, kActSlab),
                      make_smem_desc_sw128_mn(a_base + ks * 2048, kActSlab), IDESC_DW, (it | ks) != 0);
          umma_commit(empty);
          umma_commit(dx_full);
        }
        __syncwarp();
      }
      mbar_wait_b(dx_full, (uint32_t)(it & 1));
      tc_fence_after();
      // [dagg | droot]: 64 columns (two TMEM chunks) -> 32 packed bf16 words per row, stored through the warp's staging
      // tile so that an instruction writes whole 128-byte row segments.
#pragma unroll
      for (int c = 0; c < 2 * kC / 64; ++c) {
        uint32_t v[32], w[32];
        tmem_ld32(lane_base + T_DX + c * 64, v);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) w[j] = pack_bf16x2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
        tmem_ld32(lane_base + T_DX + c * 64 + 32, v);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) w[16 + j] = pack_bf16x2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
        __nv_bfloat16* dst = (c < kC / 64) ? p.dagg_out : p.droot_out;
        warp_store_rows32(stage, w, reinterpret_cast<uint32_t*>(dst) + (size_t)node0 * (kC / 2) + (c & 1) * 32, kC / 2, rows_valid, lane);
      }
      tc_fence_before();
      mbar_arrive_warp(dx_free);
    }
    // dW partial [C out][2C]: lane = out feature
    float* dst = p.dw_part + ((size_t)blockIdx.x * kC + row) * (2 * kC);
    if (my_tiles > 0) {
#pragma unroll 1
      for (int c = 0; c < 2 * kC / 32; ++c) {
        uint32_t v[32];
        tmem_ld32(lane_base + T_DW + c * 32, v);
        tmem_wait_ld();
        warp_store_rows32(stage, v, reinterpret_cast<uint32_t*>(dst - (size_t)lane * (2 * kC)) + c * 32, 2 * kC, 32, lane);
      }
    } else {
      for (int j = 0; j < 2 * kC; ++j) dst[j] = 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kCbMmaWarp) tmem_dealloc<512>(tmem);
}

// ====================================================================== aggregation backward (+ sums for the bn backward)
// dh[j] = droot[j] + sum_{e: src(e) = j} w_e dagg[dst(e)]   (CSR by source; for mean aggregation w already carries
// 1/deg(dst)); warp per node, lane = 4 channels; writes dh IN PLACE over droot.  Also accumulates sum dh and
// sum dh xhat of the PREVIOUS block (z_prev, its mean / invstd) per block.
// The neighbour rows (256 B of bf16) are fetched by the TMA engine into a per-warp shared-memory slot (one
// cp.async.bulk per row, all of a node's rows in flight at once, no registers tied up), like the forward gather.
constexpr int kAggSlotRows = 22;
constexpr uint32_t kAggRowB = kC * 2, kAggSlotB = kAggSlotRows * kAggRowB;
template <int ACT>
__global__ void __launch_bounds__(256, 3) gnn_agg_bwd_kernel(const __nv_bfloat16* __restrict__ dagg, GnnGraph g, __nv_bfloat16* __restrict__ dh,
                                                          const float* __restrict__ z_prev, const float* __restrict__ mu_prev,
                                                          const float* __restrict__ r_prev, int64_t M, float* __restrict__ partials) {
  extern __shared__ __align__(128) uint8_t smem_agg[];
  uint8_t* slots = smem_agg;                                                // [8 warps][22 rows][256 B]
  float* red = reinterpret_cast<float*>(smem_agg + 8 * kAggSlotB);          // [8][2][C]
  uint64_t* gbar = reinterpret_cast<uint64_t*>(red + 8 * 2 * kC);           // [8]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < 8) mbar_init(&gbar[threadIdx.x], 1);
  fence_mbar_init();
  __syncthreads();
  const uint8_t* src = reinterpret_cast<const uint8_t*>(dagg);
  uint8_t* slot = slots + warp * kAggSlotB;
  uint64_t* bar = &gbar[warp];
  uint32_t gphase = 0;
  const float4 mu = __ldg(reinterpret_cast<const float4*>(mu_prev) + lane), rs = __ldg(reinterpret_cast<const float4*>(r_prev) + lane);
  float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
  const int64_t nwarps = (int64_t)gridDim.x * 8;
  int64_t node = (int64_t)blockIdx.x * 8 + warp;
  // Software pipeline over the warp's nodes (the loop is a chain of dependent global loads otherwise — row pointers ->
  // neighbour ids -> rows, and the node's own dh / z rows; ncu showed ~20 % of the samples on their first uses): the row
  // pointers are loaded TWO nodes ahead, the node's dh / z rows and the neighbour ids ONE node ahead.
  int pb = 0, pe = 0, nb = 0, ne = 0;     // [pb, pe): this node's CSR slots, [nb, ne): the next node's  (E < 2^31)
  if (node < M) { pb = (int)__ldg(g.rowptr + node); pe = (int)__ldg(g.rowptr + node + 1); }
  if (node + nwarps < M) { nb = (int)__ldg(g.rowptr + node + nwarps); ne = (int)__ldg(g.rowptr + node + nwarps + 1); }
  int cnt = (pe - pb < kAggSlotRows) ? pe - pb : kAggSlotRows;
  int myc = lane < cnt ? __ldg(g.col + pb + lane) : 0;
  float myw = (g.w && lane < cnt) ? __ldg(g.w + pb + lane) : 1.f;
  uint2 dh_next = make_uint2(0u, 0u);
  float4 z_next = make_float4(0.f, 0.f, 0.f, 0.f);
  if (node < M) {
    dh_next = *(reinterpret_cast<const uint2*>(dh + (size_t)node * kC) + lane);
    z_next = __ldg(reinterpret_cast<const float4*>(z_prev + (size_t)node * kC) + lane);
  }
  for (; node < M; node += nwarps) {
    const uint2 acc0 = dh_next;
    const float4 z = z_next;
    int n2b = 0, n2e = 0;
    if (node + nwarps < M) {
      // (every node is read and written by exactly one warp, once: the early read of the next node's dh is safe)
      dh_next = *(reinterpret_cast<const uint2*>(dh + (size_t)(node + nwarps) * kC) + lane);
      z_next = __ldg(reinterpret_cast<const float4*>(z_prev + (size_t)(node + nwarps) * kC) + lane);
      if (node + 2 * nwarps < M) { n2b = (int)__ldg(g.rowptr + node + 2 * nwarps); n2e = (int)__ldg(g.rowptr + node + 2 * nwarps + 1); }
    }
    float acc[4];
    bool first = true;
    const int deg = pe - pb;
    int done = 0;
    for (;;) {
      if (cnt > 0) {
        if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)cnt * kAggRowB);
        __syncwarp();
        if (lane < cnt) bulk_g2s(slot + lane * kAggRowB, src + (size_t)myc * kAggRowB, kAggRowB, bar);
      }
      const int ccnt = cnt;
      const float cw = myw;
      done += cnt;
      const bool next_node = done >= deg;
      const int npb = next_node ? nb : pb + done, npe = next_node ? ne : pe;
      cnt = (npe - npb < kAggSlotRows) ? npe - npb : kAggSlotRows;
      myc = lane < cnt ? __ldg(g.col + npb + lane) : 0;
      myw = (g.w && lane < cnt) ? __ldg(g.w + npb + lane) : 1.f;
      if (first) {
        acc[0] = bf16_lo(acc0.x); acc[1] = bf16_hi(acc0.x); acc[2] = bf16_lo(acc0.y); acc[3] = bf16_hi(acc0.y);
        first = false;
      }
      if (ccnt > 0) {
        mbar_wait_b(bar, gphase);
        gphase ^= 1;
        slot_reduce<(int)kAggRowB>(slot, ccnt, lane, g.w != nullptr, cw, acc);
        __syncwarp();
      }
      if (next_node) { pb = nb; pe = ne; nb = n2b; ne = n2e; break; }
    }
    *(reinterpret_cast<uint2*>(dh + (size_t)node * kC) + lane) = make_uint2(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]));
    s1[0] += acc[0]; s1[1] += acc[1]; s1[2] += acc[2]; s1[3] += acc[3];
    s2[0] += acc[0] * (actf<ACT>(z.x) - mu.x) * rs.x; s2[1] += acc[1] * (actf<ACT>(z.y) - mu.y) * rs.y;
    s2[2] += acc[2] * (actf<ACT>(z.z) - mu.z) * rs.z; s2[3] += acc[3] * (actf<ACT>(z.w) - mu.w) * rs.w;
  }
  *reinterpret_cast<float4*>(&red[(warp * 2 + 0) * kC + 4 * lane]) = make_float4(s1[0], s1[1], s1[2], s1[3]);
  *reinterpret_cast<float4*>(&red[(warp * 2 + 1) * kC + 4 * lane]) = make_float4(s2[0], s2[1], s2[2], s2[3]);
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * kC; i += 256) {
    float s = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) s += red[(w8 * 2 + i / kC) * kC + i % kC];
    partials[(size_t)blockIdx.x * 2 * kC + i] = s;
  }
}

// ====================================================================== conv1 backward (K = 2F): CUDA cores
// dz1 = s (dh - c1 - xhat c2) act'(z1);  dW_rel1[c,f] += dz1[c] agg1[f],  dW_root1[c,f] += dz1[c] x[f],  db1[c] += dz1[c]
// per-block partial [C][2F+1] (rel | root | bias).
template <int ACT, int FP>
__global__ void __launch_bounds__(256) gnn_conv1_bwd_kernel(const __nv_bfloat16* __restrict__ dh, const float* __restrict__ z, BnBack bn,
                                                            const float* __restrict__ agg, const float* __restrict__ x, int F,
                                                            int64_t M, float* __restrict__ partials) {
  extern __shared__ float red1[];   // [8][C][2 FP + 1]
  constexpr int NA = 2 * FP + 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float4 mu = __ldg(reinterpret_cast<const float4*>(bn.mean) + lane), rs = __ldg(reinterpret_cast<const float4*>(bn.invstd) + lane);
  const float4 sc = __ldg(reinterpret_cast<const float4*>(bn.scale) + lane), c1 = __ldg(reinterpret_cast<const float4*>(bn.c1) + lane);
  const float4 c2 = __ldg(reinterpret_cast<const float4*>(bn.c2) + lane);
  float acc[4][NA];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int f = 0; f < NA; ++f) acc[j][f] = 0.f;
  const int64_t nwarps = (int64_t)gridDim.x * 8;
  // two nodes per iteration: their row loads are independent (the loop is bound by load latency otherwise)
  for (int64_t node0 = (int64_t)blockIdx.x * 8 + warp; node0 < M; node0 += 2 * nwarps) {
    float4 g[2], zz[2];
    uint2 gb[2];
    float in[2][2 * FP];
    bool ok[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int64_t node = node0 + h * nwarps;
      ok[h] = node < M;
      zz[h] = make_float4(0.f, 0.f, 0.f, 0.f);
      gb[h] = make_uint2(0u, 0u);
#pragma unroll
      for (int f = 0; f < 2 * FP; ++f) in[h][f] = 0.f;
      if (ok[h]) {
        gb[h] = __ldg(reinterpret_cast<const uint2*>(dh + (size_t)node * kC) + lane);
        zz[h] = __ldg(reinterpret_cast<const float4*>(z + (size_t)node * kC) + lane);
#pragma unroll
        for (int f = 0; f < FP; ++f)
          if (f < F) { in[h][f] = __ldg(agg + node * F + f); in[h][FP + f] = __ldg(x + node * F + f); }
      }
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (!ok[h]) continue;
      g[h] = make_float4(bf16_lo(gb[h].x), bf16_hi(gb[h].x), bf16_lo(gb[h].y), bf16_hi(gb[h].y));
      float dz[4], a;
      a = actf<ACT>(zz[h].x); dz[0] = sc.x * (g[h].x - c1.x - (a - mu.x) * rs.x * c2.x) * actg<ACT>(zz[h].x, a);
      a = actf<ACT>(zz[h].y); dz[1] = sc.y * (g[h].y - c1.y - (a - mu.y) * rs.y * c2.y) * actg<ACT>(zz[h].y, a);
      a = actf<ACT>(zz[h].z); dz[2] = sc.z * (g[h].z - c1.z - (a - mu.z) * rs.z * c2.z) * actg<ACT>(zz[h].z, a);
      a = actf<ACT>(zz[h].w); dz[3] = sc.w * (g[h].w - c1.w - (a - mu.w) * rs.w * c2.w) * actg<ACT>(zz[h].w, a);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int f = 0; f < 2 * FP; ++f) acc[j][f] = fmaf(dz[j], in[h][f], acc[j][f]);
        acc[j][2 * FP] += dz[j];
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int f = 0; f < NA; ++f) red1[(warp * kC + 4 * lane + j) * NA + f] = acc[j][f];
  __syncthreads();
  const int W = 2 * F + 1;
  for (int i = threadIdx.x; i < kC * W; i += 256) {
    const int c = i / W, f = i % W;
    const int slot = f < F ? f : (f < 2 * F ? FP + (f - F) : 2 * FP);
    float s = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) s += red1[(w8 * kC + c) * NA + slot];
    partials[(size_t)blockIdx.x * kC * W + i] = s;
  }
}

int gnn_grid(int64_t num_tiles);

}  // namespace gnn
}  // namespace pcc

using namespace pcc;
using namespace pcc::gnn;

#define GNN_ACT_DISPATCH(act, ...)                        \
  switch (act) {                                           \
    case PCC_ACT_RELU: { constexpr int A = PCC_ACT_RELU; __VA_ARGS__; break; } \
    case PCC_ACT_GELU: { constexpr int A = PCC_ACT_GELU; __VA_ARGS__; break; } \
    case PCC_ACT_TANH: { constexpr int A = PCC_ACT_TANH; __VA_ARGS__; break; } \
    default: return fail(__func__, "activation must be tanh / relu / gelu (graph_net.py:38-43)"); \
  }

extern "C" int pcc_gnn_bn_bwd_finalize(const float* partials, int nblk, int Cn, int64_t rows, float* c1, float* c2,
                                       float* dgamma, float* dbeta, int device, void* stream) {
  PCC_ENTER(device);
  PCC_K(gnn_bn_bwd_finalize_kernel)<<<cdiv(Cn, 32), 256, 0, (cudaStream_t)stream>>>(partials, nblk, Cn, rows, c1, c2, dgamma, dbeta);
  return check_launch(__func__);
}

extern "C" int pcc_gnn_reduce(const float* part, int nblk, int64_t count, float* out, int device, void* stream) {
  PCC_ENTER(device);
  if (count == 0) return 0;
  PCC_K(gnn_reduce_kernel)<<<(unsigned)cdiv(count, 256), 256, 0, (cudaStream_t)stream>>>(part, nblk, count, out);
  return check_launch(__func__);
}

extern "C" int pcc_gnn_fc1_bwd(const void* h_in_bf16, const void* packed, const float* bias, const int64_t* membership,
                               const float* gs, const float* kap, const float* lam, const float* mu3, const float* r3,
                               const float* z_prev, const float* mu_prev, const float* r_prev, int64_t M, int act,
                               void* dh_out_bf16, float* stat_part, float* dw_part, float* db_part, int* nblk_out, int device,
                               void* stream) {
  PCC_ENTER(device);
  Fc1BwdParams p{};
  p.h_in = (const __nv_bfloat16*)h_in_bf16;
  p.wimg = (const uint8_t*)packed + 2 * kC * kC * 2;
  p.bias = bias; p.membership = membership; p.gs = gs; p.kap = kap; p.lam = lam; p.mu3 = mu3; p.r3 = r3;
  p.z_prev = z_prev; p.mu_prev = mu_prev; p.r_prev = r_prev;
  p.dh_out = (__nv_bfloat16*)dh_out_bf16; p.stat_part = stat_part; p.dw_part = dw_part; p.db_part = db_part;
  p.M = M; p.num_tiles = cdiv(M, kTile);
  const int grid = gnn_grid(p.num_tiles);
  *nblk_out = grid;
  if (grid == 0) return 0;
  const int smem_bytes = 2 * kHImgB + kFcWImgB + kDzImg + (5 * kFc + 2 * kC + 8 * kC + 4 * kFc) * 4 + 128;
  {
    ProfScope prof(7, (cudaStream_t)stream);
    GNN_ACT_DISPATCH(act, {
      auto kern = gnn_fc1_bwd_kernel<A>;
      PCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
      PCC_K(kern)<<<grid, kFbThreads, smem_bytes, (cudaStream_t)stream>>>(p);
    });
  }
  return check_launch(__func__);
}

extern "C" int pcc_gnn_pool_bwd_prep(const float* G, const float* P, const float* mu, const float* rinv, const float* s,
                                     const int64_t* counts, int64_t B, int Cn, int64_t M, int use_scale, float* gs, float* kap,
                                     float* lam, float* dgamma, float* dbeta, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(Cn > 0 && M > 0, "empty problem");
  PCC_K(gnn_pool_bwd_prep_kernel)<<<(unsigned)cdiv(Cn, 32), 1024, 0, (cudaStream_t)stream>>>(G, P, mu, rinv, s, counts, B, Cn, M, use_scale,
                                                                                        gs, kap, lam, dgamma, dbeta);
  return check_launch(__func__);
}

extern "C" int pcc_gnn_conv_bwd(const void* dh_bf16, const int64_t* membership, const float* dh_graph, const float* z, const float* bn_mean, const float* bn_invstd,
                                const float* bn_scale, const float* bn_c1, const float* bn_c2, const void* agg_bf16,
                                const void* h_in_bf16, const void* packed, int64_t M, int act, void* dagg_out_bf16,
                                void* droot_out_bf16, float* dw_part, float* db_part, int* nblk_out, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE((dh_bf16 != nullptr) != (dh_graph != nullptr), "exactly one of dh / dh_graph");
  PCC_REQUIRE(dh_graph == nullptr || membership != nullptr, "dh_graph needs the membership vector");
  ConvBwdParams p{};
  p.dh = (const __nv_bfloat16*)dh_bf16; p.z = z; p.membership = membership; p.dh_graph = dh_graph;
  p.bn = BnBack{bn_mean, bn_invstd, bn_scale, bn_c1, bn_c2};
  p.agg = (const __nv_bfloat16*)agg_bf16; p.h_in = (const __nv_bfloat16*)h_in_bf16;
  p.wimg = (const uint8_t*)packed;
  p.dagg_out = (__nv_bfloat16*)dagg_out_bf16; p.droot_out = (__nv_bfloat16*)droot_out_bf16; p.dw_part = dw_part; p.db_part = db_part;
  p.M = M; p.num_tiles = cdiv(M, kTile);
  const int grid = gnn_grid(p.num_tiles);
  *nblk_out = grid;
  if (grid == 0) return 0;
  const int smem_bytes = kDz2Img + kAinImg + kCwImg + (5 * kC + kCbLoadWarps * kC) * 4 + 128 + 4 * kStageWords * 4;
  {
    ProfScope prof(4, (cudaStream_t)stream);
    GNN_ACT_DISPATCH(act, {
      auto kern = gnn_conv_bwd_kernel<A>;
      PCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
      PCC_K(kern)<<<grid, kCbThreads, smem_bytes, (cudaStream_t)stream>>>(p);
    });
  }
  return check_launch(__func__);
}

extern "C" int pcc_gnn_agg_bwd(const void* dagg_bf16, const int64_t* rowptr_src, const int32_t* col_src, const float* w_src,
                               void* dh_inout_bf16, const float* z_prev, const float* mu_prev, const float* r_prev, int64_t M,
                               int act, float* partials, int* nblk_out, int device, void* stream) {
  PCC_ENTER(device);
  int blocks = 1;
  GnnGraph g{rowptr_src, col_src, w_src, 0};
  {
    ProfScope prof(5, (cudaStream_t)stream);
    const int smem_bytes = 8 * kAggSlotB + 8 * 2 * kC * 4 + 64;
    GNN_ACT_DISPATCH(act, {
      auto kern = gnn_agg_bwd_kernel<A>;
      PCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
      blocks = gnn_resident_blocks((const void*)kern, 256, smem_bytes, cdiv(M, 8));
      *nblk_out = blocks;
      PCC_K(kern)<<<blocks, 256, smem_bytes, (cudaStream_t)stream>>>((const __nv_bfloat16*)dagg_bf16, g, (__nv_bfloat16*)dh_inout_bf16, z_prev, mu_prev,
                                                                     r_prev, M, partials);
    });
  }
  return check_launch(__func__);
}

extern "C" int pcc_gnn_conv1_bwd(const void* dh_bf16, const float* z, const float* bn_mean, const float* bn_invstd,
                                 const float* bn_scale, const float* bn_c1, const float* bn_c2, const float* agg, const float* x,
                                 int F, int64_t M, int act, float* partials, int* nblk_out, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(F >= 1 && F <= 8, "fused conv1 needs input_dim <= 8");
  int blocks = 1;
  BnBack bn{bn_mean, bn_invstd, bn_scale, bn_c1, bn_c2};
  const int smem_bytes = 8 * kC * (F <= 4 ? 9 : 17) * 4;
  GNN_ACT_DISPATCH(act, {
    auto kern = F <= 4 ? gnn_conv1_bwd_kernel<A, 4> : gnn_conv1_bwd_kernel<A, 8>;
    PCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    blocks = gnn_resident_blocks((const void*)kern, 256, smem_bytes, cdiv(M, 8 * 16) < 592 ? cdiv(M, 8 * 16) : 592);   // (caller: 592 partials)
    *nblk_out = blocks;
    PCC_K(kern)<<<blocks, 256, smem_bytes, (cudaStream_t)stream>>>((const __nv_bfloat16*)dh_bf16, z, bn, agg, x, F, M, partials);
  });
  return check_launch(__func__);
}
