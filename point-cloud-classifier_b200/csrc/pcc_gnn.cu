// Fused bf16 GraphNet path, forward kernels + the CUDA-core pieces shared with the backward (see pcc_gnn.cuh).
//   reference: /root/reference/models/graph_net.py:73-92 (conv1/act/bn1, conv2/act/bn2, fc1/act/bn3, global_mean_pool);
//   GraphConv semantics: out_i = lin_rel(sum_{e: dst(e)=i} w_e x[src(e)]) + lin_root(x_i)   (PyG, restated in
//   oracle/graphnet_oracle.py).
#include "pcc_gnn.cuh"

namespace pcc {
namespace gnn {

// ------------------------------------------------------------------ weight images
// conv image: [C rows = out feature][2C cols = (lin_rel in | lin_root in)] bf16, SWIZZLE_128B slabs of C rows x 64 cols
// fc1 image : [256 rows = out feature][C cols = in feature]
__global__ void gnn_pack_kernel(const float* __restrict__ w_rel, const float* __restrict__ w_root, const float* __restrict__ w_fc1,
                                uint8_t* __restrict__ conv_img, uint8_t* __restrict__ fc1_img) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // one thread per 16-byte chunk (8 elements)
  const int conv_chunks = kC * (2 * kC / 8), fc_chunks = kFc * (kC / 8);
  if (i < conv_chunks) {
    const int row = i % kC, kc = i / kC;                 // kc = 8-column chunk index inside the 2C columns
    const float* src = (kc * 8 < kC) ? (w_rel + (size_t)row * kC + kc * 8) : (w_root + (size_t)row * kC + (kc * 8 - kC));
    uint32_t q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = pack_bf16x2(__ldg(src + 2 * j), __ldg(src + 2 * j + 1));
    const uint32_t off = (uint32_t)(kc >> 3) * (kC * 128u) + (uint32_t)row * 128u + ((uint32_t)((kc & 7) ^ (row & 7)) << 4);
    *reinterpret_cast<uint4*>(conv_img + off) = make_uint4(q[0], q[1], q[2], q[3]);
  } else if (w_fc1 && i < conv_chunks + fc_chunks) {
    const int t = i - conv_chunks;
    const int row = t % kFc, kc = t / kFc;
    const float* src = w_fc1 + (size_t)row * kC + kc * 8;
    uint32_t q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = pack_bf16x2(__ldg(src + 2 * j), __ldg(src + 2 * j + 1));
    const uint32_t off = (uint32_t)(kc >> 3) * (kFc * 128u) + (uint32_t)row * 128u + ((uint32_t)((kc & 7) ^ (row & 7)) << 4);
    *reinterpret_cast<uint4*>(fc1_img + off) = make_uint4(q[0], q[1], q[2], q[3]);
  }
}

// ------------------------------------------------------------------ conv1 (K = 2F <= 16): CUDA cores
// Block = 256 nodes per iteration, two phases.  (A) thread = node: gather-reduce of the node's neighbours (F <= 8
// floats per row, independent loads -> deep memory-level parallelism, no shuffles), aggregate and own row parked in
// shared memory.  (B) warp = 32 of those nodes in turn, lane = output channels lane + 32 j: z = b + W_rel agg + W_root x
// from broadcast shared-memory reads, coalesced 128-byte stores of z1, per-lane column sums of act(z1), act(z1)^2
// (BatchNorm statistics).  Writes agg1 (kept for the weight gradient).
template <int ACT, int FP>
__global__ void __launch_bounds__(256) gnn_conv1_fwd_kernel(const float* __restrict__ x, int F, GnnGraph g,
                                                            const float* __restrict__ w_rel, const float* __restrict__ w_root,
                                                            const float* __restrict__ bias, int64_t M, float* __restrict__ agg_out,
                                                            float* __restrict__ z_out, float* __restrict__ partials) {
  constexpr int CPL = kC / 32;
  __shared__ float red[8][2][kC];
  __shared__ float aS[256][FP], xS[256][FP];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float wr[CPL][FP], wo[CPL][FP], bb[CPL];
#pragma unroll
  for (int j = 0; j < CPL; ++j) {
    const int c = lane + 32 * j;
    bb[j] = __ldg(bias + c);
#pragma unroll
    for (int f = 0; f < FP; ++f) {
      wr[j][f] = f < F ? __ldg(w_rel + c * F + f) : 0.f;
      wo[j][f] = f < F ? __ldg(w_root + c * F + f) : 0.f;
    }
  }
  float s1[CPL] = {}, s2[CPL] = {};
  const int64_t nchunks = (M + 255) / 256;
  for (int64_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
    const int64_t node = chunk * 256 + threadIdx.x;
    float a[FP], xs[FP];
#pragma unroll
    for (int f = 0; f < FP; ++f) a[f] = xs[f] = 0.f;
    if (node < M) {
      const int64_t pb = __ldg(g.rowptr + node), pe = __ldg(g.rowptr + node + 1);
#pragma unroll 4
      for (int64_t p = pb; p < pe; ++p) {
        const int64_t sidx = (int64_t)__ldg(g.col + p);
        const float we = g.w ? __ldg(g.w + p) : 1.f;
#pragma unroll
        for (int f = 0; f < FP; ++f)
          if (f < F) a[f] = fmaf(we, __ldg(x + sidx * F + f), a[f]);
      }
      const float inv = (g.mean && pe > pb) ? 1.f / (float)(pe - pb) : 1.f;
#pragma unroll
      for (int f = 0; f < FP; ++f) {
        a[f] *= inv;
        if (f < F) { xs[f] = __ldg(x + node * F + f); agg_out[node * F + f] = a[f]; }
      }
    }
    __syncthreads();   // phase B of the previous chunk has finished reading the shared arrays
#pragma unroll
    for (int f = 0; f < FP; ++f) { aS[threadIdx.x][f] = a[f]; xS[threadIdx.x][f] = xs[f]; }
    __syncthreads();
    const int64_t base = chunk * 256 + warp * 32;
    const int nn = (int)((M - base < 32) ? (M - base < 0 ? 0 : M - base) : 32);
#pragma unroll 2
    for (int i = 0; i < nn; ++i) {
      float av[FP], xv[FP];
#pragma unroll
      for (int f = 0; f < FP; ++f) { av[f] = aS[warp * 32 + i][f]; xv[f] = xS[warp * 32 + i][f]; }
#pragma unroll
      for (int j = 0; j < CPL; ++j) {
        float z = bb[j];
#pragma unroll
        for (int f = 0; f < FP; ++f) z = fmaf(wr[j][f], av[f], fmaf(wo[j][f], xv[f], z));
        z_out[(base + i) * kC + lane + 32 * j] = z;
        const float act = actf<ACT>(z);
        s1[j] += act;
        s2[j] += act * act;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < CPL; ++j) { red[warp][0][lane + 32 * j] = s1[j]; red[warp][1][lane + 32 * j] = s2[j]; }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * kC; i += 256) {
    float s = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) s += red[w8][i / kC][i % kC];
    partials[(size_t)blockIdx.x * 2 * kC + i] = s;
  }
}
// ------------------------------------------------------------------ BatchNorm: partial sums -> scale / shift (+ running stats)
// partials [nblk][2][Cn] = per-block sums of a, a^2 over the rows; train-mode BatchNorm1d (graph_net.py:76,84,89):
// mean, biased variance; running stats with momentum and the unbiased variance.
// block = 8 partial groups x 32 channels: coalesced 128-byte reads of the partial rows, 8-way split of the nblk loop
__global__ void __launch_bounds__(256) gnn_bn_finalize_kernel(const float* __restrict__ partials, int nblk, int Cn, int64_t rows,
                                       const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float momentum,
                                       float* __restrict__ running_mean, float* __restrict__ running_var,
                                       float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean_out,
                                       float* __restrict__ invstd_out) {
  __shared__ double red[8][2][32];
  const int cl = threadIdx.x & 31, gq = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  double s1 = 0.0, s2 = 0.0;
  if (c < Cn) {
    int b = gq;
    for (; b + 24 < nblk; b += 32) {   // four independent loads per sum in flight
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
  const double n = (double)rows;
  const double mean = s1 / n;
  double var = s2 / n - mean * mean;
  if (var < 0.0) var = 0.0;
  const float invstd = (float)(1.0 / sqrt(var + (double)eps));
  const float sc = gamma[c] * invstd;
  scale[c] = sc;
  shift[c] = beta[c] - (float)mean * sc;
  mean_out[c] = (float)mean;
  invstd_out[c] = invstd;
  if (running_mean) {
    const double unbiased = rows > 1 ? var * n / (n - 1.0) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}
// eval mode: scale / shift from the running statistics
__global__ void gnn_bn_eval_kernel(const float* __restrict__ running_mean, const float* __restrict__ running_var,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int Cn,
                                   float* __restrict__ scale, float* __restrict__ shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Cn) return;
  const float invstd = rsqrtf(running_var[c] + eps);
  scale[c] = gamma[c] * invstd;
  shift[c] = beta[c] - running_mean[c] * gamma[c] * invstd;
}

// per-graph mean + BatchNorm affine of the pooled sums: P = psum / max(n_g, 1), y = P * scale + shift   ([B, Cn] tensors;
// global_mean_pool commutes with the affine, graph_net.py:89-92 / :96).  A graph without nodes pools to y = 0, as
// global_mean_pool of the normalised rows does: the affine is applied per node, so an empty graph never receives the shift.
__global__ void gnn_pool_affine_kernel(const float* __restrict__ psum, const int64_t* __restrict__ counts,
                                       const float* __restrict__ scale, const float* __restrict__ shift, int64_t B, int Cn,
                                       float* __restrict__ P, float* __restrict__ y) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= B * Cn) return;
  const int64_t b = i / Cn;
  const int c = (int)(i % Cn);
  const int64_t n = counts[b];
  const float pv = psum[i] / (float)(n > 0 ? n : 1);
  P[i] = pv;
  y[i] = n > 0 ? fmaf(pv, scale[c], shift[c]) : 0.f;
}

// h = bf16( act(z) * scale + shift ), 8 elements per thread
template <int ACT>
__global__ void __launch_bounds__(256) gnn_bn_apply_kernel(const float* __restrict__ z, const float* __restrict__ scale,
                                                           const float* __restrict__ shift, int64_t total8,
                                                           __nv_bfloat16* __restrict__ h) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= total8) return;
  const int c0 = (int)((i * 8) % kC);
  const float4 a = __ldg(reinterpret_cast<const float4*>(z) + 2 * i), b = __ldg(reinterpret_cast<const float4*>(z) + 2 * i + 1);
  const float4 s0 = __ldg(reinterpret_cast<const float4*>(scale + c0)), s1 = __ldg(reinterpret_cast<const float4*>(scale + c0 + 4));
  const float4 t0 = __ldg(reinterpret_cast<const float4*>(shift + c0)), t1 = __ldg(reinterpret_cast<const float4*>(shift + c0 + 4));
  uint4 o;
  o.x = pack_bf16x2(fmaf(actf<ACT>(a.x), s0.x, t0.x), fmaf(actf<ACT>(a.y), s0.y, t0.y));
  o.y = pack_bf16x2(fmaf(actf<ACT>(a.z), s0.z, t0.z), fmaf(actf<ACT>(a.w), s0.w, t0.w));
  o.z = pack_bf16x2(fmaf(actf<ACT>(b.x), s1.x, t1.x), fmaf(actf<ACT>(b.y), s1.y, t1.y));
  o.w = pack_bf16x2(fmaf(actf<ACT>(b.z), s1.z, t1.z), fmaf(actf<ACT>(b.w), s1.w, t1.w));
  reinterpret_cast<uint4*>(h)[i] = o;
}

// ====================================================================== conv2: gather + tcgen05 GEMM + BatchNorm partials
// Persistent, one CTA per SM, 128-node tiles.
//   warps 0-15 : CSR gather-reduce.  The neighbour rows (256 B of bf16 each) are fetched by the TMA engine: the lanes of
//                a warp issue one cp.async.bulk per neighbour into the warp's shared-memory slot (21 rows) and wait on
//                the slot's mbarrier, so a node's rows are ALL in flight at once and no register holds in-flight data
//                (ncu on the register-gather version: every memory unit below 25 % of peak, the loop was bound by the
//                ~1.2k-cycle L2 latency times the few loads a thread can keep in registers).  The next node's neighbour
//                ids are prefetched while the rows land.  Reduced rows go as bf16 into the SW128 A image [agg | h] of
//                the tile and into the kept copy of agg.
//   warp 20    : one thread issues the [128 x 2C] x [2C x C] MMAs (weights resident in shared memory) into one of two
//                TMEM accumulators;
//   warps 16-19: TMEM -> + bias -> z (fp32, HBM) and the column sums of act(z), act(z)^2 (transposed warp reductions).
constexpr int kLoadWarps = 16, kEpiWarp0 = 16, kMmaWarpG = 20, kConvThreads = 21 * 32;
constexpr uint32_t kAImg = 2 * kC * kTile * 2;   // [128 rows][2C cols] bf16 = 64 KB
constexpr uint32_t kWImg = 2 * kC * kC * 2;      // 64 KB
constexpr int kSlotRows = 21;                    // neighbour rows per gather slot (k = 20 fits in one round)
constexpr uint32_t kRowB = kC * 2;               // 256 B
constexpr uint32_t kSlotB = kSlotRows * kRowB;

struct ConvFwdParams {
  const __nv_bfloat16* h_in;
  GnnGraph g;
  const uint8_t* wimg;
  const float* bias;
  __nv_bfloat16* agg_out;
  float* z_out;
  float* partials;   // [grid][2][C]
  const int64_t* membership;   // optional (with psum): graph of every node
  float* psum;                 // optional [B,C]: per-graph sums of act(z) (global_mean_pool straight after the block)
  int64_t M, num_tiles;
};

template <int ACT>
__global__ void __launch_bounds__(kConvThreads, 1) gnn_conv_fwd_kernel(const ConvFwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* Aimg = smem;                       // 64 KB (single buffer: the MMA of a tile takes ~0.5k cycles, its gather >10k)
  uint8_t* Wimg = smem + kAImg;               // 64 KB
  uint8_t* slots = smem + kAImg + kWImg;      // 16 x 21 rows x 256 B
  float* biasS = reinterpret_cast<float*>(slots + kLoadWarps * kSlotB);     // [C]
  float* scratch = biasS + kC;                                              // [4][2][C]
  uint64_t* bars = reinterpret_cast<uint64_t*>(scratch + 4 * 2 * kC);
  uint64_t* full = bars;          // A image written (16 warp arrivals)
  uint64_t* empty = bars + 1;     // MMAs that read the image complete
  uint64_t* acc_full = bars + 2;  // [2]
  uint64_t* acc_empty = bars + 4; // [2] 4 warp arrivals
  uint64_t* wbar = bars + 6;
  uint64_t* gbar = bars + 7;      // [16] gather slot of warp w landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 7 + kLoadWarps);
  uint32_t* stage_all = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(bars) + 256);   // [4 warps] 2 KB staging tiles
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    mbar_init(full, kLoadWarps); mbar_init(empty, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4); }
    for (int i = 0; i < kLoadWarps; ++i) mbar_init(&gbar[i], 1);
    mbar_init(wbar, 1);
    fence_mbar_init();
    mbar_arrive_expect_tx(wbar, kWImg);
    for (int s = 0; s < 4; ++s) bulk_g2s(Wimg + s * (kWImg / 4), p.wimg + (size_t)s * (kWImg / 4), kWImg / 4, wbar);
  }
  for (int i = threadIdx.x; i < kC; i += kConvThreads) biasS[i] = __ldg(p.bias + i);
  if (warp == kMmaWarpG) tmem_alloc<256>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp < kLoadWarps) {
    // ===================== gather warps
    const uint8_t* hin = reinterpret_cast<const uint8_t*>(p.h_in);
    uint8_t* slot = slots + warp * kSlotB;
    uint64_t* bar = &gbar[warp];
    uint32_t gphase = 0;
    constexpr int NPW = kTile / kLoadWarps;   // 8 nodes per warp and tile: rows warp + 16 i
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int64_t n0 = tile * kTile;
      // row pointers of this warp's 8 nodes: lane i < 8 holds node i's [pb, pe)
      int64_t pbv = 0, pev = 0;
      if (lane < NPW && n0 + warp + kLoadWarps * lane < p.M) {
        pbv = __ldg(p.g.rowptr + n0 + warp + kLoadWarps * lane);
        pev = __ldg(p.g.rowptr + n0 + warp + kLoadWarps * lane + 1);
      }
      // neighbour ids / weights of node 0, chunk 0 (lane = CSR slot)
      int64_t pb = __shfl_sync(0xffffffffu, pbv, 0), pe = __shfl_sync(0xffffffffu, pev, 0);
      int cnt = (int)((pe - pb < kSlotRows) ? pe - pb : kSlotRows);
      int myc = lane < cnt ? __ldg(p.g.col + pb + lane) : 0;
      float myw = (p.g.w && lane < cnt) ? __ldg(p.g.w + pb + lane) : 1.f;
#pragma unroll 1
      for (int i = 0; i < NPW; ++i) {
        const int r = warp + kLoadWarps * i;
        const bool ok = n0 + r < p.M;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        const int64_t deg = pe - pb;
        // root row of the node: issued early, used last
        uint2 root = make_uint2(0u, 0u);
        if (ok) root = __ldg(reinterpret_cast<const uint2*>(hin + (size_t)(n0 + r) * kRowB) + lane);
        int64_t done = 0;
        for (;;) {
          // ---- issue this chunk's row copies (TMA engine), then prefetch the ids of the NEXT chunk / node
          if (cnt > 0) {
            if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)cnt * kRowB);
            __syncwarp();
            if (lane < cnt) bulk_g2s(slot + lane * kRowB, hin + (size_t)myc * kRowB, kRowB, bar);
          }
          const int ccnt = cnt;
          const float cw = myw;
          done += cnt;
          int64_t npb = pb + done, npe = pe;
          bool next_node = false;
          if (done >= deg) {   // this node is complete after this chunk: next = node i + 1
            next_node = true;
            const int ni = (i + 1 < NPW) ? i + 1 : 0;
            npb = __shfl_sync(0xffffffffu, pbv, ni);
            npe = __shfl_sync(0xffffffffu, pev, ni);
            if (i + 1 >= NPW) { npb = 0; npe = 0; }
          }
          cnt = (int)((npe - npb < kSlotRows) ? npe - npb : kSlotRows);
          myc = lane < cnt ? __ldg(p.g.col + npb + lane) : 0;
          myw = (p.g.w && lane < cnt) ? __ldg(p.g.w + npb + lane) : 1.f;
          // ---- reduce the landed rows: lane owns 4 channels (8 bytes of every row)
          if (ccnt > 0) {
            mbar_wait_b(bar, gphase);
            gphase ^= 1;
            slot_reduce<(int)kRowB>(slot, ccnt, lane, p.g.w != nullptr, cw, acc);
            __syncwarp();   // every lane has read the slot before the next chunk's copies overwrite it
          }
          if (next_node) { pb = npb; pe = npe; break; }
        }
        if (p.g.mean && deg > 0) {
          const float inv = 1.f / (float)deg;
          acc[0] *= inv; acc[1] *= inv; acc[2] *= inv; acc[3] *= inv;
        }
        const uint2 ag = make_uint2(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]));
        if (ok) reinterpret_cast<uint2*>(p.agg_out + (size_t)(n0 + r) * kC)[lane] = ag;
        // the A image is free once the MMAs of the previous tile have completed
        if (i == 0 && it >= 1) mbar_wait_b(empty, (uint32_t)((it - 1) & 1));
        const int col = 4 * lane;
        *reinterpret_cast<uint2*>(Aimg + act_chunk_off(r, col) + ((col & 7) << 1)) = ag;
        *reinterpret_cast<uint2*>(Aimg + act_chunk_off(r, kC + col) + ((col & 7) << 1)) = root;
      }
      fence_proxy_async();
      mbar_arrive_warp(full);
    }
  } else if (warp == kMmaWarpG) {
    // ===================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t IDESC = make_idesc_bf16(128, kC, 0, 0);
      mbar_wait_b(wbar, 0);
      const uint32_t a_base = smem_u32(Aimg), w_base = smem_u32(Wimg);
      int it = 0;
      for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1, k = it >> 1;
        mbar_wait_b(full, (uint32_t)(it & 1));
        if (k >= 1) mbar_wait_b(&acc_empty[buf], (uint32_t)((k - 1) & 1));
        tc_fence_after();
#pragma unroll
        for (int s = 0; s < 2 * kC / 64; ++s)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_bf16(tmem + buf * kC, make_smem_desc_sw128_k(a_base + s * kActSlab + ks * 32),
                      make_smem_desc_sw128_k(w_base + s * (kC * 128) + ks * 32), IDESC, (s | ks) != 0);
        umma_commit(empty);
        umma_commit(&acc_full[buf]);
      }
    }
  } else {
    // ===================== epilogue warps 16-19
    const int q = warp & 3;
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
    float st[kC / 16][2];
#pragma unroll
    for (int c = 0; c < kC / 16; ++c) st[c][0] = st[c][1] = 0.f;
    uint32_t* stage = stage_all + q * kStage16Words;
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1, k = it >> 1;
      mbar_wait_b(&acc_full[buf], (uint32_t)(k & 1));
      tc_fence_after();
      const int64_t node0 = tile * kTile + q * 32;
      const int64_t node = node0 + lane;
      const bool valid = node < p.M;
      const int rows_valid = (int)((p.M - node0) < 32 ? (p.M - node0 < 0 ? 0 : p.M - node0) : 32);
      // optional per-graph sums (the block is followed by global_mean_pool): like the fc1 kernel, one atomic per column
      // when the warp's 32 rows belong to one graph, per-row atomics otherwise
      int64_t gph = -1, g0 = -1;
      bool uniform = false;
      if (p.psum) {
        gph = valid ? __ldg(p.membership + node) : -1;
        g0 = __shfl_sync(0xffffffffu, gph, 0);
        uniform = __all_sync(0xffffffffu, gph == g0) && g0 >= 0;
      }
#pragma unroll
      for (int c = 0; c < kC / 16; ++c) {
        uint32_t v[16];
        tmem_ld16(lane_base + buf * kC + c * 16, v);
        tmem_wait_ld();
        float a1[16], a2[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float z = __uint_as_float(v[j]) + biasS[c * 16 + j];
          v[j] = __float_as_uint(z);
          const float a = valid ? actf<ACT>(z) : 0.f;
          a1[j] = a;
          a2[j] = a * a;
        }
        warp_store_rows16(stage, v, reinterpret_cast<uint32_t*>(p.z_out) + (size_t)node0 * kC + c * 16, kC, rows_valid, lane);
        if (p.psum && !uniform && valid) {
#pragma unroll
          for (int j = 0; j < 16; ++j) atomicAdd(p.psum + gph * kC + c * 16 + j, a1[j]);
        }
        const float cs = warp_transpose_sum16(a1, lane);
        st[c][0] += cs;
        st[c][1] += warp_transpose_sum16(a2, lane);
        if (p.psum && uniform && lane < 16) atomicAdd(p.psum + g0 * kC + c * 16 + lane, cs);
      }
      tc_fence_before();
      mbar_arrive_warp(&acc_empty[buf]);
    }
    if (lane < 16) {
#pragma unroll
      for (int c = 0; c < kC / 16; ++c) {
        scratch[(q * 2 + 0) * kC + c * 16 + lane] = st[c][0];
        scratch[(q * 2 + 1) * kC + c * 16 + lane] = st[c][1];
      }
    }
    asm volatile("bar.sync 2, 128;" ::: "memory");
    const int t = threadIdx.x - kEpiWarp0 * 32;   // 0..127
    for (int i = t; i < 2 * kC; i += 128) {
      const int which = i / kC, c = i % kC;
      p.partials[(size_t)blockIdx.x * 2 * kC + i] = scratch[(0 * 2 + which) * kC + c] + scratch[(1 * 2 + which) * kC + c] +
                                                     scratch[(2 * 2 + which) * kC + c] + scratch[(3 * 2 + which) * kC + c];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarpG) tmem_dealloc<256>(tmem);
}

// ====================================================================== fc1 + act + BatchNorm partials + per-graph sums
// z3 = h2 Wfc1^T + b (N = 256), a3 = act(z3): only the column sums of a3, a3^2 over all nodes (bn3 statistics) and the
// per-graph sums of a3 leave the SM — global_mean_pool(bn3(a3)) = bn3_affine(mean_graph(a3)) (graph_net.py:88-92).
// Warps 0-3: h2 tile (bf16 rows) -> SW128 image, double buffered; warp 12: MMA (two 256-column accumulators);
// warps 4-11: epilogue (lane quarter = warp & 3, column half = (warp - 4) >> 2).
// 4 loader warps, 16 epilogue warps (lane quarter x 64-column part: the kernel is bound by its epilogue — activation, two
// transposed column sums and the per-graph sums of 128 x 256 outputs per tile), 1 MMA warp
constexpr int kFcLoadWarps = 4, kFcEpiWarp0 = 4, kFcEpiWarps = 16, kFcMmaWarp = 20, kFcThreads = 21 * 32;
constexpr int kFcChunks = kFc / 16 / (kFcEpiWarps / 4);   // 16-column chunks per epilogue warp
constexpr uint32_t kHImg = kC * kTile * 2;       // 32 KB
constexpr uint32_t kFcWImg = kFc * kC * 2;       // 64 KB

struct Fc1FwdParams {
  const __nv_bfloat16* h_in;   // [M,C]
  const uint8_t* wimg;         // [256][C] image
  const float* bias;           // [256]
  const int64_t* membership;   // [M] graph of every node
  float* psum;                 // [B,256] per-graph sums of a3 (zeroed by the caller)
  float* partials;             // [grid][2][256]
  int64_t M, num_tiles;
};

// h tile (rows [tile*128, +128) of a bf16 [M,C] matrix) -> SW128 image; `nw` warps cooperate
__device__ __forceinline__ void load_h_tile(const __nv_bfloat16* __restrict__ h, int64_t tile, int64_t M, uint8_t* img,
                                            int warp, int lane, int nw) {
  // 128 rows x 16 chunks of 16 B; a warp covers 2 rows per step
  for (int c = warp * 32 + lane; c < kTile * (kC / 8); c += nw * 32) {
    const int r = c >> 4, kc = c & 15;
    const int64_t node = tile * kTile + r;
    const uint4 v = node < M ? __ldg(reinterpret_cast<const uint4*>(h + (size_t)node * kC) + kc) : make_uint4(0u, 0u, 0u, 0u);
    *reinterpret_cast<uint4*>(img + act_chunk_off(r, kc * 8)) = v;
  }
}

template <int ACT>
__global__ void __launch_bounds__(kFcThreads, 1) gnn_fc1_pool_fwd_kernel(const Fc1FwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* Himg = smem;                       // 2 x 32 KB
  uint8_t* Wimg = smem + 2 * kHImg;           // 64 KB
  float* biasS = reinterpret_cast<float*>(smem + 2 * kHImg + kFcWImg);      // [256]
  float* scratch = biasS + kFc;                                             // [4][2][256]
  uint64_t* bars = reinterpret_cast<uint64_t*>(scratch + 4 * 2 * kFc);
  uint64_t* full = bars;          // [2]
  uint64_t* empty = bars + 2;     // [2]
  uint64_t* acc_full = bars + 4;  // [2]
  uint64_t* acc_empty = bars + 6; // [2] 8 warp arrivals
  uint64_t* wbar = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&full[i], kFcLoadWarps); mbar_init(&empty[i], 1); mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], kFcEpiWarps); }
    mbar_init(wbar, 1);
    fence_mbar_init();
    mbar_arrive_expect_tx(wbar, kFcWImg);
    for (int s = 0; s < 4; ++s) bulk_g2s(Wimg + s * (kFcWImg / 4), p.wimg + (size_t)s * (kFcWImg / 4), kFcWImg / 4, wbar);
  }
  for (int i = threadIdx.x; i < kFc; i += kFcThreads) biasS[i] = __ldg(p.bias + i);
  if (warp == kFcMmaWarp) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp < kFcLoadWarps) {
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1, k = it >> 1;
      if (k >= 1) mbar_wait_b(&empty[buf], (uint32_t)((k - 1) & 1));
      load_h_tile(p.h_in, tile, p.M, Himg + buf * kHImg, warp, lane, kFcLoadWarps);
      fence_proxy_async();
      mbar_arrive_warp(&full[buf]);
    }
  } else if (warp == kFcMmaWarp) {
    if (lane == 0) {
      constexpr uint32_t IDESC = make_idesc_bf16(128, kFc, 0, 0);
      mbar_wait_b(wbar, 0);
      const uint32_t h_base = smem_u32(Himg), w_base = smem_u32(Wimg);
      int it = 0;
      for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1, k = it >> 1;
        mbar_wait_b(&full[buf], (uint32_t)(k & 1));
        if (k >= 1) mbar_wait_b(&acc_empty[buf], (uint32_t)((k - 1) & 1));
        tc_fence_after();
#pragma unroll
        for (int s = 0; s < kC / 64; ++s)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_bf16(tmem + buf * kFc, make_smem_desc_sw128_k(h_base + buf * kHImg + s * kActSlab + ks * 32),
                      make_smem_desc_sw128_k(w_base + s * (kFc * 128) + ks * 32), IDESC, (s | ks) != 0);
        umma_commit(&empty[buf]);
        umma_commit(&acc_full[buf]);
      }
    }
  } else {
    const int q = warp & 3, part = (warp - kFcEpiWarp0) >> 2;   // column part of kFcChunks * 16
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
    float st[kFcChunks][2];
#pragma unroll
    for (int c = 0; c < kFcChunks; ++c) st[c][0] = st[c][1] = 0.f;
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1, k = it >> 1;
      const int64_t node = tile * kTile + q * 32 + lane;
      const bool valid = node < p.M;
      const int64_t gph = valid ? __ldg(p.membership + node) : -1;
      // the 32 rows of this warp usually belong to one graph: then the per-graph sums come out of the same
      // transposed reduction as the statistics (one atomic per column); otherwise every row adds its own values
      const int64_t g0 = __shfl_sync(0xffffffffu, gph, 0);
      const bool uniform = __all_sync(0xffffffffu, gph == g0) && g0 >= 0;
      mbar_wait_b(&acc_full[buf], (uint32_t)(k & 1));
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < kFcChunks; ++c) {
        const int col0 = (part * kFcChunks + c) * 16;
        uint32_t v[16];
        tmem_ld16(lane_base + buf * kFc + col0, v);
        tmem_wait_ld();
        float a1[16], a2[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float a = valid ? actf<ACT>(__uint_as_float(v[j]) + biasS[col0 + j]) : 0.f;
          a1[j] = a;
          a2[j] = a * a;
        }
        if (!uniform && valid) {
#pragma unroll
          for (int j = 0; j < 16; ++j) atomicAdd(p.psum + gph * kFc + col0 + j, a1[j]);
        }
        const float cs = warp_transpose_sum16(a1, lane);
        st[c][0] += cs;
        st[c][1] += warp_transpose_sum16(a2, lane);
        if (uniform && lane < 16) atomicAdd(p.psum + g0 * kFc + col0 + lane, cs);
      }
      tc_fence_before();
      mbar_arrive_warp(&acc_empty[buf]);
    }
    if (lane < 16) {
#pragma unroll
      for (int c = 0; c < kFcChunks; ++c) {
        scratch[(q * 2 + 0) * kFc + (part * kFcChunks + c) * 16 + lane] = st[c][0];
        scratch[(q * 2 + 1) * kFc + (part * kFcChunks + c) * 16 + lane] = st[c][1];
      }
    }
    asm volatile("bar.sync 2, %0;" ::"n"(kFcEpiWarps * 32) : "memory");
    const int t = threadIdx.x - kFcEpiWarp0 * 32;   // 0..511
    for (int i = t; i < 2 * kFc; i += kFcEpiWarps * 32) {
      const int which = i / kFc, c = i % kFc;
      p.partials[(size_t)blockIdx.x * 2 * kFc + i] = scratch[(0 * 2 + which) * kFc + c] + scratch[(1 * 2 + which) * kFc + c] +
                                                      scratch[(2 * 2 + which) * kFc + c] + scratch[(3 * 2 + which) * kFc + c];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kFcMmaWarp) tmem_dealloc<512>(tmem);
}

// grid of a grid-stride CUDA-core kernel: every CTA resident at once (a 592-block launch of a kernel that fits 3 CTAs per SM
// ran 1.33 waves: the last third of the blocks had the chip to itself at a third of the occupancy)
int gnn_resident_blocks(const void* kern, int threads, int smem_bytes, int64_t want) {
  int dev = 0, sms = 148, occ = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, (size_t)smem_bytes) != cudaSuccess || occ < 1) occ = 1;
  const int64_t cap = (int64_t)occ * sms;
  int64_t b = want < cap ? want : cap;
  if (b > 1184) b = 1184;   // pcc_gnn_max_blocks
  return (int)(b < 1 ? 1 : b);
}

int gnn_grid(int64_t num_tiles) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return (int)(num_tiles < sms ? num_tiles : sms);
}

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

extern "C" int64_t pcc_gnn_packed_bytes(void) { return (int64_t)kWImg + kFcWImg; }
extern "C" int pcc_gnn_max_blocks(void) { return 1184; }

extern "C" int pcc_gnn_pack_weights(const float* w_rel2, const float* w_root2, const float* w_fc1, void* packed, int device,
                                    void* stream) {
  PCC_ENTER(device);
  const int total = kC * (2 * kC / 8) + kFc * (kC / 8);
  PCC_K(gnn_pack_kernel)<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(w_rel2, w_root2, w_fc1, (uint8_t*)packed,
                                                                            (uint8_t*)packed + kWImg);
  return check_launch(__func__);
}

extern "C" int pcc_gnn_conv1_fwd(const float* x, int F, const int64_t* rowptr, const int32_t* col, const float* w, int mean,
                                 const float* w_rel, const float* w_root, const float* bias, int64_t M, int act, float* agg_out,
                                 float* z_out, float* partials, int* nblk_out, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(F >= 1 && F <= 8, "fused conv1 needs input_dim <= 8");
  int blocks = 1;
  GnnGraph g{rowptr, col, w, mean};
  GNN_ACT_DISPATCH(act, {
    auto kern = F <= 4 ? gnn_conv1_fwd_kernel<A, 4> : gnn_conv1_fwd_kernel<A, 8>;
    blocks = (int)(cdiv(M, 256) < 592 ? cdiv(M, 256) : 592);   // (measured: 592 blocks 52 us, one resident wave of 444 57 us)
    if (blocks < 1) blocks = 1;
    PCC_K(kern)<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, F, g, w_rel, w_root, bias, M, agg_out, z_out, partials);
  });
  *nblk_out = blocks;
  return check_launch(__func__);
}

extern "C" int pcc_gnn_bn_finalize(const float* partials, int nblk, int Cn, int64_t rows, const float* gamma, const float* beta,
                                   float eps, float momentum, float* running_mean, float* running_var, float* scale,
                                   float* shift, float* mean_out, float* invstd_out, int device, void* stream) {
  PCC_ENTER(device);
  PCC_K(gnn_bn_finalize_kernel)<<<cdiv(Cn, 32), 256, 0, (cudaStream_t)stream>>>(partials, nblk, Cn, rows, gamma, beta, eps, momentum,
                                                                                running_mean, running_var, scale, shift, mean_out,
                                                                                invstd_out);
  return check_launch(__func__);
}

extern "C" int pcc_gnn_bn_eval(const float* running_mean, const float* running_var, const float* gamma, const float* beta,
                               float eps, int Cn, float* scale, float* shift, int device, void* stream) {
  PCC_ENTER(device);
  PCC_K(gnn_bn_eval_kernel)<<<cdiv(Cn, 128), 128, 0, (cudaStream_t)stream>>>(running_mean, running_var, gamma, beta, eps, Cn, scale, shift);
  return check_launch(__func__);
}

extern "C" int pcc_gnn_pool_affine(const float* psum, const int64_t* counts, const float* scale, const float* shift, int64_t B,
                                   int Cn, float* P, float* y, int device, void* stream) {
  PCC_ENTER(device);
  if (B * Cn == 0) return 0;
  PCC_K(gnn_pool_affine_kernel)<<<(unsigned)cdiv(B * Cn, 256), 256, 0, (cudaStream_t)stream>>>(psum, counts, scale, shift, B, Cn, P, y);
  return check_launch(__func__);
}

extern "C" int pcc_gnn_bn_apply(const float* z, const float* scale, const float* shift, int64_t M, int act, void* h_bf16,
                                int device, void* stream) {
  PCC_ENTER(device);
  const int64_t total8 = M * kC / 8;
  if (total8 == 0) return 0;
  GNN_ACT_DISPATCH(act, {
    auto kern = gnn_bn_apply_kernel<A>;
    PCC_K(kern)<<<(unsigned)cdiv(total8, 256), 256, 0, (cudaStream_t)stream>>>(z, scale, shift, total8, (__nv_bfloat16*)h_bf16);
  });
  return check_launch(__func__);
}

extern "C" int pcc_gnn_conv_fwd(const void* h_in_bf16, const int64_t* rowptr, const int32_t* col, const float* w, int mean,
                                const void* packed, const float* bias, int64_t M, int act, void* agg_out_bf16, float* z_out,
                                float* partials, const int64_t* membership, float* psum, int64_t B, int* nblk_out, int device,
                                void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(psum == nullptr || membership != nullptr, "psum needs the membership vector");
  if (psum) PCC_CUDA(cudaMemsetAsync(psum, 0, (size_t)B * kC * sizeof(float), (cudaStream_t)stream));
  ConvFwdParams p{};
  p.membership = membership;
  p.psum = psum;
  p.h_in = (const __nv_bfloat16*)h_in_bf16;
  p.g = GnnGraph{rowptr, col, w, mean};
  p.wimg = (const uint8_t*)packed;
  p.bias = bias;
  p.agg_out = (__nv_bfloat16*)agg_out_bf16;
  p.z_out = z_out;
  p.partials = partials;
  p.M = M;
  p.num_tiles = cdiv(M, kTile);
  const int grid = gnn_grid(p.num_tiles);
  *nblk_out = grid;
  if (grid == 0) return 0;
  const int smem_bytes = kAImg + kWImg + kLoadWarps * kSlotB + (kC + 8 * kC) * 4 + 256 + 4 * kStage16Words * 4;
  {
    ProfScope prof(3, (cudaStream_t)stream);
    GNN_ACT_DISPATCH(act, {
      auto kern = gnn_conv_fwd_kernel<A>;
      PCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
      PCC_K(kern)<<<grid, kConvThreads, smem_bytes, (cudaStream_t)stream>>>(p);
    });
  }
  return check_launch(__func__);
}

extern "C" int pcc_gnn_fc1_pool_fwd(const void* h_in_bf16, const void* packed, const float* bias, const int64_t* membership,
                                    int64_t M, int64_t B, int act, float* psum, float* partials, int* nblk_out, int device,
                                    void* stream) {
  PCC_ENTER(device);
  Fc1FwdParams p{};
  p.h_in = (const __nv_bfloat16*)h_in_bf16;
  p.wimg = (const uint8_t*)packed + kWImg;
  p.bias = bias;
  p.membership = membership;
  p.psum = psum;
  p.partials = partials;
  p.M = M;
  p.num_tiles = cdiv(M, kTile);
  PCC_CUDA(cudaMemsetAsync(psum, 0, (size_t)B * kFc * sizeof(float), (cudaStream_t)stream));
  const int grid = gnn_grid(p.num_tiles);
  *nblk_out = grid;
  if (grid == 0) return 0;
  const int smem_bytes = 2 * kHImg + kFcWImg + (kFc + 8 * kFc) * 4 + 128;
  GNN_ACT_DISPATCH(act, {
    auto kern = gnn_fc1_pool_fwd_kernel<A>;
    PCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    PCC_K(kern)<<<grid, kFcThreads, smem_bytes, (cudaStream_t)stream>>>(p);
  });
  return check_launch(__func__);
}
