// Fused DeepSets phi backward on tcgen05 / TMEM (sm_100a): autograd of
// /root/reference/models/deep_sets.py:89-106 in two kernels.
//
//  K1 "chain" (persistent, 128-point tiles): recompute the forward per tile (activations
//     never stored by the forward), build dZ of the final Linear from the pooled gradient
//     (+ argmax rows for max pooling), then walk the layers backwards:
//        dZ_l = dH_l * act'(z_l)            (epilogue: TMEM x TMEM -> bf16 blob in smem)
//        dH_{l-1} = dZ_l W_l (+ dH_l for a ResidualBlock: MMA accumulates onto dH_l in TMEM)
//     The operand blobs needed by the weight gradients (h_{l-1}, dZ_l) are pushed to a
//     staging area with cp.async.bulk stores straight from the smem operand images.
//     (TMEM holds exactly one H x H fp32 matrix, so the weight gradients of several
//     layers cannot stay resident next to the chain's accumulators; DESIGN.md §3.)
//  K2 "wgrad": dW_l = sum_tiles dZ_l^T h_{l-1} with both operands read as MN-major views of
//     the staged blobs, fp32 accumulation in TMEM across all tiles of a CTA, one partial
//     per CTA, column sums (db) on the epilogue warps; a small kernel reduces the partials.
#include "pcc_fused.cuh"
#include "pcc_head.cuh"

namespace pcc {

constexpr int kRingB = 3;  // weight slabs (K = 64, H rows) in flight in the chain kernel

struct BwdParams {
  const float* x;
  const int64_t* offsets;
  int64_t n, B, num_tiles;
  int d, L, pooling, res_mask;
  const uint8_t* wpack;
  uint32_t w_off[kMaxLayers], wt_off[kMaxLayers];
  const float* bias[kMaxLayers];
  const float* dpooled;
  const int32_t* argmax;
  uint8_t* stage_h[kMaxLayers];  // h_l images,  l = 0..L-2, [num_tiles] x SW128 [H/64][128][64] bf16
  uint8_t* stage_g[kMaxLayers];  // dZ_l images, l = 0..L-1
  float* part_w[kMaxLayers];     // per-CTA partial dW_l [grid][H][K_l]  (K_0 = 16)
  float* part_b[kMaxLayers];     // per-CTA partial db_l [grid][H]
  int virt;                      // 1: max pooling on pre-gathered argmax rows (row b*H+f is THE argmax row of (b, f));
                                 // 2: sum / mean pooling commuted with the final Linear: dpooled holds
                                 //    G = dpooled W_{L-1} [B, H] and dH_lh[row] = scale(row) * G[set(row)]
  int nbig;                      // H x H layers whose weight gradient is a GEMM over the staged images
  const int32_t* row_set;        // [n] set of each row (-1: none), seg_prep_kernel
  const float* row_scale;        // [n] pooled-gradient scale of the row's set
  long long* trace;              // optional (debug) event trace of CTA 0
};

__device__ __forceinline__ void trace_b(long long* trace, int role, int& n, int id) {
  if (trace && blockIdx.x == 0 && n < 2047) {
    trace[role * 4096 + 2 * n] = id;
    trace[role * 4096 + 2 * n + 1] = clock64();
    ++n;
  }
}

struct BwdSmem {
  uint32_t bufG, bufH, ring, bias, bars, total;
};
__host__ __device__ inline BwdSmem bwd_smem(int H, int L) {
  BwdSmem s;
  uint32_t o = 0;
  s.bufG = o; o += kTileM * H * 2;   // dZ image (A operand of the dgrad GEMMs)
  s.bufH = o; o += kTileM * H * 2;   // h image; its first 4 KB double as the layer-0 operand (x tile)
  s.ring = o; o += kRingB * w_slab_bytes(H);
  s.bias = o; o += (uint32_t)(L - 1) * H * 4;  // biases of the hidden layers 0..L-2
  s.bars = o; o += 128;
  s.total = o;
  return s;
}

// ====================================================================== K1: chain
// Per 128-row tile (lh = L-2 is the last hidden layer; L is 2 or 3):
//   E: x tile -> bufH head                                   | M: z_0 = x W_0^T            -> accA
//   E: dZ_{L-1} from the pooled gradient -> bufG (staged)     | M: dH_lh = dZ_{L-1} W_{L-1} -> accB
//   L = 3 only:  E: h_0 = act(z_0 + b_0) -> bufH (staged)     | M: z_1 = h_0 W_1^T          -> accA
//   E: ONE pass over (accA, accB): h_lh -> bufH and dZ_lh = dH_lh * act'(z_lh) -> bufG (both staged)
//   L = 3 only:  E: x tile -> bufH head again                 | M: dH_0 = dZ_1 W_1 (+ dH_1 for a ResidualBlock:
//                                                                  the MMA accumulates onto accB), z_0 -> accA
//                E: dZ_0 = dH_0 * act'(z_0) -> bufG (staged)
// so the dgrad of the final layer runs under the h_0 epilogue and z of the last hidden layer is read
// from TMEM once for both of its uses.  Max pooling with L = 3 (`pipe` below) hands the h_0 and dZ_1 images
// over slab by slab and rotates the two accumulators, so that z_1, dH_0 and the next tile's z_0 run under the
// epilogue passes; with ReLU, dZ_0 takes act'(z_0) from bits kept by the h_0 pass instead of a second z_0 GEMM.
template <int H, int ACT, bool PIPE>
__global__ void __launch_bounds__(kThreads, 1) phi_bwd_chain_kernel(const BwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const BwdSmem lay = bwd_smem(H, p.L);
  uint8_t* bufG = smem + lay.bufG;
  uint8_t* bufH = smem + lay.bufH;
  uint8_t* ring = smem + lay.ring;
  float* biasS = reinterpret_cast<float*>(smem + lay.bias);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + lay.bars);
  uint64_t* full = bars;
  uint64_t* empty = bars + kRingB;
  uint64_t* a_ready = bars + 2 * kRingB;      // an operand image is ready (epilogue warps -> MMA thread)
  uint64_t* accA_ready = bars + 2 * kRingB + 1;  // z in accA complete
  uint64_t* accB_ready = bars + 2 * kRingB + 2;  // dH in accB complete
  uint64_t* wf_ready = bars + 2 * kRingB + 3;    // virtual-row mode: rows of the final weight image landed in bufG
  uint64_t* slab_ready = bars + 2 * kRingB + 4;  // [4] max pooling, L = 3: 64-column slab s of h_0 / dZ_1 written
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kRingB + 8);

  constexpr uint32_t SLAB = w_slab_bytes(H);
  constexpr uint32_t X_LBO = kTileM * 16;
  constexpr uint32_t W0_LBO = H * 16;
  constexpr uint32_t BLOB = kTileM * H * 2;
  constexpr int NSLAB = H / 64;
  constexpr int NCHUNK = H / 32;
  constexpr uint32_t ACC_A = 0, ACC_B = 256;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = p.L;
  const int lh = L - 2;

  for (int i = threadIdx.x; i < (L - 1) * H; i += kThreads) biasS[i] = __ldg(p.bias[i / H] + (i % H));
  if (threadIdx.x == 0) {
    for (int i = 0; i < kRingB; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(a_ready, kEpiWarps);
    mbar_init(accA_ready, 1);
    mbar_init(accB_ready, 1);
    mbar_init(wf_ready, 1);
    if (PIPE)
      for (int i = 0; i < 4; ++i) mbar_init(&slab_ready[i], kEpiWarps);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_wait();  // the prologue read only parameters; rows, gradients and images come from the predecessors in the stream
  // Virtual-row mode (max pooling, rows pre-gathered: row b*H + f is the argmax row of (b, f)): the gradient of
  // the final Linear's output is one-hot per row, dZ_{L-1}[row] = dpooled[row] * e_f, so
  //   dH_lh[row, :] = dpooled[row] * W_{L-1}[f, :]      (a scaled weight row: no dgrad GEMM, no dZ_{L-1} image)
  //   dW_{L-1}[f, :] = sum_b dpooled[b, f] * h_lh[b*H + f, :]   (final_wgrad_virtual_kernel, no GEMM either)
  // The 128 weight rows a tile needs are one contiguous 16 KB piece of every K slab of the packed image.
  // Mode 2 (sum / mean): the final Linear was applied AFTER pooling (forward kernel, poolh), so its dgrad is the
  // [B, H] product G computed by the host and dH_lh of a row is its set's row of G times the pooling scale: the
  // same per-tile flow as mode 1 with the dH image built from G; h_lh is not needed by any weight gradient.
  const bool virt = p.virt != 0;     // no per-point dgrad / wgrad GEMM for the final Linear
  const bool vmax = p.virt == 1, bcast = p.virt == 2;
  // bcast3 (sum / mean pooling commuted with the final Linear, two hidden layers): the pooled gradient of a row is read
  // straight from the [B,H] matrix G in the dZ_1 pass, which leaves the gradient image buffer free during the h_0
  // epilogue: that epilogue also stores act'(z_0) there (bf16), so the tile needs neither a second z_0 GEMM nor a second
  // activation evaluation for dZ_0; dZ_1 is written over h_0 (already staged) and feeds the dgrad from there.
  const bool bcast3 = bcast && p.L == 3;
  // pipe (max pooling, two hidden layers): every GEMM runs under the epilogue pass that feeds it.  The two 256-column
  // accumulators rotate: tile t holds z_0 and then dH_0 in X, z_1 in Y, and X / Y swap every tile, so
  //   h_0 pass (reads X)        | z_1 = h_0 W_1^T -> Y, K slab s issued as soon as h_0 slab s is written
  //   h_1 / dZ_1 pass (reads Y) | dH_0 = dZ_1 W_1 -> X, K slab s issued as soon as dZ_1 slab s is written
  //   dZ_0 pass (reads X)       | z_0 of the next tile -> Y (ReLU; its x tile is staged before this pass)
  // Within each GEMM the K order is that of a plain gemm(), so the accumulators hold the same bits.  A template
  // parameter (the host sets it exactly when p.virt == 1 and p.L == 3), so the other modes compile without it.
  constexpr bool pipe = PIPE;
  // ReLU: act'(z_0 + b_0) is the predicate z_0 + b_0 > 0, which the h_0 pass keeps as a bit mask in registers (every
  // thread owns the same row and column chunks in the h_0 and dZ_0 passes), so z_0 is not recomputed for dZ_0.  Other
  // activations recompute z_0 into Y after the h_1 / dZ_1 pass.
  constexpr bool mask0 = PIPE && ACT == PCC_ACT_RELU;
  // wait trace of the producer and the MMA thread (tools/trace_bwd.py): pipelined variant only, so that the other modes
  // compile without it
  long long* const wtrace = PIPE ? p.trace : nullptr;

  if (warp == kProdWarp) {
    // ===================== producer: weight slabs in consumption order
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      int tn = 0;
      auto push = [&](const uint8_t* src, uint32_t bytes) {
        trace_b(wtrace, 2, tn, 30);   // ring slot wait: begin / end
        mbar_wait(&empty[stage], phase ^ 1);
        trace_b(wtrace, 2, tn, 31);
        mbar_arrive_expect_tx(&full[stage], bytes);
        bulk_g2s(ring + stage * SLAB, src, bytes, &full[stage]);
        if (++stage == kRingB) { stage = 0; phase ^= 1; }
      };
      auto push_layer = [&](uint32_t off) { for (int s = 0; s < NSLAB; ++s) push(p.wpack + off + (size_t)s * SLAB, SLAB); };
      for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        push(p.wpack + p.w_off[0], (kK0 / 8) * W0_LBO);        // z_0
        if (!virt) push_layer(p.wt_off[L - 1]);                 // dgrad of the final layer
        if (L == 3) {
          push_layer(p.w_off[1]);                               // z_1
          push_layer(p.wt_off[1]);                              // dgrad of layer 1
          if (!bcast3 && !mask0) push(p.wpack + p.w_off[0], (kK0 / 8) * W0_LBO);      // z_0 again
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t IDESC = make_idesc_bf16(128, H, 0, 0);
      uint32_t stage = 0, phase = 0, a_phase = 0;
      int tn = 0;
      const uint32_t g_base = smem_u32(bufG), h_base = smem_u32(bufH), r_base = smem_u32(ring);
      // trace ids of the MMA thread: 40/41 operand hand-over wait begin/end, 42/43 weight slab wait begin/end
      auto wait_a = [&]() {
        trace_b(wtrace, 1, tn, 40);
        mbar_wait(a_ready, a_phase);
        trace_b(wtrace, 1, tn, 41);
        a_phase ^= 1;
        tc_fence_after();
      };
      auto wait_full = [&]() {
        trace_b(wtrace, 1, tn, 42);
        mbar_wait(&full[stage], phase);
        trace_b(wtrace, 1, tn, 43);
        tc_fence_after();
      };
      // D[acc] (+)= act[:, K slab s] (SW128 image) * streamed weight slab^T
      auto gemm_slab = [&](uint32_t act_base, uint32_t acc_col, int s, bool accumulate_first) {
        wait_full();
        const uint32_t w_slab = r_base + stage * SLAB;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          umma_bf16(tmem + acc_col, make_smem_desc_sw128_k(act_base + s * kActSlab + ks * 32),
                    make_smem_desc_sw128_k(w_slab + ks * 32), IDESC, ((s | ks) != 0) || accumulate_first);
        umma_commit(&empty[stage]);
        if (++stage == kRingB) { stage = 0; phase ^= 1; }
      };
      // D[acc] (+)= act[128 x H] * streamed weight image^T
      auto gemm = [&](uint32_t act_base, uint32_t acc_col, bool accumulate_first) {
        for (int s = 0; s < NSLAB; ++s) gemm_slab(act_base, acc_col, s, accumulate_first);
      };
      // z_0 = x tile (un-swizzled image at the head of bufH) * W_0^T -> acc
      auto gemm0 = [&](uint32_t acc_col) {
        wait_full();
        umma_bf16(tmem + acc_col, make_smem_desc(h_base, X_LBO, 128), make_smem_desc(r_base + stage * SLAB, W0_LBO, 128),
                  IDESC, 0);
        umma_commit(&empty[stage]);
        if (++stage == kRingB) { stage = 0; phase ^= 1; }
      };
      if (pipe) {
        const bool res = (p.res_mask >> 1) & 1;
        uint32_t sl_phase = 0, accX = ACC_A;
        auto wait_slab = [&](int s) {  // trace ids 44/45: slab hand-over wait begin/end
          trace_b(wtrace, 1, tn, 44);
          mbar_wait(&slab_ready[s], sl_phase);
          trace_b(wtrace, 1, tn, 45);
          tc_fence_after();
        };
        for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
          const uint32_t accY = ACC_A + ACC_B - accX;
          wait_a();                                 // x tile staged (ReLU: during the previous tile's h_1 / dZ_1 pass)
          gemm0(accX);
          umma_commit(accA_ready);
          for (int s = 0; s < NSLAB; ++s) {         // z_1 under the h_0 pass; X is free once its last slab is handed over
            wait_slab(s);
            gemm_slab(h_base, accY, s, false);
          }
          sl_phase ^= 1;
          umma_commit(accA_ready);
          // ResidualBlock: dH_1 is stored into X during the dZ_1 pass and the dgrad accumulates onto all of it
          if (res)
            for (int s = 0; s < NSLAB; ++s) wait_slab(s);
          for (int s = 0; s < NSLAB; ++s) {         // dH_0 (+ dH_1) under the h_1 / dZ_1 pass
            wait_slab(s);
            gemm_slab(g_base, accX, s, res);
          }
          sl_phase ^= 1;
          umma_commit(accB_ready);
          if (!mask0) {
            wait_a();                               // x tile staged again
            gemm0(accY);                            // z_0 again, into Y (read by the h_1 / dZ_1 pass before)
            umma_commit(accA_ready);
          }
          accX = accY;
        }
      } else
      for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        wait_a();                                   // x tile staged
        gemm0(ACC_A);
        umma_commit(accA_ready);
        if (!virt) {
          wait_a();                                 // dZ of the final layer built
          gemm(g_base, ACC_B, false);               // dH_lh
          umma_commit(accB_ready);
        }
        if (L == 3) {
          wait_a();                                 // h_0 image written
          gemm(h_base, ACC_A, false);               // z_1
          umma_commit(accA_ready);
          wait_a();                                 // dZ_1 image written (bcast3: into bufH, over h_0)
          gemm(bcast3 ? h_base : g_base, ACC_B, (p.res_mask >> 1) & 1);  // dH_0 (+ dH_1)
          umma_commit(accB_ready);
          if (!bcast3) {
            wait_a();                               // x tile staged again
            gemm0(ACC_A);                           // z_0 again
            umma_commit(accA_ready);
          }
        }
      }
    }
  } else {
    // ===================== epilogue warps 0-7
    const int quarter = warp & 3, grp = warp >> 2;
    const int r = quarter * 32 + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(quarter * 32) << 16);
    uint32_t phA = 0, phB = 0, wf_phase = 0;
    const int d = p.d;
    float xcur[kK0] = {}, xnext[kK0];
    auto load_x = [&](int64_t tile) {
      const int64_t row = tile * kTileM + r;
#pragma unroll
      for (int j = 0; j < kK0; ++j)
        xnext[j] = (grp == 0 && j < d && row < p.n && tile < p.num_tiles) ? __ldg(p.x + row * d + j) : 0.f;
    };
    auto stage_x = [&](const float (&xv)[kK0]) {  // x tile -> un-swizzled [2][128][8] image at the head of bufH
      if (grp == 0) {
        *reinterpret_cast<uint4*>(bufH + r * 16) = make_uint4(pack_bf16x2(xv[0], xv[1]), pack_bf16x2(xv[2], xv[3]),
                                                              pack_bf16x2(xv[4], xv[5]), pack_bf16x2(xv[6], xv[7]));
        *reinterpret_cast<uint4*>(bufH + X_LBO + r * 16) =
            make_uint4(pack_bf16x2(xv[8], xv[9]), pack_bf16x2(xv[10], xv[11]), pack_bf16x2(xv[12], xv[13]),
                       pack_bf16x2(xv[14], xv[15]));
      }
    };
    // mask0: the next x tile as bf16 pairs (the packing of stage_x).  It is loaded just before the z_1 wait and staged
    // after the h_1 / dZ_1 pass; the loads issue together and only 8 registers stay live (a float prefetch at the
    // start of the tile was spilled load by load, each spill store waiting for its load)
    uint32_t xpk[kK0 / 2];
    auto load_xpk = [&](int64_t tile) {
      const int64_t row = tile * kTileM + r;
      float v[kK0];
#pragma unroll
      for (int j = 0; j < kK0; ++j)
        v[j] = (grp == 0 && j < d && row < p.n && tile < p.num_tiles) ? __ldg(p.x + row * d + j) : 0.f;
#pragma unroll
      for (int k = 0; k < kK0 / 2; ++k) xpk[k] = pack_bf16x2(v[2 * k], v[2 * k + 1]);
    };
    auto stage_xpk = [&]() {
      if (grp == 0) {
        *reinterpret_cast<uint4*>(bufH + r * 16) = make_uint4(xpk[0], xpk[1], xpk[2], xpk[3]);
        *reinterpret_cast<uint4*>(bufH + X_LBO + r * 16) = make_uint4(xpk[4], xpk[5], xpk[6], xpk[7]);
      }
    };
    // buffer hand-over with the bulk stores issued by thread 0
    auto acquire = [&]() {  // every earlier bulk store has finished reading its smem source
      if (threadIdx.x == 0) bulk_wait_read0();
      asm volatile("bar.sync 1, 256;" ::: "memory");
    };
    auto store_blob = [&](uint8_t* gdst, const uint8_t* sbuf) {
      fence_proxy_async();
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (threadIdx.x == 0) { bulk_s2g(gdst, sbuf, BLOB); bulk_commit(); }
    };
    // slab-wise staging: `count` finished 64-column slabs (16 KB each, contiguous in the image) leave for the
    // staging area while the epilogue works on the next ones, so the buffer hand-over waits stay short
    auto store_slabs = [&](uint8_t* gdst, const uint8_t* sbuf, int s0, int count, uint8_t* gdst2, const uint8_t* sbuf2) {
      fence_proxy_async();
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (threadIdx.x == 0) {
        bulk_s2g(gdst + (size_t)s0 * kActSlab, sbuf + (size_t)s0 * kActSlab, (uint32_t)count * kActSlab);
        if (gdst2) bulk_s2g(gdst2 + (size_t)s0 * kActSlab, sbuf2 + (size_t)s0 * kActSlab, (uint32_t)count * kActSlab);
        bulk_commit();
      }
    };
    auto wait_A = [&]() { mbar_wait(accA_ready, phA); phA ^= 1; tc_fence_after(); };
    auto wait_B = [&]() { mbar_wait(accB_ready, phB); phB ^= 1; tc_fence_after(); };
    auto arrive_a = [&]() { tc_fence_before(); fence_proxy_async(); mbar_arrive_warp(a_ready); };
    auto arrive_slab = [&](int s) { tc_fence_before(); fence_proxy_async(); mbar_arrive_warp(&slab_ready[s]); };
    // h = [old +] act(z + b) for one 8-column group (packed-pair math: two columns per instruction); returns the
    // predicates z + b > 0 (ReLU: act'(z + b)) as bits 0..7
    auto h_chunk8 = [&](const uint32_t* z, const float* bl, uint8_t* dst, bool res) -> uint32_t {
      const float4 b0 = *reinterpret_cast<const float4*>(bl);
      const float4 b1 = *reinterpret_cast<const float4*>(bl + 4);
      const uint64_t bb[4] = {f32x2(b0.x, b0.y), f32x2(b0.z, b0.w), f32x2(b1.x, b1.y), f32x2(b1.z, b1.w)};
      uint4 old = make_uint4(0u, 0u, 0u, 0u);
      if (res) old = *reinterpret_cast<const uint4*>(dst);
      const uint32_t oo[4] = {old.x, old.y, old.z, old.w};
      uint32_t pk[4], m = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint64_t zb = fadd2(f32x2(__uint_as_float(z[2 * j]), __uint_as_float(z[2 * j + 1])), bb[j]);
        float lo, hi;
        f32x2_unpack(zb, lo, hi);
        m |= (lo > 0.f ? 1u : 0u) << (2 * j) | (hi > 0.f ? 1u : 0u) << (2 * j + 1);
        uint64_t o = act2<ACT>(zb);
        if (res) o = fadd2(o, bf16x2_to_f32x2(oo[j]));
        pk[j] = pack_bf16x2_pair(o);
      }
      *reinterpret_cast<uint4*>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      return m;
    };
    // ReLU: dZ = dH * act'(z + b) for one 8-column group, act' given as the bits 0..7 of m: the same product as dz_chunk8
    auto dzm_chunk8 = [&](const uint32_t* g, uint32_t m, uint8_t* dst) {
      uint32_t pk[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint64_t da = f32x2((m >> (2 * j)) & 1u ? 1.f : 0.f, (m >> (2 * j + 1)) & 1u ? 1.f : 0.f);
        pk[j] = pack_bf16x2_pair(fmul2(f32x2(__uint_as_float(g[2 * j]), __uint_as_float(g[2 * j + 1])), da));
      }
      *reinterpret_cast<uint4*>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    };
    // h = act(z + b) -> hdst and act'(z + b) -> dadst (both bf16) for one 8-column group
    auto hda_chunk8 = [&](const uint32_t* z, const float* bl, uint8_t* hdst, uint8_t* dadst) {
      const float4 b0 = *reinterpret_cast<const float4*>(bl);
      const float4 b1 = *reinterpret_cast<const float4*>(bl + 4);
      const uint64_t bb[4] = {f32x2(b0.x, b0.y), f32x2(b0.z, b0.w), f32x2(b1.x, b1.y), f32x2(b1.z, b1.w)};
      uint32_t ph[4], pd[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint64_t a, da;
        act_and_grad2<ACT>(fadd2(f32x2(__uint_as_float(z[2 * j]), __uint_as_float(z[2 * j + 1])), bb[j]), a, da);
        ph[j] = pack_bf16x2_pair(a);
        pd[j] = pack_bf16x2_pair(da);
      }
      *reinterpret_cast<uint4*>(hdst) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
      *reinterpret_cast<uint4*>(dadst) = make_uint4(pd[0], pd[1], pd[2], pd[3]);
    };
    // dZ = dH * act'(z + b) for one 8-column group
    auto dz_chunk8 = [&](const uint32_t* z, const uint32_t* g, const float* bl, uint8_t* dst) {
      const float4 b0 = *reinterpret_cast<const float4*>(bl);
      const float4 b1 = *reinterpret_cast<const float4*>(bl + 4);
      const uint64_t bb[4] = {f32x2(b0.x, b0.y), f32x2(b0.z, b0.w), f32x2(b1.x, b1.y), f32x2(b1.z, b1.w)};
      uint32_t pk[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint64_t a, da;
        act_and_grad2<ACT>(fadd2(f32x2(__uint_as_float(z[2 * j]), __uint_as_float(z[2 * j + 1])), bb[j]), a, da);
        pk[j] = pack_bf16x2_pair(fmul2(f32x2(__uint_as_float(g[2 * j]), __uint_as_float(g[2 * j + 1])), da));
      }
      *reinterpret_cast<uint4*>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    };
    // both at once (the activation and its derivative share their transcendental)
    auto hdz_chunk8 = [&](const uint32_t* z, const uint32_t* g, const float* bl, uint8_t* hdst, uint8_t* gdst, bool res) {
      const float4 b0 = *reinterpret_cast<const float4*>(bl);
      const float4 b1 = *reinterpret_cast<const float4*>(bl + 4);
      const uint64_t bb[4] = {f32x2(b0.x, b0.y), f32x2(b0.z, b0.w), f32x2(b1.x, b1.y), f32x2(b1.z, b1.w)};
      uint4 old = make_uint4(0u, 0u, 0u, 0u);
      if (res) old = *reinterpret_cast<const uint4*>(hdst);
      const uint32_t oo[4] = {old.x, old.y, old.z, old.w};
      uint32_t ph[4], pg[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint64_t a, da;
        act_and_grad2<ACT>(fadd2(f32x2(__uint_as_float(z[2 * j]), __uint_as_float(z[2 * j + 1])), bb[j]), a, da);
        if (res) a = fadd2(a, bf16x2_to_f32x2(oo[j]));
        ph[j] = pack_bf16x2_pair(a);
        pg[j] = pack_bf16x2_pair(fmul2(f32x2(__uint_as_float(g[2 * j]), __uint_as_float(g[2 * j + 1])), da));
      }
      *reinterpret_cast<uint4*>(hdst) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
      *reinterpret_cast<uint4*>(gdst) = make_uint4(pg[0], pg[1], pg[2], pg[3]);
    };

    if (mask0) load_xpk(blockIdx.x);
    else load_x(blockIdx.x);
    int tn = 0;
    const bool tr0 = threadIdx.x == 0;
#define TRE(id) do { if (tr0) trace_b(p.trace, 0, tn, id); } while (0)
    uint32_t accX = ACC_A;  // pipe: the accumulator of z_0 and dH_0 in this tile (the other one, Y, holds z_1)
    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int64_t r0 = tile * kTileM;
      const int64_t row = r0 + r;
      const uint32_t accY = ACC_A + ACC_B - accX;
      // layer-0 act' bits of this thread's chunks grp, grp + 2, ... in order (mask0; bit j of an entry = column j)
      uint32_t mk[NCHUNK / 2];
      if (!mask0) {
#pragma unroll
        for (int j = 0; j < kK0; ++j) xcur[j] = xnext[j];
      }
      TRE(0);
      if (!mask0 || tile == blockIdx.x) {
        // bufH is free: its last staging store (h_lh) was waited for before dZ_0 / at the previous tile
        if (mask0) stage_xpk();
        else stage_x(xcur);
        arrive_a();     // (mask0: staged after the previous tile's h_1 / dZ_1 pass)
      }
      TRE(2);
      if (!mask0) load_x(tile + gridDim.x);
      // set of this thread's row (for the pooled-gradient scatter), precomputed; virtual-row mode: the row's
      // pooled gradient itself
      const int64_t myset = (!vmax && row < p.n) ? (int64_t)__ldg(p.row_set + row) : -1;
      const float scale = (!vmax && row < p.n) ? __ldg(p.row_scale + row) : 0.f;
      float gs = (vmax && !mask0) ? ((row < p.n) ? __ldg(p.dpooled + row) : 0.f) : 1.f;  // mask0: under the z_1 wait

      // rows f0 .. f0+127 of the final weight image -> bufG (same SW128 layout as an activation image); thread 0, once
      // the previous tile's dZ_0 store has finished reading bufG
      auto load_wrows = [&]() {
        const uint32_t f0 = (uint32_t)(r0 % H);
        mbar_arrive_expect_tx(wf_ready, NSLAB * kActSlab);
        for (int s = 0; s < NSLAB; ++s)
          bulk_g2s(bufG + s * kActSlab, p.wpack + p.w_off[L - 1] + (size_t)s * SLAB + (size_t)f0 * 128, kActSlab, wf_ready);
      };

      // ---- dZ of the final Linear from the pooled gradient (autograd of deep_sets.py:96-106)
      if (!pipe) acquire();  // the previous tile's dZ_0 store has finished reading bufG (pipe: during the h_0 pass)
      TRE(1);
      if (vmax) {
        if (!pipe && threadIdx.x == 0) load_wrows();
      } else if (!bcast3) {
        // the pooled-gradient rows of the sets that intersect this tile are staged one set at a time in a
        // scratch area of bufH (free until the h_0 epilogue) and broadcast from shared memory; a thread
        // writes its row when its own set is staged.  (Per-thread global loads here were latency bound:
        // 6.6k cycles per tile.)
        float* gS = reinterpret_cast<float*>(bufH + 16384);
        int* aS = reinterpret_cast<int*>(bufH + 16384 + H * 4);
        const int64_t last_row = (r0 + kTileM - 1 < p.n - 1) ? r0 + kTileM - 1 : p.n - 1;
        const int64_t b_lo = __ldg(p.row_set + r0), b_hi = __ldg(p.row_set + last_row);
        const bool is_max = (p.pooling == PCC_POOL_MAX) && !bcast;
        if (myset < 0) {  // rows past the last set carry no gradient
          for (int kc = grp; kc < H / 8; kc += 2)
            *reinterpret_cast<uint4*>(bufG + act_chunk_off(r, kc * 8)) = make_uint4(0u, 0u, 0u, 0u);
        }
        for (int64_t b = (b_lo < 0 ? 0 : b_lo); b <= b_hi; ++b) {
          asm volatile("bar.sync 1, 256;" ::: "memory");  // previous set's scratch fully consumed
          for (int i = threadIdx.x; i < H; i += kEpiThreads) {
            gS[i] = __ldg(p.dpooled + b * H + i);
            if (is_max) aS[i] = __ldg(p.argmax + b * H + i);
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (myset == b) {
            const int rr = (int)row;
#pragma unroll 2
            for (int kc = grp; kc < H / 8; kc += 2) {
              const float4 g0 = *reinterpret_cast<const float4*>(gS + kc * 8);
              const float4 g1 = *reinterpret_cast<const float4*>(gS + kc * 8 + 4);
              float o[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
              if (is_max) {
                const int4 a0 = *reinterpret_cast<const int4*>(aS + kc * 8);
                const int4 a1 = *reinterpret_cast<const int4*>(aS + kc * 8 + 4);
                o[0] = a0.x == rr ? o[0] : 0.f; o[1] = a0.y == rr ? o[1] : 0.f; o[2] = a0.z == rr ? o[2] : 0.f;
                o[3] = a0.w == rr ? o[3] : 0.f; o[4] = a1.x == rr ? o[4] : 0.f; o[5] = a1.y == rr ? o[5] : 0.f;
                o[6] = a1.z == rr ? o[6] : 0.f; o[7] = a1.w == rr ? o[7] : 0.f;
              } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] *= scale;
              }
              *reinterpret_cast<uint4*>(bufG + act_chunk_off(r, kc * 8)) =
                  make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
            }
          }
        }
      }
      TRE(3);
      if (!virt) {
        store_blob(p.stage_g[L - 1] + (size_t)tile * BLOB, bufG);
        arrive_a();
      }
      TRE(4);

      // ---- L = 3: h_0 = act(z_0 + b_0) -> bufH (over the x tile), staged; TMEM loads one chunk ahead
      if (bcast3) {
        wait_A();
        TRE(5);
        const float* bl = biasS;
#pragma unroll 1
        for (int c = grp; c < NCHUNK; c += 2) {
          uint32_t z[32];
          tmem_ld32(lane_base + ACC_A + c * 32, z);
          tmem_wait_ld();
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint32_t off = act_chunk_off(r, c * 32 + q * 8);
            hda_chunk8(z + q * 8, bl + c * 32 + q * 8, bufH + off, bufG + off);
          }
          store_slabs(p.stage_h[0] + (size_t)tile * BLOB, bufH, c >> 1, 1, nullptr, nullptr);
        }
        TRE(6);
        arrive_a();
        TRE(7);
      } else if (L == 3) {
        wait_A();
        TRE(5);
        const float* bl = biasS;
        uint32_t va[32], vb[32];
        // one chunk of h_0; mask0 keeps its act' bits
        auto h_chunk32 = [&](const uint32_t (&z)[32], int c) {
          uint32_t m = 0;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            m |= h_chunk8(z + q * 8, bl + c * 32 + q * 8, bufH + act_chunk_off(r, c * 32 + q * 8), false) << (8 * q);
          if (mask0) {
#pragma unroll
            for (int k = 0; k + 1 < NCHUNK / 2; ++k) mk[k] = mk[k + 1];
            mk[NCHUNK / 2 - 1] = m;
          }
        };
        tmem_ld32(lane_base + accX + grp * 32, va);
#pragma unroll 1
        for (int c = grp; c < NCHUNK; c += 4) {
          tmem_wait_ld();
          if (c + 2 < NCHUNK) tmem_ld32(lane_base + accX + (c + 2) * 32, vb);
          h_chunk32(va, c);
          if (pipe) arrive_slab(c >> 1);  // the z_1 MMAs of this K slab can start
          if (c + 2 < NCHUNK) {
            tmem_wait_ld();
            if (c + 4 < NCHUNK) tmem_ld32(lane_base + accX + (c + 4) * 32, va);
            h_chunk32(vb, c + 2);
            if (pipe) arrive_slab((c + 2) >> 1);
          }
          // the two groups together have finished slabs (c - grp) / 2 and + 1
          store_slabs(p.stage_h[0] + (size_t)tile * BLOB, bufH, (c - grp) >> 1, (c + 2 < NCHUNK) ? 2 : 1, nullptr, nullptr);
          // pipe: the dZ_0 store of the previous tile has long drained, so the weight rows that the h_1 / dZ_1 pass
          // reads are fetched here instead of holding up the start of the tile (all but the h_0 store just issued)
          if (pipe && c == grp && threadIdx.x == 0) {
            bulk_wait_read1();
            load_wrows();
          }
        }
        TRE(6);
        if (!pipe) arrive_a();
        if (mask0) {  // needed after the z_1 wait at the earliest
          load_xpk(tile + gridDim.x);
          gs = (row < p.n) ? __ldg(p.dpooled + row) : 0.f;
        }
        TRE(7);
      }

      // ---- one pass over z_lh (accA) and dH_lh (accB): h_lh -> bufH, dZ_lh -> bufG, both staged
      if (!virt) wait_B();
      TRE(8);
      wait_A();
      TRE(9);
      acquire();  // staging stores of h_0 (bufH) and dZ_{L-1} (bufG) have finished reading
      TRE(10);
      if (bcast3) {
        const bool res = (p.res_mask >> lh) & 1;
        const float* bl = biasS + lh * H;
        const float* grow = p.dpooled + (myset < 0 ? 0 : myset) * H;   // G row of this thread's set ([B,H] fp32, L2 resident)
        const float sc = myset < 0 ? 0.f : scale;
        uint32_t gn[32];
        auto load_g = [&](int c, uint32_t (&dst)[32]) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 t4 = __ldg(reinterpret_cast<const float4*>(grow + c * 32) + j);   // raw: scaled at use, so the
            dst[4 * j] = __float_as_uint(t4.x); dst[4 * j + 1] = __float_as_uint(t4.y);    // loads stay in flight
            dst[4 * j + 2] = __float_as_uint(t4.z); dst[4 * j + 3] = __float_as_uint(t4.w);
          }
        };
        load_g(grp, gn);
#pragma unroll 1
        for (int c = grp; c < NCHUNK; c += 2) {
          uint32_t z[32], g[32];
          tmem_ld32(lane_base + ACC_A + c * 32, z);
#pragma unroll
          for (int j = 0; j < 32; ++j) g[j] = __float_as_uint(sc * __uint_as_float(gn[j]));
          if (c + 2 < NCHUNK) load_g(c + 2, gn);     // next chunk's gradient row in flight during this chunk's math
          if (res) tmem_st32(lane_base + ACC_B + c * 32, g);
          tmem_wait_ld();
#pragma unroll
          for (int q = 0; q < 4; ++q)
            dz_chunk8(z + q * 8, g + q * 8, bl + c * 32 + q * 8, bufH + act_chunk_off(r, c * 32 + q * 8));
          // (one 64 KB store per image instead of slab-wise stores was tried: the passes get shorter but the store then
          // competes with the GEMM that reads the same buffer — z_1 wait 2.2k -> 3.7k cycles — and the step got slower)
          store_slabs(p.stage_g[lh] + (size_t)tile * BLOB, bufH, c >> 1, 1, nullptr, nullptr);
        }
        if (res) tmem_wait_st();
      } else if (virt) {
        if (vmax) {
          mbar_wait(wf_ready, wf_phase);
          wf_phase ^= 1;
        }
        const bool res = (p.res_mask >> lh) & 1;
        const float* bl = biasS + lh * H;
        const uint32_t zacc = pipe ? accY : ACC_A, gacc = pipe ? accX : ACC_B;
#pragma unroll 1
        for (int c = grp; c < NCHUNK; c += 2) {
          uint32_t z[32], g[32];
          tmem_ld32(lane_base + zacc + c * 32, z);
          // dH_lh chunk: mode 1: W_{L-1}[f, 32 columns] * dpooled[row]; mode 2: the image built from G (overwritten below)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint4 wv = *reinterpret_cast<const uint4*>(bufG + act_chunk_off(r, c * 32 + q * 8));
            g[q * 8 + 0] = __float_as_uint(gs * bf16_lo(wv.x)); g[q * 8 + 1] = __float_as_uint(gs * bf16_hi(wv.x));
            g[q * 8 + 2] = __float_as_uint(gs * bf16_lo(wv.y)); g[q * 8 + 3] = __float_as_uint(gs * bf16_hi(wv.y));
            g[q * 8 + 4] = __float_as_uint(gs * bf16_lo(wv.z)); g[q * 8 + 5] = __float_as_uint(gs * bf16_hi(wv.z));
            g[q * 8 + 6] = __float_as_uint(gs * bf16_lo(wv.w)); g[q * 8 + 7] = __float_as_uint(gs * bf16_hi(wv.w));
          }
          // ResidualBlock: dH_{lh-1} = dZ_lh W_lh + dH_lh — the dgrad MMA accumulates onto accB, so dH_lh goes there
          if (res) tmem_st32(lane_base + gacc + c * 32, g);
          tmem_wait_ld();
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint32_t off = act_chunk_off(r, c * 32 + q * 8);
            if (bcast) dz_chunk8(z + q * 8, g + q * 8, bl + c * 32 + q * 8, bufG + off);
            else hdz_chunk8(z + q * 8, g + q * 8, bl + c * 32 + q * 8, bufH + off, bufG + off, res);
          }
          if (pipe) {  // the dgrad MMAs of this K slab can start (ResidualBlock: once dH_1 is in X, see the MMA thread)
            if (res) tmem_wait_st();
            arrive_slab(c >> 1);
          }
          if (bcast) store_slabs(p.stage_g[lh] + (size_t)tile * BLOB, bufG, c >> 1, 1, nullptr, nullptr);
          else store_slabs(p.stage_h[lh] + (size_t)tile * BLOB, bufH, c >> 1, 1, p.stage_g[lh] + (size_t)tile * BLOB, bufG);
        }
        if (res) tmem_wait_st();
      } else {
        const bool res = (p.res_mask >> lh) & 1;
        const float* bl = biasS + lh * H;
#pragma unroll 1
        for (int c = grp; c < NCHUNK; c += 2) {
          uint32_t z[32], g[32];
          tmem_ld32(lane_base + ACC_A + c * 32, z);
          tmem_ld32(lane_base + ACC_B + c * 32, g);
          tmem_wait_ld();
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint32_t off = act_chunk_off(r, c * 32 + q * 8);
            hdz_chunk8(z + q * 8, g + q * 8, bl + c * 32 + q * 8, bufH + off, bufG + off, res);
          }
          store_slabs(p.stage_h[lh] + (size_t)tile * BLOB, bufH, c >> 1, 1, p.stage_g[lh] + (size_t)tile * BLOB, bufG);
        }
      }
      TRE(11);
      TRE(12);

      if (L == 3) {
        if (!pipe) arrive_a();  // dZ_1 image complete: the dgrad of layer 1 can start while the staging stores drain
        // h_1 staged out of bufH: its head can take the x tile again.  Slab-wise stores: only the last slab pair can
        // still be in flight; mask0 lets it drain under the dgrad (the x image lies in slab 0, bufG is acquired below)
        if (threadIdx.x == 0) {
          if (mask0) bulk_wait_read1();
          else bulk_wait_read0();
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        TRE(13);
        if (bcast3) {
          // ---- dZ_0 = dH_0 * act'(z_0) with act'(z_0) kept (bf16) in bufG by the h_0 epilogue: in place
          wait_B();
          TRE(14);
          TRE(15);
#pragma unroll 1
          for (int c = grp; c < NCHUNK; c += 2) {
            uint32_t g[32];
            tmem_ld32(lane_base + ACC_B + c * 32, g);
            tmem_wait_ld();
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              uint8_t* dst = bufG + act_chunk_off(r, c * 32 + q * 8);
              const uint4 da = *reinterpret_cast<const uint4*>(dst);
              const uint32_t dd[4] = {da.x, da.y, da.z, da.w};
              uint32_t pk[4];
#pragma unroll
              for (int j = 0; j < 4; ++j)
                pk[j] = pack_bf16x2_pair(fmul2(f32x2(__uint_as_float(g[q * 8 + 2 * j]), __uint_as_float(g[q * 8 + 2 * j + 1])),
                                               bf16x2_to_f32x2(dd[j])));
              *reinterpret_cast<uint4*>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
            store_slabs(p.stage_g[0] + (size_t)tile * BLOB, bufG, c >> 1, 1, nullptr, nullptr);
          }
        } else if (mask0) {
          // the next tile's x -> bufH head: its z_0 GEMM (into Y) runs under this pass
          if (tile + gridDim.x < p.num_tiles) {
            stage_xpk();
            arrive_a();
          }
          // ---- dZ_0 = dH_0 * act'(z_0 + b_0) with act' from the h_0 pass's bits -> bufG (the dgrad has read it), staged
          wait_B();
          TRE(14);
          acquire();  // the last dZ_1 store has finished reading bufG
          TRE(15);
#pragma unroll 1
          for (int c = grp; c < NCHUNK; c += 2) {
            uint32_t g[32];
            tmem_ld32(lane_base + accX + c * 32, g);
            const uint32_t m = mk[0];
#pragma unroll
            for (int k = 0; k + 1 < NCHUNK / 2; ++k) mk[k] = mk[k + 1];
            tmem_wait_ld();
#pragma unroll
            for (int q = 0; q < 4; ++q) dzm_chunk8(g + q * 8, m >> (8 * q), bufG + act_chunk_off(r, c * 32 + q * 8));
            store_slabs(p.stage_g[0] + (size_t)tile * BLOB, bufG, c >> 1, 1, nullptr, nullptr);
          }
        } else {
          stage_x(xcur);
          arrive_a();
          // ---- dZ_0 = dH_0 * act'(z_0 + b_0) -> bufG, staged (pipe: z_0 recomputed into Y, dH_0 in X)
          wait_B();
          wait_A();
          TRE(14);
          acquire();
          TRE(15);
          const float* bl = biasS;
          const uint32_t zacc = pipe ? accY : ACC_A, gacc = pipe ? accX : ACC_B;
#pragma unroll 1
          for (int c = grp; c < NCHUNK; c += 2) {
            uint32_t z[32], g[32];
            tmem_ld32(lane_base + zacc + c * 32, z);
            tmem_ld32(lane_base + gacc + c * 32, g);
            tmem_wait_ld();
#pragma unroll
            for (int q = 0; q < 4; ++q)
              dz_chunk8(z + q * 8, g + q * 8, bl + c * 32 + q * 8, bufG + act_chunk_off(r, c * 32 + q * 8));
            store_slabs(p.stage_g[0] + (size_t)tile * BLOB, bufG, c >> 1, 1, nullptr, nullptr);
          }
        }
        TRE(16);
        TRE(17);
      }
      if (pipe) accX = accY;
    }
#undef TRE
    if (threadIdx.x == 0) bulk_wait0();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc<512>(tmem);
}

// ====================================================================== K2: wgrad
// staged images travel through the ring as HALF images (64 of a tile's 128 rows = 4 of the 8 K steps): six 32 KB
// slots instead of three 64 KB ones keep the same bytes in shared memory but let the loads of the next one and a
// half tiles overlap the MMAs of the current half instead of waiting for a whole image to drain
constexpr int kSlots = 6;

// Work split of the wgrad kernel.  Each CTA runs two jobs: (0) ONE of the H x H layers (layers 1..L-1
// are dealt round-robin over the CTAs) on every members-th tile, (1) layer 0 (K = 16) on every grid-th
// tile.  A CTA therefore flushes one big partial instead of one per layer, and the partial count per
// big layer is grid / (L-1).
struct WgradJob {
  int layer;
  int64_t first, stride;
  int slot;  // index of this CTA's partial inside the layer's partial array
};
// nbig = number of H x H layers handled as GEMM jobs: layers 1 .. nbig (L-1, or L-2 in virtual-row mode)
__host__ __device__ inline int wgrad_members(int grid, int nbig, int layer) {  // CTAs that work on `layer`
  if (layer == 0) return grid;
  return (grid - (layer - 1) + nbig - 1) / nbig;
}
__device__ inline WgradJob wgrad_job(int j, int cta, int grid, int nbig) {
  WgradJob w;
  if (j == 0) {
    w.layer = 1 + cta % nbig;
    w.first = cta / nbig;
    w.stride = wgrad_members(grid, nbig, w.layer);
    w.slot = cta / nbig;
  } else {
    w.layer = 0; w.first = cta; w.stride = grid; w.slot = cta;
  }
  return w;
}

// Tiles are consumed in DESCENDING order: the chain kernel wrote the images in ascending order just before, so the
// high tiles are the ones still in L2 (reading upwards starts with the evicted ones and pushes the rest out).
__device__ __forceinline__ int64_t wgrad_last_tile(const WgradJob& jb, int64_t num_tiles) {
  if (jb.first >= num_tiles) return jb.first - jb.stride;  // no tile: the loop condition fails at once
  return jb.first + (num_tiles - 1 - jb.first) / jb.stride * jb.stride;
}

template <int H>
__global__ void __launch_bounds__(kThreads, 1) phi_wgrad_kernel(const BwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr uint32_t BLOB = kTileM * H * 2;
  constexpr uint32_t HBLOB = BLOB / 2;       // half image: rows [64 hf, +64) of every 64-column slab, packed
  constexpr uint32_t HSLAB = kActSlab / 2;   // 64 rows x 128 B
  constexpr int NSL = H / 64;                // slabs per image
  constexpr uint32_t XBLOB = kTileM * kK0 * 2;
  constexpr int HALVES = H / 128;
  constexpr int CH = H / 8;            // 16-byte feature chunks per image row
  constexpr int CPW = CH / kEpiWarps;  // chunks per epilogue warp for the db column sums
  uint8_t* slots = smem;                                   // kSlots half images (1024-aligned)
  uint8_t* bufX = smem + kSlots * HBLOB;                   // 2 x-images (tile parity)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kSlots * HBLOB + 2 * XBLOB);
  uint64_t* full = bars;                       // [kSlots]
  uint64_t* empty = bars + kSlots;             // [kSlots] count 1 (MMA commit) + 256 (epilogue readers)
  uint64_t* x_full = bars + 2 * kSlots;        // [2] count 256
  uint64_t* x_empty = bars + 2 * kSlots + 2;   // [2] count 1
  uint64_t* acc_ready = bars + 2 * kSlots + 4;
  uint64_t* acc_free = bars + 2 * kSlots + 5;  // count 256
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kSlots + 6);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j0 = (p.nbig == 0) ? 1 : 0;  // no H x H GEMM job (one hidden layer in virtual-row mode): layer 0 only
  if (threadIdx.x == 0) {
    for (int i = 0; i < kSlots; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1 + kEpiWarps); }
    for (int i = 0; i < 2; ++i) { mbar_init(&x_full[i], kEpiWarps); mbar_init(&x_empty[i], 1); }
    mbar_init(acc_ready, 1);
    mbar_init(acc_free, kEpiWarps);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_wait();  // barriers and TMEM are set up while the predecessor drains; the images below are its output

  if (warp == kProdWarp) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      auto push = [&](const uint8_t* src, int hf) {
        mbar_wait(&empty[stage], phase ^ 1);
        mbar_arrive_expect_tx(&full[stage], HBLOB);
        for (int sl = 0; sl < NSL; ++sl)
          bulk_g2s(slots + stage * HBLOB + sl * HSLAB, src + (size_t)sl * kActSlab + (size_t)hf * HSLAB, HSLAB, &full[stage]);
        if (++stage == kSlots) { stage = 0; phase ^= 1; }
      };
      for (int j = 1; j >= j0; --j) {  // layer 0 first: its accumulator flush (32 columns) is the short one to wait for
        const WgradJob jb = wgrad_job(j, blockIdx.x, gridDim.x, p.nbig);
        const int l = jb.layer;
        for (int64_t tile = wgrad_last_tile(jb, p.num_tiles); tile >= jb.first; tile -= jb.stride) {
          for (int hf = 0; hf < 2; ++hf) {
            push(p.stage_g[l] + (size_t)tile * BLOB, hf);
            if (l >= 1) push(p.stage_h[l - 1] + (size_t)tile * BLOB, hf);
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, xpar = 0, xphase = 0 /* bit i = phase of x buffer i */, free_phase = 0;
      const uint32_t s_base = smem_u32(slots), x_base = smem_u32(bufX);
      for (int j = 1; j >= j0; --j) {  // layer 0 first: its accumulator flush (32 columns) is the short one to wait for
        const WgradJob jb = wgrad_job(j, blockIdx.x, gridDim.x, p.nbig);
        const int l = jb.layer;
        const int Np = (l == 0) ? kK0 : H;
        const uint32_t idesc = make_idesc_bf16(128, Np, 1, 1);
        if (j < 1) { mbar_wait(acc_free, free_phase); free_phase ^= 1; tc_fence_after(); }
        bool first = true;
        for (int64_t tile = wgrad_last_tile(jb, p.num_tiles); tile >= jb.first; tile -= jb.stride) {
          uint32_t x_addr = 0;
          if (l == 0) {
            mbar_wait(&x_full[xpar], (xphase >> xpar) & 1);
            xphase ^= 1u << xpar;
            x_addr = x_base + xpar * XBLOB;
          }
          for (int hf = 0; hf < 2; ++hf) {
            const uint32_t g_stage = stage;
            mbar_wait(&full[stage], phase);
            if (++stage == kSlots) { stage = 0; phase ^= 1; }
            uint32_t in_addr = 0, in_stage = 0;
            if (l >= 1) {
              in_stage = stage;
              mbar_wait(&full[stage], phase);
              if (++stage == kSlots) { stage = 0; phase ^= 1; }
              in_addr = s_base + in_stage * HBLOB;
            }
            tc_fence_after();
            const uint32_t g_addr = s_base + g_stage * HBLOB;
            // D[out(128 per half), in] += dZ^T (MN-major view of the dZ half image) * In (MN-major view)
#pragma unroll
            for (int o = 0; o < HALVES; ++o)
              for (int ks = 0; ks < kTileM / 32; ++ks) {
                const uint64_t a_desc = make_smem_desc_sw128_mn(g_addr + o * (2 * HSLAB) + ks * 2048, HSLAB);
                const uint64_t b_desc = (l >= 1) ? make_smem_desc_sw128_mn(in_addr + ks * 2048, HSLAB)
                                                 : make_smem_desc(x_addr + (hf * (kTileM / 32) + ks) * 256, 128, kTileM * 16);
                umma_bf16(tmem + o * Np, a_desc, b_desc, idesc, !(first && hf == 0 && ks == 0));
              }
            umma_commit(&empty[g_stage]);
            if (l >= 1) umma_commit(&empty[in_stage]);
          }
          first = false;
          if (l == 0) { umma_commit(&x_empty[xpar]); xpar ^= 1; }
        }
        umma_commit(acc_ready);
      }
    }
  } else {
    // ===================== epilogue warps: db column sums, x images for layer 0, TMEM flush
    const int quarter = warp & 3, grp = warp >> 2;
    const int r = quarter * 32 + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(quarter * 32) << 16);
    uint32_t stage = 0, phase = 0, xpar = 0, xphase = 0, acc_phase = 0;
    const int d = p.d;
    for (int j = 1; j >= j0; --j) {  // layer 0 first: its accumulator flush (32 columns) is the short one to wait for
      const WgradJob jb = wgrad_job(j, blockIdx.x, gridDim.x, p.nbig);
      const int l = jb.layer;
      const int Np = (l == 0) ? kK0 : H;
      float dbacc[CPW][8];
#pragma unroll
      for (int i = 0; i < CPW; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) dbacc[i][j] = 0.f;
      for (int64_t tile = wgrad_last_tile(jb, p.num_tiles); tile >= jb.first; tile -= jb.stride) {
        if (l == 0) {  // x tile -> [2][128][8] bf16 image (group 0 owns the rows)
          mbar_wait(&x_empty[xpar], ((xphase >> xpar) & 1) ^ 1);
          xphase ^= 1u << xpar;
          if (grp == 0) {
            const int64_t row = tile * kTileM + r;
            float xr[kK0];
#pragma unroll
            for (int j = 0; j < kK0; ++j) xr[j] = (j < d && row < p.n) ? __ldg(p.x + row * d + j) : 0.f;
            uint8_t* xb = bufX + xpar * XBLOB;
            *reinterpret_cast<uint4*>(xb + r * 16) = make_uint4(pack_bf16x2(xr[0], xr[1]), pack_bf16x2(xr[2], xr[3]),
                                                                pack_bf16x2(xr[4], xr[5]), pack_bf16x2(xr[6], xr[7]));
            *reinterpret_cast<uint4*>(xb + kTileM * 16 + r * 16) =
                make_uint4(pack_bf16x2(xr[8], xr[9]), pack_bf16x2(xr[10], xr[11]), pack_bf16x2(xr[12], xr[13]),
                           pack_bf16x2(xr[14], xr[15]));
          }
          fence_proxy_async();
          mbar_arrive_warp(&x_full[xpar]);
          xpar ^= 1;
        }
        // column sums of the dZ half images: warp w owns chunks w, w+8, ...; lane owns rows lane, lane+32 of the half
        for (int hf = 0; hf < 2; ++hf) {
          mbar_wait(&full[stage], phase);
          const uint8_t* gb = slots + stage * HBLOB;
#pragma unroll
          for (int i = 0; i < CPW; ++i) {
            const int c = warp + kEpiWarps * i;
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
              const int rw = lane + 32 * rr;
              const uint4 u = *reinterpret_cast<const uint4*>(gb + (uint32_t)(c >> 3) * HSLAB + (uint32_t)rw * 128u +
                                                              ((uint32_t)((c & 7) ^ (rw & 7)) << 4));
              dbacc[i][0] += bf16_lo(u.x); dbacc[i][1] += bf16_hi(u.x); dbacc[i][2] += bf16_lo(u.y); dbacc[i][3] += bf16_hi(u.y);
              dbacc[i][4] += bf16_lo(u.z); dbacc[i][5] += bf16_hi(u.z); dbacc[i][6] += bf16_lo(u.w); dbacc[i][7] += bf16_hi(u.w);
            }
          }
          mbar_arrive_warp(&empty[stage]);
          if (++stage == kSlots) { stage = 0; phase ^= 1; }
          if (l >= 1) {  // the input half image is only read by the tensor core; wait for THIS use of the slot
            // to be filled before releasing it, otherwise the arrival could land in the previous phase
            mbar_wait(&full[stage], phase);
            mbar_arrive_warp(&empty[stage]);
            if (++stage == kSlots) { stage = 0; phase ^= 1; }
          }
        }
      }
      // ---- db partial: reduce over lanes, lane 0 writes
      float* pb = p.part_b[l] + (size_t)jb.slot * H;
#pragma unroll
      for (int i = 0; i < CPW; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float s = warp_sum(dbacc[i][j]);
          if (lane == 0) pb[(warp + kEpiWarps * i) * 8 + j] = s;
        }
      // ---- dW partial: TMEM -> global; the two warp groups split the (half, 32-column chunk) items
      mbar_wait(acc_ready, acc_phase);
      acc_phase ^= 1;
      tc_fence_after();
      // partial layout: [k (Np)][row (H)] — thread = row, so every store of a warp is one coalesced 128 B line
      float* pw = p.part_w[l] + (size_t)jb.slot * H * Np;
      const int nchunk = (Np < 32) ? 1 : Np / 32;
      const int ncol = (Np < 32) ? Np : 32;
#pragma unroll 1
      for (int item = grp; item < HALVES * nchunk; item += 2) {
        const int o = item / nchunk, c = item % nchunk;
        uint32_t v[32];
        tmem_ld32(lane_base + o * Np + c * 32, v);
        tmem_wait_ld();
        float* dst = pw + (size_t)(c * 32) * H + (o * 128 + r);
        const bool has_tiles = jb.first < p.num_tiles;  // a CTA without tiles for this job contributes zeros
#pragma unroll
        for (int q = 0; q < 32; ++q)
          if (q < ncol) dst[(size_t)q * H] = has_tiles ? __uint_as_float(v[q]) : 0.f;
      }
      tc_fence_before();
      mbar_arrive_warp(acc_free);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc<512>(tmem);
}

// Virtual-row mode: weight gradient of the final Linear without a GEMM.  dZ_{L-1}[b*H + f] = dpooled[b, f] * e_f, so
//   dW_{L-1}[f, :] = sum_b dpooled[b, f] * h_lh[b*H + f, :]      db_{L-1}[f] = sum_b dpooled[b, f]
// One CTA per output feature f; thread = (8-column chunk, b group); the h rows come from the staged SW128 images.
constexpr int kFwvThreads = 512;
template <int H>
__global__ void __launch_bounds__(kFwvThreads) final_wgrad_virtual_kernel(const uint8_t* __restrict__ stage_h,
                                                                  const float* __restrict__ dpooled, int64_t B,
                                                                  float* __restrict__ dw, float* __restrict__ db) {
  pdl_enter();
  constexpr int CH = H / 8, NG = kFwvThreads / CH;
  constexpr uint32_t BLOB = kTileM * H * 2;
  __shared__ float red[NG][CH][8];
  __shared__ float redb[NG];
  const int f = blockIdx.x;
  const int kc = threadIdx.x % CH, bg = threadIdx.x / CH;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  float gsum = 0.f;
  // 8 independent (gradient, row chunk) loads in flight per thread: the loop is latency bound
  // highest sets first: their rows were written last by the chain kernel and are the likeliest to still be in L2
  for (int64_t b0 = (B - 1) / (8 * NG) * (8 * NG) + bg; b0 >= 0; b0 -= 8 * NG) {
    float g[8];
    uint4 u[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int64_t b = b0 + (int64_t)i * NG;
      const int64_t row = (b < B ? b : 0) * H + f;
      g[i] = (b < B) ? __ldg(dpooled + row) : 0.f;
      u[i] = __ldg(reinterpret_cast<const uint4*>(stage_h + (size_t)(row / kTileM) * BLOB +
                                                  act_chunk_off((int)(row % kTileM), kc * 8)));
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      acc[0] = fmaf(g[i], bf16_lo(u[i].x), acc[0]); acc[1] = fmaf(g[i], bf16_hi(u[i].x), acc[1]);
      acc[2] = fmaf(g[i], bf16_lo(u[i].y), acc[2]); acc[3] = fmaf(g[i], bf16_hi(u[i].y), acc[3]);
      acc[4] = fmaf(g[i], bf16_lo(u[i].z), acc[4]); acc[5] = fmaf(g[i], bf16_hi(u[i].z), acc[5]);
      acc[6] = fmaf(g[i], bf16_lo(u[i].w), acc[6]); acc[7] = fmaf(g[i], bf16_hi(u[i].w), acc[7]);
      gsum += g[i];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[bg][kc][j] = acc[j];
  if (kc == 0) redb[bg] = gsum;
  __syncthreads();
  if (threadIdx.x < H) {
    const int c = threadIdx.x >> 3, j = threadIdx.x & 7;
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < NG; ++g) s += red[g][c][j];
    dw[(size_t)f * H + threadIdx.x] = s;
  }
  if (threadIdx.x == 0) {
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < NG; ++g) s += redb[g];
    db[f] = s;
  }
}

// sum the per-CTA partials of ALL layers in one launch: dW_l[H, K] (K = real in-features), db_l[H].
// Partials are stored [k][row]; one thread owns 4 consecutive rows of one k (float4 loads), the 8 thread
// groups of a block split the partial range and combine through shared memory.
struct ReduceParams {
  const float* part_w[kMaxLayers];
  const float* part_b[kMaxLayers];
  float* dw[kMaxLayers];
  float* db[kMaxLayers];
  int Kp[kMaxLayers], K[kMaxLayers], np[kMaxLayers];
  int vec_begin[kMaxLayers + 1];  // first float4 work item of each layer: (Kp + 1) * H / 4 items (last k = bias)
  int L, H;
};
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const ReduceParams p) {
  pdl_enter();
  __shared__ float4 red[8][32];
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int item = blockIdx.x * 32 + lane;
  int l = 0;
  while (l + 1 < p.L && item >= p.vec_begin[l + 1]) ++l;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  const int local = item - p.vec_begin[l];
  const int vec_per_k = p.H / 4;
  const int k = local / vec_per_k, row4 = (local % vec_per_k) * 4;
  const bool valid = item < p.vec_begin[p.L];
  const bool is_bias = valid && (k == p.Kp[l]);
  if (valid) {
    const float* src = is_bias ? p.part_b[l] + row4 : p.part_w[l] + (size_t)k * p.H + row4;
    const size_t stride = is_bias ? (size_t)p.H : (size_t)p.H * p.Kp[l];
    for (int c = g; c < p.np[l]; c += 8) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(src + c * stride));
      s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
    }
  }
  red[g][lane] = s;
  __syncthreads();
  if (g == 0 && valid) {
    float4 t = red[0][lane];
#pragma unroll
    for (int j = 1; j < 8; ++j) { t.x += red[j][lane].x; t.y += red[j][lane].y; t.z += red[j][lane].z; t.w += red[j][lane].w; }
    if (is_bias) {
      *reinterpret_cast<float4*>(p.db[l] + row4) = t;
    } else if (k < p.K[l]) {
      float* dst = p.dw[l] + (size_t)row4 * p.K[l] + k;
      dst[0] = t.x; dst[(size_t)p.K[l]] = t.y; dst[2 * (size_t)p.K[l]] = t.z; dst[3 * (size_t)p.K[l]] = t.w;
    }
  }
}

__global__ void zero_f32_kernel_b(float* p, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0.f;
}

// ------------------------------------------------------------------ host side
struct BwdWs {
  int64_t stage_h[kMaxLayers], stage_g[kMaxLayers], part_w[kMaxLayers], part_b[kMaxLayers];
  int64_t row_set, row_scale, gmat, bscale;
  int64_t total;
  int grid;
};
constexpr int kGridCap = 160;  // upper bound on persistent CTAs used for sizing the partial buffers
static BwdWs bwd_ws(const pcc_phi_desc* d, int64_t n, int sms, int64_t B = 0) {
  BwdWs w{};
  const int H = d->hidden, L = d->n_layers;
  const int64_t tiles = cdiv(n, kTileM);
  if (sms > kGridCap) sms = kGridCap;
  w.grid = (int)(tiles < sms ? tiles : sms);
  if (w.grid < L - 1) w.grid = L - 1;  // the wgrad kernel deals the H x H layers round-robin over the CTAs
  if (w.grid < 1) w.grid = 1;
  int64_t o = 0;
  auto take = [&](int64_t bytes) { int64_t at = o; o = (o + bytes + 255) / 256 * 256; return at; };
  const int64_t blob = (int64_t)kTileM * H * 2;
  for (int l = 0; l <= L - 2; ++l) w.stage_h[l] = take(tiles * blob);
  for (int l = 0; l < L; ++l) w.stage_g[l] = take(tiles * blob);
  for (int l = 0; l < L; ++l) {
    w.part_w[l] = take((int64_t)kGridCap * H * ((l == 0) ? kK0 : H) * 4);
    w.part_b[l] = take((int64_t)kGridCap * H * 4);
  }
  w.row_set = take(n * 4);
  w.row_scale = take(n * 4);
  w.gmat = take(B * H * 4);
  w.bscale = take(B * 4);
  w.total = o;
  return w;
}

int64_t phi_bwd_workspace_bytes(const pcc_phi_desc* d, int64_t n, int64_t B) { return bwd_ws(d, n, kGridCap, B).total; }

// bscale[b] = n_b * rs_b (sqrt(n) for sum pooling, 1 for mean): the factor of the final bias inside pooled[b]
__global__ void set_bscale_kernel(const int64_t* __restrict__ offsets, int64_t B, int pooling, float* __restrict__ bscale) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float n = (float)(offsets[b + 1] - offsets[b]);
  bscale[b] = (n <= 0.f) ? 0.f : (pooling == PCC_POOL_SUM ? sqrtf(n) : 1.f);
}

static int g_bwd_pipe = 1;  // pcc_debug_set_bwd_pipe: 0 runs max pooling with two hidden layers on the serial schedule

template <int H, int ACT>
static int launch_chain(const BwdParams& p, int grid, cudaStream_t st) {
  const BwdSmem lay = bwd_smem(H, p.L);
  auto kern = (p.virt == 1 && p.L == 3 && g_bwd_pipe) ? phi_bwd_chain_kernel<H, ACT, true>
                                                       : phi_bwd_chain_kernel<H, ACT, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.total);
  if (e != cudaSuccess) return fail("pcc_deepsets_phi_pool_bwd", cudaGetErrorString(e));
  {
    ProfScope prof(1, st);
    launch_dep(kern, dim3(grid), dim3(kThreads), lay.total, st, p);
  }
  return 0;
}
template <int H>
static int launch_wgrad(const BwdParams& p, int grid, cudaStream_t st) {
  const int smem_bytes = kSlots * (kTileM * H * 2 / 2) + 2 * kTileM * kK0 * 2 + 256;
  auto kern = phi_wgrad_kernel<H>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
  if (e != cudaSuccess) return fail("pcc_deepsets_phi_pool_bwd", cudaGetErrorString(e));
  {
    ProfScope prof(2, st);
    launch_dep(kern, dim3(grid), dim3(kThreads), smem_bytes, st, p);
  }
  return 0;
}

}  // namespace pcc

using namespace pcc;

extern "C" int pcc_debug_set_bwd_pipe(int on) {
  pcc::g_bwd_pipe = on ? 1 : 0;
  return 0;
}

extern "C" int pcc_deepsets_phi_pool_bwd(const pcc_phi_desc* d, const float* x, const int64_t* offsets, int64_t n,
                                         int64_t B, const float* dpooled, const int32_t* argmax, float* const* dw,
                                         float* const* db, void* ws, const void* wpack, int device, void* stream) {
  PCC_ENTER(device);
  if (check_phi_desc(d, __func__) != 0) return -1;
  cudaStream_t st = (cudaStream_t)stream;
  const int H = d->hidden, L = d->n_layers;
  // max pooling with argmax == NULL: the caller passes the B*H argmax rows themselves (row b*H + f = argmax row
  // of (b, f)); offsets are not read
  const bool virt = d->pooling == PCC_POOL_MAX && argmax == nullptr;
  PCC_REQUIRE(!virt || n == B * H, "max pooling without argmax: x must hold the B*H gathered argmax rows");
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  const BwdWs wl = bwd_ws(d, n, sms, B);
  uint8_t* wsb = (uint8_t*)ws;
  const int64_t tiles = cdiv(n, kTileM);
  // sum / mean pooling with the aux buffer of the forward (argmax slot = ph [B, H] fp32): commuted final Linear
  const bool bcast = d->pooling != PCC_POOL_MAX && argmax != nullptr;
  if (tiles == 0) {
    for (int l = 0; l < L; ++l) {
      const int64_t cnt = (int64_t)H * (l == 0 ? d->input_dim : H);
      PCC_K(zero_f32_kernel_b)<<<(unsigned)cdiv(cnt, 256), 256, 0, st>>>(dw[l], cnt);
      PCC_K(zero_f32_kernel_b)<<<(unsigned)cdiv(H, 256), 256, 0, st>>>(db[l], H);
    }
    return check_launch(__func__);
  }

  PCC_REQUIRE(wpack != nullptr, "packed weight images of the forward pass required");
  const PackLayout pl = pack_layout(L, H);

  BwdParams p{};
  p.x = x; p.offsets = offsets; p.n = n; p.B = B; p.num_tiles = tiles;
  p.d = d->input_dim; p.L = L; p.pooling = d->pooling; p.res_mask = d->residual_mask;
  p.wpack = (const uint8_t*)wpack; p.dpooled = dpooled; p.argmax = argmax;
  for (int l = 0; l < L; ++l) {
    p.w_off[l] = pl.w_off[l]; p.wt_off[l] = pl.wt_off[l]; p.bias[l] = d->b[l];
    p.stage_g[l] = wsb + wl.stage_g[l];
    if (l <= L - 2) p.stage_h[l] = wsb + wl.stage_h[l];
    p.part_w[l] = (float*)(wsb + wl.part_w[l]);
    p.part_b[l] = (float*)(wsb + wl.part_b[l]);
  }
  p.trace = (long long*)debug_trace_buffer();
  p.row_set = (const int32_t*)(wsb + wl.row_set);
  p.row_scale = (const float*)(wsb + wl.row_scale);
  p.virt = virt ? 1 : (bcast ? 2 : 0);
  p.nbig = (virt || bcast) ? L - 2 : L - 1;
  if (bcast) {
    // dW_{L-1} = dpooled^T ph, db_{L-1} = sum_b bscale_b dpooled[b], G = dpooled W_{L-1}: three [B, H]-sized products
    float* bscale = (float*)(wsb + wl.bscale);
    float* G = (float*)(wsb + wl.gmat);
    const float* ph = reinterpret_cast<const float*>(argmax);
    PCC_K(set_bscale_kernel)<<<(unsigned)cdiv(B, 256), 256, 0, st>>>(offsets, B, d->pooling, bscale);
    HeadTileParams hp{};
    hp.act = PCC_ACT_RELU;
    HeadTileProb& pw = hp.prob[0];
    pw.A = HeadOperand{dpooled, nullptr, 1, H, 0, 0, 0};
    pw.B = HeadOperand{ph, nullptr, 1, H, 0, 0, 0};
    pw.I = H; pw.J = H; pw.KK = (int)B;
    pw.C = dw[L - 1]; pw.ldc = H; pw.colsum = db[L - 1]; pw.colsum_w = bscale;
    head_set_tiles(pw);
    HeadTileProb& pg = hp.prob[1];
    pg.A = HeadOperand{dpooled, nullptr, H, 1, 0, 0, 0};
    pg.B = HeadOperand{d->w[L - 1], nullptr, 1, H, 0, 0, 0};
    pg.I = (int)B; pg.J = H; pg.KK = H;
    pg.C = G; pg.ldc = H;
    head_set_tiles(pg);
    launch_head_tiles(hp, pw.tiles + pg.tiles, st);
    p.dpooled = G;
    p.argmax = nullptr;
  }
  if (!virt)  // (also in mode 2: row -> set and pooling scale)
    PCC_K(seg_prep_kernel)<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(offsets, n, B, tiles, d->pooling, nullptr,
                                                                  (int32_t*)(wsb + wl.row_set), (float*)(wsb + wl.row_scale));
  int rc = 0;
#define PCC_DISPATCH(HH)                                                                 \
  switch (d->act) {                                                                      \
    case PCC_ACT_RELU: rc = launch_chain<HH, PCC_ACT_RELU>(p, wl.grid, st); break;       \
    case PCC_ACT_GELU: rc = launch_chain<HH, PCC_ACT_GELU>(p, wl.grid, st); break;       \
    default: rc = launch_chain<HH, PCC_ACT_SILU>(p, wl.grid, st); break;                 \
  }
  if (H == 256) { PCC_DISPATCH(256) } else { PCC_DISPATCH(128) }
#undef PCC_DISPATCH
  if (rc != 0) return rc;
  if (virt) {  // final Linear: scaled row sums instead of a GEMM; right after the chain, while its h images are in L2
    auto fk = (H == 256) ? final_wgrad_virtual_kernel<256> : final_wgrad_virtual_kernel<128>;
    launch_dep(fk, dim3(H), dim3(kFwvThreads), 0, st, p.stage_h[L - 2], dpooled, B, dw[L - 1], db[L - 1]);
  }
  rc = (H == 256) ? launch_wgrad<256>(p, wl.grid, st) : launch_wgrad<128>(p, wl.grid, st);
  if (rc != 0) return rc;
  ReduceParams rp{};
  const int Lr = (virt || bcast) ? L - 1 : L;  // layers whose per-CTA partials are reduced
  rp.L = Lr; rp.H = H;
  int items = 0;
  for (int l = 0; l < Lr; ++l) {
    rp.part_w[l] = p.part_w[l]; rp.part_b[l] = p.part_b[l]; rp.dw[l] = dw[l]; rp.db[l] = db[l];
    rp.K[l] = (l == 0) ? d->input_dim : H;
    rp.Kp[l] = (l == 0) ? kK0 : H;
    rp.np[l] = wgrad_members(wl.grid, p.nbig, l);
    rp.vec_begin[l] = items;
    items += (rp.Kp[l] + 1) * (H / 4);
  }
  rp.vec_begin[Lr] = items;
  launch_dep(wgrad_reduce_kernel, dim3((unsigned)cdiv(items, 32)), dim3(256), 0, st, rp);
  return check_launch(__func__);
}
