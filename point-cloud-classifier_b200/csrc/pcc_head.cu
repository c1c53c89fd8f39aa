// rho head (set encoder): [Linear + act] x (0..3) + Linear, M = batch rows.
//   reference: /root/reference/models/deep_sets.py:112 (self.rho(pooled)) with the layer stack of :59-72
//   (no LayerNorm variant) and its autograd.
// The head is tiny (0.07 GFLOP per train step at the yaml shape), so what matters is the LENGTH of the
// dependent chain, not throughput.  An earlier version ran one CTA per 4 rows through all layers in a
// single launch: every CTA streamed every weight matrix through a latency-bound loop and the weight
// gradients needed ~1M vector atomics (16 us forward, 30 us backward, warm).  Here every layer is ONE
// launch of 32x32 output tiles spread over the whole chip (a 256x256x256 layer = 64 CTAs, K loop of 4
// tiles), with all elementwise work folded into the operand loads:
//   forward  layer l : z_l = f(in) W_l^T + b_l          f = act for l > 0 (input is the saved z_{l-1})
//   backward layer l : dz_l = g_l * act'(z_l) built on load (g_L-1 = dy), and in the SAME launch
//                        dW_l = dz_l^T in_l , db_l = colsum(dz_l)      (tiles over [N_l, K_l])
//                        g_{l-1} = dz_l W_l                            (tiles over [M,   K_l])
// No atomics, no zero-fill launches, bitwise deterministic.
#include "pcc_head.cuh"
#include "pcc_tf32.cuh"

namespace pcc {

constexpr int kHeadMaxDim = 1024;
constexpr int kHeadMaxLayers = 4;
constexpr int kHT = 32;    // output tile edge
constexpr int kHThreads = 256;

// One 32 x 32 output tile per CTA, K consumed in chunks of 256.  The kernel runs once per CTA with 8 warps on an
// otherwise empty SM, so it is bound by dependent-latency chains, not by throughput (tools/head_micro.py: 3.2 us
// fixed + a per-K slope that did not depend on the instruction mix until the chains were broken):
//   * 128-bit operand loads along each operand's contiguous direction, 8 per thread, operand and chunk: a 256-wide
//     layer is ONE round trip, the next chunk's loads are in flight under the math of the current one;
//   * no transposition: an operand contiguous along kk is staged as [i][kk] (rows of 260 floats), one contiguous
//     along i as [kk][i] (rows of 40 floats) — both conflict free for the float4 stores AND for the k-strided
//     fragment loads; the activation / act' transforms happen in registers on the way;
//   * 8 warps, one m16n8 output tile each, 3xTF32 mma.sync (x = hi + lo, a b ~ a_hi b_hi + a_hi b_lo + a_lo b_hi,
//     error ~2^-21 relative: fp32-grade, the parity path depends on it), four K steps unrolled with six
//     independent accumulator fragments so that LDS -> cvt -> HMMA chains of different steps overlap.
constexpr int kHC = 256;            // K chunk
constexpr int kHSk = kHC + 4;       // row of an [i][kk] staged operand
constexpr int kHSi = kHT + 8;       // row of a [kk][i] staged operand
constexpr int kHOp = (kHT * kHSk > kHC * kHSi) ? kHT * kHSk : kHC * kHSi;  // floats per staged operand
constexpr int kHNV = kHT * kHC / 4 / kHThreads;  // float4 per thread, operand and chunk (8)
constexpr int kHeadSmem = 3 * kHOp * (int)sizeof(float);  // A, B, act' argument

template <int ACT>
__global__ void __launch_bounds__(kHThreads) head_tile_kernel(const HeadTileParams hp) {
  pdl_enter();
  extern __shared__ __align__(16) float smem_f[];
  float* As = smem_f;
  float* Bs = smem_f + kHOp;
  int t = blockIdx.x;
  const bool second = t >= hp.prob[0].tiles;
  if (second) t -= hp.prob[0].tiles;
  const HeadTileProb& pr = second ? hp.prob[1] : hp.prob[0];
  const int I = pr.I, J = pr.J, KK = pr.KK;
  const int i0 = (t / pr.tiles_j) * kHT, j0 = (t % pr.tiles_j) * kHT;
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int wm = (warp & 1) * 16, wn = (warp >> 1) * 8;  // 16 x 8 output tile of this warp
  const int fg = lane >> 2, ft = lane & 3;              // mma fragment coordinates
  const float* __restrict__ ap = pr.A.p;
  const float* __restrict__ aq = pr.A.q;
  const float* __restrict__ bp = pr.B.p;
  const int a_mode = pr.A.mode, b_mode = pr.B.mode;
  const bool a_kc = pr.A.sk == 1, b_kc = pr.B.sk == 1;  // contiguous along kk (else along i)
  const int64_t a_ld = a_kc ? pr.A.si : pr.A.sk, q_ld = a_kc ? pr.A.qi : pr.A.qk, b_ld = b_kc ? pr.B.si : pr.B.sk;
  const bool a_vec = (a_ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(ap) & 15) == 0);
  const bool q_vec = (q_ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(aq) & 15) == 0);
  const bool b_vec = (b_ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(bp) & 15) == 0);
  // float4 e (0..7) of this thread inside an operand chunk: kk-contiguous: row i = (tid >> 6) + 4 e, kk = 4 (tid & 63);
  // i-contiguous: row kk = (tid >> 3) + 32 e, i = 4 (tid & 7).  (major, minor) = (row, offset inside the row)
  const int a_maj = a_kc ? (tid >> 6) : (tid >> 3), a_mstep = a_kc ? 4 : 32, a_min = a_kc ? 4 * (tid & 63) : 4 * (tid & 7);
  const int b_maj = b_kc ? (tid >> 6) : (tid >> 3), b_mstep = b_kc ? 4 : 32, b_min = b_kc ? 4 * (tid & 63) : 4 * (tid & 7);
  const int a_srow = a_kc ? kHSk : kHSi, b_srow = b_kc ? kHSk : kHSi;
  // fragment strides: element (i, k) of a staged operand
  const int a_fi = a_kc ? kHSk : 1, a_fk = a_kc ? 1 : kHSi, b_fi = b_kc ? kHSk : 1, b_fk = b_kc ? 1 : kHSi;

  // staging: the operand (and act' argument) float4s go global -> shared with 16-byte cp.async from ROLLED loops
  // (all of a chunk's loads in flight, no registers held, little code: this kernel runs once per CTA and every
  // instruction is an instruction-cache miss); operands that are not 16-byte loadable take a scalar path
  float* Qs = smem_f + 2 * kHOp;
  auto stage_operand = [&](const float* __restrict__ gp, float* sdst, bool kc, bool vec, int64_t ld, int maj0, int mstep,
                           int mn, int srow, int lim_row, int lim_vec, int row0, int vec0) {
    // row0 / vec0: global index of the first row / first vector component of this thread's float4 0
#pragma unroll 1
    for (int e = 0; e < kHNV; ++e) {
      const int maj = maj0 + e * mstep;
      const int grow = row0 + e * mstep, gvec = vec0;
      const int lim = lim_vec - gvec;
      const int nv = (grow < lim_row) ? (lim > 4 ? 4 : (lim < 0 ? 0 : lim)) : 0;
      float* d = sdst + maj * srow + mn;
      const float* g = gp + (int64_t)grow * ld + gvec;
      if (vec && nv == 4) {
        const uint32_t da = (uint32_t)__cvta_generic_to_shared(d);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(da), "l"(g) : "memory");
      } else {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (nv > 0) v.x = __ldg(g);
        if (nv > 1) v.y = __ldg(g + 1);
        if (nv > 2) v.z = __ldg(g + 2);
        if (nv > 3) v.w = __ldg(g + 3);
        *reinterpret_cast<float4*>(d) = v;
      }
    }
  };
  auto fetch = [&](int k0) {
    // kk-contiguous: rows = i (limit I / J), vector along kk (limit KK); i-contiguous: rows = kk, vector along i
    stage_operand(ap, As, a_kc, a_vec, a_ld, a_maj, a_mstep, a_min, a_srow, a_kc ? I : KK, a_kc ? KK : I,
                  a_kc ? i0 + a_maj : k0 + a_maj, a_kc ? k0 + a_min : i0 + a_min);
    if (a_mode == 2)
      stage_operand(aq, Qs, a_kc, q_vec, q_ld, a_maj, a_mstep, a_min, a_srow, a_kc ? I : KK, a_kc ? KK : I,
                    a_kc ? i0 + a_maj : k0 + a_maj, a_kc ? k0 + a_min : i0 + a_min);
    stage_operand(bp, Bs, b_kc, b_vec, b_ld, b_maj, b_mstep, b_min, b_srow, b_kc ? J : KK, b_kc ? KK : J,
                  b_kc ? j0 + b_maj : k0 + b_maj, b_kc ? k0 + b_min : j0 + b_min);
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  auto transform = [&]() {  // in place, on the float4s this thread staged
    if (a_mode == 0 && b_mode == 0) return;
#pragma unroll 1
    for (int e = 0; e < kHNV; ++e) {
      float4* pa = reinterpret_cast<float4*>(As + (a_maj + e * a_mstep) * a_srow + a_min);
      if (a_mode == 1) {
        float4 v = *pa;
        v.x = act_fwd(ACT, v.x); v.y = act_fwd(ACT, v.y); v.z = act_fwd(ACT, v.z); v.w = act_fwd(ACT, v.w);
        *pa = v;
      } else if (a_mode == 2) {
        float4 v = *pa;
        const float4 q = *reinterpret_cast<const float4*>(Qs + (a_maj + e * a_mstep) * a_srow + a_min);
        v.x *= act_grad(ACT, q.x); v.y *= act_grad(ACT, q.y); v.z *= act_grad(ACT, q.z); v.w *= act_grad(ACT, q.w);
        *pa = v;
      }
      if (b_mode == 1) {
        float4* pb = reinterpret_cast<float4*>(Bs + (b_maj + e * b_mstep) * b_srow + b_min);
        float4 v = *pb;
        v.x = act_fwd(ACT, v.x); v.y = act_fwd(ACT, v.y); v.z = act_fwd(ACT, v.z); v.w = act_fwd(ACT, v.w);
        *pb = v;
      }
    }
  };

  // six independent accumulator fragments (3 product terms x even / odd k step) keep the HMMA latency chains
  // short; fragment layout c0 (g, 2t), c1 (g, 2t+1), c2 (g+8, 2t), c3 (g+8, 2t+1)
  float acc[6][4];
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  float csum = 0.f;
  const bool want_colsum = pr.colsum != nullptr && j0 == 0;

#pragma unroll 1
  for (int k0 = 0; k0 < KK; k0 += kHC) {
    if (k0 > 0) __syncthreads();  // the previous chunk has been consumed
    fetch(k0);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    transform();
    __syncthreads();
    const int kend = (KK - k0 < kHC) ? ((KK - k0 + 31) & ~31) : kHC;  // zero filled beyond KK
    const float* ar = As + (wm + fg) * a_fi + ft * a_fk;
    const float* br = Bs + (wn + fg) * b_fi + ft * b_fk;
#pragma unroll 1
    for (int k32 = 0; k32 < kend; k32 += 32) {
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const int k8 = k32 + 8 * h;
        const float av[4] = {ar[k8 * a_fk], ar[k8 * a_fk + 8 * a_fi], ar[(k8 + 4) * a_fk], ar[(k8 + 4) * a_fk + 8 * a_fi]};
        const float bv[2] = {br[k8 * b_fk], br[(k8 + 4) * b_fk]};
        uint32_t ah[4], al[4], bh[2], bl[2];
#pragma unroll
        for (int i = 0; i < 4; ++i) split_tf32(av[i], ah[i], al[i]);
#pragma unroll
        for (int i = 0; i < 2; ++i) split_tf32(bv[i], bh[i], bl[i]);
        mma_tf32(acc[3 * (h & 1) + 0], al, bh);
        mma_tf32(acc[3 * (h & 1) + 1], ah, bl);
        mma_tf32(acc[3 * (h & 1) + 2], ah, bh);
      }
    }
    if (want_colsum && tid < kHT) {
      const float* ac = As + tid * a_fi;
      if (pr.colsum_w) {
#pragma unroll 4
        for (int k = 0; k < kend; ++k) csum += ac[k * a_fk] * (k0 + k < KK ? __ldg(pr.colsum_w + k0 + k) : 0.f);
      } else {
#pragma unroll 4
        for (int k = 0; k < kend; ++k) csum += ac[k * a_fk];
      }
    }
  }

  // ---- store: each warp owns its 16 x 8 outputs
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int i = i0 + wm + fg + (e >> 1) * 8, j = j0 + wn + 2 * ft + (e & 1);
    if (i < I && j < J) {
      float v = ((acc[0][e] + acc[3][e]) + (acc[1][e] + acc[4][e])) + (acc[2][e] + acc[5][e]);  // small terms first
      if (pr.row_scale) v *= __ldg(pr.row_scale + i);
      if (pr.bias) v += (pr.bias_scale ? __ldg(pr.bias_scale + i) : 1.f) * __ldg(pr.bias + j);
      pr.C[(int64_t)i * pr.ldc + j] = v;
    }
  }
  if (want_colsum && tid < kHT && i0 + tid < I) pr.colsum[i0 + tid] = csum;
}

void launch_head_tiles(const HeadTileParams& hp, int tiles, cudaStream_t st) {
  if (tiles <= 0) return;
  auto kern = head_tile_kernel<PCC_ACT_TANH>;
  switch (hp.act) {
    case PCC_ACT_RELU: kern = head_tile_kernel<PCC_ACT_RELU>; break;
    case PCC_ACT_GELU: kern = head_tile_kernel<PCC_ACT_GELU>; break;
    case PCC_ACT_SILU: kern = head_tile_kernel<PCC_ACT_SILU>; break;
    default: break;
  }
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kHeadSmem);
  launch_dep(kern, dim3(tiles), dim3(kHThreads), kHeadSmem, st, hp);
}

static int check_head(const pcc_head_desc* d, const char* where) {
  if (!d) return fail(where, "null descriptor");
  if (d->n_layers < 1 || d->n_layers > kHeadMaxLayers) return fail(where, "head needs 1..4 layers");
  for (int l = 0; l <= d->n_layers; ++l)
    if (d->dims[l] < 1 || d->dims[l] > kHeadMaxDim) return fail(where, "head widths must be in [1,1024]");
  if (d->act != PCC_ACT_RELU && d->act != PCC_ACT_GELU && d->act != PCC_ACT_SILU && d->act != PCC_ACT_TANH)
    return fail(where, "head activation must be relu/gelu/silu/tanh");
  return 0;
}

struct HeadGeom {
  int zoff[kHeadMaxLayers];
  int zwidth, maxhid;
};
static HeadGeom head_geom(const pcc_head_desc* d) {
  HeadGeom g{};
  int off = 0, mh = 1;
  for (int l = 0; l < d->n_layers - 1; ++l) {
    g.zoff[l] = off;
    off += d->dims[l + 1];
    if (d->dims[l + 1] > mh) mh = d->dims[l + 1];
  }
  g.zwidth = off;
  g.maxhid = mh;
  return g;
}

void head_set_tiles(HeadTileProb& p) {
  p.tiles_j = (int)cdiv(p.J, kHT);
  p.tiles = (int)cdiv(p.I, kHT) * p.tiles_j;
}
static void set_tiles(HeadTileProb& p) { head_set_tiles(p); }

}  // namespace pcc

using namespace pcc;

extern "C" int pcc_mlp_head_supported(const pcc_head_desc* d) { return check_head(d, __func__); }

extern "C" int64_t pcc_mlp_head_workspace_bytes(const pcc_head_desc* d, int64_t M) {
  if (check_head(d, __func__) != 0) return -1;
  const HeadGeom g = head_geom(d);
  return 2 * (M > 0 ? M : 1) * (int64_t)g.maxhid * (int64_t)sizeof(float);
}

extern "C" int pcc_mlp_head_fwd(const pcc_head_desc* d, const float* x, float* y, float* zsave, int64_t M, int device,
                                void* stream) {
  PCC_ENTER(device);
  if (check_head(d, __func__) != 0) return -1;
  PCC_REQUIRE(M < (int64_t)0x7fffffff, "row count exceeds int32");
  if (M == 0) return 0;
  const HeadGeom g = head_geom(d);
  const int L = d->n_layers;
  for (int l = 0; l < L; ++l) {
    const int K = d->dims[l], N = d->dims[l + 1];
    HeadTileParams hp{};
    hp.act = d->act;
    HeadTileProb& p = hp.prob[0];
    if (l == 0) p.A = HeadOperand{x, nullptr, K, 1, 0, 0, 0};
    else p.A = HeadOperand{zsave + g.zoff[l - 1], nullptr, g.zwidth, 1, 0, 0, 1};
    p.B = HeadOperand{d->w[l], nullptr, K, 1, 0, 0, 0};
    p.I = (int)M; p.J = N; p.KK = K;
    if (l < L - 1) { p.C = zsave + g.zoff[l]; p.ldc = g.zwidth; } else { p.C = y; p.ldc = N; }
    p.bias = d->b[l];
    set_tiles(p);
    launch_head_tiles(hp, p.tiles, (cudaStream_t)stream);
  }
  return check_launch(__func__);
}

extern "C" int pcc_mlp_head_bwd(const pcc_head_desc* d, const float* x, const float* zsave, const float* dy, float* dx,
                                float* const* dw, float* const* db, void* ws, int64_t M, int device, void* stream) {
  PCC_ENTER(device);
  if (check_head(d, __func__) != 0) return -1;
  PCC_REQUIRE(M < (int64_t)0x7fffffff, "row count exceeds int32");
  const HeadGeom g = head_geom(d);
  const int L = d->n_layers;
  PCC_REQUIRE(L == 1 || ws != nullptr || M == 0, "workspace required (pcc_mlp_head_workspace_bytes)");
  float* gbuf[2] = {(float*)ws, (float*)ws + (M > 0 ? M : 1) * (int64_t)g.maxhid};
  for (int l = L - 1; l >= 0; --l) {
    const int K = d->dims[l], N = d->dims[l + 1];
    HeadTileParams hp{};
    hp.act = d->act;
    // dz_l(r, u): dy for the final layer, g_l * act'(z_l) for hidden layers
    const float* gsrc = (l == L - 1) ? dy : gbuf[l & 1];
    const int64_t gld = N;
    const float* zq = (l == L - 1) ? nullptr : zsave + g.zoff[l];
    const int dzmode = (l == L - 1) ? 0 : 2;
    // ---- dW_l[u][k] = sum_r dz(r,u) in(r,k); db_l[u] = sum_r dz(r,u)
    HeadTileProb& pw = hp.prob[0];
    pw.A = HeadOperand{gsrc, zq, 1, gld, 1, g.zwidth, dzmode};
    if (l == 0) pw.B = HeadOperand{x, nullptr, 1, K, 0, 0, 0};
    else pw.B = HeadOperand{zsave + g.zoff[l - 1], nullptr, 1, g.zwidth, 0, 0, 1};
    pw.I = N; pw.J = K; pw.KK = (int)M;
    pw.C = dw[l]; pw.ldc = K; pw.bias = nullptr; pw.colsum = db[l];
    set_tiles(pw);
    // ---- g_{l-1}[r][k] = sum_u dz(r,u) W_l[u][k]
    HeadTileProb& pd = hp.prob[1];
    float* dst = (l == 0) ? dx : gbuf[(l - 1) & 1];
    if (dst != nullptr && M > 0) {
      pd.A = HeadOperand{gsrc, zq, gld, 1, g.zwidth, 1, dzmode};
      pd.B = HeadOperand{d->w[l], nullptr, 1, K, 0, 0, 0};
      pd.I = (int)M; pd.J = K; pd.KK = N;
      pd.C = dst; pd.ldc = K;
      set_tiles(pd);
    }
    launch_head_tiles(hp, pw.tiles + pd.tiles, (cudaStream_t)stream);
  }
  return check_launch(__func__);
}
