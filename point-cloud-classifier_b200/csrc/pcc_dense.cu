// fp32 SIMT dense path: Linear fwd / dgrad / wgrad with fused epilogues, activation
// backward, LayerNorm, BatchNorm1d.  This is the exact-fp32 ("parity") path and the
// path for shapes the fused tcgen05 kernel does not take (LayerNorm inside phi, rho
// head, GraphNet dense layers).
//   reference call sites: /root/reference/models/deep_sets.py:89,112,156-160;
//   /root/reference/models/graph_net.py:73-102 (lin_rel/lin_root, fc1/fc2, bn1-3).
#include "pcc_common.cuh"
#include "pcc_tf32.cuh"

namespace pcc {

struct GemmArgs {
  const float* A;
  const float* B;
  float* C;
  int64_t M, N, K;  // C[M,N] = A[M,K] * B[K,N]
  int64_t lda, ldb, ldc;
  const float* bias;      // [N] or null
  const float* pre_add;   // [M,N] (ld = ldc) or null, added before the activation
  const float* residual;  // [M,N] (ld = ldc) or null, added after the activation
  float* z_out;           // [M,N] (ld = ldc) or null
  int act;
  int accumulate;   // C += result
  int atomic;       // split-K partial sums: atomicAdd into C
  int tf32x1;       // one TF32 MMA per product (operands rounded to 10 mantissa bits) instead of the 3xTF32 split
  int64_t k_chunk;  // K range per blockIdx.z
};

// library-wide precision of the dense (pcc_linear_*) path: 0 = fp32-grade 3xTF32 (default, parity mode),
// 1 = single TF32 (~1e-3 relative, better than the bf16 operands of the fused DeepSets path; 3x fewer MMAs)
static int g_dense_tf32x1 = 0;

// four consecutive floats p[0..3]; `nvalid` leading ones are in range; one 128-bit load when possible
__device__ __forceinline__ float4 gemm_ld4(const float* p, bool vec, int nvalid) {
  if (vec && nvalid == 4) return __ldg(reinterpret_cast<const float4*>(p));
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (nvalid > 0) v.x = __ldg(p);
  if (nvalid > 1) v.y = __ldg(p + 1);
  if (nvalid > 2) v.z = __ldg(p + 2);
  if (nvalid > 3) v.w = __ldg(p + 3);
  return v;
}

// A_T=false: A(m,k)=A[m*lda+k] ; A_T=true: A(m,k)=A[k*lda+m]
// B_T=false: B(k,n)=B[k*ldb+n] ; B_T=true: B(k,n)=B[n*ldb+k]
// 256 threads = 8 warps laid out 2 (M) x 4 (N); a warp owns a (BM/2) x (BN/4) sub-tile as m16n8 fragments.
// Operands are staged without transposition — one contiguous along k as [row][k] (stride BK+4), one contiguous
// along its row index as [k][row] (stride B+8): 128-bit global loads and stores either way, and both layouts are
// conflict free for the k-strided fragment loads.  The next K step's loads are in flight (registers) under the
// math of the current one.  TM / TN are unused legacy parameters (the tile shape is BM x BN x BK).
template <int BM, int BN, int BK, int TM, int TN, bool A_T, bool B_T>
__global__ void __launch_bounds__(256, 2) sgemm_kernel(GemmArgs p) {
  constexpr int NT = 256;
  constexpr int WM = BM / 2, WN = BN / 4;      // warp tile
  constexpr int MT = WM / 16, NTL = WN / 8;    // m16 / n8 fragments per warp
  constexpr bool A_KC = !A_T, B_KC = B_T;      // contiguous along k
  constexpr int ASZ = A_KC ? BM * (BK + 4) : BK * (BM + 8);
  constexpr int BSZ = B_KC ? BN * (BK + 4) : BK * (BN + 8);
  constexpr int AV = BM * BK / 4 / NT, BV = BN * BK / 4 / NT;  // float4 per thread and K step
  __shared__ __align__(16) float As[ASZ];
  __shared__ __align__(16) float Bs[BSZ];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm0 = (warp & 1) * WM, wn0 = (warp >> 1) * WN;
  const int fg = lane >> 2, ft = lane & 3;
  const int64_t m0 = (int64_t)blockIdx.y * BM, n0 = (int64_t)blockIdx.x * BN;
  const int64_t kbeg = (int64_t)blockIdx.z * p.k_chunk;
  const int64_t kend = (kbeg + p.k_chunk < p.K) ? kbeg + p.k_chunk : p.K;
  const bool a_vec = (p.lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.A) & 15) == 0);
  const bool b_vec = (p.ldb % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.B) & 15) == 0);
  // element (row, k) of a staged operand
  constexpr int A_FR = A_KC ? BK + 4 : 1, A_FK = A_KC ? 1 : BM + 8;
  constexpr int B_FR = B_KC ? BK + 4 : 1, B_FK = B_KC ? 1 : BN + 8;

  float4 ra[AV], rb[BV];
  auto fetch = [&](int64_t k0) {
#pragma unroll
    for (int e = 0; e < AV; ++e) {
      const int id = tid + NT * e;
      int row, k;
      if (A_KC) { row = id / (BK / 4); k = 4 * (id % (BK / 4)); } else { k = id / (BM / 4); row = 4 * (id % (BM / 4)); }
      const int64_t gr = m0 + row, gk = k0 + k;
      const int64_t lim = A_KC ? kend - gk : p.M - gr;
      const bool ok = A_KC ? (gr < p.M) : (gk < kend);
      const int nv = ok ? (lim > 4 ? 4 : (lim < 0 ? 0 : (int)lim)) : 0;
      ra[e] = gemm_ld4(p.A + (nv ? (A_KC ? gr * p.lda + gk : gk * p.lda + gr) : 0), a_vec, nv);
    }
#pragma unroll
    for (int e = 0; e < BV; ++e) {
      const int id = tid + NT * e;
      int row, k;
      if (B_KC) { row = id / (BK / 4); k = 4 * (id % (BK / 4)); } else { k = id / (BN / 4); row = 4 * (id % (BN / 4)); }
      const int64_t gr = n0 + row, gk = k0 + k;
      const int64_t lim = B_KC ? kend - gk : p.N - gr;
      const bool ok = B_KC ? (gr < p.N) : (gk < kend);
      const int nv = ok ? (lim > 4 ? 4 : (lim < 0 ? 0 : (int)lim)) : 0;
      rb[e] = gemm_ld4(p.B + (nv ? (B_KC ? gr * p.ldb + gk : gk * p.ldb + gr) : 0), b_vec, nv);
    }
  };
  auto stage = [&]() {
#pragma unroll
    for (int e = 0; e < AV; ++e) {
      const int id = tid + NT * e;
      if (A_KC) *reinterpret_cast<float4*>(As + (id / (BK / 4)) * (BK + 4) + 4 * (id % (BK / 4))) = ra[e];
      else *reinterpret_cast<float4*>(As + (id / (BM / 4)) * (BM + 8) + 4 * (id % (BM / 4))) = ra[e];
    }
#pragma unroll
    for (int e = 0; e < BV; ++e) {
      const int id = tid + NT * e;
      if (B_KC) *reinterpret_cast<float4*>(Bs + (id / (BK / 4)) * (BK + 4) + 4 * (id % (BK / 4))) = rb[e];
      else *reinterpret_cast<float4*>(Bs + (id / (BN / 4)) * (BN + 8) + 4 * (id % (BN / 4))) = rb[e];
    }
  };

  float acc[MT][NTL][4];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < NTL; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.f;

  if (kbeg < kend) fetch(kbeg);
  for (int64_t k0 = kbeg; k0 < kend; k0 += BK) {
    if (k0 > kbeg) __syncthreads();  // the previous tiles have been consumed
    stage();
    __syncthreads();
    if (k0 + BK < kend) fetch(k0 + BK);
    const float* ar = As + (wm0 + fg) * A_FR + ft * A_FK;
    const float* br = Bs + (wn0 + fg) * B_FR + ft * B_FK;
#pragma unroll
    for (int k8 = 0; k8 < BK; k8 += 8) {
      uint32_t bh[NTL][2], bl[NTL][2];
#pragma unroll
      for (int j = 0; j < NTL; ++j) {
        split_tf32(br[j * 8 * B_FR + k8 * B_FK], bh[j][0], bl[j][0]);
        split_tf32(br[j * 8 * B_FR + (k8 + 4) * B_FK], bh[j][1], bl[j][1]);
      }
#pragma unroll
      for (int i = 0; i < MT; ++i) {
        uint32_t ah[4], al[4];
        split_tf32(ar[(i * 16) * A_FR + k8 * A_FK], ah[0], al[0]);
        split_tf32(ar[(i * 16 + 8) * A_FR + k8 * A_FK], ah[1], al[1]);
        split_tf32(ar[(i * 16) * A_FR + (k8 + 4) * A_FK], ah[2], al[2]);
        split_tf32(ar[(i * 16 + 8) * A_FR + (k8 + 4) * A_FK], ah[3], al[3]);
#pragma unroll
        for (int j = 0; j < NTL; ++j) {
          if (!p.tf32x1) {
            mma_tf32(acc[i][j], al, bh[j]);
            mma_tf32(acc[i][j], ah, bl[j]);
          }
          mma_tf32(acc[i][j], ah, bh[j]);
        }
      }
    }
  }

  // fragment element e: row = fg + 8 (e >> 1), column = 2 ft + (e & 1)
#pragma unroll
  for (int i = 0; i < MT; ++i) {
#pragma unroll
    for (int e2 = 0; e2 < 2; ++e2) {
      const int64_t gm = m0 + wm0 + i * 16 + fg + 8 * e2;
      if (gm >= p.M) continue;
#pragma unroll
      for (int j = 0; j < NTL; ++j) {
#pragma unroll
        for (int e1 = 0; e1 < 2; ++e1) {
          const int64_t gn = n0 + wn0 + j * 8 + 2 * ft + e1;
          if (gn >= p.N) continue;
          const int64_t o = gm * p.ldc + gn;
          float v = acc[i][j][e2 * 2 + e1];
          if (p.atomic) {
            atomicAdd(p.C + o, v);
            continue;
          }
          if (p.bias) v += __ldg(p.bias + gn);
          if (p.pre_add) v += __ldg(p.pre_add + o);
          if (p.z_out) p.z_out[o] = v;
          v = act_fwd(p.act, v);
          if (p.residual) v += __ldg(p.residual + o);
          if (p.accumulate) v += p.C[o];
          p.C[o] = v;
        }
      }
    }
  }
}

// Small problems (rho head, M = batch): 32x32 output tile per CTA, 256 threads (2x2 per thread),
// so a 256x256x256 layer spreads over 64 CTAs with a short K loop instead of 4 long-running ones.
template <bool A_T, bool B_T>
__global__ void __launch_bounds__(256) sgemm_small_kernel(GemmArgs p) {
  __shared__ float As[32][33];
  __shared__ float Bs[32][33];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t m0 = (int64_t)blockIdx.y * 32, n0 = (int64_t)blockIdx.x * 32;
  const int64_t kbeg = (int64_t)blockIdx.z * p.k_chunk;
  const int64_t kend = (kbeg + p.k_chunk < p.K) ? kbeg + p.k_chunk : p.K;
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  // global -> registers one K tile ahead of the math (the K loop is short: latency, not bandwidth, bound)
  float ra[4], rb[4];
  auto fetch = [&](int64_t k0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int i = tid + 256 * j;
      int m, k;
      if (A_T) { m = i & 31; k = i >> 5; } else { m = i >> 5; k = i & 31; }
      const int64_t gm = m0 + m, gk = k0 + k;
      ra[j] = (gm < p.M && gk < kend) ? (A_T ? __ldg(p.A + gk * p.lda + gm) : __ldg(p.A + gm * p.lda + gk)) : 0.f;
      int n, kb;
      if (B_T) { n = i >> 5; kb = i & 31; } else { n = i & 31; kb = i >> 5; }
      const int64_t gn = n0 + n, gkb = k0 + kb;
      rb[j] = (gn < p.N && gkb < kend) ? (B_T ? __ldg(p.B + gn * p.ldb + gkb) : __ldg(p.B + gkb * p.ldb + gn)) : 0.f;
    }
  };
  fetch(kbeg);
  for (int64_t k0 = kbeg; k0 < kend; k0 += 32) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int i = tid + 256 * j;
      if (A_T) As[i >> 5][i & 31] = ra[j]; else As[i & 31][i >> 5] = ra[j];
      if (B_T) Bs[i & 31][i >> 5] = rb[j]; else Bs[i >> 5][i & 31] = rb[j];
    }
    __syncthreads();
    if (k0 + 32 < kend) fetch(k0 + 32);
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      const float a0 = As[k][ty], a1 = As[k][ty + 16], b0 = Bs[k][tx], b1 = Bs[k][tx + 16];
      acc[0][0] = fmaf(a0, b0, acc[0][0]); acc[0][1] = fmaf(a0, b1, acc[0][1]);
      acc[1][0] = fmaf(a1, b0, acc[1][0]); acc[1][1] = fmaf(a1, b1, acc[1][1]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int64_t gm = m0 + ty + 16 * i;
    if (gm >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int64_t gn = n0 + tx + 16 * j;
      if (gn >= p.N) continue;
      const int64_t o = gm * p.ldc + gn;
      float v = acc[i][j];
      if (p.atomic) { atomicAdd(p.C + o, v); continue; }
      if (p.bias) v += __ldg(p.bias + gn);
      if (p.pre_add) v += __ldg(p.pre_add + o);
      if (p.z_out) p.z_out[o] = v;
      v = act_fwd(p.act, v);
      if (p.residual) v += __ldg(p.residual + o);
      if (p.accumulate) v += p.C[o];
      p.C[o] = v;
    }
  }
}

// tile configuration (0 = 128x128, 1 = 64x64, 2 = 32x32 small kernel) and split-K factor of a problem
static void plan_gemm(const GemmArgs& p, int64_t want_split, int* cfg_out, int64_t* split_out, int64_t* k_chunk_out);

template <bool A_T, bool B_T>
static int launch_gemm(GemmArgs p, int64_t want_split, cudaStream_t st) {
  if (p.M == 0 || p.N == 0) return 0;
  int cfg;
  int64_t split;
  plan_gemm(p, want_split, &cfg, &split, &p.k_chunk);
  p.atomic = split > 1 ? 1 : 0;
  p.tf32x1 = g_dense_tf32x1;
  if (cfg == 0) {
    dim3 grid((unsigned)cdiv(p.N, 128), (unsigned)cdiv(p.M, 128), (unsigned)split);
    pcc::note_launch(1), sgemm_kernel<128, 128, 32, 8, 8, A_T, B_T><<<grid, 256, 0, st>>>(p);
  } else if (cfg == 1) {
    dim3 grid((unsigned)cdiv(p.N, 64), (unsigned)cdiv(p.M, 64), (unsigned)split);
    pcc::note_launch(1), sgemm_kernel<64, 64, 32, 4, 4, A_T, B_T><<<grid, 256, 0, st>>>(p);
  } else {
    dim3 grid((unsigned)cdiv(p.N, 32), (unsigned)cdiv(p.M, 32), (unsigned)split);
    pcc::note_launch(1), sgemm_small_kernel<A_T, B_T><<<grid, 256, 0, st>>>(p);
  }
  return 0;
}

static void plan_gemm(const GemmArgs& p, int64_t want_split, int* cfg_out, int64_t* split_out, int64_t* k_chunk_out) {
  const int64_t tiles[3] = {cdiv(p.M, 128) * cdiv(p.N, 128), cdiv(p.M, 64) * cdiv(p.N, 64),
                            cdiv(p.M, 32) * cdiv(p.N, 32)};
  const int64_t min_mn = p.M < p.N ? p.M : p.N;
  int cfg = min_mn <= 32 ? 2 : (min_mn <= 64 ? 1 : 0);  // do not waste a big tile on a thin matrix
  if (p.M * p.N <= 512 * 512) cfg = 2;                  // head-sized outputs: many small CTAs
  int64_t split = 1;
  if (want_split > 1) {
    // reduction-dominated (wgrad): spread K over ~2 waves of CTAs.  With a long reduction the output tile should
    // be as large as the output allows: a [128 x 128] weight gradient over 262k rows read through 32 x 32 tiles
    // re-reads both operands four times (1 GB instead of 268 MB)
    if (p.K >= 8192) cfg = min_mn >= 128 ? 0 : (min_mn >= 64 ? 1 : 2);
    split = cdiv(296, tiles[cfg]);
    int64_t max_split = cdiv(p.K, 256);
    if (split > max_split) split = max_split;
    if (split < 1) split = 1;
  } else {
    while (cfg < 2 && tiles[cfg] < 120) ++cfg;
  }
  int64_t k_chunk = cdiv(cdiv(p.K, split), 32) * 32;
  if (k_chunk == 0) k_chunk = 32;
  split = cdiv(p.K, k_chunk);
  if (split < 1) split = 1;
  *cfg_out = cfg; *split_out = split; *k_chunk_out = k_chunk;
}

// ------------------------------------------------------------------ small kernels
__global__ void zero_f32_kernel(float* p, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0.f;
}

// column sums of dy[M,N] -> db[N] (atomic accumulate): block = 32 columns x 8 row lanes over a 256-row slab
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ dy, int64_t M, int64_t N,
                                                     float* __restrict__ db, int direct) {
  __shared__ float red[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int64_t c = (int64_t)blockIdx.x * 32 + cx;
  const int64_t r0 = (int64_t)blockIdx.y * 256;
  const int64_t r1 = r0 + 256 < M ? r0 + 256 : M;
  float s = 0.f;
  if (c < N)
    for (int64_t r = r0 + ry; r < r1; r += 8) s += __ldg(dy + r * N + c);
  red[ry][cx] = s;
  __syncthreads();
  if (ry == 0 && c < N) {
    float t = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) t += red[j][cx];
    if (direct) db[c] = t; else atomicAdd(db + c, t);
  }
}

__global__ void act_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ z, float* __restrict__ dz,
                               int64_t count, int act) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
    dz[i] = dy[i] * act_grad(act, z[i]);
}

// ------------------------------------------------------------------ LayerNorm (warp per row)
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const float* __restrict__ z, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta,
                                                            const float* __restrict__ residual, float* __restrict__ y,
                                                            float* __restrict__ mean_o, float* __restrict__ rstd_o,
                                                            int64_t M, int64_t H, int act, float eps) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= M) return;
  const float* zr = z + row * H;
  float s = 0.f;
  for (int64_t c = lane; c < H; c += 32) s += zr[c];
  const float mu = warp_sum(s) / (float)H;
  float v = 0.f;
  for (int64_t c = lane; c < H; c += 32) {
    float d = zr[c] - mu;
    v += d * d;
  }
  const float rstd = rsqrtf(warp_sum(v) / (float)H + eps);
  if (lane == 0) {
    mean_o[row] = mu;
    rstd_o[row] = rstd;
  }
  for (int64_t c = lane; c < H; c += 32) {
    float u = (zr[c] - mu) * rstd * __ldg(gamma + c) + __ldg(beta + c);
    float o = act_fwd(act, u);
    if (residual) o += residual[row * H + c];
    y[row * H + c] = o;
  }
}

// dz written; dgamma/dbeta accumulated (block-level smem reduction, then atomics)
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ z,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta,
                                                            const float* __restrict__ mean, const float* __restrict__ rstd,
                                                            float* __restrict__ dz, float* __restrict__ dgamma,
                                                            float* __restrict__ dbeta, int64_t M, int64_t H, int act,
                                                            int rows_per_block) {
  extern __shared__ float sm[];  // [2][H] partial dgamma / dbeta
  float* s_dg = sm;
  float* s_db = sm + H;
  for (int64_t c = threadIdx.x; c < 2 * H; c += blockDim.x) sm[c] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t rbeg = (int64_t)blockIdx.x * rows_per_block;
  const int64_t rend = rbeg + rows_per_block < M ? rbeg + rows_per_block : M;
  for (int64_t row = rbeg + wid; row < rend; row += 8) {
    const float mu = mean[row], rs = rstd[row];
    const float* zr = z + row * H;
    const float* gr = dy + row * H;
    float s1 = 0.f, s2 = 0.f;
    for (int64_t c = lane; c < H; c += 32) {
      float xh = (zr[c] - mu) * rs;
      float g = __ldg(gamma + c);
      float u = xh * g + __ldg(beta + c);
      float du = gr[c] * act_grad(act, u);
      float dxh = du * g;
      s1 += dxh;
      s2 += dxh * xh;
      atomicAdd(&s_dg[c], du * xh);
      atomicAdd(&s_db[c], du);
    }
    s1 = warp_sum(s1) / (float)H;
    s2 = warp_sum(s2) / (float)H;
    for (int64_t c = lane; c < H; c += 32) {
      float xh = (zr[c] - mu) * rs;
      float g = __ldg(gamma + c);
      float u = xh * g + __ldg(beta + c);
      float dxh = gr[c] * act_grad(act, u) * g;
      dz[row * H + c] = rs * (dxh - s1 - xh * s2);
    }
  }
  __syncthreads();
  for (int64_t c = threadIdx.x; c < H; c += blockDim.x) {
    atomicAdd(dgamma + c, s_dg[c]);
    atomicAdd(dbeta + c, s_db[c]);
  }
}

// ------------------------------------------------------------------ BatchNorm1d
// pass 1: column sums -> ws[0:C]; pass 2: sum (x-mean)^2 -> ws[C:2C]; finalize; apply.
__global__ void __launch_bounds__(256) bn_colsum_kernel(const float* __restrict__ x, int64_t n, int64_t C,
                                                        const float* __restrict__ mean, float* __restrict__ out) {
  const int64_t r0 = (int64_t)blockIdx.y * 256;
  const int64_t r1 = r0 + 256 < n ? r0 + 256 : n;
  for (int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x; c < C; c += (int64_t)gridDim.x * 256) {
    float s = 0.f;
    if (mean) {
      const float mu = mean[c];
      for (int64_t r = r0; r < r1; ++r) {
        float d = __ldg(x + r * C + c) - mu;
        s += d * d;
      }
    } else {
      for (int64_t r = r0; r < r1; ++r) s += __ldg(x + r * C + c);
    }
    atomicAdd(out + c, s);
  }
}

__global__ void bn_mean_finalize_kernel(float* sum_to_mean, int64_t C, float inv_n) {
  int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c < C) sum_to_mean[c] *= inv_n;
}

// ssq and invstd may alias (the sum of squares is replaced by 1/std in place)
__global__ void bn_var_finalize_kernel(const float* mean, const float* ssq, float* invstd, float* running_mean,
                                       float* running_var, int64_t C, int64_t n, float momentum, float eps) {
  int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float s = ssq[c];
  float var = s / (float)n;
  invstd[c] = rsqrtf(var + eps);
  if (running_mean) {
    float unbiased = n > 1 ? s / (float)(n - 1) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean[c];
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * unbiased;
  }
}

__global__ void bn_apply_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                const float* __restrict__ beta, const float* __restrict__ mean,
                                const float* __restrict__ invstd_or_var, float* __restrict__ y, int64_t total,
                                int64_t C, float eps, int is_var) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t c = i % C;
    float is = is_var ? rsqrtf(invstd_or_var[c] + eps) : invstd_or_var[c];
    y[i] = (x[i] - mean[c]) * is * gamma[c] + beta[c];
  }
}

// backward pass 1: dbeta = sum dy ; dgamma = sum dy * xhat
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                            const float* __restrict__ mean,
                                                            const float* __restrict__ invstd, int64_t n, int64_t C,
                                                            float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int64_t r0 = (int64_t)blockIdx.y * 256;
  const int64_t r1 = r0 + 256 < n ? r0 + 256 : n;
  for (int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x; c < C; c += (int64_t)gridDim.x * 256) {
    const float mu = mean[c], is = invstd[c];
    float sg = 0.f, sb = 0.f;
    for (int64_t r = r0; r < r1; ++r) {
      float g = __ldg(dy + r * C + c);
      sb += g;
      sg += g * (__ldg(x + r * C + c) - mu) * is;
    }
    atomicAdd(dgamma + c, sg);
    atomicAdd(dbeta + c, sb);
  }
}

__global__ void bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                    const float* __restrict__ gamma, const float* __restrict__ mean,
                                    const float* __restrict__ invstd, const float* __restrict__ dgamma,
                                    const float* __restrict__ dbeta, float* __restrict__ dx, int64_t total, int64_t C,
                                    float inv_n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t c = i % C;
    float is = invstd[c];
    float xh = (x[i] - mean[c]) * is;
    dx[i] = gamma[c] * is * (dy[i] - dbeta[c] * inv_n - xh * dgamma[c] * inv_n);
  }
}

static inline unsigned ew_blocks(int64_t total) {
  int64_t b = cdiv(total, 256);
  return (unsigned)(b < 148 * 16 ? (b < 1 ? 1 : b) : 148 * 16);
}

}  // namespace pcc

using namespace pcc;

extern "C" int pcc_set_dense_precision(int mode) {
  if (mode != 0 && mode != 1) return fail(__func__, "mode must be 0 (fp32-grade 3xTF32) or 1 (single TF32)");
  pcc::g_dense_tf32x1 = mode;
  return 0;
}

extern "C" int pcc_linear_fwd(const float* x, const float* w, const float* bias, const float* pre_add,
                              const float* residual, float* y, float* z_out, int64_t M, int64_t N, int64_t K, int act,
                              int accumulate, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(!(accumulate && act != PCC_ACT_NONE), "accumulate requires act NONE");
  GemmArgs p{};
  p.A = x; p.B = w; p.C = y; p.M = M; p.N = N; p.K = K; p.lda = K; p.ldb = K; p.ldc = N;
  p.bias = bias; p.pre_add = pre_add; p.residual = residual; p.z_out = z_out; p.act = act;
  p.accumulate = accumulate;
  launch_gemm<false, true>(p, 1, (cudaStream_t)stream);
  return check_launch(__func__);
}

extern "C" int pcc_linear_bwd_data(const float* dy, const float* w, const float* residual, float* dx, int64_t M,
                                   int64_t N, int64_t K, int device, void* stream) {
  PCC_ENTER(device);
  GemmArgs p{};  // dx[M,K] = dy[M,N] * w[N,K]
  p.A = dy; p.B = w; p.C = dx; p.M = M; p.N = K; p.K = N; p.lda = N; p.ldb = K; p.ldc = K;
  p.residual = residual; p.act = PCC_ACT_NONE;
  launch_gemm<false, false>(p, 1, (cudaStream_t)stream);
  return check_launch(__func__);
}

extern "C" int pcc_linear_bwd_weight(const float* dy, const float* x, float* dw, float* db, int64_t M, int64_t N,
                                     int64_t K, int accumulate, int device, void* stream) {
  PCC_ENTER(device);
  cudaStream_t st = (cudaStream_t)stream;
  GemmArgs p{};  // dw[N,K] = dy^T[N,M] * x[M,K]  (reduction over M)
  p.A = dy; p.B = x; p.C = dw; p.M = N; p.N = K; p.K = M; p.lda = N; p.ldb = K; p.ldc = K;
  p.act = PCC_ACT_NONE;
  int cfg;
  int64_t split, k_chunk;
  plan_gemm(p, 2, &cfg, &split, &k_chunk);
  const bool single_slab = cdiv(M, 256) <= 1;
  // zero only what will be accumulated into with atomics (split-K partials / multi-slab column sums)
  if (!accumulate && (split > 1 || M == 0)) PCC_K(zero_f32_kernel)<<<(unsigned)cdiv(N * K, 256), 256, 0, st>>>(dw, N * K);
  if (!accumulate && db && (!single_slab || M == 0)) PCC_K(zero_f32_kernel)<<<(unsigned)cdiv(N, 256), 256, 0, st>>>(db, N);
  if (M > 0) {
    p.accumulate = accumulate;  // split == 1: plain store (or += when accumulating); split > 1: atomics
    launch_gemm<true, false>(p, 2, st);
    if (db) {
      dim3 grid((unsigned)cdiv(N, 32), (unsigned)cdiv(M, 256));
      PCC_K(colsum_kernel)<<<grid, 256, 0, st>>>(dy, M, N, db, (single_slab && !accumulate) ? 1 : 0);
    }
  }
  return check_launch(__func__);
}

extern "C" int pcc_act_bwd(const float* dy, const float* z, float* dz, int64_t count, int act, int device,
                           void* stream) {
  PCC_ENTER(device);
  if (count == 0) return 0;
  PCC_K(act_bwd_kernel)<<<ew_blocks(count), 256, 0, (cudaStream_t)stream>>>(dy, z, dz, count, act);
  return check_launch(__func__);
}

extern "C" int pcc_layernorm_fwd(const float* z, const float* gamma, const float* beta, const float* residual,
                                 float* y, float* mean, float* rstd, int64_t M, int64_t H, int act, float eps,
                                 int device, void* stream) {
  PCC_ENTER(device);
  if (M == 0) return 0;
  PCC_K(layernorm_fwd_kernel)<<<(unsigned)cdiv(M, 8), 256, 0, (cudaStream_t)stream>>>(z, gamma, beta, residual, y, mean,
                                                                                 rstd, M, H, act, eps);
  return check_launch(__func__);
}

extern "C" int pcc_layernorm_bwd(const float* dy, const float* z, const float* gamma, const float* beta,
                                 const float* mean, const float* rstd, float* dz, float* dgamma, float* dbeta,
                                 int64_t M, int64_t H, int act, int device, void* stream) {
  PCC_ENTER(device);
  if (M == 0) return 0;
  PCC_REQUIRE(H <= 4096, "LayerNorm width > 4096 unsupported");
  const int rows_per_block = 64;
  PCC_K(layernorm_bwd_kernel)<<<(unsigned)cdiv(M, rows_per_block), 256, 2 * H * sizeof(float), (cudaStream_t)stream>>>(
      dy, z, gamma, beta, mean, rstd, dz, dgamma, dbeta, M, H, act, rows_per_block);
  return check_launch(__func__);
}

extern "C" int pcc_batchnorm_fwd_train(const float* x, const float* gamma, const float* beta, float* y,
                                       float* save_mean, float* save_invstd, float* running_mean,
                                       float* running_var, int64_t n, int64_t C, float momentum, float eps,
                                       int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(n > 0, "BatchNorm1d training needs at least one row");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned cb = (unsigned)cdiv(C, 256);
  dim3 grid(cb, (unsigned)cdiv(n, 256));
  PCC_K(zero_f32_kernel)<<<cb, 256, 0, st>>>(save_mean, C);
  PCC_K(zero_f32_kernel)<<<cb, 256, 0, st>>>(save_invstd, C);
  PCC_K(bn_colsum_kernel)<<<grid, 256, 0, st>>>(x, n, C, nullptr, save_mean);
  PCC_K(bn_mean_finalize_kernel)<<<cb, 256, 0, st>>>(save_mean, C, 1.f / (float)n);
  PCC_K(bn_colsum_kernel)<<<grid, 256, 0, st>>>(x, n, C, save_mean, save_invstd);  // holds ssq until finalize
  PCC_K(bn_var_finalize_kernel)<<<cb, 256, 0, st>>>(save_mean, save_invstd, save_invstd, running_mean, running_var, C, n,
                                             momentum, eps);
  PCC_K(bn_apply_kernel)<<<ew_blocks(n * C), 256, 0, st>>>(x, gamma, beta, save_mean, save_invstd, y, n * C, C, eps, 0);
  return check_launch(__func__);
}

extern "C" int pcc_batchnorm_fwd_eval(const float* x, const float* gamma, const float* beta,
                                      const float* running_mean, const float* running_var, float* y, int64_t n,
                                      int64_t C, float eps, int device, void* stream) {
  PCC_ENTER(device);
  if (n == 0) return 0;
  PCC_K(bn_apply_kernel)<<<ew_blocks(n * C), 256, 0, (cudaStream_t)stream>>>(x, gamma, beta, running_mean, running_var, y,
                                                                        n * C, C, eps, 1);
  return check_launch(__func__);
}

extern "C" int pcc_batchnorm_bwd(const float* dy, const float* x, const float* gamma, const float* save_mean,
                                 const float* save_invstd, float* dx, float* dgamma, float* dbeta, int64_t n,
                                 int64_t C, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(n > 0, "BatchNorm1d backward needs at least one row");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned cb = (unsigned)cdiv(C, 256);
  PCC_K(zero_f32_kernel)<<<cb, 256, 0, st>>>(dgamma, C);
  PCC_K(zero_f32_kernel)<<<cb, 256, 0, st>>>(dbeta, C);
  dim3 grid(cb, (unsigned)cdiv(n, 256));
  PCC_K(bn_bwd_reduce_kernel)<<<grid, 256, 0, st>>>(dy, x, save_mean, save_invstd, n, C, dgamma, dbeta);
  PCC_K(bn_bwd_apply_kernel)<<<ew_blocks(n * C), 256, 0, st>>>(dy, x, gamma, save_mean, save_invstd, dgamma, dbeta, dx, n * C,
                                                        C, 1.f / (float)n);
  return check_launch(__func__);
}
