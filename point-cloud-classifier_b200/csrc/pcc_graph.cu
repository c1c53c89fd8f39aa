// Graph neighbour stage: CSR build, GraphConv neighbour aggregation fwd/bwd, kNN.
//   reference: PyG GraphConv.propagate called at /root/reference/models/graph_net.py:73,82
//   (gather x[src] -> optional scalar edge weight -> scatter-aggr at dst); batch layout
//   from /root/reference/utils/data.py:1228-1261.  kNN has no reference counterpart
//   (semantics: oracle/knn_oracle.py).
// HBM/L2-bound gather-reduce: one thread group per node, 128-bit channel loads, no
// [E,C] message tensor is ever materialised.
#include "pcc_common.cuh"
#include "pcc_scan.cuh"

namespace pcc {

// ------------------------------------------------------------------ CSR build
__global__ void csr_zero_kernel(int64_t* rowptr, int64_t n1) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n1) rowptr[i] = 0;
}
__global__ void csr_count_kernel(const int64_t* __restrict__ keys, int64_t E, int64_t n,
                                 unsigned long long* __restrict__ counts) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < E) {
    int64_t k = keys[e];
    if (k >= 0 && k < n) atomicAdd(&counts[k], 1ull);
  }
}
__global__ void csr_copy_kernel(const int64_t* __restrict__ rowptr, unsigned long long* __restrict__ cursor, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) cursor[i] = (unsigned long long)rowptr[i];
}
__global__ void csr_fill_kernel(const int64_t* __restrict__ keys, int64_t E, int64_t n,
                                unsigned long long* __restrict__ cursor, int32_t* __restrict__ perm) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e < E) {
    int64_t k = keys[e];
    if (k >= 0 && k < n) {
      unsigned long long pos = atomicAdd(&cursor[k], 1ull);
      perm[pos] = (int32_t)e;
    }
  }
}
// restore ascending edge order inside each row (makes float summation order reproducible): one warp per row,
// rows of up to 32 entries (kNN graphs: k <= 32) by a bitonic sort across the lanes (coalesced load / store),
// longer rows by an insertion sort on lane 0
__global__ void __launch_bounds__(256) csr_sort_rows_kernel(const int64_t* __restrict__ rowptr, int32_t* __restrict__ perm, int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (i >= n) return;
  const int64_t s = rowptr[i], e = rowptr[i + 1];
  const int64_t len = e - s;
  if (len < 2) return;
  if (len <= 32) {
    int v = lane < len ? perm[s + lane] : 0x7fffffff;
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1)
#pragma unroll
      for (int j = k >> 1; j > 0; j >>= 1) {
        const int other = __shfl_xor_sync(0xffffffffu, v, j);
        const bool up = (lane & k) == 0, lower = (lane & j) == 0;
        v = (lower == up) ? min(v, other) : max(v, other);
      }
    if (lane < len) perm[s + lane] = v;
    return;
  }
  if (lane != 0 || len > 4096) return;
  for (int64_t a = s + 1; a < e; ++a) {
    int32_t v = perm[a];
    int64_t b = a - 1;
    while (b >= s && perm[b] > v) {
      perm[b + 1] = perm[b];
      --b;
    }
    perm[b + 1] = v;
  }
}

// ------------------------------------------------------------------ CSR transpose (by target -> by source)
// Input: CSR by target with int32 neighbour ids (col_d[p] = source of slot p; the slots of target i are
// [rowptr_d[i], rowptr_d[i+1]), or [i k, (i+1) k) when k_uniform > 0, e.g. a kNN graph).  Output: rowptr_s[n+1] and
// col_s[E] = TARGET ids grouped by source, ascending inside a row (deterministic).  No edge-id permutation, no int64
// index traffic: the backward aggregation of the fused GraphNet path reads exactly these two arrays.
__global__ void csrt_count_kernel(const int32_t* __restrict__ col_d, int64_t E, int64_t n, unsigned long long* __restrict__ counts) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p < E) {
    const int s = col_d[p];
    if (s >= 0 && s < n) atomicAdd(&counts[s], 1ull);
  }
}
__global__ void csrt_fill_kernel(const int32_t* __restrict__ col_d, const int64_t* __restrict__ rowptr_d, int64_t E, int64_t n,
                                 int k_uniform, unsigned long long* __restrict__ cursor, int32_t* __restrict__ col_s) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= E) return;
  const int s = col_d[p];
  if (s < 0 || s >= n) return;
  int64_t t;
  if (k_uniform > 0) {
    t = p / k_uniform;
  } else {   // target of slot p: last i with rowptr_d[i] <= p
    int64_t lo = 0, hi = n;
    while (hi - lo > 1) {
      const int64_t mid = (lo + hi) >> 1;
      if (__ldg(rowptr_d + mid) <= p) lo = mid; else hi = mid;
    }
    t = lo;
  }
  const unsigned long long pos = atomicAdd(&cursor[s], 1ull);
  col_s[pos] = (int32_t)t;
}

// ---- block-diagonal simple graphs (a kNN graph over a batch of clouds): one CTA per cloud, everything in shared memory.
// Preconditions: uniform k slots per target, every neighbour of a node lies in the node's own cloud, no repeated edge
// (violations trap: the caller built the graph).  Then the cloud's edges occupy the same slot range [o k, (o + nc) k)
// in both CSRs and the transpose is local to the cloud:
//   1. in-degree of every source: shared-memory histogram, block scan -> rowptr_s;
//   2. for blocks of S sources: a bitmap [S][nc bits] over the targets, one atomicOr per edge, then thread = source
//      enumerates the set bits of its row — ascending target order for free, no sort, no global atomics.  S = all sources of the
//      cloud when nc <= ~1250 (one pass), fewer for larger clouds (several passes over the cloud's edge slots).
// The kernel is bound by instruction issue (ncu: 42 M warp instructions in its first version, 57 % issue utilisation), so
// the loops are written for instruction count: no division, no modulo in the hot paths, dynamic trip counts.
// 256 clouds of 1024 points, k = 20: ~20 us against ~180 us for count + scan + fill + row sort in global memory.
constexpr int kCsrtBlkThreads = 1024;
constexpr int kCsrtBlkSmem = 200 * 1024;
__global__ void __launch_bounds__(kCsrtBlkThreads, 1) csrt_block_kernel(const int32_t* __restrict__ col_d, int k,
                                                                         const int64_t* __restrict__ offsets, int64_t n,
                                                                         int64_t* __restrict__ rowptr_s, int32_t* __restrict__ col_s) {
  extern __shared__ __align__(16) uint32_t csrt_smem[];
  __shared__ int warp_tot[32];
  const int64_t o = offsets[blockIdx.x];
  const int nc = (int)(offsets[blockIdx.x + 1] - o);
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) rowptr_s[n] = n * (int64_t)k;
  if (nc <= 0) return;
  const int W = (nc + 31) >> 5;                       // bitmap words per source row
  int* cnt = reinterpret_cast<int*>(csrt_smem);       // [nc + 1] in-degree, then exclusive offsets
  uint32_t* bm = csrt_smem + ((nc + 1 + 3) & ~3);
  const int avail_words = kCsrtBlkSmem / 4 - ((nc + 1 + 3) & ~3);
  if (avail_words < W) __trap();                      // cloud beyond ~50k points
  const int S = avail_words / W < nc ? avail_words / W : nc;
  const int tid = threadIdx.x;
  const int64_t e0 = o * (int64_t)k;
  // ---- 1. in-degrees.  thread = target; its k slots are consecutive.  The slots are read four at a time BEFORE the
  //         shared-memory atomics that use them (a load-atomic-load-atomic chain exposes every load's latency).
  for (int i = tid; i <= nc; i += kCsrtBlkThreads) cnt[i] = 0;
  __syncthreads();
  for (int t = tid; t < nc; t += kCsrtBlkThreads) {
    const int32_t* slots = col_d + e0 + (int64_t)t * k;
    for (int j0 = 0; j0 < k; j0 += 4) {
      int v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = (j0 + u < k) ? slots[j0 + u] - (int)o : -1;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (j0 + u < k) {
          if (v[u] < 0 || v[u] >= nc) __trap();       // neighbour outside the cloud (or a missing neighbour)
          atomicAdd(&cnt[v[u]], 1);
        }
      }
    }
  }
  __syncthreads();
  // block exclusive scan, thread = contiguous range of `per` sources
  {
    const int per = (nc + kCsrtBlkThreads - 1) / kCsrtBlkThreads;
    const int b = tid * per, e = (b + per < nc) ? b + per : nc;
    int local = 0;
    for (int i = b; i < e; ++i) local += cnt[i];
    int incl = local;
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      int t = lane < kCsrtBlkThreads / 32 ? warp_tot[lane] : 0;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, t, d);
        if (lane >= d) t += u;
      }
      warp_tot[lane] = t;   // inclusive over warps
    }
    __syncthreads();
    int run = incl - local + (warp > 0 ? warp_tot[warp - 1] : 0);
    for (int i = b; i < e; ++i) {
      const int c = cnt[i];
      cnt[i] = run;
      rowptr_s[o + i] = e0 + run;
      run += c;
    }
    if (tid == kCsrtBlkThreads - 1) cnt[nc] = warp_tot[kCsrtBlkThreads / 32 - 1];
    __syncthreads();
  }
  // ---- 2. bitmap passes
  for (int s0 = 0; s0 < nc; s0 += S) {
    const int sn = (s0 + S < nc) ? S : nc - s0;
    for (int i = tid; i < sn * W; i += kCsrtBlkThreads) bm[i] = 0u;
    __syncthreads();
    for (int t = tid; t < nc; t += kCsrtBlkThreads) {
      const int32_t* slots = col_d + e0 + (int64_t)t * k;
      const int tw = t >> 5;
      const uint32_t bit = 1u << (t & 31);
      for (int j0 = 0; j0 < k; j0 += 4) {
        int v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = (j0 + u < k) ? slots[j0 + u] - (int)o - s0 : -1;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int r = v[u];
          if (r >= 0 && r < sn) {
            int w = tw + (W == 32 ? (r & 31) : r % W);   // word index rotated by the row: the lanes of a warp (same word
            if (w >= W) w -= W;                          // column, different rows) hit different banks, and so do the
            atomicOr(&bm[r * W + w], bit);               // row scans below
          }
        }
      }
    }
    __syncthreads();
    // thread = source row: set bits in ascending word / bit order = ascending target order
    for (int r = tid; r < sn; r += kCsrtBlkThreads) {
      int pos = cnt[s0 + r];
      const int end = cnt[s0 + r + 1];
      const uint32_t* row = bm + r * W;
      int w = (W == 32) ? (r & 31) : r % W;
      int32_t* out = col_s + e0;
      const int base = (int)o;
      for (int j = 0; j < W; ++j) {
        uint32_t word = row[w];
        if (++w == W) w = 0;
        while (word) {
          const int b = __ffs(word) - 1;
          word &= word - 1;
          if (pos < end) out[pos] = base + j * 32 + b;
          ++pos;
        }
      }
      if (pos != end) __trap();                       // repeated edge
    }
    __syncthreads();
  }
}

// ---- by-target position of every by-source entry of such a graph (max aggregation's backward reads the winner mask
// of an edge at its CSR-by-target position).  Thread = by-target slot p = (target t = p / k, source j = col_d[p]); the
// entry (j -> t) of the by-source CSR is the unique t in j's row (ascending targets, simple graph): a binary search.
__global__ void csrt_pos_kernel(const int32_t* __restrict__ col_d, int k, int64_t E, const int64_t* __restrict__ rowptr_s,
                                const int32_t* __restrict__ col_s, int32_t* __restrict__ pos_s) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= E) return;
  const int j = __ldg(col_d + p);
  const int t = (int)(p / k);
  int64_t lo = __ldg(rowptr_s + j), hi = __ldg(rowptr_s + j + 1);
  const int64_t end = hi;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(col_s + mid) < t) lo = mid + 1; else hi = mid;
  }
  if (lo >= end || __ldg(col_s + lo) != t) __trap();   // not the transpose of col_d
  pos_s[lo] = (int32_t)p;
}

// ------------------------------------------------------------------ aggregation
// tpn threads per node, each owning float4 channel groups c = 4*(lane + it*tpn)
template <bool VEC4>
__global__ void __launch_bounds__(256) graph_aggregate_fwd_kernel(const float* __restrict__ x,
                                                                  const int64_t* __restrict__ src,
                                                                  const float* __restrict__ w,
                                                                  const int64_t* __restrict__ rowptr,
                                                                  const int32_t* __restrict__ perm, int64_t n,
                                                                  int64_t C, int aggr, int tpn,
                                                                  float* __restrict__ out,
                                                                  int32_t* __restrict__ arg_edge) {
  const int npb = 256 / tpn;
  const int64_t node = (int64_t)blockIdx.x * npb + threadIdx.x / tpn;
  const int lane = threadIdx.x % tpn;
  if (node >= n) return;
  const int64_t pb = rowptr[node], pe = rowptr[node + 1];
  constexpr int W = VEC4 ? 4 : 1;
  for (int64_t c = (int64_t)lane * W; c < C; c += (int64_t)tpn * W) {
    float acc[W];
    int arg[W];
#pragma unroll
    for (int j = 0; j < W; ++j) { acc[j] = (aggr == PCC_POOL_MAX) ? -INFINITY : 0.f; arg[j] = -1; }
    for (int64_t p = pb; p < pe; ++p) {
      const int e = __ldg(perm + p);
      const int64_t s = __ldg(src + e);
      const float we = w ? __ldg(w + e) : 1.f;
      float v[W];
      if (VEC4) {
        float4 t = __ldg(reinterpret_cast<const float4*>(x + s * C + c));
        v[0] = t.x; v[1 % W] = t.y; v[2 % W] = t.z; v[3 % W] = t.w;
      } else {
        v[0] = __ldg(x + s * C + c);
      }
#pragma unroll
      for (int j = 0; j < W; ++j) {
        float m = v[j] * we;
        if (aggr == PCC_POOL_MAX) {
          if (m > acc[j] || arg[j] < 0) { acc[j] = m; arg[j] = e; }
        } else {
          acc[j] += m;
        }
      }
    }
    const float inv = (aggr == PCC_POOL_MEAN && pe > pb) ? 1.f / (float)(pe - pb) : 1.f;
#pragma unroll
    for (int j = 0; j < W; ++j) {
      float r = acc[j];
      if (aggr == PCC_POOL_MAX) {
        if (arg[j] < 0) r = 0.f;
        arg_edge[node * C + c + j] = arg[j];
      } else {
        r *= inv;
      }
      out[node * C + c + j] = r;
    }
  }
}

template <bool VEC4>
__global__ void __launch_bounds__(256) graph_aggregate_bwd_kernel(const float* __restrict__ g,
                                                                  const int64_t* __restrict__ dst,
                                                                  const float* __restrict__ w,
                                                                  const int64_t* __restrict__ rowptr_src,
                                                                  const int32_t* __restrict__ perm_src,
                                                                  const int64_t* __restrict__ rowptr_dst,
                                                                  const int32_t* __restrict__ arg_edge, int64_t n,
                                                                  int64_t C, int aggr, int tpn,
                                                                  float* __restrict__ dx) {
  const int npb = 256 / tpn;
  const int64_t node = (int64_t)blockIdx.x * npb + threadIdx.x / tpn;
  const int lane = threadIdx.x % tpn;
  if (node >= n) return;
  const int64_t pb = rowptr_src[node], pe = rowptr_src[node + 1];
  constexpr int W = VEC4 ? 4 : 1;
  for (int64_t c = (int64_t)lane * W; c < C; c += (int64_t)tpn * W) {
    float acc[W];
#pragma unroll
    for (int j = 0; j < W; ++j) acc[j] = 0.f;
    for (int64_t p = pb; p < pe; ++p) {
      const int e = __ldg(perm_src + p);
      const int64_t t = __ldg(dst + e);
      float we = w ? __ldg(w + e) : 1.f;
      if (aggr == PCC_POOL_MEAN) we /= (float)(rowptr_dst[t + 1] - rowptr_dst[t]);
      float v[W];
      if (VEC4) {
        float4 q = __ldg(reinterpret_cast<const float4*>(g + t * C + c));
        v[0] = q.x; v[1 % W] = q.y; v[2 % W] = q.z; v[3 % W] = q.w;
      } else {
        v[0] = __ldg(g + t * C + c);
      }
#pragma unroll
      for (int j = 0; j < W; ++j) {
        if (aggr == PCC_POOL_MAX) {
          if (__ldg(arg_edge + t * C + c + j) == e) acc[j] += v[j] * we;
        } else {
          acc[j] += v[j] * we;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < W; ++j) dx[node * C + c + j] = acc[j];
  }
}

static inline int threads_per_node(int64_t C, bool vec4) {
  int64_t groups = vec4 ? C / 4 : C;
  int t = 1;
  while (t < 32 && t < groups) t <<= 1;
  return t;
}

// ------------------------------------------------------------------ kNN, shared-memory tiled
// CTA = 256 consecutive query points; for every cloud the CTA's queries belong to, the cloud's points stream through a
// shared-memory tile ({x, y, z} as float4, 1024 candidates) that ALL warps read (one broadcast LDS.128 per candidate
// instead of per-lane global loads).  Thread = one query: its running top-K lives in REGISTERS as a sorted list of
// (fp32 bits of d2, candidate id) — d2 >= 0, so the unsigned order of the bits is the order of the distances, and the
// ascending scan order makes a stable insertion reproduce the oracle's (d2, id) order (ties -> lower id).  A candidate that
// beats the thread's current K-th distance is appended to a small per-thread queue in shared memory; the queues are
// drained warp-wide (unrolled insertion chain, ~5 instructions per list slot) only when some lane's queue fills, so the
// divergent insertion cost is paid once per several accepted candidates instead of once per candidate.  Distances use
// the oracle's arithmetic (no FMA contraction): results are bit-exact.
constexpr int kKnnTile = 1024;
template <int K, int kKnnQ>
__global__ void __launch_bounds__(256) knn_tiled_kernel(const float* __restrict__ pos, int64_t pos_stride,
                                                        const int64_t* __restrict__ offsets, int64_t n, int64_t B, int k,
                                                        int64_t* __restrict__ nbr, float* __restrict__ d2o,
                                                        int32_t* __restrict__ nbr32) {
  __shared__ float4 tile[kKnnTile];
  __shared__ unsigned long long queue[kKnnQ][256];
  const int tid = threadIdx.x;
  const int64_t q = (int64_t)blockIdx.x * 256 + tid;
  const bool valid = q < n;
  auto cloud_of = [&](int64_t r) {
    int64_t lo = 0, hi = B;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (__ldg(offsets + mid + 1) <= r) lo = mid + 1; else hi = mid;
    }
    return lo;
  };
  const int64_t q_first = (int64_t)blockIdx.x * 256;
  const int64_t q_last = (q_first + 255 < n - 1) ? q_first + 255 : n - 1;
  const int64_t b_first = cloud_of(q_first), b_last = cloud_of(q_last);
  // Sorted top-K list as two register arrays (distance bits, candidate id).  Candidates arrive in ASCENDING id order (tiles
  // and slots are scanned in order, a lane's queue is drained in order), so a candidate's id is larger than every id
  // already in the list: the (d2, id) order the oracle defines reduces to "insert after every entry with d2 <= mine"
  // — compares on the 32-bit distance bits only, and a stable insertion keeps equal distances in id order.
  unsigned ld[K], li[K];
#pragma unroll
  for (int s = 0; s < K; ++s) { ld[s] = 0xffffffffu; li[s] = 0xffffffffu; }
  int cnt = 0;
  auto drain = [&]() {
    const int m = __reduce_max_sync(0xffffffffu, cnt);
    for (int i = 0; i < m; ++i) {
      const unsigned long long key = (i < cnt) ? queue[i][tid] : ~0ull;
      const unsigned kd = (unsigned)(key >> 32), ki = (unsigned)key;
      if (kd < ld[K - 1]) {
        // new[s] = (kd < ld[s-1]) ? old[s-1] : ((kd < ld[s]) ? key : old[s]), from the bottom up
        bool below = true;   // kd < ld[s] (true for s = K-1 by the test above)
#pragma unroll
        for (int s = K - 1; s >= 1; --s) {
          const bool above = kd < ld[s - 1];
          ld[s] = above ? ld[s - 1] : (below ? kd : ld[s]);
          li[s] = above ? li[s - 1] : (below ? ki : li[s]);
          below = above;
        }
        if (below) { ld[0] = kd; li[0] = ki; }
      }
    }
    cnt = 0;
  };
  for (int64_t b = b_first; b <= b_last && b < B; ++b) {
    const int64_t cs = __ldg(offsets + b), ce = __ldg(offsets + b + 1);
    const bool active = valid && q >= cs && q < ce;
    float qx = 0.f, qy = 0.f, qz = 0.f;
    if (active) {
      qx = __ldg(pos + q * pos_stride); qy = __ldg(pos + q * pos_stride + 1); qz = __ldg(pos + q * pos_stride + 2);
    }
    const bool warp_active = __any_sync(0xffffffffu, active);
    for (int64_t t0 = cs; t0 < ce; t0 += kKnnTile) {
      const int tn = (int)((ce - t0 < kKnnTile) ? ce - t0 : kKnnTile);
      __syncthreads();
      for (int i = tid; i < tn; i += 256) {
        const float* pp = pos + (t0 + i) * pos_stride;
        tile[i] = make_float4(__ldg(pp), __ldg(pp + 1), __ldg(pp + 2), 0.f);
      }
      __syncthreads();
      if (!warp_active) continue;
      const unsigned self = (unsigned)(q - t0);   // position of the query inside this tile (or out of range)
      // Per candidate: one broadcast LDS.128, the oracle's 8 flops and ONE compare of the distance bits against the bits
      // of the K-th distance (0 for an inactive lane: never taken); the self test and the queue append sit behind that
      // rarely taken branch.
      unsigned thr1 = 0u;
      auto refresh = [&]() { thr1 = active ? ld[K - 1] : 0u; };
      refresh();
      auto dist_bits = [&](int j) {
        const float4 c = tile[j];
        const float dx = c.x - qx, dy = c.y - qy, dz = c.z - qz;
        return __float_as_uint(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
      };
      auto accept = [&](int j, unsigned bits) {
        if (bits < thr1 && (unsigned)j != self) {
          queue[cnt][tid] = ((unsigned long long)bits << 32) | (unsigned long long)(unsigned)(t0 + j);
          ++cnt;
        }
      };
      auto consider = [&](int j) {
        const unsigned bits = dist_bits(j);
        if (bits < thr1) accept(j, bits);
      };
      const int tn4 = tn & ~3;
      for (int j0 = 0; j0 < tn4; j0 += 4) {
        // four candidates per branch: the distances are independent, one test covers the group
        const unsigned b0 = dist_bits(j0), b1 = dist_bits(j0 + 1), b2 = dist_bits(j0 + 2), b3 = dist_bits(j0 + 3);
        if ((b0 < thr1) | (b1 < thr1) | (b2 < thr1) | (b3 < thr1)) {
          accept(j0, b0); accept(j0 + 1, b1); accept(j0 + 2, b2); accept(j0 + 3, b3);
        }
        if (__any_sync(0xffffffffu, cnt > kKnnQ - 4)) { drain(); refresh(); }
      }
      for (int j = tn4; j < tn; ++j) consider(j);
      if (__any_sync(0xffffffffu, cnt > kKnnQ - 4)) { drain(); refresh(); }
    }
    if (warp_active) drain();
  }
  if (valid) {
#pragma unroll
    for (int s = 0; s < K; ++s) {
      if (s < k) {
        const bool ok = li[s] != 0xffffffffu;
        nbr[q * k + s] = ok ? (int64_t)li[s] : -1;
        d2o[q * k + s] = ok ? __uint_as_float(ld[s]) : INFINITY;
        if (nbr32) nbr32[q * k + s] = ok ? (int32_t)li[s] : -1;
      }
    }
  }
}

__global__ void knn_edges_kernel(const int64_t* __restrict__ nbr, int64_t total, int k, int64_t* __restrict__ ei) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < total) {
    ei[i] = nbr[i];
    ei[total + i] = i / k;
  }
}

}  // namespace pcc

using namespace pcc;

extern "C" int64_t pcc_csr_workspace_bytes(int64_t n, int64_t E) {
  (void)E;
  return (n + cdiv(n + 1, 1024) + 8) * (int64_t)sizeof(int64_t);
}

extern "C" int pcc_csr_build(const int64_t* keys, int64_t E, int64_t n, int64_t* rowptr, int32_t* perm, void* ws,
                             int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(E < (int64_t)0x7fffffff, "edge count exceeds int32 range");
  cudaStream_t st = (cudaStream_t)stream;
  int64_t* scan_ws = (int64_t*)ws;
  unsigned long long* cursor = (unsigned long long*)(scan_ws + cdiv(n + 1, 1024) + 4);
  PCC_K(csr_zero_kernel)<<<(unsigned)cdiv(n + 1, 256), 256, 0, st>>>(rowptr, n + 1);
  if (E > 0) PCC_K(csr_count_kernel)<<<(unsigned)cdiv(E, 256), 256, 0, st>>>(keys, E, n, (unsigned long long*)rowptr);
  exclusive_scan_i64(rowptr, n + 1, scan_ws, st);
  if (E > 0 && n > 0) {
    PCC_K(csr_copy_kernel)<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(rowptr, cursor, n);
    PCC_K(csr_fill_kernel)<<<(unsigned)cdiv(E, 256), 256, 0, st>>>(keys, E, n, cursor, perm);
    PCC_K(csr_sort_rows_kernel)<<<(unsigned)cdiv(n, 8), 256, 0, st>>>(rowptr, perm, n);
  }
  return check_launch(__func__);
}

extern "C" int pcc_csr_transpose(const int32_t* col_d, const int64_t* rowptr_d, int64_t E, int64_t n, int k_uniform,
                                 int64_t* rowptr_s, int32_t* col_s, void* ws, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(E < (int64_t)0x7fffffff && n < (int64_t)0x7fffffff, "edge / node count exceeds int32 range");
  PCC_REQUIRE(k_uniform > 0 || rowptr_d != nullptr, "rowptr_d required unless every target has k_uniform slots");
  cudaStream_t st = (cudaStream_t)stream;
  int64_t* scan_ws = (int64_t*)ws;
  unsigned long long* cursor = (unsigned long long*)(scan_ws + cdiv(n + 1, 1024) + 4);
  PCC_K(csr_zero_kernel)<<<(unsigned)cdiv(n + 1, 256), 256, 0, st>>>(rowptr_s, n + 1);
  if (E > 0) PCC_K(csrt_count_kernel)<<<(unsigned)cdiv(E, 256), 256, 0, st>>>(col_d, E, n, (unsigned long long*)rowptr_s);
  exclusive_scan_i64(rowptr_s, n + 1, scan_ws, st);
  if (E > 0 && n > 0) {
    PCC_K(csr_copy_kernel)<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(rowptr_s, cursor, n);
    PCC_K(csrt_fill_kernel)<<<(unsigned)cdiv(E, 256), 256, 0, st>>>(col_d, rowptr_d, E, n, k_uniform, cursor, col_s);
    PCC_K(csr_sort_rows_kernel)<<<(unsigned)cdiv(n, 8), 256, 0, st>>>(rowptr_s, col_s, n);
  }
  return check_launch(__func__);
}

extern "C" int pcc_csr_transpose_blocks(const int32_t* col_d, int k, const int64_t* offsets, int64_t B, int64_t n,
                                        int64_t* rowptr_s, int32_t* col_s, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(k >= 1, "k must be positive");
  PCC_REQUIRE(n * (int64_t)k < (int64_t)0x7fffffff, "edge count exceeds int32 range");
  if (B == 0) {
    PCC_K(csr_zero_kernel)<<<1, 32, 0, (cudaStream_t)stream>>>(rowptr_s, n + 1);
    return check_launch(__func__);
  }
  PCC_CUDA(cudaFuncSetAttribute(csrt_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCsrtBlkSmem));
  PCC_K(csrt_block_kernel)<<<(unsigned)B, kCsrtBlkThreads, kCsrtBlkSmem, (cudaStream_t)stream>>>(col_d, k, offsets, n, rowptr_s, col_s);
  return check_launch(__func__);
}

extern "C" int pcc_csr_transpose_pos(const int32_t* col_d, int k, int64_t n, const int64_t* rowptr_s, const int32_t* col_s,
                                     int32_t* pos_s, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(k >= 1, "k must be positive");
  PCC_REQUIRE(n * (int64_t)k < (int64_t)0x7fffffff, "edge count exceeds int32 range");
  const int64_t E = n * (int64_t)k;
  if (E == 0) return 0;
  PCC_K(csrt_pos_kernel)<<<(unsigned)cdiv(E, 256), 256, 0, (cudaStream_t)stream>>>(col_d, k, E, rowptr_s, col_s, pos_s);
  return check_launch(__func__);
}

extern "C" int pcc_graph_aggregate_fwd(const float* x, const int64_t* src, const float* w, const int64_t* rowptr,
                                       const int32_t* perm, int64_t n, int64_t C, int aggr, float* out,
                                       int32_t* arg_edge, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(aggr == PCC_POOL_ADD || aggr == PCC_POOL_MEAN || aggr == PCC_POOL_MAX, "aggr must be add/mean/max");
  PCC_REQUIRE(aggr != PCC_POOL_MAX || arg_edge != nullptr, "arg_edge buffer required for max aggregation");
  if (n == 0 || C == 0) return 0;
  const bool vec4 = (C % 4 == 0) && (((uintptr_t)x & 15) == 0);
  const int tpn = threads_per_node(C, vec4);
  const unsigned grid = (unsigned)cdiv(n, 256 / tpn);
  if (vec4)
    pcc::note_launch(1), graph_aggregate_fwd_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(x, src, w, rowptr, perm, n, C, aggr, tpn,
                                                                             out, arg_edge);
  else
    pcc::note_launch(1), graph_aggregate_fwd_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(x, src, w, rowptr, perm, n, C, aggr, tpn,
                                                                              out, arg_edge);
  return check_launch(__func__);
}

extern "C" int pcc_graph_aggregate_bwd(const float* g, const int64_t* dst, const float* w, const int64_t* rowptr_src,
                                       const int32_t* perm_src, const int64_t* rowptr_dst, const int32_t* arg_edge,
                                       int64_t n, int64_t C, int aggr, float* dx, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(aggr == PCC_POOL_ADD || aggr == PCC_POOL_MEAN || aggr == PCC_POOL_MAX, "aggr must be add/mean/max");
  PCC_REQUIRE(aggr != PCC_POOL_MAX || arg_edge != nullptr, "arg_edge buffer required for max aggregation");
  PCC_REQUIRE(aggr != PCC_POOL_MEAN || rowptr_dst != nullptr, "rowptr_dst required for mean aggregation");
  if (n == 0 || C == 0) return 0;
  const bool vec4 = (C % 4 == 0) && (((uintptr_t)g & 15) == 0);
  const int tpn = threads_per_node(C, vec4);
  const unsigned grid = (unsigned)cdiv(n, 256 / tpn);
  if (vec4)
    pcc::note_launch(1), graph_aggregate_bwd_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(g, dst, w, rowptr_src, perm_src,
                                                                             rowptr_dst, arg_edge, n, C, aggr, tpn, dx);
  else
    pcc::note_launch(1), graph_aggregate_bwd_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(g, dst, w, rowptr_src, perm_src,
                                                                              rowptr_dst, arg_edge, n, C, aggr, tpn, dx);
  return check_launch(__func__);
}

extern "C" int pcc_knn(const float* pos, int64_t pos_stride, const int64_t* offsets, int64_t n, int64_t B, int k,
                       int64_t* nbr, float* d2, int32_t* nbr32, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(k >= 1 && k <= 32, "k must be in [1,32]");
  PCC_REQUIRE(n < (int64_t)0x7fffffff, "point count exceeds int32 range");
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope prof(6, st);
  const unsigned grid = (unsigned)cdiv(n, 256);
  pcc::note_launch(1);
  // queue depth 16 (measured at N = 1024: depth 8 0.478 ms, 12 0.440 ms, 16 0.430 ms)
  if (k <= 8) knn_tiled_kernel<8, 16><<<grid, 256, 0, st>>>(pos, pos_stride, offsets, n, B, k, nbr, d2, nbr32);
  else if (k <= 16) knn_tiled_kernel<16, 16><<<grid, 256, 0, st>>>(pos, pos_stride, offsets, n, B, k, nbr, d2, nbr32);
  else if (k <= 20) knn_tiled_kernel<20, 16><<<grid, 256, 0, st>>>(pos, pos_stride, offsets, n, B, k, nbr, d2, nbr32);
  else knn_tiled_kernel<32, 16><<<grid, 256, 0, st>>>(pos, pos_stride, offsets, n, B, k, nbr, d2, nbr32);
  return check_launch(__func__);
}

extern "C" int pcc_knn_edges(const int64_t* nbr, int64_t n, int k, int64_t* edge_index, int device, void* stream) {
  PCC_ENTER(device);
  const int64_t total = n * k;
  if (total == 0) return 0;
  PCC_K(knn_edges_kernel)<<<(unsigned)cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(nbr, total, k, edge_index);
  return check_launch(__func__);
}

// ====================================================================== Gaussian edge weights
//   reference: /root/reference/utils/data.py:835-845 (Step2PointGraph._compute_weights), one call per graph (:814):
//     dists = ||pos[src] - pos[dst]||  (float32),  sigma = median(dists) + eps,  w = exp(-dists^2 / (2 sigma^2)).
//   Device version for batched graphs (edges of graph g = [eoff[g], eoff[g+1])): distances once, an EXACT per-graph
//   median by radix selection on the float bit patterns (distances are >= 0, so the uint32 order is the float
//   order; np.median = mean of the two middle order statistics for an even count), then the weights.  All
//   arithmetic in fp32 with round-to-nearest and no FMA contraction, like numpy.
namespace pcc {

__global__ void edge_dist_kernel(const float* __restrict__ pos, int64_t pos_stride, const int64_t* __restrict__ edges,
                                 int64_t E, float* __restrict__ dist) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int64_t s = edges[e], t = edges[E + e];
  const float dx = __fsub_rn(pos[s * pos_stride + 0], pos[t * pos_stride + 0]);
  const float dy = __fsub_rn(pos[s * pos_stride + 1], pos[t * pos_stride + 1]);
  const float dz = __fsub_rn(pos[s * pos_stride + 2], pos[t * pos_stride + 2]);
  const float ss = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
  dist[e] = __fsqrt_rn(ss);
}

// order statistic `rank` (0-based) of d[0..m): 4 passes of 8-bit radix selection, one CTA per graph
__device__ uint32_t radix_select_u32(const float* __restrict__ d, int64_t m, int64_t rank, unsigned int* hist /*[256]*/) {
  uint32_t prefix = 0, mask = 0;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int64_t i = threadIdx.x; i < m; i += blockDim.x) {
      const uint32_t u = __float_as_uint(d[i]);
      if ((u & mask) == prefix) atomicAdd(&hist[(u >> shift) & 255u], 1u);
    }
    __syncthreads();
    // every thread walks the 256 bins (cheap, keeps the result uniform without another broadcast)
    int64_t cum = 0;
    uint32_t bin = 0;
    for (int b = 0; b < 256; ++b) {
      const int64_t c = hist[b];
      if (cum + c > rank) { bin = (uint32_t)b; break; }
      cum += c;
    }
    rank -= cum;
    prefix |= bin << shift;
    mask |= 255u << shift;
    __syncthreads();
  }
  return prefix;
}

__global__ void __launch_bounds__(1024) edge_sigma_kernel(const float* __restrict__ dist, const int64_t* __restrict__ eoff,
                                                          float eps, float* __restrict__ sigma) {
  __shared__ unsigned int hist[256];
  const int64_t g = blockIdx.x;
  const int64_t lo = eoff[g], m = eoff[g + 1] - lo;
  if (m <= 0) {
    if (threadIdx.x == 0) sigma[g] = __int_as_float(0x7fc00000);  // np.median of an empty array: nan
    return;
  }
  const float* d = dist + lo;
  float med;
  if (m & 1) {
    med = __uint_as_float(radix_select_u32(d, m, m / 2, hist));
  } else {
    const float a = __uint_as_float(radix_select_u32(d, m, m / 2 - 1, hist));
    const float b = __uint_as_float(radix_select_u32(d, m, m / 2, hist));
    med = __fmul_rn(__fadd_rn(a, b), 0.5f);  // np.mean of the two middle elements, float32
  }
  if (threadIdx.x == 0) sigma[g] = __fadd_rn(med, eps);
}

__global__ void edge_weight_kernel(const float* __restrict__ dist, const int64_t* __restrict__ eoff, int64_t G, int64_t E,
                                   const float* __restrict__ sigma, float* __restrict__ w) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  int64_t lo = 0, hi = G;  // graph of edge e: last g with eoff[g] <= e
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (eoff[mid] <= e) lo = mid; else hi = mid;
  }
  const float s = sigma[lo], d = dist[e];
  const float den = __fmul_rn(2.f, __fmul_rn(s, s));
  w[e] = expf(-__fdiv_rn(__fmul_rn(d, d), den));
}

}  // namespace pcc

extern "C" int64_t pcc_edge_weights_workspace_bytes(int64_t E, int64_t G) {
  return ((E > 0 ? E : 1) * 4 + 255) / 256 * 256 + ((G > 0 ? G : 1) * 4 + 255) / 256 * 256;
}

extern "C" int pcc_edge_weights(const float* pos, int64_t pos_stride, const int64_t* edges, int64_t E,
                                const int64_t* edge_offsets, int64_t G, float eps, float* weights, float* sigma_out,
                                void* ws, int device, void* stream) {
  PCC_ENTER(device);
  PCC_REQUIRE(E >= 0 && G >= 0 && pos_stride >= 3, "bad sizes");
  if (E == 0 || G == 0) return 0;
  PCC_REQUIRE(ws != nullptr, "workspace required (pcc_edge_weights_workspace_bytes)");
  cudaStream_t st = (cudaStream_t)stream;
  float* dist = (float*)ws;
  float* sigma = sigma_out ? sigma_out : (float*)((uint8_t*)ws + (E * 4 + 255) / 256 * 256);
  PCC_K(edge_dist_kernel)<<<(unsigned)cdiv(E, 256), 256, 0, st>>>(pos, pos_stride, edges, E, dist);
  PCC_K(edge_sigma_kernel)<<<(unsigned)G, 1024, 0, st>>>(dist, edge_offsets, eps, sigma);
  PCC_K(edge_weight_kernel)<<<(unsigned)cdiv(E, 256), 256, 0, st>>>(dist, edge_offsets, G, E, sigma, weights);
  return check_launch(__func__);
}
