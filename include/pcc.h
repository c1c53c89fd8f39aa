/* pcc.h — C ABI of libpcc.so, the B200 (sm_100a) point-set encoder hot path.
 *
 * Drop-in boundary (SURVEY.md §8b): the reference has no native layer; its hot path is
 * the sequence of torch / torch_geometric library calls made by
 *   /root/reference/models/deep_sets.py:81-114   (DeepSets._forward_sparse)
 *   /root/reference/models/graph_net.py:65-104   (GraphNet.forward)
 * and their autograd.  Every entry point below replaces one of those call sites (cited
 * per function).  The Python host side (point-cloud-classifier_b200/pcc_b200) binds
 * them with ctypes; see INTEGRATION.md for the stub.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; pcc_last_error() gives the
 *     thread-local message.  No CPU fallback exists: a call without a usable CUDA
 *     device fails.
 *   - all pointers are DEVICE pointers unless the name ends in _host.  The caller
 *     (PyTorch) owns every buffer: inputs, outputs, saved-for-backward and workspace.
 *     The library never allocates persistent device memory.
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no internal
 *     synchronisation.  `device` is made current for the duration of the call.
 *   - matrices are dense row-major fp32 unless stated; index arrays are int64
 *     (torch.long) on the boundary, as the reference collate functions produce them
 *     (/root/reference/utils/data.py:651-663, :1228-1261).
 *   - re-entrant and stateless: forward is called from the Python main thread,
 *     backward from PyTorch's autograd worker thread.
 */
#ifndef PCC_H_
#define PCC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* activation ids: deep_sets.py:21-26 (relu/gelu/silu), graph_net.py:38-43 (tanh/relu/gelu) */
enum { PCC_ACT_NONE = 0, PCC_ACT_RELU = 1, PCC_ACT_GELU = 2, PCC_ACT_SILU = 3, PCC_ACT_TANH = 4 };
/* pooling ids: deep_sets.py:96-104.  SUM is the reference's sum/sqrt(n) (:99); ADD is a
 * plain sum (PyG aggr="add", graph_net.py:50). */
enum { PCC_POOL_SUM = 0, PCC_POOL_MEAN = 1, PCC_POOL_MAX = 2, PCC_POOL_ADD = 3 };

const char* pcc_last_error(void);
int pcc_version(void);
/* 0 if `device` is an sm_100 part this library can run on, <0 (with message) otherwise */
int pcc_check_device(int device);

/* ---- segment bookkeeping: replaces torch.bincount + counts.tolist() + torch.split
 *      (deep_sets.py:91-92) without the host sync.  offsets[B+1] = exclusive scan of the
 *      histogram of idx (values >= B are ignored).  Also used for PyG `batch` vectors. */
int pcc_segment_offsets(const int64_t* idx, int64_t n, int64_t B, int64_t* offsets, int device, void* stream);
/* max over an int64 vector (num_sets = max+1 when the caller does not know B) */
int pcc_index_max(const int64_t* idx, int64_t n, int64_t* out_max, int device, void* stream);

/* ---- ragged pooling: replaces the python loop deep_sets.py:94-106 and PyG
 *      global_mean_pool (graph_net.py:92,96).  x[n,H] -> pooled[B,H]; argmax[B,H]
 *      (int32 global row id, first occurrence on ties) is written for PCC_POOL_MAX only.
 *      Empty segments give 0 (reference: NaN / error; never produced by the collate). */
int pcc_segment_pool_fwd(const float* x, const int64_t* offsets, int64_t n, int64_t B, int64_t H, int pooling,
                         float* pooled, int32_t* argmax, int device, void* stream);
/* backward of the above (autograd of deep_sets.py:96-106): dx[n,H] fully written */
int pcc_segment_pool_bwd(const float* dpooled, const int64_t* offsets, const int32_t* argmax, int64_t n, int64_t B,
                         int64_t H, int pooling, float* dx, int device, void* stream);

/* precision of the large-tile dense kernels behind pcc_linear_*: 0 (default) = fp32-grade 3xTF32 mma.sync
 * (x = hi + lo split, error ~2^-21 per product: the parity mode), 1 = single TF32 (operands rounded to 10 mantissa
 * bits, ~1e-3 relative, 3x fewer MMAs).  Library-wide switch; the small-tile (batch-sized) kernels stay exact fp32. */
int pcc_set_dense_precision(int mode);
/* ---- dense layer, fp32-grade path (3xTF32 `mma.sync` with a hi / lo operand split; small shapes exact fp32 FFMA): replaces nn.Linear (+ fused activation / residual)
 *      inside phi / rho (deep_sets.py:89,112), GraphConv's lin_rel / lin_root and fc1 /
 *      fc2 (graph_net.py:73,82,87,98,102).
 *      y[M,N] = residual[M,N]? + act( x[M,K] · w[N,K]^T + bias[N]? + pre_add[M,N]? );
 *      z_out (optional) receives the pre-activation.  pre_add is how GraphConv's
 *      lin_rel(agg) + lin_root(x) shares one activation.  accumulate!=0 adds into y
 *      instead of overwriting (act must be NONE then). */
int pcc_linear_fwd(const float* x, const float* w, const float* bias, const float* pre_add, const float* residual,
                   float* y, float* z_out, int64_t M, int64_t N, int64_t K, int act, int accumulate, int device,
                   void* stream);
/* dx[M,K] = residual[M,K]? + dy[M,N] · w[N,K] */
int pcc_linear_bwd_data(const float* dy, const float* w, const float* residual, float* dx, int64_t M, int64_t N,
                        int64_t K, int device, void* stream);
/* dw[N,K] (+)= dy[M,N]^T · x[M,K];  db[N] (+)= column sums of dy (db may be NULL).
 * accumulate==0 overwrites (the function zeroes the outputs itself). */
int pcc_linear_bwd_weight(const float* dy, const float* x, float* dw, float* db, int64_t M, int64_t N, int64_t K,
                          int accumulate, int device, void* stream);
/* dz = dy * act'(z) elementwise over `count` values (autograd of the activation) */
int pcc_act_bwd(const float* dy, const float* z, float* dz, int64_t count, int act, int device, void* stream);

/* ---- LayerNorm over the last dim (deep_sets.py:50-51,65-66,153), fused with the
 *      following activation and the residual add of ResidualBlock (:156-160):
 *      y = residual? + act( (z-mean)*rstd*gamma + beta ).  mean/rstd [M] are saved. */
int pcc_layernorm_fwd(const float* z, const float* gamma, const float* beta, const float* residual, float* y,
                      float* mean, float* rstd, int64_t M, int64_t H, int act, float eps, int device, void* stream);
/* dz[M,H] written; dgamma/dbeta[H] accumulated with atomics (caller zeroes them). */
int pcc_layernorm_bwd(const float* dy, const float* z, const float* gamma, const float* beta, const float* mean,
                      const float* rstd, float* dz, float* dgamma, float* dbeta, int64_t M, int64_t H, int act,
                      int device, void* stream);

/* ---- BatchNorm1d over rows (graph_net.py:76,84,89,100).  Training: batch statistics
 *      (biased variance) + running-stat update (momentum, unbiased variance).
 *      stats_ws: 2*C floats of workspace. */
int pcc_batchnorm_fwd_train(const float* x, const float* gamma, const float* beta, float* y, float* save_mean,
                            float* save_invstd, float* running_mean, float* running_var, int64_t n, int64_t C,
                            float momentum, float eps, int device, void* stream);
int pcc_batchnorm_fwd_eval(const float* x, const float* gamma, const float* beta, const float* running_mean,
                           const float* running_var, float* y, int64_t n, int64_t C, float eps, int device,
                           void* stream);
/* dx written; dgamma/dbeta[C] overwritten. ws: 2*C floats. */
int pcc_batchnorm_bwd(const float* dy, const float* x, const float* gamma, const float* save_mean,
                      const float* save_invstd, float* dx, float* dgamma, float* dbeta, int64_t n, int64_t C,
                      int device, void* stream);

/* ---- graph stage -------------------------------------------------------------------
 * CSR by key: rowptr[n+1], perm[E] = edge ids grouped by key (ascending edge id inside a
 * group, so results are run-to-run deterministic).  Replaces the sort inside PyG's
 * scatter (GraphConv.propagate, graph_net.py:73,82).  ws: workspace of
 * pcc_csr_workspace_bytes(n, E) bytes. */
int64_t pcc_csr_workspace_bytes(int64_t n, int64_t E);
int pcc_csr_build(const int64_t* keys, int64_t E, int64_t n, int64_t* rowptr, int32_t* perm, void* ws, int device,
                  void* stream);
/* transpose of a CSR by target with int32 neighbour ids (col_d[p] = source of slot p; slots of target i =
 * [rowptr_d[i], rowptr_d[i+1]) or, with k_uniform > 0, [i k, (i+1) k) — a kNN graph): rowptr_s[n+1], col_s[E] = target ids
 * grouped by source, ascending inside a row.  ws: pcc_csr_workspace_bytes(n, E).  Feeds pcc_gnn_agg_bwd. */
int pcc_csr_transpose(const int32_t* col_d, const int64_t* rowptr_d, int64_t E, int64_t n, int k_uniform, int64_t* rowptr_s,
                      int32_t* col_s, void* ws, int device, void* stream);
/* the same transpose for a block-diagonal simple graph with k slots per target (a kNN graph over a batch of clouds:
 * offsets[B+1] = node range of every cloud, all neighbours of a node in the node's cloud, no repeated edge — violations
 * trap): one CTA per cloud in shared memory, no workspace, no sort. */
int pcc_csr_transpose_blocks(const int32_t* col_d, int k, const int64_t* offsets, int64_t B, int64_t n, int64_t* rowptr_s,
                             int32_t* col_s, int device, void* stream);
/* for such a transpose (k slots per target, no repeated edge, rows of col_s ascending): pos_s[E = n k] = the by-target slot
 * of every by-source entry, pos_s[q] = t k + s where col_s[q] = t and col_d[t k + s] is the row's source (a missing entry
 * traps).  Feeds pcc_gnn_agg_bwd with max aggregation. */
int pcc_csr_transpose_pos(const int32_t* col_d, int k, int64_t n, const int64_t* rowptr_s, const int32_t* col_s, int32_t* pos_s,
                          int device, void* stream);
/* out[i,:] = aggr_{e in in(i)} w_e * x[src(e),:]   (aggr: PCC_POOL_ADD / MEAN / MAX);
 * rowptr/perm = CSR by TARGET.  arg_edge[n,C] (int32 edge id, -1 if none) for MAX only. */
int pcc_graph_aggregate_fwd(const float* x, const int64_t* src, const float* w, const int64_t* rowptr,
                            const int32_t* perm, int64_t n, int64_t C, int aggr, float* out, int32_t* arg_edge,
                            int device, void* stream);
/* dx[j,:] = sum_{e in out(j)} w_e * scale(dst e) * g[dst(e),:]  (MAX: only where
 * arg_edge[dst,c]==e); rowptr_src/perm_src = CSR by SOURCE; rowptr_dst gives in-degrees
 * for MEAN. */
int pcc_graph_aggregate_bwd(const float* g, const int64_t* dst, const float* w, const int64_t* rowptr_src,
                            const int32_t* perm_src, const int64_t* rowptr_dst, const int32_t* arg_edge, int64_t n,
                            int64_t C, int aggr, float* dx, int device, void* stream);

/* kNN graph build (north_star; no reference counterpart — semantics defined by
 * oracle/knn_oracle.py).  pos: row r at pos + r*pos_stride floats, 3 coordinates.
 * nbr[n,k] global neighbour ids (-1 pad), d2[n,k] squared distances (inf pad), both
 * ascending by (d2, id).  k <= 32.  nbr32 (optional): the same table as int32 — the CSR-by-target column array the fused
 * GraphNet kernels read (k slots per node), written by the same launch. */
int pcc_knn(const float* pos, int64_t pos_stride, const int64_t* offsets, int64_t n, int64_t B, int k, int64_t* nbr,
            float* d2, int32_t* nbr32, int device, void* stream);
/* edge_index[2,n*k] from nbr (row0 = neighbour, row1 = centre); all slots must be valid */
int pcc_knn_edges(const int64_t* nbr, int64_t n, int k, int64_t* edge_index, int device, void* stream);
/* Gaussian edge weights of the reference's graph dataset (/root/reference/utils/data.py:835-845,
 * Step2PointGraph._compute_weights, called once per graph at :814) for a batch of graphs on device:
 * d_e = ||pos[src_e] - pos[dst_e]|| (fp32), sigma_g = median over the graph's edges + eps (exact order statistics,
 * mean of the two middle ones for an even count, like np.median), w_e = exp(-d_e^2 / (2 sigma_g^2)).
 * pos: xyz at pos[i * pos_stride + 0..2]; edges [2,E] (node-offset, graphs back to back, utils/data.py:1228-1261);
 * edge_offsets [G+1]: first edge of every graph; sigma_out [G] optional; ws: pcc_edge_weights_workspace_bytes. */
int64_t pcc_edge_weights_workspace_bytes(int64_t E, int64_t G);
int pcc_edge_weights(const float* pos, int64_t pos_stride, const int64_t* edges, int64_t E, const int64_t* edge_offsets,
                     int64_t G, float eps, float* weights, float* sigma_out, void* ws, int device, void* stream);

/* ---- device-side collate helpers (SURVEY §8f rank 2).  pcc_expand_segments: idx[i] = segment of row i from
 *      offsets[B+1] — the `cat(full((n_i,), i))` of /root/reference/utils/data.py:658-659 (_collate_sparse) and
 *      :1245 (_graph_collate membership) without the per-sample loop.  pcc_offset_edges: per-graph local edge lists
 *      stored back to back -> batched edge_index (edges_i + node offset, utils/data.py:1240). */
int pcc_expand_segments(const int64_t* offsets, int64_t B, int64_t n, int64_t* idx, int device, void* stream);
int pcc_offset_edges(const int64_t* edges, int64_t E, const int64_t* edge_offsets, const int64_t* node_offsets, int64_t G,
                     int64_t* out, int device, void* stream);

/* ---- fused DeepSets phi + pool, tcgen05 / TMEM path (bf16 operands, fp32 accumulate).
 *      Replaces deep_sets.py:89-106 and its autograd in two launches; per-point
 *      activations never reach HBM.  See DESIGN.md §3 for the layer descriptor. */
typedef struct {
  int32_t n_layers;      /* hidden layers + the final Linear(H,H) (deep_sets.py:55); <= 6 */
  int32_t input_dim;     /* d <= 16 */
  int32_t hidden;        /* H in {64,128,256}: every phi width equal (after layer 0) */
  int32_t act;           /* PCC_ACT_RELU / GELU / SILU */
  int32_t pooling;       /* PCC_POOL_SUM / MEAN / MAX */
  int32_t residual_mask; /* bit l set: layer l is a ResidualBlock (deep_sets.py:149-160) */
  const float* w[6];     /* fp32 [out,in] row-major, nn.Linear layout */
  const float* b[6];
} pcc_phi_desc;

/* 0 when the fused path supports the descriptor; <0 with a reason otherwise */
int pcc_phi_fused_supported(const pcc_phi_desc* d);
int64_t pcc_phi_fused_workspace_bytes(const pcc_phi_desc* d, int64_t n, int64_t B);
/* bytes of the packed bf16 weight images (forward + transposed) the forward writes and the backward reads */
int64_t pcc_phi_packed_bytes(const pcc_phi_desc* d);
/* x[n,d] fp32, offsets[B+1] -> pooled[B,H] (+ argmax[B,H] for MAX).  For SUM / MEAN a non-NULL `argmax` is an
 * aux [B,H] fp32 buffer: the kernel then pools the last hidden activations (sum_i (W h_i + b) = W sum_i h_i + n b),
 * applies the final Linear to the [B,H] result and leaves the scaled pooled activations in aux for the backward.
 * ws: workspace; wpack: caller buffer of
 * pcc_phi_packed_bytes() that RECEIVES the packed weight images (keep it for the backward of the same step). */
int pcc_deepsets_phi_pool_fwd(const pcc_phi_desc* d, const float* x, const int64_t* offsets, int64_t n, int64_t B,
                              float* pooled, int32_t* argmax, void* ws, void* wpack, int device, void* stream);
/* dpooled[B,H] -> dw[l] / db[l] (fp32, OVERWRITTEN) for every phi layer; recomputes the
 * forward per tile.  dw/db arrays follow d->w / d->b order.  wpack: the images written by the forward of
 * the same parameters.
 * Max pooling with argmax == NULL ("virtual rows"): x holds the B*H gathered argmax rows (row b*H + f is the
 * argmax row of (b, f); n == B*H, offsets unused).  The gradient of the final Linear's output is then one-hot
 * per row, and the library skips that layer's dgrad and wgrad GEMMs (scaled weight rows / scaled row sums).
 * Sum / mean pooling with argmax != NULL: the buffer is the aux [B,H] fp32 array the forward filled when it was
 * given one (pooled hidden activations; pooling commuted with the final Linear); the backward then needs no
 * per-point GEMM for the final Linear either.  argmax == NULL keeps the plain per-point formulation. */
int pcc_deepsets_phi_pool_bwd(const pcc_phi_desc* d, const float* x, const int64_t* offsets, int64_t n, int64_t B,
                              const float* dpooled, const int32_t* argmax, float* const* dw, float* const* db,
                              void* ws, const void* wpack, int device, void* stream);

/* ---- set-encoder head: rho = [Linear + act] x (n_layers-1) + Linear over M = batch rows
 *      (deep_sets.py:112 with the stack of :59-72, no LayerNorm).  One launch per layer and direction
 *      (32x32 output tiles over the whole chip; activation, act' and the bias gradient are folded into the
 *      operand loads), no atomics: results are bitwise reproducible.
 *      zsave[M, sum of hidden widths] keeps the pre-activations for the backward.  dw / db are OVERWRITTEN.
 *      ws (backward): pcc_mlp_head_workspace_bytes(d, M) bytes of scratch, may be null for n_layers == 1. */
typedef struct {
  int32_t n_layers;   /* hidden layers + final Linear, 1..4 */
  int32_t dims[5];    /* dims[0] = input width, dims[l+1] = output width of layer l; <= 1024 */
  int32_t act;        /* PCC_ACT_RELU / GELU / SILU / TANH (hidden layers) */
  const float* w[4];  /* fp32 [out, in], nn.Linear layout */
  const float* b[4];
} pcc_head_desc;
int pcc_mlp_head_supported(const pcc_head_desc* d);
int64_t pcc_mlp_head_workspace_bytes(const pcc_head_desc* d, int64_t M);
int pcc_mlp_head_fwd(const pcc_head_desc* d, const float* x, float* y, float* zsave, int64_t M, int device,
                     void* stream);
int pcc_mlp_head_bwd(const pcc_head_desc* d, const float* x, const float* zsave, const float* dy, float* dx,
                     float* const* dw, float* const* db, void* ws, int64_t M, int device, void* stream);

/* ---- fused bf16 GraphNet path (tcgen05 / TMEM): the neighbour stage of /root/reference/models/graph_net.py:73-92 for
 *      hidden_dim = 128 (configs/graph_net.yaml), deepchem_style = true, aggregation add / mean / max (`aggr` =
 *      PCC_POOL_ADD / MEAN / MAX), activations tanh / relu / gelu.  Pipeline and data layout: DESIGN.md section 4 (GraphNet) and csrc/pcc_gnn.cuh.  CSR arguments: rowptr[M+1]
 *      int64, col[E] int32 = neighbour node per CSR slot, w[E] fp32 edge weight per slot or NULL.  *_bf16 = bf16 [M,128]
 *      row-major.  "partials" are per-CTA partial sums, [nblk][...]; *nblk_out (host int) receives the block count used.
 *      Every buffer is caller-owned.
 *   pcc_gnn_pack_weights : conv2 lin_rel / lin_root [128,128] and fc1 [256,128] fp32 -> packed bf16 operand images
 *                          (pcc_gnn_packed_bytes() bytes); w_fc1 may be NULL.
 *   pcc_gnn_conv1_fwd    : GraphConv 1 (graph_net.py:73; K = 2 input_dim <= 16, CUDA cores): agg_out[M,F], z_out[M,128],
 *                          partials [nblk][2][128] = sums of act(z), act(z)^2 (BatchNorm statistics, :76).  MAX: agg = max
 *                          of the fp32 products w_e x[src(e)], 0 for a node without in-edges.
 *   pcc_gnn_bn_finalize  : partial sums -> scale = gamma*invstd, shift = beta - mean*scale, mean, invstd; updates the
 *                          running statistics (momentum, unbiased variance) when the pointers are non-NULL.
 *   pcc_gnn_bn_eval      : scale / shift from the running statistics (eval mode).
 *   pcc_gnn_bn_apply     : h = bf16(act(z)*scale + shift)            (activation BEFORE BatchNorm, graph_net.py:75-76)
 *   pcc_gnn_conv_fwd     : GraphConv 2 (:82) in ONE kernel: CSR gather-reduce of bf16 neighbour rows into the shared-
 *                          memory A image [agg | h], tcgen05 GEMM with [W_rel ; W_root], z (fp32) + BatchNorm partial
 *                          sums in the epilogue; agg_out keeps the aggregate for the weight gradient.  Optional
 *                          membership + psum[B,128]: per-graph sums of act(z) (deepchem_style = false pools right after
 *                          the block, graph_net.py:96: mean pooling commutes with the BatchNorm affine).
 *                          MAX: agg[i][c] = max over the row of i of the fp32 products w_e h[src(e)][c] (0 without in-edges),
 *                          then rounded to bf16.  Ties: the FIRST position of the row wins (lowest CSR-by-target slot).
 *                          win (optional, MAX only, training): winner masks, 16 bytes per CSR-by-target position p =
 *                          4 uint32 words; bit (c % 32) of word (c / 32) is set when channel c of the row's target took its
 *                          max from position p.  Every position is written (all-zero masks included).
 *   pcc_gnn_fc1_pool_fwd : fc1 + act + bn3 statistics + global_mean_pool (:87-92): psum[B,256] = per-graph sums of
 *                          act(fc1(h)), partials [nblk][2][256]; the per-node [M,256] tensor never reaches HBM. */
int64_t pcc_gnn_packed_bytes(void);
int pcc_gnn_max_blocks(void);
int pcc_gnn_pack_weights(const float* w_rel2, const float* w_root2, const float* w_fc1, void* packed, int device, void* stream);
int pcc_gnn_conv1_fwd(const float* x, int F, const int64_t* rowptr, const int32_t* col, const float* w, int aggr,
                      const float* w_rel, const float* w_root, const float* bias, int64_t M, int act, float* agg_out,
                      float* z_out, float* partials, int* nblk_out, int device, void* stream);
int pcc_gnn_bn_finalize(const float* partials, int nblk, int Cn, int64_t rows, const float* gamma, const float* beta,
                        float eps, float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                        float* mean_out, float* invstd_out, int device, void* stream);
int pcc_gnn_bn_eval(const float* running_mean, const float* running_var, const float* gamma, const float* beta, float eps,
                    int Cn, float* scale, float* shift, int device, void* stream);
int pcc_gnn_bn_apply(const float* z, const float* scale, const float* shift, int64_t M, int act, void* h_bf16, int device,
                     void* stream);
int pcc_gnn_conv_fwd(const void* h_in_bf16, const int64_t* rowptr, const int32_t* col, const float* w, int aggr,
                     const void* packed, const float* bias, int64_t M, int act, void* agg_out_bf16, float* z_out,
                     float* partials, const int64_t* membership, float* psum, int64_t B, void* win, int* nblk_out, int device,
                     void* stream);
/* graph-sized glue of the pooled outputs: P = psum / max(n_g, 1), y = P * scale + shift (mean pool commuted with the affine) */
int pcc_gnn_pool_affine(const float* psum, const int64_t* counts, const float* scale, const float* shift, int64_t B, int Cn,
                        float* P, float* y, int device, void* stream);
int pcc_gnn_fc1_pool_fwd(const void* h_in_bf16, const void* packed, const float* bias, const int64_t* membership, int64_t M,
                         int64_t B, int act, float* psum, float* partials, int* nblk_out, int device, void* stream);
/*   backward (autograd of the above).  One block z = A W^T + b, a = act(z), h = a*scale + shift has
 *      dz = scale (dh - c1 - xhat c2) act'(z),  c1 = sum(dh)/M,  c2 = sum(dh xhat)/M,  xhat = (a - mean) invstd;
 *   the kernel that produces a gradient tensor dh also accumulates the two sums (partials [nblk][2][128]) — from its fp32
 *   values; the [M,128] gradient tensors themselves travel between the kernels in bf16 (they are GEMM / gather operands,
 *   rounded to bf16 by their consumer anyway; the traffic, not the arithmetic, bounds these kernels).
 *   pcc_gnn_bn_bwd_finalize : partial sums -> c1, c2, dgamma, dbeta.
 *   pcc_gnn_reduce          : out[i] = sum_b part[b*count + i] (weight-gradient partials).
 *   pcc_gnn_fc1_bwd         : recomputes z3 per tile; dz3 = (gs[graph] - kap - lam*xhat3) act'(z3) (gs / kap / lam carry the
 *                             mean-pool + bn3 backward, computed by the caller from [B,256]-sized data); dh_out = dz3 Wfc1
 *                             (bf16) + its bn2 sums; dw_part [nblk][256][128], db_part [nblk][256].
 *   pcc_gnn_conv_bwd        : dz in the operand prologue (dh [M,128] bf16, or dh_graph [B,128] fp32 + membership when the gradient is
 *                             the same row for every node of a graph: mean pooling straight after the block); dagg_out | droot_out (bf16) = dz [W_rel | W_root];
 *                             dw_part [nblk][128][256] = dz^T [agg | h_in] accumulated in TMEM; db_part [nblk][128].
 *   pcc_gnn_agg_bwd         : dh_inout[j] += sum_{e: src(e)=j} w_e dagg[dst(e)] (CSR by source) + the bn sums of the
 *                             previous block (z_prev, its mean / invstd).  ADD / MEAN: w_src carries 1/deg(dst) for mean.
 *                             MAX: only the channels edge e won count, win[pos_src[q]] (.) dagg[dst(e)], pos_src[E] =
 *                             CSR-by-target position of every by-source entry q, win = the masks of pcc_gnn_conv_fwd.
 *   pcc_gnn_conv1_bwd       : partials [nblk][128][2F+1] = (dW_rel | dW_root | db) of GraphConv 1. */
/* backward of the same glue from G = dL/dy [B, Cn]: gs = G f / n_g, kap = f sum(G) / M, lam = f sum(G xhat(P)) / M,
 * dgamma = sum(G xhat), dbeta = sum(G)   (f = s, or 1 with use_scale = 0) */
int pcc_gnn_pool_bwd_prep(const float* G, const float* P, const float* mu, const float* rinv, const float* s,
                          const int64_t* counts, int64_t B, int Cn, int64_t M, int use_scale, float* gs, float* kap, float* lam,
                          float* dgamma, float* dbeta, int device, void* stream);
int pcc_gnn_bn_bwd_finalize(const float* partials, int nblk, int Cn, int64_t rows, float* c1, float* c2, float* dgamma,
                            float* dbeta, int device, void* stream);
int pcc_gnn_reduce(const float* part, int nblk, int64_t count, float* out, int device, void* stream);
int pcc_gnn_fc1_bwd(const void* h_in_bf16, const void* packed, const float* bias, const int64_t* membership, const float* gs,
                    const float* kap, const float* lam, const float* mu3, const float* r3, const float* z_prev,
                    const float* mu_prev, const float* r_prev, int64_t M, int act, void* dh_out_bf16, float* stat_part,
                    float* dw_part, float* db_part, int* nblk_out, int device, void* stream);
int pcc_gnn_conv_bwd(const void* dh_bf16, const int64_t* membership, const float* dh_graph, const float* z, const float* bn_mean, const float* bn_invstd, const float* bn_scale,
                     const float* bn_c1, const float* bn_c2, const void* agg_bf16, const void* h_in_bf16, const void* packed,
                     int64_t M, int act, void* dagg_out_bf16, void* droot_out_bf16, float* dw_part, float* db_part, int* nblk_out,
                     int device, void* stream);
int pcc_gnn_agg_bwd(const void* dagg_bf16, const int64_t* rowptr_src, const int32_t* col_src, const float* w_src, int aggr,
                    const int32_t* pos_src, const void* win, void* dh_inout_bf16, const float* z_prev, const float* mu_prev,
                    const float* r_prev, int64_t M, int act, float* partials, int* nblk_out, int device, void* stream);
int pcc_gnn_conv1_bwd(const void* dh_bf16, const float* z, const float* bn_mean, const float* bn_invstd, const float* bn_scale,
                      const float* bn_c1, const float* bn_c2, const float* agg, const float* x, int F, int64_t M, int act,
                      float* partials, int* nblk_out, int device, void* stream);

/* ---- loss and row gather.
 *      pcc_bce_logits: nn.BCEWithLogitsLoss(reduction="mean") forward AND its gradient in one pass
 *      (/root/reference/models/wrapper.py:38,64-67): loss[1], dlogits[count] = (sigmoid(z) - y) / count.
 *      pcc_gather_rows: out[i,:] = x[clamp(idx[i]),:] for rows of d floats (argmax-row backward of max
 *      pooling, DESIGN.md §4).  Optional g_in / g_out [count]: g_out[i] = idx[i] >= 0 ? g_in[i] : 0 — the pooled
 *      gradient with the entries of empty sets (argmax -1, autograd routes nothing there) zeroed. */
int pcc_bce_logits(const float* logits, const float* target, int64_t count, float* loss, float* dlogits, int device,
                   void* stream);
int pcc_gather_rows(const float* x, const int32_t* idx, int64_t count, int d, int64_t n, float* out,
                    const float* g_in, float* g_out, int device, void* stream);

/* ---- accounting / measurement helpers used by bench.py.
 *      pcc_launch_count: kernels launched by this library since the last reset.
 *      pcc_prof_*: CUDA-event brackets around the three fused kernels, recorded on the launching
 *      stream (slot 0 = phi+pool forward, 1 = backward chain, 2 = wgrad).  Not for use under CUDA
 *      graph capture. */
int64_t pcc_launch_count(int reset);
int pcc_prof_enable(int on);
int pcc_prof_read(int slot, double* ms_total, int64_t* count);

/* ---- diagnostics: one-CTA tcgen05 GEMM on integer data, out[128,64] fp32.
 *      mode 0 = K-major operands (forward), 1 = MN-major B (dgrad), 2 = MN-major A and B
 *      (wgrad).  Expected values: tests/test_fused_gpu.py. */
int pcc_selftest_umma(int mode, float* out, int device, void* stream);
/* FP32 FMA throughput probe (roofline denominator of the kNN kernel): `blocks` blocks of 256 threads, 16 * iters
 * flops per thread; out[blocks*256].  The caller times it with CUDA events (tools/bench_knn.py). */
int pcc_selftest_fp32_peak(float* out, int blocks, int iters, int device, void* stream);
/* ---- fused multi-tensor Adam / AdamW step (SURVEY §8f rank 3): torch.optim.Adam / AdamW as constructed at
 *      /root/reference/models/wrapper.py:30-33 (default betas / eps; weight_decay 0 / 0.01), every parameter
 *      tensor in one launch.  table (device, [n_tensors][4] int64): {param pointer, grad pointer (0 = no gradient:
 *      skipped), numel, offset of the tensor's moments inside exp_avg / exp_avg_sq [total]} sorted by offset;
 *      step: device int64 scalar, incremented by the call (bias corrections use the incremented value);
 *      decoupled: 1 = AdamW, 0 = Adam (L2 term added to the gradient).  Capturable in a CUDA graph. */
int pcc_adam_step(const int64_t* table, int n_tensors, int64_t total, float* exp_avg, float* exp_avg_sq, int64_t* step,
                  float lr, float beta1, float beta2, float eps, float weight_decay, int decoupled, int device,
                  void* stream);

/* ---- gradient all-reduce over NVLink / NVSwitch peer memory (one process per GPU, one node; SURVEY.md §8e).
 *      One-shot: every rank stages its flat fp32 bucket in CUDA-IPC memory mapped by all peers, publishes a
 *      sequence number to every peer with a system-scope release, then sums all ranks' staging buffers in rank
 *      order (bitwise identical results everywhere) and writes scale * sum back into its bucket.  A plain kernel:
 *      capturable into the CUDA graph of the train step (an NCCL call is not, on this stack).
 *      pcc_peer_alloc: region = 1 KB of flags + 2 staging buffers of buf_bytes, allocated with cudaMalloc by the
 *      library (IPC export needs it — the one exception to caller-owned memory) + its 64-byte IPC handle;
 *      pcc_peer_open / _close map / unmap a peer's region; pcc_peer_free releases the local one.
 *      pcc_peer_allreduce: n % 4 == 0, 4 n <= buf_bytes, bucket 16-byte aligned; regions[world] in rank order;
 *      counters = 16 zeroed bytes of local device memory that persist across calls; every rank calls it the same
 *      number of times with the same n. */
int pcc_peer_alloc(int64_t buf_bytes, void** region, void* ipc_handle_64, int device);
int pcc_peer_open(const void* ipc_handle_64, void** region, int device);
int pcc_peer_close(void* region, int device);
int pcc_peer_free(void* region, int device);
int pcc_peer_allreduce(float* bucket, int64_t n, void* const* regions, int64_t buf_bytes, int rank, int world,
                       float scale, void* counters, int device, void* stream);

/* optional event trace of CTA 0 of the fused forward kernel into a device buffer of 3*4096 int64
 * (role, (id, clock64) pairs); NULL disables.  Development aid. */
int pcc_debug_set_trace(void* device_buf);
/* forward kernel selection for H = 256 without commuted pooling: 1 = CTA-pair kernel (cta_group::2, default; env
 * PCC_FWD_PAIR=0 disables), 0 = one CTA per SM.  Both compute the same function; tests compare them. */
int pcc_debug_set_fwd_pair(int on);
/* backward chain schedule for max pooling with two hidden layers: 1 = pipelined (the GEMMs run under the epilogue
 * passes, default), 0 = serial (one GEMM after another).  Both compute the same function; tests compare them. */
int pcc_debug_set_bwd_pipe(int on);
/* programmatic dependent launch between the kernels of the DeepSets train step (griddepcontrol: a kernel is
 * scheduled while its predecessor drains and waits for it before its first global access): 1 = on (default; env
 * PCC_PDL=0 disables), 0 = plain stream-ordered launches.  Same results either way; tests compare them. */
int pcc_debug_set_pdl(int on);

#ifdef __cplusplus
}
#endif
#endif /* PCC_H_ */
