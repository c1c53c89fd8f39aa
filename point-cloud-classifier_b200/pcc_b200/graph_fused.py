"""Host side of the fused bf16 GraphNet path (pcc_gnn_* in libpcc.so): GraphConv -> act -> BatchNorm1d (twice),
fc1 -> act -> bn3 -> global_mean_pool of /root/reference/models/graph_net.py:73-92 and their autograd as ONE
autograd Function over tcgen05 kernels.  bf16 operands (normalised activations h, aggregates, weights), fp32
accumulation, fp32 pre-activations and BatchNorm statistics.  Stated tolerance: tests/test_graph_fused_gpu.py.

Supported: hidden_dim 128 or 64 (64 runs the 128-wide kernels on zero-padded parameters: padded channels stay exactly 0
through conv / act / BatchNorm), deepchem_style True (fc1 per node, then mean pool) and False (mean pool straight after
conv2; fc1 / bn3 / fc2 then run on [B, .] tensors through the layer-wise ops), local_pooling add / mean / max,
input_dim <= 8, tanh / relu / gelu (configs/graph_net.yaml is inside).  hidden_dim 256 takes the fp32 layer-wise path.

Max aggregation: agg_i[c] = max_{e: dst(e)=i} w_e h[src(e)][c] (the product in fp32), 0 for a node without in-edges.
Ties go to the FIRST edge: the lowest position in the target's CSR-by-target row (the lowest edge id of an edge list,
the kNN slot order of a neighbour table), and the whole gradient of agg_i[c] goes to that edge.  In this mode h1 is
bf16, so exact ties between neighbours are common; the fp32 path applies the same rule.  Training writes one 16-byte
winner mask per edge in the conv2 forward (pcc_gnn_conv_fwd) that the aggregation backward reads at the edge's
CSR-by-target position (FusedGraph.by_src).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L
from ._lib import ACT, call, ptr

C_HID, C_FC = 128, 256


def supported(input_dim: int, hidden_dim: int, act: str, aggr: str, deepchem: bool) -> bool:
    return hidden_dim in (64, C_HID) and aggr in ("add", "mean", "max") and 1 <= input_dim <= 8 and act in ("tanh", "relu", "gelu")


class FusedGraph:
    """CSR views of a batched edge list in the layout the fused kernels read: rowptr int64 [n+1], col int32 [E]
    (neighbour node per slot), w fp32 [E] or None.  by_dst feeds the forward aggregation, by_src its transpose (for max
    aggregation with the CSR-by-target position of every by-source entry)."""

    def __init__(self, edges: Optional[torch.Tensor], n: int, weights: Optional[torch.Tensor], aggr: str, by_dst=None, k_uniform: int = 0,
                 block_offsets: Optional[torch.Tensor] = None):
        from .functional import GraphCSR
        self.n, self.aggr = n, aggr
        if edges is None and (by_dst is None or block_offsets is None or weights is not None):
            raise ValueError("a graph without an edge list needs by_dst and block_offsets (an unweighted kNN neighbour table)")
        self.E = edges.shape[1] if edges is not None else by_dst[1].numel()
        if self.E >= 2 ** 31 or n >= 2 ** 31:
            raise ValueError("the fused GraphNet kernels index nodes and edges with int32")
        self.k_uniform = k_uniform
        self.block_offsets = block_offsets           # [B+1] node range per cloud of a block-diagonal simple graph, or None
        weights = L.f32c(weights) if weights is not None else None    # the kernels read fp32 weights
        csr = None
        if by_dst is not None:                       # e.g. a kNN graph: k consecutive edges per target, already grouped
            self.rowptr_d, self.col_d = by_dst
            self.w_d = weights
            perm_d = None                            # slot p of by_dst is edge p
        else:
            csr = GraphCSR(edges, n)
            self.rowptr_d, perm_d = csr.by_dst
            pl = perm_d.long()
            self.col_d = edges[0][pl].to(torch.int32)
            self.w_d = weights[pl].contiguous() if weights is not None else None
        self._edges, self._weights, self._csr, self._perm_d = edges, weights, csr, perm_d
        self._src = None

    def by_src(self):
        """(rowptr_s int64 [n+1], col_s int32 [E] = target per slot, w_s fp32 [E] or None, pos_s): w_s folds 1 / deg(target)
        for mean; pos_s (max only, else None) int32 [E] = the CSR-by-target position of every by-source entry."""
        if self._src is None and self._weights is None and self.block_offsets is not None and self.k_uniform > 0:
            # kNN graph: per-cloud transpose in shared memory (pcc_csr_transpose_blocks); mean folds 1 / deg = 1 / k
            dev = L.require_cuda(self.col_d, self.block_offsets)
            rowptr_s = torch.empty(self.n + 1, dtype=torch.int64, device=self.col_d.device)
            col_s = torch.empty(max(self.E, 1), dtype=torch.int32, device=self.col_d.device)
            call("pcc_csr_transpose_blocks", ptr(self.col_d), int(self.k_uniform), ptr(self.block_offsets),
                 self.block_offsets.numel() - 1, self.n, ptr(rowptr_s), ptr(col_s), dev, L.stream_ptr(dev))
            w_s = pos_s = None
            if self.aggr == "mean":
                w_s = torch.full((max(self.E, 1),), 1.0 / self.k_uniform, dtype=torch.float32, device=self.col_d.device)
            if self.aggr == "max":
                pos_s = torch.empty(max(self.E, 1), dtype=torch.int32, device=self.col_d.device)
                call("pcc_csr_transpose_pos", ptr(self.col_d), int(self.k_uniform), self.n, ptr(rowptr_s), ptr(col_s), ptr(pos_s),
                     dev, L.stream_ptr(dev))
            self._src = (rowptr_s, col_s, w_s, pos_s)
        if self._src is None and self._weights is None and self.aggr == "add":
            # unweighted sum aggregation: transpose the int32 CSR directly (no edge-id permutation, no int64 index ops)
            dev = L.require_cuda(self.col_d)
            rowptr_s = torch.empty(self.n + 1, dtype=torch.int64, device=self.col_d.device)
            col_s = torch.empty(max(self.E, 1), dtype=torch.int32, device=self.col_d.device)
            ws = torch.empty(call("pcc_csr_workspace_bytes", self.n, self.E), dtype=torch.uint8, device=self.col_d.device)
            call("pcc_csr_transpose", ptr(self.col_d), ptr(self.rowptr_d), self.E, self.n, int(self.k_uniform), ptr(rowptr_s),
                 ptr(col_s), ptr(ws), dev, L.stream_ptr(dev))
            self._src = (rowptr_s, col_s, None, None)
        if self._src is None:
            from .functional import GraphCSR
            csr = self._csr or GraphCSR(self._edges, self.n)
            rowptr_s, perm_s = csr.by_src
            pl = perm_s.long()
            dst = self._edges[1][pl]
            col_s = dst.to(torch.int32)
            w_s = self._weights[pl] if self._weights is not None else None
            if self.aggr == "mean":                  # d agg_i / d x_j = w_e / deg(i)
                deg = (self.rowptr_d[1:] - self.rowptr_d[:-1]).clamp(min=1).to(torch.float32)
                inv = (1.0 / deg)[dst]
                w_s = inv if w_s is None else w_s * inv
            pos_s = None
            if self.aggr == "max":                   # by-target position of edge perm_s[q]: inv(perm_d)[perm_s[q]]
                if self._perm_d is None:
                    pos_s = perm_s
                else:
                    inv_d = torch.empty_like(self._perm_d)     # (both permutations hold max(E, 1) entries)
                    inv_d[self._perm_d[:self.E].long()] = torch.arange(self.E, dtype=torch.int32, device=inv_d.device)
                    pos_s = inv_d[pl] if self.E > 0 else inv_d
            self._src = (rowptr_s, col_s, w_s.contiguous() if w_s is not None else None, pos_s)
        return self._src


def _nblk():
    return C.c_int(0)


def _pad(t: torch.Tensor, shape, fill: float = 0.0) -> torch.Tensor:
    """t zero-extended (or `fill`-extended) to `shape` (hidden_dim 64 -> the 128-wide kernels)"""
    if tuple(t.shape) == tuple(shape):
        return L.f32c(t)
    out = torch.full(shape, fill, dtype=torch.float32, device=t.device)
    out[tuple(slice(0, n) for n in t.shape)] = t
    return out


class GraphNetFusedFn(torch.autograd.Function):
    """deepchem_style=True : (x, 14 params) -> y3[B,256] = bn3-normalised, mean-pooled act(fc1(.)) — everything before fc2.
    deepchem_style=False: (x, 10 params) -> pooled[B,hidden] = global_mean_pool(bn2(act(conv2(.)))) — everything before fc1.
    meta = (act, training, eps, momentum, deepchem, hidden, grad): grad = autograd was recording at the call (forward
    itself runs without it), so that max aggregation writes its winner masks only for a step that can run a backward."""

    @staticmethod
    def forward(ctx, x, membership, graph: FusedGraph, counts, meta, bufs, *params):
        act, training, eps, momentum, deepchem, Cr, grad = meta
        if deepchem:
            (w_rel1, b_rel1, w_root1, w_rel2, b_rel2, w_root2, g1, be1, g2, be2, w_fc1, b_fc1, g3, be3) = params
        else:
            (w_rel1, b_rel1, w_root1, w_rel2, b_rel2, w_root2, g1, be1, g2, be2) = params
            w_fc1 = b_fc1 = g3 = be3 = None
        x = L.f32c(x)
        membership = L.i64c(membership)              # the kernels read int64 graph ids
        dev = L.require_cuda(x, membership, *params)
        st = L.stream_ptr(dev)
        M, F = x.shape
        B = counts.numel()
        A = ACT[act]
        Ch = C_HID
        # hidden_dim 64: zero-padded parameters (gamma / beta padded with 0: the padded channels are 0 after every block)
        w_rel1, w_root1 = _pad(w_rel1, (Ch, F)), _pad(w_root1, (Ch, F))
        b_rel1, b_rel2 = _pad(b_rel1, (Ch,)), _pad(b_rel2, (Ch,))
        w_rel2, w_root2 = _pad(w_rel2, (Ch, Ch)), _pad(w_root2, (Ch, Ch))
        g1, be1, g2, be2 = _pad(g1, (Ch,)), _pad(be1, (Ch,)), _pad(g2, (Ch,)), _pad(be2, (Ch,))
        if deepchem:
            w_fc1, b_fc1, g3, be3 = _pad(w_fc1, (C_FC, Ch)), L.f32c(b_fc1), L.f32c(g3), L.f32c(be3)
        aggr = L.POOL[graph.aggr]
        f32 = dict(dtype=torch.float32, device=x.device)
        bf = dict(dtype=torch.bfloat16, device=x.device)
        nmax = call("pcc_gnn_max_blocks")
        part = torch.empty(nmax * 2 * C_FC, **f32)
        packed = torch.empty(call("pcc_gnn_packed_bytes"), dtype=torch.uint8, device=x.device)
        call("pcc_gnn_pack_weights", ptr(w_rel2), ptr(w_root2), ptr(w_fc1), ptr(packed), dev, st)

        def bn(layer, Cn, gamma, beta, nblk, rows):
            rm, rv = bufs[layer]
            real = rm.numel()
            rmp, rvp = (rm, rv) if real == Cn else (_pad(rm, (Cn,)), _pad(rv, (Cn,), 1.0))
            sc, sh, mu, rs = (torch.empty(Cn, **f32) for _ in range(4))
            if training:
                call("pcc_gnn_bn_finalize", ptr(part), nblk, Cn, rows, ptr(gamma), ptr(beta), eps, momentum, ptr(rmp), ptr(rvp),
                     ptr(sc), ptr(sh), ptr(mu), ptr(rs), dev, st)
                if real != Cn:
                    rm.copy_(rmp[:real])
                    rv.copy_(rvp[:real])
            else:
                call("pcc_gnn_bn_eval", ptr(rmp), ptr(rvp), ptr(gamma), ptr(beta), eps, Cn, ptr(sc), ptr(sh), dev, st)
                mu, rs = rmp, torch.rsqrt(rvp + eps)
            return sc, sh, mu, rs

        # ---- conv1 -> act -> bn1
        agg1 = torch.empty((M, F), **f32)
        z1 = torch.empty((M, Ch), **f32)
        nb = _nblk()
        call("pcc_gnn_conv1_fwd", ptr(x), F, ptr(graph.rowptr_d), ptr(graph.col_d), ptr(graph.w_d), aggr, ptr(w_rel1), ptr(w_root1),
             ptr(b_rel1), M, A, ptr(agg1), ptr(z1), ptr(part), C.byref(nb), dev, st)
        s1, t1, mu1, r1 = bn(0, Ch, g1, be1, nb.value, M)
        h1 = torch.empty((M, Ch), **bf)
        call("pcc_gnn_bn_apply", ptr(z1), ptr(s1), ptr(t1), M, A, ptr(h1), dev, st)
        # ---- conv2 -> act -> bn2 (gather + GEMM + statistics in one kernel; + per-graph sums when the pool follows at once)
        agg2 = torch.empty((M, Ch), **bf)
        z2 = torch.empty((M, Ch), **f32)
        psum2 = None if deepchem else torch.empty((B, Ch), **f32)
        # max aggregation: winner masks (16 bytes per edge) only when this step will run a backward
        win = None
        if graph.aggr == "max" and training and grad and any(ctx.needs_input_grad):
            win = torch.empty((max(graph.E, 1), 16), dtype=torch.uint8, device=x.device)
        call("pcc_gnn_conv_fwd", ptr(h1), ptr(graph.rowptr_d), ptr(graph.col_d), ptr(graph.w_d), aggr, ptr(packed), ptr(b_rel2), M, A,
             ptr(agg2), ptr(z2), ptr(part), ptr(membership) if not deepchem else None, ptr(psum2), B, ptr(win), C.byref(nb), dev, st)
        ctx.win = win
        s2, t2, mu2, r2 = bn(1, Ch, g2, be2, nb.value, M)
        counts = L.i64c(counts)
        ctx.graph, ctx.meta, ctx.shapes = graph, meta, (M, F, B)
        if not deepchem:
            # global_mean_pool(bn2(a2)) = bn2_affine(mean_graph(a2)): graph_net.py:96 with the pool commuted with the affine
            P2, out = torch.empty((B, Ch), **f32), torch.empty((B, Ch), **f32)
            call("pcc_gnn_pool_affine", ptr(psum2), ptr(counts), ptr(s2), ptr(t2), B, Ch, ptr(P2), ptr(out), dev, st)
            ctx.save_for_backward(x, membership, agg1, z1, h1, agg2, z2, P2, counts, packed, s1, mu1, r1, s2, mu2, r2)
            return out[:, :Cr].contiguous() if Cr != Ch else out
        h2 = torch.empty((M, Ch), **bf)
        call("pcc_gnn_bn_apply", ptr(z2), ptr(s2), ptr(t2), M, A, ptr(h2), dev, st)
        # ---- fc1 -> act -> bn3 -> global_mean_pool: only per-graph sums and the statistics leave the kernel
        psum = torch.empty((B, C_FC), **f32)
        call("pcc_gnn_fc1_pool_fwd", ptr(h2), ptr(packed), ptr(b_fc1), ptr(membership), M, B, A, ptr(psum), ptr(part), C.byref(nb),
             dev, st)
        s3, t3, mu3, r3 = bn(2, C_FC, g3, be3, nb.value, M)
        P, y3 = torch.empty((B, C_FC), **f32), torch.empty((B, C_FC), **f32)
        call("pcc_gnn_pool_affine", ptr(psum), ptr(counts), ptr(s3), ptr(t3), B, C_FC, ptr(P), ptr(y3), dev, st)
        ctx.save_for_backward(x, membership, agg1, z1, h1, agg2, z2, h2, P, counts, packed, b_fc1,
                              s1, mu1, r1, s2, mu2, r2, s3, mu3, r3)
        return y3

    @staticmethod
    def backward(ctx, G):
        act, training, eps, momentum, deepchem, Cr, _ = ctx.meta
        if not training:
            raise RuntimeError("the fused GraphNet backward uses batch statistics: call it in train() mode")
        graph = ctx.graph
        M, F, B = ctx.shapes
        Ch = C_HID
        G = L.f32c(G)
        dev = L.require_cuda(G)
        st = L.stream_ptr(dev)
        A = ACT[act]
        f32 = dict(dtype=torch.float32, device=G.device)
        nmax = call("pcc_gnn_max_blocks")
        nb = _nblk()
        stat = torch.empty(nmax * 2 * Ch, **f32)
        dagg2 = torch.empty((M, Ch), dtype=torch.bfloat16, device=G.device)
        droot = torch.empty((M, Ch), dtype=torch.bfloat16, device=G.device)   # becomes dh1 in place (pcc_gnn_agg_bwd)
        cw_part = torch.empty(148 * Ch * 2 * Ch, **f32)
        cb_part = torch.empty(148 * Ch, **f32)
        if deepchem:
            (x, membership, agg1, z1, h1, agg2, z2, h2, P, counts, packed, b_fc1,
             s1, mu1, r1, s2, mu2, r2, s3, mu3, r3) = ctx.saved_tensors
            # ---- bn3 + mean-pool backward: per-graph / per-channel terms (graph-sized tensors, one launch)
            gs = torch.empty((B, C_FC), **f32)
            kap, lam, d_g3, d_be3 = (torch.empty(C_FC, **f32) for _ in range(4))
            call("pcc_gnn_pool_bwd_prep", ptr(G), ptr(P), ptr(mu3), ptr(r3), ptr(s3), ptr(counts), B, C_FC, M, 1, ptr(gs), ptr(kap),
                 ptr(lam), ptr(d_g3), ptr(d_be3), dev, st)
            # ---- fc1 backward (+ bn2 sums)
            dh2 = torch.empty((M, Ch), dtype=torch.bfloat16, device=G.device)
            dw_part = torch.empty(148 * C_FC * Ch, **f32)
            db_part = torch.empty(148 * C_FC, **f32)
            call("pcc_gnn_fc1_bwd", ptr(h2), ptr(packed), ptr(b_fc1), ptr(membership), ptr(gs), ptr(kap), ptr(lam), ptr(mu3), ptr(r3),
                 ptr(z2), ptr(mu2), ptr(r2), M, A, ptr(dh2), ptr(stat), ptr(dw_part), ptr(db_part), C.byref(nb), dev, st)
            d_wfc1 = torch.empty((C_FC, Ch), **f32)
            d_bfc1 = torch.empty(C_FC, **f32)
            call("pcc_gnn_reduce", ptr(dw_part), nb.value, C_FC * Ch, ptr(d_wfc1), dev, st)
            call("pcc_gnn_reduce", ptr(db_part), nb.value, C_FC, ptr(d_bfc1), dev, st)
            c1, c2, d_g2, d_be2 = (torch.empty(Ch, **f32) for _ in range(4))
            call("pcc_gnn_bn_bwd_finalize", ptr(stat), nb.value, Ch, M, ptr(c1), ptr(c2), ptr(d_g2), ptr(d_be2), dev, st)
            # ---- conv2 backward: dz2 in the prologue, [dagg2 | droot] and dW in one kernel
            call("pcc_gnn_conv_bwd", ptr(dh2), None, None, ptr(z2), ptr(mu2), ptr(r2), ptr(s2), ptr(c1), ptr(c2), ptr(agg2), ptr(h1),
                 ptr(packed), M, A, ptr(dagg2), ptr(droot), ptr(cw_part), ptr(cb_part), C.byref(nb), dev, st)
        else:
            (x, membership, agg1, z1, h1, agg2, z2, P2, counts, packed, s1, mu1, r1, s2, mu2, r2) = ctx.saved_tensors
            if Cr != Ch:
                G = _pad(G, (B, Ch))
            # the gradient of h2 is the same row for every node of a graph: dh2[i] = G[g(i)] / n_g, so the two bn2 sums are
            # graph-sized reductions and the conv backward reads the row through the membership vector
            gsb = torch.empty((B, Ch), **f32)
            c1, c2, d_g2, d_be2 = (torch.empty(Ch, **f32) for _ in range(4))
            call("pcc_gnn_pool_bwd_prep", ptr(G), ptr(P2), ptr(mu2), ptr(r2), ptr(s2), ptr(counts), B, Ch, M, 0, ptr(gsb), ptr(c1),
                 ptr(c2), ptr(d_g2), ptr(d_be2), dev, st)
            call("pcc_gnn_conv_bwd", None, ptr(membership), ptr(gsb), ptr(z2), ptr(mu2), ptr(r2), ptr(s2), ptr(c1), ptr(c2), ptr(agg2),
                 ptr(h1), ptr(packed), M, A, ptr(dagg2), ptr(droot), ptr(cw_part), ptr(cb_part), C.byref(nb), dev, st)
        d_w2 = torch.empty((Ch, 2 * Ch), **f32)
        d_b2 = torch.empty(Ch, **f32)
        call("pcc_gnn_reduce", ptr(cw_part), nb.value, Ch * 2 * Ch, ptr(d_w2), dev, st)
        call("pcc_gnn_reduce", ptr(cb_part), nb.value, Ch, ptr(d_b2), dev, st)
        d_wrel2, d_wroot2 = d_w2[:Cr, :Cr].contiguous(), d_w2[:Cr, Ch:Ch + Cr].contiguous()
        # ---- dh1 = droot + A^T dagg2 (+ bn1 sums)
        rowptr_s, col_s, w_s, pos_s = graph.by_src()
        call("pcc_gnn_agg_bwd", ptr(dagg2), ptr(rowptr_s), ptr(col_s), ptr(w_s), L.POOL[graph.aggr], ptr(pos_s), ptr(ctx.win), ptr(droot),
             ptr(z1), ptr(mu1), ptr(r1), M, A, ptr(stat), C.byref(nb), dev, st)
        c1b, c2b, d_g1, d_be1 = (torch.empty(Ch, **f32) for _ in range(4))
        call("pcc_gnn_bn_bwd_finalize", ptr(stat), nb.value, Ch, M, ptr(c1b), ptr(c2b), ptr(d_g1), ptr(d_be1), dev, st)
        # ---- conv1 backward (weights only: x needs no gradient)
        W1 = 2 * F + 1
        p1 = torch.empty(592 * Ch * W1, **f32)
        call("pcc_gnn_conv1_bwd", ptr(droot), ptr(z1), ptr(mu1), ptr(r1), ptr(s1), ptr(c1b), ptr(c2b), ptr(agg1), ptr(x), F, M, A,
             ptr(p1), C.byref(nb), dev, st)
        d1 = torch.empty((Ch, W1), **f32)
        call("pcc_gnn_reduce", ptr(p1), nb.value, Ch * W1, ptr(d1), dev, st)
        d_wrel1, d_wroot1, d_b1 = d1[:Cr, :F].contiguous(), d1[:Cr, F:2 * F].contiguous(), d1[:Cr, 2 * F].contiguous()
        grads = [d_wrel1, d_b1, d_wroot1, d_wrel2, d_b2[:Cr].contiguous(), d_wroot2, d_g1[:Cr].contiguous(), d_be1[:Cr].contiguous(),
                 d_g2[:Cr].contiguous(), d_be2[:Cr].contiguous()]
        if deepchem:
            grads += [d_wfc1[:, :Cr].contiguous(), d_bfc1, d_g3, d_be3]
        return (None, None, None, None, None, None) + tuple(grads)
