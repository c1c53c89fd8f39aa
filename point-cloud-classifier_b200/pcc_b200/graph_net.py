"""B200-native GraphNet — drop-in for /root/reference/models/graph_net.py.

Same constructor kwargs (graph_net.py:10-22) and `forward(x, membership, edges,
weights=None)` (:65); same `state_dict` layout (`conv{1,2}.lin_rel.{weight,bias}`,
`conv{1,2}.lin_root.weight`, `bn{1,2,3}.*`, `fc1.*`, `fc2.*`).  `GraphConv` below is a
parameter container with PyG's parameter names; the arithmetic (neighbour aggregation,
dense layers, BatchNorm1d, segmented mean pool) runs in libpcc.so.  No CPU fallback and
no torch_geometric dependency.

Out of scope (SURVEY.md §2 row 3): `use_gat=True` (GATConv) and `sag_pool=True`
(SAGPooling) raise NotImplementedError instead of silently computing something else.
BatchNorm statistics are per process (per replica under data parallelism), as with
torch DDP's default.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn

from . import functional as PF
from . import graph_fused as GF


class GraphConv(nn.Module):
    """Parameter container with torch_geometric.nn.GraphConv's names:
    out_i = lin_rel(aggr_j w_ji x_j) + lin_root(x_i); lin_rel has the bias."""

    def __init__(self, in_channels: int, out_channels: int, aggr: str = "add"):
        super().__init__()
        if aggr not in ("add", "mean", "max"):
            raise ValueError("aggr must be 'add', 'mean' or 'max'")
        self.in_channels, self.out_channels, self.aggr = in_channels, out_channels, aggr
        self.lin_rel = nn.Linear(in_channels, out_channels, bias=True)
        self.lin_root = nn.Linear(in_channels, out_channels, bias=False)

    def forward(self, x, csr: PF.GraphCSR, weights, act: str):
        """act( lin_rel(agg) + lin_root(x) ) with the activation of graph_net.py:75,83 fused in."""
        agg = PF.graph_aggregate(x, weights, csr, self.aggr)
        root = PF.linear_act(x, self.lin_root.weight, None, None, "none")
        return PF.linear_act(agg, self.lin_rel.weight, self.lin_rel.bias, None, act, pre_add=root)


class GraphNet(nn.Module):

    def __init__(self,
                 input_dim,
                 hidden_dim,
                 output_dim,
                 activation,
                 use_gat=False,
                 gat_heads=4,
                 sag_pool=False,
                 pool_ratio=0.5,
                 local_pooling="add",
                 global_pooling="mean",
                 deepchem_style=False,
                 precision: Optional[str] = None):
        super().__init__()
        import os
        self.precision = precision or os.environ.get("PCC_GRAPH_PRECISION", "fp32")
        if self.precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        if use_gat:
            raise NotImplementedError("use_gat=True (GATConv, graph_net.py:47-48) is outside the B200 hot path")
        if sag_pool:
            raise NotImplementedError("sag_pool=True (SAGPooling, graph_net.py:57-58) is outside the B200 hot path")
        # the reference selects self.global_pooling here (:26-31) but forward never uses it
        # (:92,:96 hard-code global_mean_pool); kept for attribute compatibility.
        self.global_pooling = global_pooling
        self.deepchem_style = deepchem_style
        self.local_pooling = local_pooling
        self.sag_pool = sag_pool
        self.use_gat = use_gat

        if activation == "tanh":
            self.activation = nn.Tanh()
        elif activation == "relu":
            self.activation = nn.ReLU()
        elif activation == "gelu":
            self.activation = nn.GELU()
        self._act_name = activation

        self.conv1 = GraphConv(input_dim, hidden_dim, aggr=self.local_pooling)
        self.conv2 = GraphConv(hidden_dim, hidden_dim, aggr=self.local_pooling)
        self.bn1 = nn.BatchNorm1d(hidden_dim)
        self.bn2 = nn.BatchNorm1d(hidden_dim)
        self.fc1 = nn.Linear(hidden_dim, 256)
        self.bn3 = nn.BatchNorm1d(256)
        self.fc2 = nn.Linear(256, output_dim)
        self.last_path = None   # "fused-bf16" | "fp32": which kernels the last forward used

    def forward(self, x, membership, edges, weights=None, num_graphs: Optional[int] = None,
                edges_sorted_by_target: bool = False, simple_graph: bool = False):
        """edges_sorted_by_target: the edge list holds the same number of consecutive edges for every target node, in node
        order (a kNN graph).  simple_graph: additionally no edge is repeated (lets the bf16 path transpose the graph per
        cloud in shared memory; a violation traps)."""
        if not x.is_cuda:
            raise RuntimeError("pcc_b200.GraphNet runs on CUDA tensors only (sm_100a kernels, no CPU fallback)")
        if not hasattr(self, "activation"):
            raise AttributeError("'GraphNet' object has no attribute 'activation'")
        act = self._act_name
        n = x.shape[0]
        if num_graphs is None:
            num_graphs = PF.index_max(membership) + 1
        offsets = PF.segment_offsets(membership, num_graphs)
        if self.precision == "bf16" and self.fused_supported(x.shape[1]):
            return self._forward_fused(x, membership, edges, weights, offsets, edges_sorted_by_target, simple_graph)
        self.last_path = "fp32"
        csr = PF.GraphCSR(edges, n)

        h = self.conv1(x, csr, weights, act)
        h = PF.batchnorm(h, self.bn1)
        h = self.conv2(h, csr, weights, act)
        h = PF.batchnorm(h, self.bn2)
        if self.deepchem_style:
            h = PF.linear_act(h, self.fc1.weight, self.fc1.bias, None, act)
            h = PF.batchnorm(h, self.bn3)
            h = PF.segment_pool(h, offsets, "mean")
        else:
            h = PF.segment_pool(h, offsets, "mean")
            h = PF.linear_act(h, self.fc1.weight, self.fc1.bias, None, act)
            h = PF.batchnorm(h, self.bn3)
        return PF.linear_act(h, self.fc2.weight, self.fc2.bias, None, "none")


class KnnGraphNet(nn.Module):
    """GraphNet on a kNN graph built on the device from the node positions (north_star: "kNN graph build, ...,
    scatter aggregation"): forward(features[n, F], membership[n]) = GraphNet(features, membership,
    knn_graph(features, membership, k)).  The reference builds its edges offline (utils/data.py:847-929); this module
    is the on-device equivalent for raw point clouds and carries the same parameters / state_dict keys under `net.`."""

    def __init__(self, k: int = 20, pos_cols=(1, 4), precision: Optional[str] = None, **graphnet_kwargs):
        super().__init__()
        self.k, self.pos_cols = k, tuple(pos_cols)
        self.net = GraphNet(**graphnet_kwargs, precision=precision)

    def forward(self, features, membership, num_graphs: Optional[int] = None):
        if num_graphs is None:
            num_graphs = PF.index_max(membership) + 1
        net = self.net
        if features.is_cuda and net.precision == "bf16" and net.fused_supported(features.shape[1]):
            # fused path: the [n, k] neighbour table IS the CSR by target (k slots per node); no edge list is materialised
            offsets = PF.segment_offsets(membership, num_graphs)
            _, _, nbr32 = PF.knn(features[:, self.pos_cols[0]:self.pos_cols[1]], offsets, self.k, with_int32=True)
            return net._forward_fused(features, membership, None, None, offsets, True, True, nbr=nbr32)
        edges, _ = knn_graph(features, membership, self.k, self.pos_cols, num_graphs)
        return net(features, membership, edges, num_graphs=num_graphs, edges_sorted_by_target=True, simple_graph=True)


def _fused_methods():
    def fused_supported(self, input_dim=None) -> bool:
        F = self.conv1.in_channels if input_dim is None else input_dim
        return GF.supported(F, self.conv2.out_channels, self._act_name, self.local_pooling, self.deepchem_style) and \
            all(isinstance(b.momentum, float) for b in (self.bn1, self.bn2, self.bn3))

    def _forward_fused(self, x, membership, edges, weights, offsets, sorted_by_target, simple_graph=False, nbr=None):
        """bf16 tcgen05 path (graph_fused.py): one autograd Function for everything before fc2.  Either an edge list
        [2, E] or (KnnGraphNet) the neighbour table nbr[n, k] of a kNN graph."""
        n = x.shape[0]
        by_dst, k = None, 0
        if nbr is not None:
            k = nbr.shape[1]
            col = nbr.reshape(-1)
            by_dst = (torch.arange(n + 1, device=x.device, dtype=torch.int64) * k,
                      col if col.dtype == torch.int32 else col.to(torch.int32))
        else:
            E = edges.shape[1]
            edges = edges if edges.dtype == torch.int64 else edges.long()
            if sorted_by_target and n > 0 and E % n == 0:      # kNN graph: k consecutive edges per target node
                k = E // n
                by_dst = (torch.arange(n + 1, device=x.device, dtype=torch.int64) * k, edges[0].to(torch.int32))
        graph = GF.FusedGraph(edges, n, weights, self.local_pooling, by_dst=by_dst, k_uniform=k,
                              block_offsets=offsets if (simple_graph and by_dst is not None) else None)
        counts = offsets[1:] - offsets[:-1]
        bns = (self.bn1, self.bn2, self.bn3)
        bufs = [(b.running_mean, b.running_var) for b in bns]
        hidden = self.conv2.out_channels
        meta = (self._act_name, self.training, float(self.bn1.eps), float(self.bn1.momentum), bool(self.deepchem_style), hidden,
                torch.is_grad_enabled())
        params = (self.conv1.lin_rel.weight, self.conv1.lin_rel.bias, self.conv1.lin_root.weight,
                  self.conv2.lin_rel.weight, self.conv2.lin_rel.bias, self.conv2.lin_root.weight,
                  self.bn1.weight, self.bn1.bias, self.bn2.weight, self.bn2.bias)
        self.last_path = "fused-bf16"
        if self.deepchem_style:
            params += (self.fc1.weight, self.fc1.bias, self.bn3.weight, self.bn3.bias)
            y3 = GF.GraphNetFusedFn.apply(x, membership, graph, counts, meta, bufs, *params)
            if self.training:
                for b in bns:
                    b.num_batches_tracked.add_(1)
            return PF.linear_act(y3, self.fc2.weight, self.fc2.bias, None, "none")
        # deepchem_style=False (graph_net.py:94-100): pool first, then fc1 -> act -> bn3 on [B, .] (layer-wise ops)
        pooled = GF.GraphNetFusedFn.apply(x, membership, graph, counts, meta, bufs[:2], *params)
        if self.training:
            for b in bns[:2]:
                b.num_batches_tracked.add_(1)
        h = PF.linear_act(pooled, self.fc1.weight, self.fc1.bias, None, self._act_name)
        h = PF.batchnorm(h, self.bn3)
        return PF.linear_act(h, self.fc2.weight, self.fc2.bias, None, "none")

    GraphNet.fused_supported = fused_supported
    GraphNet._forward_fused = _forward_fused


_fused_methods()


def knn_graph(features: torch.Tensor, membership: torch.Tensor, k: int = 20, pos_cols=(1, 4),
              num_graphs: Optional[int] = None):
    """kNN edge list in GraphConv's convention (row 0 = neighbour, row 1 = centre) over the
    position columns of the node features (cols 1:4, cf. utils/data.py:808-813, 837).
    Every cloud must have more than k points (otherwise use functional.knn and filter)."""
    if num_graphs is None:
        num_graphs = PF.index_max(membership) + 1
    offsets = PF.segment_offsets(membership, num_graphs)
    pos = features[:, pos_cols[0]:pos_cols[1]]
    nbr, d2 = PF.knn(pos, offsets, k)
    return PF.knn_edges(nbr), d2


def gaussian_edge_weights(features: torch.Tensor, edges: torch.Tensor, membership: torch.Tensor,
                          num_graphs: Optional[int] = None, pos_cols=(1, 4), eps: float = 1e-6) -> torch.Tensor:
    """Edge weights of the reference's graph dataset (utils/data.py:835-845, `use_weights: true`) computed on the
    device for a collated batch (utils/data.py:1228-1261: graphs back to back, node-offset edges): one
    sigma = median edge length + eps per graph.  The edges of a graph must be contiguous (what the collate and
    `knn_graph` produce)."""
    if num_graphs is None:
        num_graphs = PF.index_max(membership) + 1
    edge_graph = membership[edges[1]].contiguous()            # graph of every edge (by its centre node)
    edge_offsets = PF.segment_offsets(edge_graph, num_graphs)
    return PF.edge_weights(features[:, pos_cols[0]:pos_cols[1]], edges, edge_offsets, eps)
