"""Test-side restatement of the tie rule the fused bf16 GraphNet path states for max aggregation.

oracle/graphnet_oracle.py restates PyG: max aggregation through scatter_reduce("amax"), whose gradient splits evenly
among tied edges.  The product's bf16 mode (pcc_b200/graph_fused.py) states the FIRST-EDGE rule instead: among the
edges that reach the max, the one with the lowest edge id (the lowest position in the target's CSR-by-target row)
takes the whole gradient.  The forward values are the same under both rules.  With bf16 h1 exact ties between
neighbours are common, so the rule is part of that mode's stated arithmetic.

`graph_aggregate_first_edge` is the rule.  `bf16_oracle_first_edge(monkeypatch)` makes the oracle's bf16 mode
(graphnet_forward(..., operand_rounding="bf16"), which hands conv2 the rounding function q) aggregate with it; the fp32
oracle (q = None) keeps scatter_reduce.  conv1 is left to the oracle in both modes: x takes no gradient, and the
forward values do not depend on the rule."""
from typing import Optional

import torch
import torch.nn.functional as F

from oracle import graphnet_oracle as GO


def graph_aggregate_first_edge(x: torch.Tensor, edges: torch.Tensor, weights: Optional[torch.Tensor]) -> torch.Tensor:
    """agg_i = max_{e: dst(e)=i} w_e x[src(e)] (0 without in-edges); the gradient of agg_i[c] goes wholly to the lowest
    edge id that reaches the max"""
    n, C = x.shape
    src, dst = edges[0], edges[1]
    msg = x.index_select(0, src)
    if weights is not None:
        msg = msg * weights.view(-1, 1)
    E = msg.shape[0]
    idx = dst.view(-1, 1).expand(-1, C)
    best = x.new_zeros((n, C)).scatter_reduce(0, idx, msg.detach(), reduce="amax", include_self=False)
    # winner per (node, channel): the lowest edge id whose message equals the max; E (a zero row) without in-edges
    eid = torch.arange(E, device=x.device).view(-1, 1).expand(-1, C)
    cand = torch.where(msg.detach() == best.index_select(0, dst), eid, torch.full_like(eid, E))
    win = torch.full((n, C), E, dtype=torch.long, device=x.device).scatter_reduce(0, idx, cand, reduce="amin",
                                                                                 include_self=True)
    return torch.cat([msg, msg.new_zeros((1, C))]).gather(0, win)


_graphconv = GO.graphconv


def graphconv_first_edge(sd, prefix: str, x, edges, weights, aggr: str, q=None) -> torch.Tensor:
    """GO.graphconv with the first-edge rule for max aggregation in the bf16 mode (q given)"""
    if aggr != "max" or q is None:
        return _graphconv(sd, prefix, x, edges, weights, aggr, q)
    agg = graph_aggregate_first_edge(x, edges, weights)
    w_rel, w_root = sd[prefix + ".lin_rel.weight"], sd[prefix + ".lin_root.weight"]
    agg, w_rel, w_root = q(agg), q(w_rel), q(w_root)
    return F.linear(agg, w_rel, sd[prefix + ".lin_rel.bias"]) + F.linear(x, w_root)


def bf16_oracle_first_edge(monkeypatch):
    monkeypatch.setattr(GO, "graphconv", graphconv_first_edge)
