"""CPU oracle for the graph_net neighbour stage.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this file.  The product never does.

PARITY UNPINNED for the third-party pieces: the arithmetic of GraphConv and
global_mean_pool lives in `torch_geometric` (imported at
/root/reference/models/graph_net.py:5; call sites :50-51, :73, :82, :92, :96), which is
not vendored, not pinned (no requirements file / lock) and not installable here (no
network).  Their published semantics are restated below:

  GraphConv(in, out, aggr):  out_i = lin_rel( aggr_{e: dst(e)=i} w_e * x[src(e)] ) + lin_root(x_i)
      lin_rel has a bias, lin_root has none; edge_index row 0 = source j, row 1 = target i
      (flow source_to_target); aggr in add/mean/max; a node with no incoming edge
      aggregates to 0 (PyG scatter with include_self=False on a zero-filled output).
  global_mean_pool(x, batch): segment mean of rows by `batch`, size = batch.max()+1.

Pinned all the same, as far as the reference itself reaches (tests/test_oracle_golden.py, CPU):
  * the control flow, BatchNorm / Linear / activation arithmetic and state_dict keys against outputs of the
    reference's OWN models/graph_net.py, run by oracle/gen_golden_graphnet.py with an independent loop-based
    stand-in for the absent torch_geometric kernels (tests/golden/graphnet_*.npz: logits, loss, every gradient,
    running statistics, eval logits);
  * `_bn` against torch.nn.BatchNorm1d, `graph_aggregate` / `global_mean_pool` against torch.scatter_reduce
    (include_self=False on a zero-filled output), values and gradients.

Control flow follows /root/reference/models/graph_net.py:65-104 (activation BEFORE
BatchNorm, :75-76; forward hard-codes global_mean_pool in both branches, :92,:96;
fc1 width 256 hard-coded, :61).  BatchNorm1d is torch's own (train-mode batch
statistics with biased variance, running stats momentum 0.1 with unbiased variance).
The kNN graph build (north_star) has no reference counterpart at all: see knn_oracle.py.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.nn.functional as F


def _act(name: str, z: torch.Tensor) -> torch.Tensor:
    if name == "tanh":
        return torch.tanh(z)
    if name == "relu":
        return torch.relu(z)
    if name == "gelu":
        return 0.5 * z * (1.0 + torch.erf(z * (1.0 / math.sqrt(2.0))))
    raise AttributeError(f"unknown activation {name!r}")  # graph_net.py:38-43 leaves it unset


def graph_aggregate(x: torch.Tensor, edges: torch.Tensor, weights: Optional[torch.Tensor], aggr: str) -> torch.Tensor:
    n, C = x.shape
    src, dst = edges[0], edges[1]
    msg = x.index_select(0, src)
    if weights is not None:
        msg = msg * weights.view(-1, 1)
    out = x.new_zeros((n, C))
    if aggr == "add":
        out = out.index_add(0, dst, msg)
    elif aggr == "mean":
        out = out.index_add(0, dst, msg)
        deg = torch.zeros(n, dtype=x.dtype, device=x.device).index_add(0, dst, torch.ones_like(dst, dtype=x.dtype))
        out = out / deg.clamp(min=1.0).view(-1, 1)
    elif aggr == "max":
        out = out.scatter_reduce(0, dst.view(-1, 1).expand(-1, C), msg, reduce="amax", include_self=False)
    else:
        raise ValueError(f"unknown aggr {aggr!r}")
    return out


def _round_bf16_ste(t: torch.Tensor) -> torch.Tensor:
    """value rounded to bf16 (round-to-nearest-even), identity gradient"""
    return t + (t.to(torch.bfloat16).to(t.dtype) - t).detach()


def graphconv(sd, prefix: str, x, edges, weights, aggr: str, q=None) -> torch.Tensor:
    """q: operand rounding of the product's bf16 mode (aggregate and weights rounded to bf16; x arrives rounded)"""
    agg = graph_aggregate(x, edges, weights, aggr)
    w_rel, w_root = sd[prefix + ".lin_rel.weight"], sd[prefix + ".lin_root.weight"]
    if q is not None:
        agg, w_rel, w_root = q(agg), q(w_rel), q(w_root)
    return F.linear(agg, w_rel, sd[prefix + ".lin_rel.bias"]) + F.linear(x, w_root)


def global_mean_pool(x: torch.Tensor, membership: torch.Tensor, num_graphs: Optional[int] = None) -> torch.Tensor:
    """num_graphs (PyG's `size`): defaults to membership.max() + 1; a graph without nodes pools to 0"""
    B = int(membership.max()) + 1 if num_graphs is None else int(num_graphs)
    out = x.new_zeros((B, x.shape[1])).index_add(0, membership, x)
    cnt = torch.zeros(B, dtype=x.dtype, device=x.device).index_add(0, membership, torch.ones_like(membership, dtype=x.dtype))
    return out / cnt.clamp(min=1.0).view(-1, 1)


def _bn(sd, prefix: str, x: torch.Tensor, training: bool, stats_out: Optional[dict]) -> torch.Tensor:
    w, b = sd[prefix + ".weight"], sd[prefix + ".bias"]
    if training:
        mean = x.mean(dim=0)
        var = ((x - mean) ** 2).mean(dim=0)
        if stats_out is not None:
            n = x.shape[0]
            unbiased = var * (n / max(n - 1, 1))
            stats_out[prefix + ".running_mean"] = 0.9 * sd[prefix + ".running_mean"] + 0.1 * mean.detach()
            stats_out[prefix + ".running_var"] = 0.9 * sd[prefix + ".running_var"] + 0.1 * unbiased.detach()
            stats_out[prefix + ".num_batches_tracked"] = sd[prefix + ".num_batches_tracked"] + 1
    else:
        mean, var = sd[prefix + ".running_mean"], sd[prefix + ".running_var"]
    return (x - mean) * torch.rsqrt(var + 1e-5) * w + b


def graphnet_forward(sd: Dict[str, torch.Tensor], cfg: dict, x, membership, edges, weights=None,
                     training: bool = True, stats_out: Optional[dict] = None,
                     operand_rounding: Optional[str] = None, num_graphs: Optional[int] = None) -> torch.Tensor:
    """cfg keys = the reference ctor kwargs (graph_net.py:10-22); only the
    use_gat=False, sag_pool=False branch (configs/graph_net.yaml:6,8) is restated.
    operand_rounding="bf16": the STATED arithmetic of the product's bf16 GraphNet mode — the normalised activations h1
    (and h2 when fc1 runs per node, deepchem_style), the conv2 aggregate and the conv2 (/ fc1) weights are rounded to
    bf16; products and sums, pre-activations, BatchNorm statistics, conv1, the pooled tensors and the graph-level layers
    stay fp32.  Same algorithm, stated operand precision.
    num_graphs: number of graphs of the batch (default membership.max() + 1; larger values append empty graphs)."""
    if cfg.get("use_gat", False) or cfg.get("sag_pool", False):
        raise NotImplementedError("GATConv / SAGPooling branches are out of scope (SURVEY.md §2 row 3)")
    act = cfg["activation"]
    aggr = cfg.get("local_pooling", "add")
    q = _round_bf16_ste if operand_rounding == "bf16" else None
    h = graphconv(sd, "conv1", x, edges, weights, aggr)
    h = _bn(sd, "bn1", _act(act, h), training, stats_out)
    if q is not None:
        h = q(h)
    h = graphconv(sd, "conv2", h, edges, weights, aggr, q)
    h = _bn(sd, "bn2", _act(act, h), training, stats_out)
    if q is not None and cfg.get("deepchem_style", False):
        h = q(h)     # h2 feeds the fc1 tensor-core contraction (deepchem); otherwise it is pooled in fp32, never rounded
    if cfg.get("deepchem_style", False):
        h = F.linear(h, q(sd["fc1.weight"]) if q is not None else sd["fc1.weight"], sd["fc1.bias"])
        h = _bn(sd, "bn3", _act(act, h), training, stats_out)
        h = global_mean_pool(h, membership, num_graphs)
    else:
        h = global_mean_pool(h, membership, num_graphs)
        h = F.linear(h, sd["fc1.weight"], sd["fc1.bias"])
        h = _bn(sd, "bn3", _act(act, h), training, stats_out)
    return F.linear(h, sd["fc2.weight"], sd["fc2.bias"])


TRAINABLE = ("conv1.lin_rel.weight", "conv1.lin_rel.bias", "conv1.lin_root.weight",
             "conv2.lin_rel.weight", "conv2.lin_rel.bias", "conv2.lin_root.weight",
             "bn1.weight", "bn1.bias", "bn2.weight", "bn2.bias", "bn3.weight", "bn3.bias",
             "fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias")


def graphnet_train_step(sd, cfg, x, membership, edges, weights, y, operand_rounding: Optional[str] = None,
                        num_graphs: Optional[int] = None):
    leaves = {k: (v.detach().clone().requires_grad_(True) if k in TRAINABLE else v) for k, v in sd.items()}
    stats = {}
    logits = graphnet_forward(leaves, cfg, x, membership, edges, weights, training=True, stats_out=stats,
                              operand_rounding=operand_rounding, num_graphs=num_graphs)
    loss = F.binary_cross_entropy_with_logits(logits, y)
    loss.backward()
    grads = {k: leaves[k].grad for k in TRAINABLE}
    return logits.detach(), loss.detach(), grads, stats


def init_state_dict(cfg: dict, seed: int = 0, dtype=torch.float32) -> Dict[str, torch.Tensor]:
    g = torch.Generator().manual_seed(seed)
    F_in, Hd, out = cfg["input_dim"], cfg["hidden_dim"], cfg["output_dim"]

    def lin(o, i):
        bound = 1.0 / math.sqrt(i)
        return ((torch.rand(o, i, generator=g) * 2 - 1) * bound).to(dtype), \
            ((torch.rand(o, generator=g) * 2 - 1) * bound).to(dtype)

    sd = {}
    for name, (i, o) in (("conv1", (F_in, Hd)), ("conv2", (Hd, Hd))):
        w, b = lin(o, i)
        sd[f"{name}.lin_rel.weight"], sd[f"{name}.lin_rel.bias"] = w, b
        sd[f"{name}.lin_root.weight"] = lin(o, i)[0]
    for name, c in (("bn1", Hd), ("bn2", Hd), ("bn3", 256)):
        sd[f"{name}.weight"] = (1.0 + 0.1 * torch.randn(c, generator=g)).to(dtype)
        sd[f"{name}.bias"] = (0.1 * torch.randn(c, generator=g)).to(dtype)
        sd[f"{name}.running_mean"] = torch.zeros(c, dtype=dtype)
        sd[f"{name}.running_var"] = torch.ones(c, dtype=dtype)
        sd[f"{name}.num_batches_tracked"] = torch.tensor(0, dtype=torch.int64)
    sd["fc1.weight"], sd["fc1.bias"] = lin(256, Hd)
    sd["fc2.weight"], sd["fc2.bias"] = lin(out, 256)
    return sd
