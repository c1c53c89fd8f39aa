"""GPU: the fused bf16 GraphNet path (pcc_gnn_*: tcgen05 GraphConv / fc1 kernels, BatchNorm folded into producer epilogues
and consumer prologues) against the pinned oracle (oracle/graphnet_oracle.py, fp32).

Stated bf16 tolerance: the normalised activations h1 / h2, the aggregates and the conv2 / fc1 weights are rounded to bf16
(8-bit mantissa) before every tensor-core contraction; accumulation, pre-activations and BatchNorm statistics are fp32.
Two comparisons, per tensor, printed by the tests (measured on B200, profiles/r2/graph_fused_err_r2f.txt):
 (1) oracle with the SAME stated operand rounding (graphnet_oracle operand_rounding="bf16"): logits <= 1.5e-3 of max|ref|;
     gradients (relative Frobenius) <= 1.5e-2 for tanh / gelu, <= 3.3e-2 for relu (the backward additionally rounds the
     gradient tensors dz / dagg / dh that travel between its kernels to bf16, which the oracle does not model; bias
     gradients are near-cancelling sums).  Tolerances 2x measured: logits 3e-3, gradients 3e-2 (7e-2 relu).
 (2) the fp32 oracle: logits <= 7.3e-3 -> 1.5e-2; gradients <= 4.0e-2 (tanh / gelu) -> 8e-2, <= 0.14 (relu: ReLU masks
     flip where |z| is below the bf16 rounding noise, as in tests/test_fused_gpu.py) -> 0.3.
The general-graph, unsorted-membership, empty-graph and kNN-layout cases below hold the same bounds (measured on B200,
1000 W: logits <= 1.5e-3 / 1.0e-2, the latter for unsorted membership with deepchem_style=False, whose bn3 normalises over
5 graphs; gradients <= 1.3e-2 / 2.7e-2 for tanh / gelu, relu 5.9e-3 / 7.9e-2).
Two runs on the same values, once with int32 membership / float64 weights and once with int64 / fp32, agree to
SAME_LOGIT_TOL = 1e-5 in the logits (measured <= 2.3e-7) and SAME_GRAD_TOL = 5e-3 in the gradients: they are not
bit-identical because the per-graph sums use float atomics, and conv1.lin_rel.bias, a near-cancelling sum over nodes taken
after the bf16-rounded gradient tensors, moved by up to 6.4e-4 (relative Frobenius) between such runs.
The fp32 mode of the same module stays at rtol 1e-4 (tests/test_graph_gpu.py)."""
import numpy as np
import pytest
import torch

from helpers import rel_err, rel_l2
from oracle import graphnet_oracle as GO
from oracle import knn_oracle as KO

import pcc_b200

pytestmark = pytest.mark.gpu
LOGIT_TOL_Q, GRAD_TOL_Q, GRAD_TOL_Q_RELU = 3e-3, 3e-2, 7e-2   # vs the oracle with the stated bf16 operand rounding
LOGIT_TOL, GRAD_TOL, GRAD_TOL_RELU = 1.5e-2, 8e-2, 0.3   # vs the fp32 oracle
SAME_LOGIT_TOL, SAME_GRAD_TOL = 1e-5, 5e-3               # two runs on the same values, other index / weight dtypes


def _clouds(sizes, seed, F=4):
    g = torch.Generator().manual_seed(seed)
    n = sum(sizes)
    feats = torch.randn(n, F, generator=g)
    feats[:, 0] = torch.rand(n, generator=g)
    memb = torch.cat([torch.full((s,), i, dtype=torch.long) for i, s in enumerate(sizes)])
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return feats, memb, off


def _cfg(act, aggr, F=4, hidden=128, deepchem=True):
    return dict(input_dim=F, hidden_dim=hidden, output_dim=1, activation=act, use_gat=False, gat_heads=4, sag_pool=False,
                pool_ratio=0.5, local_pooling=aggr, global_pooling="mean", deepchem_style=deepchem)


def check_fused_step_against_oracles(cfg, sd, x, memb, edges, w, y, logits, grads, module, args, *, num_graphs=None,
                                     fwd_kwargs={}):
    """Compares one bf16 train step (forward + BCE + backward) that `module` ran from the parameters `sd` with the
    oracle with the stated bf16 operand rounding and with the fp32 oracle, both on the host tensors (x, memb, edges, w,
    y); then the running statistics the step left, and the eval-mode forward module(*args, num_graphs, **fwd_kwargs)
    on those statistics.  logits: the train-mode logits; grads: {GraphNet parameter name: gradient}; module: the
    GraphNet, or a KnnGraphNet (its GraphNet is module.net; `edges` is then the oracle's copy of the kNN graph it
    builds).  Prints the errors, asserts the stated tolerances and returns the eval-mode logits."""
    act = cfg["activation"]
    net = getattr(module, "net", module)
    ref_logits, _, ref_grads, ref_stats = GO.graphnet_train_step(sd, cfg, x, memb, edges, w, y, num_graphs=num_graphs)
    q_logits, _, q_grads, _ = GO.graphnet_train_step(sd, cfg, x, memb, edges, w, y, operand_rounding="bf16",
                                                     num_graphs=num_graphs)
    e_log, e_logq = rel_err(logits, ref_logits), rel_err(logits, q_logits)
    worst, worstq, rows = ("", 0.0), ("", 0.0), []
    for kname, ref in ref_grads.items():
        got = grads[kname]
        assert got is not None, kname
        e, eq = rel_l2(got, ref), rel_l2(got, q_grads[kname])
        rows.append(f"{kname}={eq:.1e}/{e:.1e}")
        if e > worst[1]:
            worst = (kname, e)
        if eq > worstq[1]:
            worstq = (kname, eq)
    hidden, deepchem = cfg["hidden_dim"], cfg["deepchem_style"]
    print(f"fused graphnet {act}/{cfg['local_pooling']}/w={w is not None}/F={cfg['input_dim']}/C={hidden}/deepchem={deepchem}/"
          f"n={x.shape[0]}/E={edges.shape[1]}/B={y.shape[0]}: logits {e_logq:.1e}/{e_log:.1e} (vs bf16-operand oracle / "
          f"fp32 oracle); worst grad {worstq[0]} {worstq[1]:.1e} / {worst[0]} {worst[1]:.1e}; " + " ".join(rows))
    assert e_logq < LOGIT_TOL_Q and e_log < LOGIT_TOL
    assert worstq[1] < (GRAD_TOL_Q_RELU if act == "relu" else GRAD_TOL_Q), worstq
    assert worst[1] < (GRAD_TOL_RELU if act == "relu" else GRAD_TOL), worst
    new_sd = net.state_dict()
    for kname, v in ref_stats.items():
        torch.testing.assert_close(new_sd[kname].cpu(), v, rtol=2e-2, atol=2e-3)
    # eval mode: running statistics
    module.eval()
    with torch.no_grad():
        ev = module(*args, num_graphs=num_graphs, **fwd_kwargs)
    sd_eval = {kk: v.cpu() for kk, v in new_sd.items()}
    ref_ev = GO.graphnet_forward(sd_eval, cfg, x, memb, edges, w, training=False, num_graphs=num_graphs)
    e_ev = rel_err(ev, ref_ev)
    print(f"  eval logits {e_ev:.1e} vs fp32 oracle on the running statistics; running statistics max |diff| "
          f"{max(float((new_sd[kname].cpu().double() - v.double()).abs().max()) for kname, v in ref_stats.items()):.1e}")
    assert e_ev < LOGIT_TOL
    return ev


def _check_fused_step(cfg, x, memb, edges, w, y, *, num_graphs=None, fwd_kwargs={}, module=None):
    """One bf16 train step (forward + BCE + backward) through check_fused_step_against_oracles.  module: a KnnGraphNet
    (called as module(x, memb); `edges` is then the oracle's copy of the kNN graph it builds), else a GraphNet is built
    from cfg and called on (x, memb, edges[, w]).  Returns the module and the train / eval logits."""
    sd = GO.init_state_dict(cfg, seed=23)
    if module is None:
        m = pcc_b200.GraphNet(**cfg, precision="bf16").cuda()
        args = [x.cuda(), memb.cuda(), edges.cuda()] + ([w.cuda()] if w is not None else [])
        net = m
    else:
        m = module.cuda()
        args = [x.cuda(), memb.cuda()]
        net = m.net
    net.load_state_dict(sd)
    m.train()
    logits = m(*args, num_graphs=num_graphs, **fwd_kwargs)
    assert net.last_path == "fused-bf16"
    torch.nn.BCEWithLogitsLoss()(logits, y.cuda()).backward()
    grads = {k: p.grad for k, p in net.named_parameters()}
    ev = check_fused_step_against_oracles(cfg, sd, x, memb, edges, w, y, logits, grads, m, args, num_graphs=num_graphs,
                                          fwd_kwargs=fwd_kwargs)
    return m, logits.detach(), ev


@pytest.mark.parametrize("act,aggr,use_w,F,sizes,k,hidden,deepchem", [
    ("tanh", "add", False, 4, [300, 200, 400, 256], 8, 128, True),       # configs/graph_net.yaml
    ("relu", "mean", True, 4, [129, 1000, 77], 6, 128, True),
    ("gelu", "add", True, 1, [64, 64, 500], 5, 128, True),
    ("tanh", "add", False, 4, [1024] * 20, 20, 128, True),               # more tiles than SMs: several tiles per CTA
    ("tanh", "add", False, 4, [300, 200, 400, 256], 8, 128, False),      # deepchem_style=False: pool straight after conv2
    ("gelu", "mean", True, 4, [129, 500, 77, 40], 6, 128, False),
    ("tanh", "add", False, 4, [300, 200, 400, 256], 8, 64, True),        # hidden_dim 64 (zero-padded to the 128-wide kernels)
    # (deepchem_style=False normalises over GRAPHS in bn3: 24 graphs keep that BatchNorm well conditioned)
    ("relu", "add", True, 1, [60, 45, 80, 33] * 6, 6, 64, False),
])
def test_fused_graphnet_train_step_matches_oracle(act, aggr, use_w, F, sizes, k, hidden, deepchem):
    cfg = _cfg(act, aggr, F, hidden, deepchem)
    feats, memb, off = _clouds(sizes, seed=21, F=max(F, 4))
    nbr, _ = KO.knn_neighbours(feats[:, 1:4].numpy(), off, k)
    edges = torch.from_numpy(KO.knn_edges(nbr))
    gen = torch.Generator().manual_seed(22)
    perm = torch.randperm(edges.shape[1], generator=gen)      # arbitrary edge order (general CSR build)
    edges = edges[:, perm].contiguous()
    x = feats[:, :F].contiguous()
    w = torch.rand(edges.shape[1], generator=gen) if use_w else None
    y = (torch.rand(len(sizes), 1, generator=gen) > 0.5).float()
    _check_fused_step(cfg, x, memb, edges, w, y)


HUB_DEGREES = (22, 42, 64, 300)   # 2, 2, 4 and 15 gather rounds of kSlotRows = 21 rows (pcc_gnn.cu)


def _general_graph(sizes, seed, fanout=500):
    """A random multigraph inside each graph of a batch stored back to back, in a random edge order:
     - background: every node receives 0..5 edges from random nodes of its graph;
     - hubs with in-degree HUB_DEGREES: one, two, three and many rounds of the forward gather;
     - two sources with out-degree `fanout` (long rows of the transposed graph in the backward);
     - nodes without in-edges: every 7th node and, when the batch spans 3 or more 128-node tiles, all of tile 1
       (nodes 128..255);
     - self loops and repeated edges.
    Returns (membership int64 [n], edges int64 [2, E])."""
    rng = np.random.default_rng(seed)
    n = int(sum(sizes))
    memb = np.repeat(np.arange(len(sizes)), sizes)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    lo, hi = off[memb], off[memb + 1]

    def same_graph(t):      # one random node of the graph of every node in t
        return lo[t] + (rng.random(len(t)) * (hi[t] - lo[t])).astype(np.int64)

    isolated = np.zeros(n, dtype=bool)
    isolated[::7] = True
    if n >= 3 * 128:
        isolated[128:256] = True
    hubs = rng.choice(np.flatnonzero(~isolated), len(HUB_DEGREES), replace=False)
    plain = ~isolated
    plain[hubs] = False                                   # the hubs keep exactly their stated in-degree
    deg = np.where(plain, rng.integers(0, 6, n), 0)
    deg[hubs] = HUB_DEGREES
    dst = np.repeat(np.arange(n), deg)
    src = same_graph(dst)
    targets = np.flatnonzero(plain)
    fan_src = rng.choice(n, 2, replace=False)
    fan_dst = np.concatenate([rng.choice(targets[memb[targets] == memb[s]], fanout) for s in fan_src])
    loops = rng.choice(targets, 20, replace=False)
    rep = rng.choice(np.flatnonzero(plain[dst]), 50, replace=False)
    src = np.concatenate([src, np.repeat(fan_src, fanout), loops, src[rep]])
    dst = np.concatenate([dst, fan_dst, loops, dst[rep]])
    order = rng.permutation(len(src))
    edges = np.stack([src[order], dst[order]])
    in_deg = np.bincount(edges[1], minlength=n)
    assert (in_deg[isolated] == 0).all() and (np.sort(in_deg[hubs]) == sorted(HUB_DEGREES)).all()
    return torch.from_numpy(memb), torch.from_numpy(edges)


def _general_inputs(sizes, F, use_w, seed, num_graphs=None):
    feats, _, _ = _clouds(sizes, seed=seed, F=max(F, 4))
    memb, edges = _general_graph(sizes, seed)
    gen = torch.Generator().manual_seed(seed + 1)
    w = torch.rand(edges.shape[1], generator=gen) if use_w else None
    y = (torch.rand(num_graphs or len(sizes), 1, generator=gen) > 0.5).float()
    return feats[:, :F].contiguous(), memb, edges, w, y


GENERAL = [300, 200, 400, 256, 180, 333]   # 1669 nodes, 14 tiles; tile 1 lies inside graph 0


@pytest.mark.parametrize("act,aggr,use_w,deepchem,hidden,sizes", [
    ("tanh", "add", False, True, 128, GENERAL),
    ("gelu", "add", True, True, 128, GENERAL),
    ("tanh", "mean", False, True, 128, GENERAL),
    ("gelu", "mean", True, True, 128, GENERAL),
    ("gelu", "add", False, False, 128, GENERAL),
    ("tanh", "add", True, False, 128, GENERAL),
    ("gelu", "mean", False, False, 128, GENERAL),
    ("tanh", "mean", True, False, 128, GENERAL),
    ("relu", "mean", True, True, 128, GENERAL),
    ("gelu", "add", True, False, 64, GENERAL),
    ("tanh", "mean", True, True, 128, [40, 50, 30]),      # M = 120: one partial tile
    ("gelu", "add", False, True, 128, [64, 65]),          # M = 129: a second tile with one row
])
def test_fused_graphnet_general_graph_matches_oracle(act, aggr, use_w, deepchem, hidden, sizes):
    """Edge lists that a kNN graph never produces: hubs that take several gather rounds, sources with hundreds of
    out-edges, nodes (and a whole tile) without in-edges, self loops, repeated edges, random edge order."""
    cfg = _cfg(act, aggr, 4, hidden, deepchem)
    x, memb, edges, w, y = _general_inputs(sizes, 4, use_w, seed=31)
    _check_fused_step(cfg, x, memb, edges, w, y)


@pytest.mark.parametrize("act,aggr,use_w,deepchem,sizes", [
    ("tanh", "add", False, True, [300, 200, 400, 256]),
    ("gelu", "mean", True, False, [150, 90, 220, 310, 170]),
])
def test_fused_graphnet_unsorted_membership_matches_oracle(act, aggr, use_w, deepchem, sizes):
    """Nodes of several graphs interleaved at random: every warp of 32 rows spans several graphs, so the per-graph sums
    of the forward take the per-row atomic branch everywhere (global_mean_pool does not require sorted membership)."""
    cfg = _cfg(act, aggr, 4, 128, deepchem)
    x, memb, edges, w, y = _general_inputs(sizes, 4, use_w, seed=41)
    pi = torch.randperm(x.shape[0], generator=torch.Generator().manual_seed(42))    # old node i -> new node pi[i]
    x2 = torch.empty_like(x)
    x2[pi] = x
    memb2 = torch.empty_like(memb)
    memb2[pi] = memb
    runs = int((memb2[1:] != memb2[:-1]).sum()) + 1
    assert runs > x.shape[0] // 2, runs
    _check_fused_step(cfg, x2, memb2, pi[edges], w, y)


@pytest.mark.parametrize("deepchem", [True, False])
def test_fused_graphnet_empty_graphs_pool_to_zero(deepchem):
    """Graphs without nodes (a gap in the membership ids, and trailing graphs through num_graphs) pool to 0, as
    global_mean_pool does: the bf16 module against both oracles in train and eval mode, the fp32 mode of the same module
    against the fp32 oracle at 1e-4 as the control."""
    sizes = [300, 0, 200, 400, 0, 256]
    B = len(sizes) + 2                                    # graphs 1, 4, 6 and 7 are empty
    empty = [1, 4, 6, 7]
    cfg = _cfg("tanh", "add", 4, 128, deepchem)
    x, memb, edges, w, y = _general_inputs(sizes, 4, True, seed=51, num_graphs=B)
    m, logits, ev = _check_fused_step(cfg, x, memb, edges, w, y, num_graphs=B)
    b2 = m.fc2.bias.detach()
    for name, out in (("train", logits), ("eval", ev)):
        print(f"empty graphs deepchem={deepchem} {name}: logits {out[empty, 0].tolist()} fc2.bias {b2.tolist()}")
    if deepchem:
        # pooled row 0 -> fc2(0) = fc2.bias, bit for bit
        for out in (logits, ev):
            assert torch.equal(out[empty], b2.expand(len(empty), -1))
    else:
        # eval: the pooled row 0 enters fc1 -> act -> bn3 (running statistics) -> fc2
        h = torch.tanh(m.fc1.bias.detach().cpu())
        h = (h - m.bn3.running_mean.cpu()) * torch.rsqrt(m.bn3.running_var.cpu() + m.bn3.eps) * m.bn3.weight.detach().cpu() \
            + m.bn3.bias.detach().cpu()
        ref = m.fc2.weight.detach().cpu() @ h + b2.cpu()
        torch.testing.assert_close(ev[empty].cpu(), ref.expand(len(empty), -1), rtol=1e-4, atol=1e-5)

    # control: the fp32 mode of the same module
    sd = GO.init_state_dict(cfg, seed=23)
    ref_logits, _, ref_grads, _ = GO.graphnet_train_step(sd, cfg, x, memb, edges, w, y, num_graphs=B)
    f = pcc_b200.GraphNet(**cfg, precision="fp32").cuda()
    f.load_state_dict(sd)
    f.train()
    args = [x.cuda(), memb.cuda(), edges.cuda(), w.cuda()]
    out = f(*args, num_graphs=B)
    assert f.last_path == "fp32"
    torch.nn.BCEWithLogitsLoss()(out, y.cuda()).backward()
    torch.testing.assert_close(out.detach().cpu(), ref_logits, rtol=1e-4, atol=1e-5)
    for kname, ref in ref_grads.items():
        got = dict(f.named_parameters())[kname].grad
        assert rel_err(got, ref) < 2e-4, (kname, rel_err(got, ref))
    f.eval()
    with torch.no_grad():
        ev32 = f(*args, num_graphs=B)
    sd_eval = {kk: v.cpu() for kk, v in f.state_dict().items()}
    torch.testing.assert_close(ev32.cpu(), GO.graphnet_forward(sd_eval, cfg, x, memb, edges, w, training=False, num_graphs=B),
                               rtol=1e-4, atol=1e-5)


KNN_SIZES = [300, 200, 400, 256]


def _knn_inputs(k, seed=61):
    feats, memb, off = _clouds(KNN_SIZES, seed=seed)
    nbr, _ = KO.knn_neighbours(feats[:, 1:4].numpy(), off, k)
    edges = torch.from_numpy(KO.knn_edges(nbr))
    n = feats.shape[0]
    # k consecutive edges per target, targets in node order, no repeated edge: what edges_sorted_by_target / simple_graph
    # and the kNN transpose take for granted
    assert edges.shape[1] == n * k
    assert torch.equal(edges[1], torch.arange(n).repeat_interleave(k))
    assert len(set(zip(edges[0].tolist(), edges[1].tolist()))) == n * k
    y = (torch.rand(len(KNN_SIZES), 1, generator=torch.Generator().manual_seed(seed + 1)) > 0.5).float()
    return feats, memb, edges, y


@pytest.mark.parametrize("aggr,k,simple", [
    ("add", 8, False),     # pcc_csr_transpose with k_uniform
    ("add", 8, True),      # per-cloud shared-memory transpose
    ("mean", 8, True),     # ... with the 1 / k weight folded in
    ("mean", 24, True),
])
def test_fused_graphnet_sorted_knn_edges_match_oracle(aggr, k, simple):
    """GraphNet.forward on a kNN edge list flagged edges_sorted_by_target (and simple_graph): the CSR views come from
    the uniform-degree transposes instead of the general CSR build."""
    feats, memb, edges, y = _knn_inputs(k)
    _check_fused_step(_cfg("gelu", aggr), feats, memb, edges, None, y,
                      fwd_kwargs=dict(edges_sorted_by_target=True, simple_graph=simple))


@pytest.mark.parametrize("aggr,k,hidden,act", [
    ("add", 8, 128, "tanh"),
    ("mean", 8, 128, "gelu"),
    ("add", 24, 128, "gelu"),    # k > 21: two gather rounds per node
    ("mean", 24, 128, "tanh"),
    ("add", 32, 128, "tanh"),
    ("mean", 32, 128, "gelu"),
    ("mean", 24, 64, "tanh"),
])
def test_knn_graphnet_bf16_matches_oracle(aggr, k, hidden, act):
    """KnnGraphNet in bf16 (device kNN build, neighbour table as the CSR by target, per-cloud transpose) against the
    oracle on the same graph: pcc_knn is bit-exact to the kNN oracle (tests/test_graph_gpu.py)."""
    feats, memb, edges, y = _knn_inputs(k)
    cfg = _cfg(act, aggr, 4, hidden)
    _check_fused_step(cfg, feats, memb, edges, None, y, module=pcc_b200.KnnGraphNet(k=k, precision="bf16", **cfg))


def _one_step(cfg, x, memb, edges, w, y):
    m = pcc_b200.GraphNet(**cfg, precision="bf16").cuda()
    m.load_state_dict(GO.init_state_dict(cfg, seed=23))
    m.train()
    logits = m(x.cuda(), memb.cuda(), edges.cuda(), w.cuda())
    assert m.last_path == "fused-bf16"
    torch.nn.BCEWithLogitsLoss()(logits, y.cuda()).backward()
    return logits.detach(), {k: p.grad for k, p in m.named_parameters()}


def _check_same_step(a, b, what):
    # not bit for bit: the per-graph sums use float atomics, so two runs of the same inputs differ (SAME_*_TOL)
    e = rel_err(b[0], a[0])
    errs = {k: rel_l2(b[1][k], g) for k, g in a[1].items()}
    print(f"{what}: logits {e:.1e}; grads " + " ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    assert e < SAME_LOGIT_TOL, e
    for k, v in errs.items():
        assert v < SAME_GRAD_TOL, (k, v)


@pytest.mark.parametrize("deepchem", [True, False])
def test_fused_graphnet_float64_weights(deepchem):
    """float64 edge weights are converted, not read as fp32 bit patterns"""
    cfg = _cfg("tanh", "mean", 4, 128, deepchem)
    x, memb, edges, w, y = _general_inputs(GENERAL, 4, True, seed=71)
    _check_same_step(_one_step(cfg, x, memb, edges, w, y), _one_step(cfg, x, memb, edges, w.double(), y), "float64 weights")


@pytest.mark.parametrize("deepchem", [True, False])
def test_fused_graphnet_int32_membership(deepchem):
    """int32 graph ids are converted, not read as int64"""
    cfg = _cfg("tanh", "add", 4, 128, deepchem)
    x, memb, edges, w, y = _general_inputs(GENERAL, 4, True, seed=72)
    _check_same_step(_one_step(cfg, x, memb, edges, w, y), _one_step(cfg, x, memb.int(), edges, w, y), "int32 membership")


def test_knn_graphnet_module_uses_fused_path_and_matches_fp32_mode():
    """KnnGraphNet (kNN build on device + GraphNet): the bf16 fused path against the fp32 mode of the same module"""
    cfg = _cfg("tanh", "add")
    feats, memb, _ = _clouds([512, 300, 700], seed=5)
    y = (torch.rand(3, 1, generator=torch.Generator().manual_seed(6)) > 0.5).float().cuda()
    torch.manual_seed(0)
    a = pcc_b200.KnnGraphNet(k=20, precision="bf16", **cfg).cuda()
    b = pcc_b200.KnnGraphNet(k=20, precision="fp32", **cfg).cuda()
    b.load_state_dict(a.state_dict())
    outs = []
    for m in (a, b):
        m.train()
        logits = m(feats.cuda(), memb.cuda(), num_graphs=3)
        torch.nn.BCEWithLogitsLoss()(logits, y).backward()
        outs.append((logits.detach(), {k: p.grad for k, p in m.named_parameters()}))
    assert a.net.last_path == "fused-bf16" and b.net.last_path == "fp32"
    assert rel_err(outs[0][0], outs[1][0]) < LOGIT_TOL
    for k, g in outs[1][1].items():
        assert rel_l2(outs[0][1][k], g) < GRAD_TOL, k


@pytest.mark.parametrize("sizes,k", [
    ([300, 200, 400, 256], 8),
    ([1024] * 5, 20),
    ([33, 1300, 21, 2900], 20),          # clouds beyond one bitmap pass (> ~1250 points)
    ([64], 5),
    ([16384, 300], 20),                  # the sweep's largest cloud: 245 bitmap passes
    ([8192, 8192], 20),
])
def test_csr_transpose_blocks_matches_numpy(sizes, k):
    """pcc_csr_transpose_blocks (per-cloud shared-memory transpose of a kNN graph) is bit-exact against a stable numpy
    transposition: rowptr by source, targets ascending inside a row — and equal to the generic pcc_csr_transpose."""
    import ctypes as C
    from pcc_b200 import _lib as L
    feats, memb, off = _clouds(sizes, seed=5)
    nbr, _ = KO.knn_neighbours(feats[:, 1:4].numpy(), off, k, rows_per_chunk=1024)
    n = feats.shape[0]
    src = nbr.reshape(-1).astype(np.int64)                 # slot p = (target p // k) <- source nbr
    tgt = np.repeat(np.arange(n, dtype=np.int64), k)
    order = np.lexsort((tgt, src))
    ref_col = tgt[order].astype(np.int32)
    ref_rowptr = np.concatenate([[0], np.cumsum(np.bincount(src, minlength=n))]).astype(np.int64)
    dev = torch.device("cuda:0")
    col_d = torch.from_numpy(src.astype(np.int32)).to(dev)
    offs = torch.from_numpy(off).to(dev)
    rowptr_s = torch.empty(n + 1, dtype=torch.int64, device=dev)
    col_s = torch.empty(n * k, dtype=torch.int32, device=dev)
    L.call("pcc_csr_transpose_blocks", L.ptr(col_d), k, L.ptr(offs), len(sizes), n, L.ptr(rowptr_s), L.ptr(col_s), 0,
           L.stream_ptr(0))
    torch.cuda.synchronize()
    assert np.array_equal(rowptr_s.cpu().numpy(), ref_rowptr)
    assert np.array_equal(col_s.cpu().numpy(), ref_col)
    # the generic transpose gives the same arrays
    rowptr_g = torch.empty(n + 1, dtype=torch.int64, device=dev)
    col_g = torch.empty(n * k, dtype=torch.int32, device=dev)
    ws = torch.empty(L.call("pcc_csr_workspace_bytes", n, n * k), dtype=torch.uint8, device=dev)
    L.call("pcc_csr_transpose", L.ptr(col_d), None, n * k, n, k, L.ptr(rowptr_g), L.ptr(col_g), L.ptr(ws), 0, L.stream_ptr(0))
    torch.cuda.synchronize()
    assert torch.equal(rowptr_g, rowptr_s) and torch.equal(col_g, col_s)
