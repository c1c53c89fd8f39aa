"""CPU: the first-edge tie rule of max aggregation (tests/graph_max_ref.py), the arithmetic the fused bf16 GraphNet path
states for local_pooling="max", against the oracle's scatter_reduce("amax").  The forward values are the oracle's;
among tied edges the lowest edge id takes the whole gradient, where scatter_reduce splits it evenly; without ties both
gradients agree.  A node without in-edges aggregates to 0 and passes no gradient."""
import torch

from graph_max_ref import bf16_oracle_first_edge, graph_aggregate_first_edge
from oracle import graphnet_oracle as GO


def _split(x, edges, w):
    return GO.graph_aggregate(x, edges, w, "max")


def _first(x, edges, w):
    return graph_aggregate_first_edge(x, edges, w)


def _grads(fn, x, edges, w, g):
    x = x.detach().clone().requires_grad_(True)
    out = fn(x, edges, w)
    (out * g).sum().backward()
    return out.detach(), x.grad


def _random_graph(n, E, seed):
    gen = torch.Generator().manual_seed(seed)
    edges = torch.stack([torch.randint(0, n, (E,), generator=gen), torch.randint(0, n, (E,), generator=gen)])
    return edges, gen


def test_forward_values_equal_scatter_reduce():
    n, C = 50, 16
    edges, gen = _random_graph(n, 300, 0)
    for x in (torch.randn(n, C, generator=gen),
              torch.randint(-3, 4, (n, C), generator=gen).float(),       # many exact ties
              -torch.rand(n, C, generator=gen) - 0.5):                    # all messages negative
        for w in (None, torch.rand(edges.shape[1], generator=gen), torch.randint(1, 3, (edges.shape[1],), generator=gen).float()):
            assert torch.equal(_first(x, edges, w), _split(x, edges, w))


def test_ties_send_the_whole_gradient_to_the_lowest_edge_id():
    # node 0 receives from nodes 1, 2, 3 (edge ids 0, 1, 2) and all three messages tie in channel 0; in channel 1 the
    # tie is between edges 1 and 2 only
    x = torch.tensor([[0.0, 0.0], [5.0, 1.0], [5.0, 7.0], [5.0, 7.0]])
    edges = torch.tensor([[1, 2, 3], [0, 0, 0]])
    g = torch.tensor([[2.0, 3.0], [0.0, 0.0], [0.0, 0.0], [0.0, 0.0]])
    out, dx = _grads(_first, x, edges, None, g)
    assert out[0].tolist() == [5.0, 7.0]
    assert dx.tolist() == [[0.0, 0.0], [2.0, 0.0], [0.0, 3.0], [0.0, 0.0]]
    _, dx_split = _grads(_split, x, edges, None, g)
    assert torch.allclose(dx_split, torch.tensor([[0.0, 0.0], [2 / 3, 0.0], [2 / 3, 1.5], [2 / 3, 1.5]]))
    # the rule follows edge ids, not node ids: reversed edge order moves the winner to node 3
    _, dx_rev = _grads(_first, x, edges.flip(1), None, g)
    assert dx_rev.tolist() == [[0.0, 0.0], [0.0, 0.0], [0.0, 0.0], [2.0, 3.0]]


def test_without_ties_the_gradient_equals_the_even_split():
    n, C = 60, 8
    edges, gen = _random_graph(n, 400, 1)
    x = torch.randn(n, C, generator=gen, dtype=torch.float64)   # continuous values: no ties
    w = torch.rand(edges.shape[1], generator=gen, dtype=torch.float64) + 0.1
    g = torch.randn(n, C, generator=gen, dtype=torch.float64)
    o1, d1 = _grads(_first, x, edges, w, g)
    o2, d2 = _grads(_split, x, edges, w, g)
    assert torch.equal(o1, o2)
    assert torch.allclose(d1, d2, rtol=0, atol=1e-12)


def test_empty_neighbourhoods_aggregate_to_zero():
    x = torch.tensor([[-4.0, 2.0], [-1.0, -3.0], [6.0, 6.0]])
    edges = torch.tensor([[0, 1], [1, 1]])                  # node 1 <- 0, 1; nodes 0 and 2 have no in-edge
    g = torch.ones(3, 2)
    out, dx = _grads(_first, x, edges, None, g)
    assert out.tolist() == [[0.0, 0.0], [-1.0, 2.0], [0.0, 0.0]]
    assert dx.tolist() == [[0.0, 1.0], [1.0, 0.0], [0.0, 0.0]]


def test_all_negative_messages_keep_their_max():
    # the running max starts at -inf: a node whose messages are all negative aggregates to the largest of them, not 0
    x = torch.tensor([[-2.0, -0.5], [-1.0, -4.0], [0.0, 0.0]])
    edges = torch.tensor([[0, 1], [2, 2]])
    out, dx = _grads(_first, x, edges, None, torch.ones(3, 2))
    assert out[2].tolist() == [-1.0, -0.5]
    assert dx.tolist() == [[0.0, 1.0], [1.0, 0.0], [0.0, 0.0]]


def test_repeated_edges():
    x = torch.tensor([[3.0, -2.0], [0.0, 0.0]])
    # equal weights: the repeated edges tie exactly; the first one (edge 0) takes the gradient
    edges = torch.tensor([[0, 0], [1, 1]])
    out, dx = _grads(_first, x, edges, torch.tensor([0.5, 0.5]), torch.tensor([[0.0, 0.0], [1.0, 1.0]]))
    assert out[1].tolist() == [1.5, -1.0]
    assert dx.tolist() == [[0.5, 0.5], [0.0, 0.0]]
    # unequal weights: the larger product wins per channel (w = 2 for the positive channel, w = 0.25 for the negative)
    out, dx = _grads(_first, x, edges, torch.tensor([0.25, 2.0]), torch.tensor([[0.0, 0.0], [1.0, 1.0]]))
    assert out[1].tolist() == [6.0, -0.5]
    assert dx.tolist() == [[2.0, 0.25], [0.0, 0.0]]
    # both repeated edges with the same weights are tied; the split rule would give each half
    _, dx_split = _grads(_split, x, edges, torch.tensor([0.5, 0.5]), torch.tensor([[0.0, 0.0], [1.0, 1.0]]))
    assert dx_split.tolist() == [[0.5, 0.5], [0.0, 0.0]]


def test_bf16_oracle_uses_the_rule_and_fp32_oracle_keeps_scatter_reduce(monkeypatch):
    """with bf16_oracle_first_edge, the bf16 oracle's conv2 aggregates with the rule; the fp32 oracle and conv1 are the
    oracle's own, and the forward values of both modes do not change"""
    cfg = dict(input_dim=2, hidden_dim=8, output_dim=1, activation="tanh", local_pooling="max", deepchem_style=True)
    sd = GO.init_state_dict(cfg, seed=0)
    x = torch.randint(-2, 3, (10, 2), generator=torch.Generator().manual_seed(3)).float()
    memb = torch.tensor([0] * 5 + [1] * 5)
    edges = torch.tensor([[1, 2, 3, 4, 0, 6, 7, 8, 9, 5, 2, 7], [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 0, 5]])
    y = torch.tensor([[1.0], [0.0]])
    before = {mode: GO.graphnet_train_step(sd, cfg, x, memb, edges, None, y, operand_rounding=mode) for mode in (None, "bf16")}
    seen = []

    def spy(x, edges, weights):
        seen.append(x.shape[1])
        return graph_aggregate_first_edge(x, edges, weights)

    bf16_oracle_first_edge(monkeypatch)
    monkeypatch.setattr("graph_max_ref.graph_aggregate_first_edge", spy)
    after = {}
    for mode in (None, "bf16"):
        seen.clear()
        after[mode] = GO.graphnet_train_step(sd, cfg, x, memb, edges, None, y, operand_rounding=mode)
        assert seen == ([] if mode is None else [8])        # conv2 only, in the bf16 mode only
        assert torch.equal(after[mode][0], before[mode][0])
    for k, g in after[None][2].items():
        assert torch.equal(g, before[None][2][k]), k
