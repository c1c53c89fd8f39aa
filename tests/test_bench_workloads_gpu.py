"""GPU: the workloads bench.py times, compared with the oracle at the shapes it times them.

The inputs come from bench's own workload objects (`bench.make_workload("ragged")`, and `DeepSetsWorkload` /
`GraphNetWorkload` built the way `bench.run_sweep` builds them), so these tests follow bench if its configs change.
Every case runs the step the way bench does: a `GraphedTrainStep` (CUDA-graph replay of forward + fused BCE loss +
backward) is captured on a DIFFERENT batch and then fed the checked batch through its static buffers.

 * `--config ragged` (configs[2]): 256 sets with log-normal sizes (232 .. 4096 points, 478,374 in all, not a multiple
   of 128), relu + sum.  Sets span up to 33 tiles, their pooled sums are combined across CTAs and sum / sqrt(n) is
   applied at n = 4096.  A second case captures the step on that layout and replays it on the same sizes in reverse
   order (same total, another tile-to-set map): the per-tile set ranges are recomputed inside the graph.
 * `--config sweep` DeepSets (configs[4]): relu + max and relu + sum, H = 256, depth 2, at N = 256 .. 16384 with
   B = 262144 / N.  At N = 256 (B * H = n) max pooling runs the full-row backward over 262,144 rows; at N = 16384 every
   set covers 128 tiles.  (relu + max at N = 1024 is the headline model, tests/test_fullsize_gpu.py.)
 * `--config sweep` GraphNet, which at N = 1024 is `--config graphnet` (configs[3]): `KnnGraphNet`, k = 20, tanh / add /
   deepchem, at N = 256, 1024, 4096 and 16384 with B = 262144 / N.  The device kNN graph equals the exact kNN oracle
   (oracle/knn_oracle.py with rows_per_chunk, spread over the host's cores) bit for bit, indices and distances, in every
   cloud; the oracle then runs on that graph.

Tolerances are the stated ones of tests/test_fused_gpu.py (DeepSets, through its `check_step_against_oracles`, plus
the loss against the bf16-operand oracle as in tests/test_fullsize_gpu.py) and tests/test_graph_fused_gpu.py
(GraphNet, through its `check_fused_step_against_oracles`: logits, all 16 gradients, the running statistics after the
one replay, which also shows that the capture's warm-up steps were rolled back, and the eval-mode logits).  Every case
prints its errors.  Measured maxima on a B200 at a 1000 W power limit, per group, vs the bf16-operand oracle / the fp32
oracle (logits: max error over max|ref|; gradients: worst relative Frobenius error over all parameters):
  ragged (both cases):  loss 3.2e-7; logits 3.2e-6 / 1.3e-3; gradients 4.1e-4 / 9.4e-3
  sweep relu + max:     loss 2.6e-7; logits 4.3e-4 / 6.1e-3 (N = 256); gradients 4.2e-3 / 6.3e-2 (phi.0.weight; the
                        fp32 figure is the ReLU-mask effect described in tests/test_fused_gpu.py)
  sweep relu + sum:     loss 8.5e-7; logits 1.7e-5 / 1.6e-3; gradients 7.1e-4 / 6.9e-3
  GraphNet (4 sizes):   logits 1.2e-4 / 4.4e-3; gradients 2.3e-2 / 2.7e-2 (the first is bn2.bias at N = 16384, B = 16, a
                        near-cancelling sum over 262,144 nodes of the bf16-rounded backward tensors; every other
                        gradient <= 9.1e-3 / 2.7e-2); running statistics max |diff| 3.5e-4; eval logits 6.3e-3
The kNN graphs matched the oracle bit for bit in every cloud.  The file ran in 50 s on that host (16 CPU cores).
"""
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "point-cloud-classifier_b200"))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
from oracle import deepsets_oracle as O  # noqa: E402
from oracle import graphnet_oracle as GO  # noqa: E402
from oracle import knn_oracle as KO  # noqa: E402
from pcc_b200 import functional as PF  # noqa: E402
from pcc_b200.train_step import GraphedTrainStep  # noqa: E402
from test_fused_gpu import LOSS_TOL, _fused_argmax, check_step_against_oracles  # noqa: E402
from test_graph_fused_gpu import check_fused_step_against_oracles  # noqa: E402

pytestmark = pytest.mark.gpu
SWEEP_POINTS = 262144                                  # bench.run_sweep: B = 262144 / N sets or clouds per step
SWEEP_N = (256, 512, 1024, 2048, 4096, 8192, 16384)


def _sweep_deepsets(pool, N):
    return bench.DeepSetsWorkload("deepsets", SWEEP_POINTS // N, N, 3, 10, "relu", pool, False)


def _check_deepsets_step(tag, wl, capture, checked):
    """bench's bf16 DeepSets step on `checked` ((x, idx), y on the host) through a GraphedTrainStep captured on
    `capture`, against the fp32 oracle and the oracle with the stated bf16 operand rounding"""
    cfg = wl.cfg
    sd = O.init_state_dict(cfg, seed=0)
    m = wl.build_model(torch.device("cuda"), "bf16")
    m.load_state_dict(sd)
    (cx, cidx), cy = capture
    (x, idx), y = checked
    gs = GraphedTrainStep(m, (cx.cuda(), cidx.cuda()), cy.cuda(), forward_kwargs=wl.forward_kwargs())
    assert gs.graph is not None and m.last_path == wl.expected_path("bf16")
    xc, ic = x.cuda(), idx.cuda()
    loss = gs.step((xc, ic), y.cuda())
    torch.cuda.synchronize()
    arg = None
    if cfg["pooling"] == "max":     # the oracle evaluates max pooling at the rows the kernel selected
        arg = _fused_argmax(m, xc, PF.segment_offsets(ic, wl.B), cfg["activation"])
    r32 = O.deepsets_train_step(sd, cfg, x, idx, y, argmax_rows=arg)
    r16 = O.deepsets_train_step(sd, cfg, x, idx, y, phi_operand_rounding="bf16", argmax_rows=arg)
    e_loss = abs(float(loss) - float(r16[1])) / abs(float(r16[1]))
    print(f"{tag}: loss {e_loss:.1e} vs bf16-operand oracle")
    assert e_loss < LOSS_TOL, e_loss
    check_step_against_oracles(tag, cfg["activation"], {k: p.grad for k, p in m.named_parameters()}, gs.logits,
                               (r32[0], r32[2]), (r16[0], r16[2]))


def test_ragged_workload_matches_oracle():
    wl = bench.make_workload("ragged")
    assert wl.B == 256 and max(wl.sizes) == 4096 and wl.points % 128 != 0
    checked, capture = wl.make_batches(2, seed=1000, pin=False)
    _check_deepsets_step(f"ragged B={wl.B} points={wl.points}", wl, capture, checked)


def test_ragged_replay_on_reversed_sizes_matches_oracle():
    """captured on the ragged layout, replayed on the same sizes in reverse order: same point count, other sets in every
    tile, so the per-tile set ranges must be recomputed by the replay"""
    wl = bench.make_workload("ragged")
    capture, ((x, idx), y) = wl.make_batches(2, seed=1000, pin=False)
    rev = torch.cat([torch.full((s,), i, dtype=torch.long) for i, s in enumerate(wl.sizes[::-1])])
    assert rev.shape == idx.shape and not torch.equal(rev, idx)
    _check_deepsets_step(f"ragged replayed on reversed sizes B={wl.B}", wl, capture, ((x, rev), y))


@pytest.mark.parametrize("pool,N", [(p, n) for p in ("max", "sum") for n in SWEEP_N if (p, n) != ("max", 1024)])
def test_sweep_deepsets_matches_oracle(pool, N):
    wl = _sweep_deepsets(pool, N)
    checked, capture = wl.make_batches(2, seed=7, pin=False)
    _check_deepsets_step(f"sweep relu/{pool} N={N} B={wl.B}", wl, capture, checked)


def _knn_reference(pos, offsets, k):
    """exact kNN of every cloud (oracle/knn_oracle.py, chunked rows), the clouds spread over the host's cores"""
    n = pos.shape[0]
    nbr = np.empty((n, k), dtype=np.int64)
    d2 = np.empty((n, k), dtype=np.float32)

    def one(b):
        s, e = int(offsets[b]), int(offsets[b + 1])
        a, c = KO.knn_neighbours(pos[s:e], np.array([0, e - s], dtype=np.int64), k, rows_per_chunk=256)
        nbr[s:e] = np.where(a >= 0, a + s, -1)
        d2[s:e] = c
    with ThreadPoolExecutor(min(os.cpu_count() or 1, 16)) as ex:
        list(ex.map(one, range(len(offsets) - 1)))
    return nbr, d2


@pytest.mark.parametrize("N", [256, 1024, 4096, 16384])
def test_sweep_graphnet_matches_oracle(N):
    wl = bench.GraphNetWorkload("graphnet", SWEEP_POINTS // N, N)
    checked, capture = wl.make_batches(2, seed=7, pin=False)
    (f, memb), y = checked
    fc, mc = f.cuda(), memb.cuda()
    off = np.arange(wl.B + 1, dtype=np.int64) * N
    # with_int32: the int32 table KnnGraphNet hands to the fused kernels comes out of the same launch
    nbr, d2, nbr32 = PF.knn(fc[:, 1:4], torch.from_numpy(off).cuda(), wl.k, with_int32=True)
    assert torch.equal(nbr32.long(), nbr)
    ref_nbr, ref_d2 = _knn_reference(f[:, 1:4].numpy(), off, wl.k)
    nbr, d2 = nbr.cpu().numpy(), d2.cpu().numpy()
    bad = np.unique(np.flatnonzero((nbr != ref_nbr).any(1) | (d2.view(np.uint32) != ref_d2.view(np.uint32)).any(1)) // N)
    print(f"sweep graphnet N={N} B={wl.B}: device kNN differs from the oracle in {len(bad)} of {wl.B} clouds")
    assert len(bad) == 0, f"clouds {bad[:10].tolist()} differ"

    sd = GO.init_state_dict(wl.cfg, seed=0)
    m = wl.build_model(torch.device("cuda"), "bf16")
    m.net.load_state_dict(sd)
    m.train()
    (cf, cm), cy = capture
    gs = GraphedTrainStep(m, (cf.cuda(), cm.cuda()), cy.cuda(), forward_kwargs=wl.forward_kwargs())
    assert gs.graph is not None and m.net.last_path == "fused-bf16"
    gs.step((fc, mc), y.cuda())
    torch.cuda.synchronize()
    edges = torch.from_numpy(KO.knn_edges(ref_nbr))
    check_fused_step_against_oracles(wl.cfg, sd, f, memb, edges, None, y, gs.logits,
                                     {k: p.grad for k, p in m.net.named_parameters()}, m, [fc, mc], num_graphs=wl.B)
