"""GPU, BASELINE.json's full sizes (B = 256 sets x N = 1024 points, H = 256).
(1) `test_graphed_train_step_matches_oracle_full_size`: the thing bench.py times — `GraphedTrainStep` (fused BCE
    loss, CUDA-graph replay of forward + loss + backward) — against the pinned oracle on the same batch: logits and
    every parameter gradient, for the headline relu + max model and the reference's yaml default (gelu + residual
    + mean, d = 6, out = 1); ~1 s of CPU per oracle evaluation.  Tolerances and their derivation: test_fused_gpu.py.
(2) size-independent properties of the reference's DeepSets (models/deep_sets.py:89-112):
  * permutation invariance: shuffling the points inside every set leaves the logits unchanged — bit-exact for max
    pooling (every point's row is computed independently and the maximum does not depend on the order), to
    accumulation-order noise for sum / mean;
  * batch independence: sets do not interact, so a batch evaluated in two halves gives the same logits and, the loss
    being a mean over sets, the full-batch gradient is the average of the two half-batch gradients;
  * the pooled maxima agree with an fp32 re-evaluation of phi on all 262,144 points within the stated bf16 tolerance."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "point-cloud-classifier_b200"))

sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pcc_b200  # noqa: E402
from oracle import deepsets_oracle as O  # noqa: E402
from pcc_b200 import functional as PF  # noqa: E402
from pcc_b200.train_step import GraphedTrainStep  # noqa: E402
from test_fused_gpu import LOSS_TOL, _fused_argmax, check_step_against_oracles  # noqa: E402

B, N, D, H, OUT = 256, 1024, 3, 256, 10
pytestmark = pytest.mark.gpu


def _model(pooling, act="relu", seed=0):
    torch.manual_seed(seed)
    return pcc_b200.DeepSets(D, [H, H], [H], OUT, act, layer_norm=False, residual_block=False, pooling=pooling,
                             precision="bf16").cuda()


def _batch(seed=1):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B * N, D, generator=g).cuda()
    idx = torch.arange(B).repeat_interleave(N).cuda()
    y = (torch.rand(B, OUT, generator=g) > 0.5).float().cuda()
    return x, idx, y


@pytest.mark.parametrize("pooling", ["max", "sum", "mean"])
def test_permutation_invariance_full_size(pooling):
    m = _model(pooling)
    x, idx, _ = _batch()
    g = torch.Generator().manual_seed(5)
    perm = torch.stack([torch.randperm(N, generator=g) + b * N for b in range(B)]).reshape(-1).cuda()
    with torch.no_grad():
        a = m(x, idx, num_sets=B)
        b = m(x[perm].contiguous(), idx, num_sets=B)
    assert m.last_path == "fused-bf16"
    if pooling == "max":
        assert torch.equal(a, b)
    else:
        torch.testing.assert_close(a, b, rtol=2e-4, atol=2e-5)


@pytest.mark.parametrize("pooling", ["max", "sum"])
def test_batch_independence_full_size(pooling):
    m = _model(pooling)
    x, idx, y = _batch(seed=2)
    lossf = torch.nn.BCEWithLogitsLoss()

    def run(xs, ids, ys, nb):
        m.zero_grad(set_to_none=True)
        logits = m(xs, ids, num_sets=nb)
        lossf(logits, ys).backward()
        return logits.detach().clone(), [p.grad.detach().clone() for p in m.parameters()]

    full_logits, full_grads = run(x, idx, y, B)
    hb = B // 2
    l0, g0 = run(x[: hb * N].contiguous(), idx[: hb * N].contiguous(), y[:hb].contiguous(), hb)
    l1, g1 = run(x[hb * N:].contiguous(), (idx[hb * N:] - hb).contiguous(), y[hb:].contiguous(), hb)
    halves = torch.cat([l0, l1])
    if pooling == "max":
        assert torch.equal(full_logits, halves)
    else:
        torch.testing.assert_close(full_logits, halves, rtol=2e-4, atol=2e-5)
    for gf, ga, gb in zip(full_grads, g0, g1):
        ref = 0.5 * (ga + gb)
        err = float((gf - ref).norm() / (ref.norm() + 1e-30))
        assert err < 2e-3, err   # same bf16 operands, different tile composition / summation order


def test_pooled_maxima_match_fp32_full_size():
    from pcc_b200 import functional as PF, fused as FZ
    m = _model("max", seed=3)
    x, idx, _ = _batch(seed=4)
    off = PF.segment_offsets(idx, B)
    with torch.no_grad():
        pooled = FZ.phi_pool(x, off, m._phi_plan, "relu", "max")
    # fp32 re-evaluation of phi on every point (the stock nn modules of the drop-in model, torch eager), then the
    # true per-set maxima
    m32 = pcc_b200.DeepSets(D, [H, H], [H], OUT, "relu", layer_norm=False, residual_block=False, pooling="max",
                            precision="fp32").cuda()
    m32.load_state_dict(m.state_dict())
    with torch.no_grad():
        h = x
        for layer in m32.phi:
            h = layer(h)
        true_max = h.view(B, N, H).max(dim=1).values
    gap = (pooled - true_max).abs().max() / true_max.abs().max()
    assert float(gap) < 3e-2   # the stated bf16 tolerance of tests/test_fused_gpu.py


FULL_CFGS = {
    "relu_max": dict(input_dim=3, phi_layers=[H, H], rho_layers=[H], output_dim=10, activation="relu", layer_norm=False,
                     residual_block=False, pooling="max"),
    "yaml_gelu_res_mean": dict(input_dim=6, phi_layers=[H, H], rho_layers=[H], output_dim=1, activation="gelu",
                               layer_norm=False, residual_block=True, pooling="mean"),
}


@pytest.mark.parametrize("name", list(FULL_CFGS))
def test_graphed_train_step_matches_oracle_full_size(name):
    cfg = FULL_CFGS[name]
    d, out = cfg["input_dim"], cfg["output_dim"]
    sd = O.init_state_dict(cfg, seed=71)
    g = torch.Generator().manual_seed(72)
    x = torch.randn(B * N, d, generator=g)
    idx = torch.arange(B).repeat_interleave(N)
    y = (torch.rand(B, out, generator=g) > 0.5).float()
    m = pcc_b200.DeepSets(**cfg, precision="bf16").cuda()
    m.load_state_dict(sd)
    xc, ic, yc = x.cuda(), idx.cuda(), y.cuda()
    # the captured step is built on a DIFFERENT batch and then fed this one through its static buffers
    gs = GraphedTrainStep(m, (torch.randn_like(xc), ic), torch.zeros_like(yc), forward_kwargs={"num_sets": B})
    assert gs.graph is not None and m.last_path == "fused-bf16"
    loss = gs.step((xc, ic), yc)
    torch.cuda.synchronize()
    arg = None
    if cfg["pooling"] == "max":
        arg = _fused_argmax(m, xc, PF.segment_offsets(ic, B), cfg["activation"])
    r32 = O.deepsets_train_step(sd, cfg, x, idx, y, argmax_rows=arg)
    r16 = O.deepsets_train_step(sd, cfg, x, idx, y, phi_operand_rounding="bf16", argmax_rows=arg)
    assert abs(float(loss) - float(r16[1])) < LOSS_TOL * abs(float(r16[1]))
    check_step_against_oracles(f"GraphedTrainStep full size {name}", cfg["activation"],
                               {k: p.grad for k, p in m.named_parameters()}, gs.logits, (r32[0], r32[2]), (r16[0], r16[2]))
