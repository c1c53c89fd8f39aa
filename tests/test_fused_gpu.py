"""GPU: the fused tcgen05 / TMEM phi+pool path (bf16 operands, fp32 accumulate).

Stated bf16 tolerance (north_star "or a stated bf16 tolerance").  The bf16 mode rounds both operands of every phi
Linear to bf16 (8-bit mantissa) and accumulates in fp32.  Two comparisons, both against the pinned oracle
(oracle/deepsets_oracle.py), per tensor, printed by every test:

 (1) oracle evaluated with the SAME stated operand rounding (`phi_operand_rounding="bf16"`: operands rounded to
     bf16, everything else fp32) — "the kernel computes what it says".  Measured on B200 (tools/grad_err_report.py,
     profiles/grad_err_r2.txt): logits <= 2.5e-3 of max|ref| (relu: <= 3e-4; gelu / silu carry the tanh.approx
     activation, 1e-3 .. 2.5e-3), parameter gradients <= 4.4e-3 relative Frobenius error over all 11 cases and both
     full-size configurations.  Tolerances = 2x measured:
         logits  max|got - ref| <= BF16_TOL * max|ref|,        BF16_TOL = 5e-3
         grads   ||got - ref||_F <= BF16_GRAD_TOL * ||ref||_F,  BF16_GRAD_TOL = 1e-2
 (2) the fp32 oracle (the reference's own arithmetic): logits <= FP32_TOL = 1.5e-2 (measured <= 6.5e-3).  Gradients:
     smooth activations (gelu / silu) <= FP32_GRAD_TOL_SMOOTH = 1e-2 (measured <= 4.4e-3); ReLU <=
     FP32_GRAD_TOL_RELU = 0.16 (measured 7.6e-3 .. 7.8e-2).  The ReLU figure is a property of bf16 operands, not of the
     kernel (comparison (1) holds to 2.9e-3 on the same cases): rounding the operands moves every pre-activation by
     ~2e-3 of its scale, so ~0.5 % of the ReLU masks flip, each flip changes one gradient term by O(1), and with
     random labels the gradient is an incoherent sum, so the relative error is ~sqrt(flip fraction) ~ 7e-2 whatever
     the batch size (rho.0.bias at B=256 shows the same 7e-2 as phi.0.weight).
Max pooling: a precision change can move an argmax between near-tied rows, so (a) argmax rows must lie in their set
and be maximal in fp32 within FP32_TOL, with > 97 % identical to the fp32 oracle's, and (b) gradients are checked
against oracles evaluated with the SAME argmax rows the kernel selected.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import ragged_batch, rel_err, rel_l2
from oracle import deepsets_oracle as O

import pcc_b200
from pcc_b200 import _lib, functional as PF, fused as FZ

pytestmark = pytest.mark.gpu
BF16_TOL = 5e-3
BF16_GRAD_TOL = 1e-2
FP32_TOL = 1.5e-2
FP32_GRAD_TOL_SMOOTH = 1e-2
FP32_GRAD_TOL_RELU = 0.16
LOSS_TOL = 2e-3   # |loss - loss of the bf16-operand oracle| <= LOSS_TOL * |that loss|, GraphedTrainStep's fused BCE


def check_step_against_oracles(tag, act, named_grads, logits, ref32, ref16):
    """ref32 / ref16 = (logits, grads) of the fp32 oracle and of the oracle with bf16 operand rounding.
    Prints the per-tensor errors and the worst case, asserts the stated tolerances."""
    e_l16, e_l32 = rel_err(logits, ref16[0]), rel_err(logits, ref32[0])
    rows, worst16, worst32 = [], ("", 0.0), ("", 0.0)
    for k, r16 in ref16[1].items():
        got = named_grads[k]
        assert got is not None, k
        e16, e32 = rel_l2(got, r16), rel_l2(got, ref32[1][k])
        rows.append(f"{k}={e16:.1e}/{e32:.1e}")
        if e16 > worst16[1]:
            worst16 = (k, e16)
        if e32 > worst32[1]:
            worst32 = (k, e32)
    print(f"{tag}: logits {e_l16:.1e}/{e_l32:.1e} (vs bf16-operand oracle / fp32 oracle); grads rel-L2 "
          f"worst {worst16[0]} {worst16[1]:.1e} / {worst32[0]} {worst32[1]:.1e}; " + " ".join(rows))
    assert e_l16 < BF16_TOL, ("logits vs bf16-operand oracle", e_l16)
    assert e_l32 < FP32_TOL, ("logits vs fp32 oracle", e_l32)
    assert worst16[1] < BF16_GRAD_TOL, ("grad vs bf16-operand oracle",) + worst16
    tol32 = FP32_GRAD_TOL_RELU if act == "relu" else FP32_GRAD_TOL_SMOOTH
    assert worst32[1] < tol32, ("grad vs fp32 oracle",) + worst32


def _st_a(i, k):
    return ((i * 3 + k * 5) % 7 - 3).astype(np.float64)


def _st_b(j, k):
    return ((j * 2 + k) % 5 - 2).astype(np.float64)


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
def test_umma_descriptor_conventions(mode):
    out = torch.full((128, 64), float("nan"), device="cuda")
    _lib.call("pcc_selftest_umma", mode, _lib.ptr(out), 0, _lib.stream_ptr(0))
    torch.cuda.synchronize()
    K = 64 if mode == 0 else 128
    i, j, k = np.arange(128)[:, None, None], np.arange(64)[None, :, None], np.arange(K)[None, None, :]
    ref = (_st_a(i, k) * _st_b(j, k)).sum(-1)
    got = out.cpu().numpy().astype(np.float64)
    assert np.array_equal(got, ref), f"mode {mode}: {np.abs(got - ref).max()} max abs diff, got[0,:4]={got[0,:4]} ref[0,:4]={ref[0,:4]}"


CASES = [
    # act, pool, residual, H, depth(hidden layers), d, sizes
    ("relu", "max", False, 256, 2, 3, [1024, 1024, 1024]),
    ("relu", "max", False, 128, 2, 3, [100, 128, 129, 1, 300, 33]),
    ("gelu", "mean", True, 256, 2, 6, [33, 1, 200, 128, 129, 64, 7, 500]),
    ("silu", "sum", True, 128, 2, 4, [31, 32, 33, 127, 128, 129, 1, 300]),
    ("relu", "sum", False, 256, 1, 3, [256, 100, 156]),
    ("gelu", "max", True, 128, 2, 7, [700, 5, 250]),
    ("silu", "sum", False, 256, 2, 6, [300, 41, 129, 1]),
    ("silu", "mean", False, 128, 1, 1, [64, 64]),
    # H = 256 + max pooling = the CTA-pair forward kernel: other activations, ResidualBlock, one hidden layer
    # (alternating final accumulators), d > 3 (two-quad layer-0 table), odd tile counts
    ("gelu", "max", True, 256, 2, 3, [300, 129, 1, 700, 64]),
    ("silu", "max", False, 256, 1, 6, [128, 128, 128, 5, 250]),
    ("relu", "max", False, 256, 1, 3, [1000, 24]),
]


def _cfg(act, pool, res, H, depth, d):
    return dict(input_dim=d, phi_layers=[H] * depth, rho_layers=[64], output_dim=3, activation=act, layer_norm=False,
                residual_block=res, pooling=pool)


@pytest.mark.parametrize("act,pool,res,H,depth,d,sizes", CASES)
def test_fused_forward_matches_oracle(act, pool, res, H, depth, d, sizes):
    cfg = _cfg(act, pool, res, H, depth, d)
    sd = O.init_state_dict(cfg, seed=31)
    x, idx = ragged_batch(sizes, d, seed=32)
    _, aux = O.deepsets_forward(sd, cfg, x, idx, return_aux=True)
    m = pcc_b200.DeepSets(**cfg, precision="bf16").cuda()
    m.load_state_dict(sd)
    assert m.fused_supported()
    off = PF.segment_offsets(idx.cuda(), len(sizes))
    with torch.no_grad():
        pooled = FZ.phi_pool(x.cuda(), off, m._phi_plan, act, pool)
    _, aux16 = O.deepsets_forward(sd, cfg, x, idx, return_aux=True, phi_operand_rounding="bf16")
    err, err16 = rel_err(pooled, aux["pooled"]), rel_err(pooled, aux16["pooled"])
    print(f"fused fwd {act}/{pool}/res={res}/H={H}/depth={depth}: pooled rel err {err16:.2e} vs bf16-operand oracle, "
          f"{err:.2e} vs fp32 oracle")
    assert err < FP32_TOL
    if pool != "max":   # (max: a near-tie can pick another row than the free-running oracle; covered with pinned rows below)
        assert err16 < BF16_TOL


def test_fused_argmax_consistent_with_fp32_oracle():
    cfg = _cfg("relu", "max", False, 256, 2, 3)
    sd = O.init_state_dict(cfg, seed=41)
    sizes = [1024, 500, 37, 1]
    x, idx = ragged_batch(sizes, 3, seed=42)
    _, aux = O.deepsets_forward(sd, cfg, x, idx, return_aux=True)
    m = pcc_b200.DeepSets(**cfg, precision="bf16").cuda()
    m.load_state_dict(sd)
    off = PF.segment_offsets(idx.cuda(), len(sizes))
    dsc = FZ._build_desc(m._phi_plan, "relu", "max", [(L["lin"].weight, L["lin"].bias) for L in m._phi_plan])
    n, B, H = x.shape[0], len(sizes), 256
    ws = torch.empty(_lib.call("pcc_phi_fused_workspace_bytes", C.byref(dsc), n, B), dtype=torch.uint8, device="cuda")
    pooled = torch.empty(B, H, device="cuda")
    arg = torch.empty(B, H, dtype=torch.int32, device="cuda")
    xc = x.cuda()
    wpack = torch.empty(_lib.call("pcc_phi_packed_bytes", C.byref(dsc)), dtype=torch.uint8, device="cuda")
    _lib.call("pcc_deepsets_phi_pool_fwd", C.byref(dsc), _lib.ptr(xc), _lib.ptr(off), n, B, _lib.ptr(pooled),
              _lib.ptr(arg), _lib.ptr(ws), _lib.ptr(wpack), 0, _lib.stream_ptr(0))
    arg = arg.cpu().long()
    offs = aux["offsets"]
    lo, hi = offs[:-1].view(B, 1), offs[1:].view(B, 1)
    assert bool(((arg >= lo) & (arg < hi)).all())           # rows lie inside their own set
    phi = aux["phi_x"]
    picked = phi[arg, torch.arange(H).expand(B, -1)]        # fp32 value at the row the kernel picked
    gap = (aux["pooled"] - picked).abs().max() / aux["pooled"].abs().max()
    assert float(gap) < FP32_TOL                            # picked rows are (near-)maximal in fp32 too
    agree = (arg == aux["argmax"]).float().mean()
    print(f"argmax agreement with fp32 oracle: {float(agree):.3f}")
    assert float(agree) > 0.97


def test_fused_large_config2_properties():
    """BASELINE config 2 (B=256, N=1024, H=256, relu+max): fused pooled values equal the
    max over points of an fp32 re-evaluation within the bf16 tolerance; argmax in range."""
    cfg = _cfg("relu", "max", False, 256, 2, 3)
    m = pcc_b200.DeepSets(**cfg, precision="bf16").cuda()
    B, N = 256, 1024
    x = torch.randn(B * N, 3, device="cuda")
    idx = torch.arange(B, device="cuda").repeat_interleave(N)
    off = PF.segment_offsets(idx, B)
    with torch.no_grad():
        pooled = FZ.phi_pool(x, off, m._phi_plan, "relu", "max")
        ref = m._mlp(m._phi_plan, x).view(B, N, -1).max(dim=1)[0]   # fp32 CUDA path
    assert rel_err(pooled, ref) < FP32_TOL


def _fused_argmax(m, x, off, act):
    """argmax rows the fused forward selects (deterministic: packed atomicMax is order independent)."""
    dsc = FZ._build_desc(m._phi_plan, act, "max", [(L["lin"].weight, L["lin"].bias) for L in m._phi_plan])
    n, B, H = x.shape[0], off.numel() - 1, dsc.hidden
    ws = torch.empty(_lib.call("pcc_phi_fused_workspace_bytes", C.byref(dsc), n, B), dtype=torch.uint8, device="cuda")
    pooled = torch.empty(B, H, device="cuda")
    arg = torch.empty(B, H, dtype=torch.int32, device="cuda")
    wpack = torch.empty(_lib.call("pcc_phi_packed_bytes", C.byref(dsc)), dtype=torch.uint8, device="cuda")
    _lib.call("pcc_deepsets_phi_pool_fwd", C.byref(dsc), _lib.ptr(x), _lib.ptr(off), n, B, _lib.ptr(pooled),
              _lib.ptr(arg), _lib.ptr(ws), _lib.ptr(wpack), 0, _lib.stream_ptr(0))
    return arg.cpu().long()


@pytest.mark.parametrize("act,pool,res,H,depth,d,sizes", CASES)
def test_fused_train_step_matches_oracle(act, pool, res, H, depth, d, sizes):
    """forward + BCEWithLogitsLoss + backward through the fused kernels vs the fp32 oracle."""
    cfg = _cfg(act, pool, res, H, depth, d)
    sd = O.init_state_dict(cfg, seed=51)
    x, idx = ragged_batch(sizes, d, seed=52)
    y = (torch.rand(len(sizes), 3, generator=torch.Generator().manual_seed(53)) > 0.5).float()
    m = pcc_b200.DeepSets(**cfg, precision="bf16").cuda()
    m.load_state_dict(sd)
    arg = None
    if pool == "max":
        off = PF.segment_offsets(idx.cuda(), len(sizes))
        arg = _fused_argmax(m, x.cuda(), off, act)
    r32 = O.deepsets_train_step(sd, cfg, x, idx, y, argmax_rows=arg)
    r16 = O.deepsets_train_step(sd, cfg, x, idx, y, phi_operand_rounding="bf16", argmax_rows=arg)
    logits = m(x.cuda(), idx.cuda())
    assert m.last_path == "fused-bf16"
    loss = torch.nn.BCEWithLogitsLoss()(logits, y.cuda())
    loss.backward()
    check_step_against_oracles(f"fused train {act}/{pool}/res={res}/H={H}/depth={depth}", act,
                               {k: p.grad for k, p in m.named_parameters()}, logits, (r32[0], r32[2]), (r16[0], r16[2]))


def test_fused_multi_tile_per_cta_backward():
    """more tiles than SMs (several tiles per persistent CTA) through fwd + bwd, H=256"""
    cfg = _cfg("relu", "mean", False, 256, 2, 3)
    sd = O.init_state_dict(cfg, seed=61)
    sizes = [1024] * 40
    x, idx = ragged_batch(sizes, 3, seed=62)
    y = (torch.rand(len(sizes), 3, generator=torch.Generator().manual_seed(63)) > 0.5).float()
    r32 = O.deepsets_train_step(sd, cfg, x, idx, y)
    r16 = O.deepsets_train_step(sd, cfg, x, idx, y, phi_operand_rounding="bf16")
    m = pcc_b200.DeepSets(**cfg, precision="bf16").cuda()
    m.load_state_dict(sd)
    logits = m(x.cuda(), idx.cuda())
    torch.nn.BCEWithLogitsLoss()(logits, y.cuda()).backward()
    check_step_against_oracles("multi-tile relu/mean", "relu", {k: p.grad for k, p in m.named_parameters()}, logits,
                               (r32[0], r32[2]), (r16[0], r16[2]))


def test_deeper_phi_falls_back_to_fp32_path():
    cfg = _cfg("relu", "max", False, 128, 3, 3)
    m = pcc_b200.DeepSets(**cfg, precision="bf16").cuda()
    assert not m.fused_supported()
    x, idx = ragged_batch([50, 60], 3, seed=1)
    m(x.cuda(), idx.cuda()).sum().backward()
    assert m.last_path == "fp32"


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [[1024] * 8, [300, 1, 129, 700, 64, 5], [128] * 3])
def test_pair_kernel_matches_single_cta_kernel(sizes):
    """H = 256 + max pooling runs on CTA pairs (cta_group::2, weight halves resident); the one-CTA kernel computes
    the same function with the same operand rounding: pooled values agree to fp32 accumulation-order noise and the
    argmax rows are the same (odd tile counts exercise the dummy second tile of the last pair)."""
    from pcc_b200 import _lib
    cfg = dict(input_dim=3, phi_layers=[256, 256], rho_layers=[64], output_dim=3, activation="relu", layer_norm=False,
               residual_block=False, pooling="max")
    torch.manual_seed(3)
    m = pcc_b200.DeepSets(**cfg, precision="bf16").cuda()
    x, idx = ragged_batch(sizes, 3, seed=11, device="cuda")
    outs = []
    try:
        for pair in (1, 0):
            _lib.call("pcc_debug_set_fwd_pair", pair)
            with torch.no_grad():
                logits = m(x, idx)
            outs.append((logits.clone(), m._last_pooled.clone() if hasattr(m, "_last_pooled") else None))
    finally:
        _lib.call("pcc_debug_set_fwd_pair", 1)
    torch.testing.assert_close(outs[0][0], outs[1][0], rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_peer_allreduce_single_rank(tmp_path):
    """The library's peer all-reduce (CUDA IPC staging + flags) on a one-rank group: alloc / kernel / free and the
    averaging arithmetic; multi-rank runs are tools/test_peer_allreduce.py (2 and 8 GPUs, bit-exact vs NCCL)."""
    import torch.distributed as dist
    from pcc_b200.distributed import PeerAllReduce, GradArena
    if not dist.is_initialized():
        dist.init_process_group("gloo", init_method=f"file://{tmp_path}/rdzv", rank=0, world_size=1)
    try:
        peer = PeerAllReduce(1001, torch.device("cuda", 0))
        a = torch.randn(peer.numel, device="cuda")
        ref = a.clone()
        for _ in range(3):          # the sequence number / staging parity advances per call
            peer.run(a)
        torch.cuda.synchronize()
        assert torch.equal(a, ref)
        peer.close()
        lin = torch.nn.Linear(5, 3).cuda()
        arena = GradArena(list(lin.parameters()))
        assert arena.numel % 4 == 0 and arena.view_for(lin.weight).shape == lin.weight.shape
        assert arena.view_for(torch.zeros(2, 2, device="cuda")) is None
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("pooling,act", [("max", "relu"), ("mean", "gelu")])
def test_dependent_launch_matches_stream_ordered_launch(pooling, act):
    """The kernels of the train step are launched with programmatic dependent launch (each one is scheduled while
    its predecessor drains and waits for it before its first global access).  Replays of the captured step over
    changing batches must give bit-identical gradients to plain stream-ordered launches of the same kernels
    (everything except the loss scalar's float atomics is order-deterministic)."""
    from pcc_b200 import _lib
    from pcc_b200.train_step import GraphedTrainStep
    B, N, d = 64, 256, 3
    batches = []
    g = torch.Generator().manual_seed(5)
    for _ in range(6):
        batches.append((torch.randn(B * N, d, generator=g).cuda(), (torch.rand(B, 2, generator=g) > 0.5).float().cuda()))
    idx = torch.arange(B, device="cuda").repeat_interleave(N)
    grads = []
    try:
        for pdl in (1, 0):
            _lib.call("pcc_debug_set_pdl", pdl)
            torch.manual_seed(1)
            m = pcc_b200.DeepSets(d, [256, 256], [256], 2, act, layer_norm=False, residual_block=False, pooling=pooling,
                                  precision="bf16").cuda()
            gs = GraphedTrainStep(m, (batches[0][0], idx), batches[0][1], forward_kwargs={"num_sets": B}, warmup=2)
            out = []
            for rep in range(3):
                for x, y in batches:
                    gs.step((x, idx), y)
                    out.append([p.grad.clone() for p in m.parameters()])
            torch.cuda.synchronize()
            grads.append(out)
    finally:
        _lib.call("pcc_debug_set_pdl", 1)
    for a, b in zip(*grads):
        for ga, gb in zip(a, b):
            assert torch.equal(ga, gb)


@pytest.mark.parametrize("pool,H", [("sum", 128), ("mean", 256), ("max", 256)])
def test_interior_empty_sets(pool, H):
    """Sets without points inside the index range (a gap in idx, or an explicit num_sets): the library defines their
    pooled row as 0 and they receive no gradient.  One 128-row tile here intersects 328 sets (64 one-point sets,
    200 EMPTY ones, 64 one-point sets): the commuted sum / mean pooling runs its pooling MMA in chunks of <= 128 sets;
    max pooling must not route the gradient of an empty set (argmax -1) to row 0."""
    d, act = 3, "gelu"
    cfg = _cfg(act, pool, False, H, 2, d)
    sd = O.init_state_dict(cfg, seed=91)
    ids = list(range(64)) + list(range(264, 328)) + [328] * 300 + [330] * 5
    num_sets = 480                                           # 149 trailing empty sets as well
    idx = torch.tensor(ids, dtype=torch.long)
    g = torch.Generator().manual_seed(92)
    x = torch.randn(len(ids), d, generator=g)
    wt = torch.randn(num_sets, H, generator=g)
    m = pcc_b200.DeepSets(**cfg, precision="bf16").cuda()
    m.load_state_dict(sd)
    off = PF.segment_offsets(idx.cuda(), num_sets)
    pooled = FZ.phi_pool(x.cuda(), off, m._phi_plan, act, pool)
    (pooled * wt.cuda()).sum().backward()
    torch.cuda.synchronize()
    # oracle on the compacted batch (non-empty sets only), same stated operand rounding
    nonempty = sorted(set(ids))
    remap = {b: i for i, b in enumerate(nonempty)}
    cidx = torch.tensor([remap[b] for b in ids], dtype=torch.long)
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
    plan = O.layer_plan("phi", d, [H, H], H, False, False)
    phi_x = O.mlp_forward(leaves, plan, act, x, "bf16", round_final_weight=(pool == "max"))
    if pool == "max":   # evaluate at the rows the kernel selected (near-ties may resolve differently, see the header)
        arg = _fused_argmax(m, x.cuda(), off, act)
        assert bool((arg[[b for b in range(num_sets) if b not in remap]] == -1).all())
        ref = phi_x[arg[nonempty], torch.arange(H).expand(len(nonempty), -1)]
    else:
        ref, _ = O.segment_pool(phi_x, O.segment_offsets(cidx), pool)
    (ref * wt[nonempty]).sum().backward()
    got = pooled.detach().cpu()
    empty = torch.ones(num_sets, dtype=torch.bool)
    empty[nonempty] = False
    assert bool((got[empty] == 0).all())
    assert rel_err(got[nonempty], ref) < BF16_TOL
    for i, Lr in enumerate(m._phi_plan):
        for nm, p in (("weight", Lr["lin"].weight), ("bias", Lr["lin"].bias)):
            r = leaves[f"{plan[i]['lin']}.{nm}"].grad
            e = rel_l2(p.grad, r)
            assert e < BF16_GRAD_TOL, (pool, plan[i]["lin"], nm, e)


def test_fused_path_refuses_input_gradient():
    m = pcc_b200.DeepSets(3, [128, 128], [64], 2, "relu", layer_norm=False, pooling="mean", precision="bf16").cuda()
    x = torch.randn(200, 3, device="cuda", requires_grad=True)
    idx = torch.arange(2, device="cuda").repeat_interleave(100)
    with pytest.raises(RuntimeError, match="gradient for x"):
        m(x, idx)
