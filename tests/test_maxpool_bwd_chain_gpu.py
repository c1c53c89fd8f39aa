"""GPU: the max-pool backward chain kernel (`phi_bwd_chain_kernel`, pcc_fused_bwd.cu) in virtual-row mode, every
compiled variant, against its serial schedule bit for bit and against an fp64 reference tile by tile.

Max pooling with two hidden layers runs its backward on B*H virtual rows (row b*H + f = the argmax row of (b, f),
gradient on feature f only) through the pipelined schedule of the chain kernel (`PIPE = true`): slab hand-overs on
mbarriers, two TMEM accumulators that swap roles every tile, ReLU act' bits kept in registers, the next x tile staged
under the dgrad.  `pcc_debug_set_bwd_pipe(0)` selects the serial schedule (`PIPE = false`) for the same call.  The
tests call `pcc_deepsets_phi_pool_bwd` directly (argmax = NULL, n = B*H) with the packed weights of one forward call.

Variant matrix (12 = H x act x ResidualBlock, d spread over 1 / 3 / 7):

    H = 128: relu d=1, relu+res d=7, gelu d=3, gelu+res d=1, silu d=7, silu+res d=3
    H = 256: relu d=3, relu+res d=1, gelu d=7, gelu+res d=3, silu d=1, silu+res d=7

Tile counts T = B*H/128 (persistent grid = min(T, SMs), SMs read from the device; 148 on a B200):
    "1"       H = 128, B = 1: the grid is raised to 2, so one chain CTA has no tile (H = 128 variants only)
    "few"     T = 37 (H = 128) / 38 (H = 256): one tile per CTA
    "sms+2"   T = SMs + 2: CTAs 0 and 1 run two tiles, the rest one
    "3sms+2"  T = 3 SMs + 2: CTAs 0 and 1 run four tiles, the rest three (both parities of the accumulator rotation)

Checks per case:
 1. every dW / db of all three layers is bit-identical between the pipelined and the serial schedule, and between
    two pipelined runs (the chain, weight-gradient and reduction kernels have no float atomics);
 2. with the pooled gradient zero outside the tiles of CTA 0 (most tiles) and of the last CTA (fewest), and exactly
    zero on some rows inside them (what the row gather leaves for an empty set), the gradients equal an fp64
    restatement of the kernel's arithmetic on those <= 7 tiles: max|got - ref| <= TOL * max|ref| per tensor.  A
    zero-gradient tile still runs through the pipeline but adds nothing, so each checked tile carries >= 1/7 of
    every gradient and a wrong slab or a stale accumulator moves it far beyond the tolerance.

The reference rounds to bf16 where the kernel does: x, W0, W1 and W2 (the packed images), h0 = bf16(act(z0 + b0)),
h1 = bf16(act(z1 + b1) [+ h0]), dZ1 = bf16(dH1 act'(z1 + b1)) with dH1 = dpooled W2[f, :], dZ0 = bf16(dH0
act'(z0 + b0)) with dH0 = dZ1 W1 [+ dH1]; dW1 = dZ1^T h0, dW0 = dZ0^T x, db from the bf16 dZ images; dW2[f] =
sum_b dpooled h1 and db2[f] = sum_b dpooled.  GELU / SiLU take the tanh form of pcc_act_bf16.cuh (exact tanh here,
tanh.approx.f32 in the kernel).

Measured on an NVIDIA B200 (148 SMs, 1000 W power limit), max|got - ref| / max|ref| over the 42 cases, and TOL = 2x
that maximum, rounded up:

    tensor   relu      gelu / silu   TOL
    dW0      2.5e-4    2.2e-3        5e-3
    db0      1.5e-4    9.6e-4        2e-3
    dW1      8.1e-7    1.1e-3        2.5e-3
    db1      6.1e-8    5.3e-4        1.2e-3
    dW2      9.3e-4    3.6e-3        7.5e-3
    db2      7.6e-8    1.1e-7        2.5e-7

The GELU / SiLU figures are the kernel's tanh.approx (relative error ~5e-4) carried through one bf16 rounding: where
it moves a value across a rounding boundary the stored activation differs by one bf16 ulp (2^-8 .. 2^-7 of it).  dW2
shows that nearly undiluted, because each of its rows sums only the <= 7 checked rows of one feature.  The whole file
(84 tests) runs in about 5 s on the B200.
"""
import contextlib
import ctypes as C
from types import SimpleNamespace

import pytest
import torch

from pcc_b200 import _lib, fused as FZ

pytestmark = pytest.mark.gpu

NAMES = ("dW0", "db0", "dW1", "db1", "dW2", "db2")
TOL = {"dW0": 5e-3, "db0": 2e-3, "dW1": 2.5e-3, "db1": 1.2e-3, "dW2": 7.5e-3, "db2": 2.5e-7}

VARIANTS = [
    # H, act, residual, d
    (128, "relu", False, 1),
    (128, "relu", True, 7),
    (128, "gelu", False, 3),
    (128, "gelu", True, 1),
    (128, "silu", False, 7),
    (128, "silu", True, 3),
    (256, "relu", False, 3),
    (256, "relu", True, 1),
    (256, "gelu", False, 7),
    (256, "gelu", True, 3),
    (256, "silu", False, 1),
    (256, "silu", True, 7),
]
TILES = ("1", "few", "sms+2", "3sms+2")
CASES = [(H, act, res, d, t) for (H, act, res, d) in VARIANTS for t in TILES if H == 128 or t != "1"]
GRID_CAP = 160  # kGridCap in pcc_fused_bwd.cu: the chain grid is min(tiles, SMs, 160), at least 2 with two hidden layers


def _ids(c):
    H, act, res, d, t = c
    return f"H{H}-{act}{'-res' if res else ''}-d{d}-T{t}"


@contextlib.contextmanager
def _bwd_pipe(on):
    _lib.call("pcc_debug_set_bwd_pipe", on)
    try:
        yield
    finally:
        _lib.call("pcc_debug_set_bwd_pipe", 1)


def _setup(H, act, res, d, tiles):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    T = {"1": 1, "few": 37, "sms+2": sms + 2, "3sms+2": 3 * sms + 2}[tiles]
    B = -(-T * 128 // H)
    n = B * H
    T = n // 128
    grid = max(min(T, sms, GRID_CAP), 2)
    g = torch.Generator().manual_seed(10 * VARIANTS.index((H, act, res, d)) + TILES.index(tiles))
    params = []
    for k in (d, H, H):
        params.append((torch.randn(H, k, generator=g) / k ** 0.5, 0.1 * torch.randn(H, generator=g)))
    x = torch.randn(n, d, generator=g)
    dp = torch.randn(n, generator=g)
    dev = [(w.cuda(), b.cuda()) for w, b in params]
    plan = [{"lin": SimpleNamespace(in_features=w.shape[1], out_features=H), "res": res and i == 1}
            for i, (w, _) in enumerate(params)]
    dsc = FZ._build_desc(plan, act, "max", dev)
    xc = x.cuda()
    off = torch.arange(0, n + 1, H, dtype=torch.int64, device="cuda")
    ws = torch.empty(_lib.call("pcc_phi_fused_workspace_bytes", C.byref(dsc), n, B), dtype=torch.uint8, device="cuda")
    wpack = torch.empty(_lib.call("pcc_phi_packed_bytes", C.byref(dsc)), dtype=torch.uint8, device="cuda")
    pooled = torch.empty(B, H, device="cuda")
    arg = torch.empty(B, H, dtype=torch.int32, device="cuda")
    _lib.call("pcc_deepsets_phi_pool_fwd", C.byref(dsc), _lib.ptr(xc), _lib.ptr(off), n, B, _lib.ptr(pooled),
              _lib.ptr(arg), _lib.ptr(ws), _lib.ptr(wpack), 0, _lib.stream_ptr(0))
    return SimpleNamespace(H=H, act=act, res=res, n=n, B=B, T=T, grid=grid, params=params, dev=dev, dsc=dsc, x=x,
                           xc=xc, dp=dp, off=off, ws=ws, wpack=wpack)


def _bwd(c, dp):
    """[dW0, db0, dW1, db1, dW2, db2] of one virtual-row backward call; outputs start as NaN, so an entry the
    library does not write fails every check"""
    grads = [torch.full_like(t, float("nan")) for pair in c.dev for t in pair]
    dw = (C.c_void_p * _lib.MAX_PHI_LAYERS)(*[grads[2 * i].data_ptr() for i in range(3)])
    db = (C.c_void_p * _lib.MAX_PHI_LAYERS)(*[grads[2 * i + 1].data_ptr() for i in range(3)])
    dpc = dp.cuda()
    _lib.call("pcc_deepsets_phi_pool_bwd", C.byref(c.dsc), _lib.ptr(c.xc), _lib.ptr(c.off), c.n, c.B, _lib.ptr(dpc),
              None, C.cast(dw, C.c_void_p), C.cast(db, C.c_void_p), _lib.ptr(c.ws), _lib.ptr(c.wpack), 0,
              _lib.stream_ptr(0))
    torch.cuda.synchronize()
    return [t.cpu() for t in grads]


def _bf(t):
    return t.to(torch.bfloat16).double()


def _act(act, z):
    """act(z) and act'(z) in fp64, the formulas of pcc_act_bf16.cuh"""
    if act == "relu":
        return z.clamp_min(0.0), (z > 0).double()
    if act == "gelu":
        c0 = 0.7978845608028654
        t = torch.tanh(c0 * z * (1.0 + 0.044715 * z * z))
        return 0.5 * z * (1.0 + t), 0.5 * (1.0 + t) + 0.5 * z * (1.0 - t * t) * c0 * (1.0 + 0.134145 * z * z)
    s = 0.5 * (1.0 + torch.tanh(0.5 * z))
    return z * s, s * (1.0 + z * (1.0 - s))


def _reference(c, dp, rows):
    """fp64 gradients of the virtual rows `rows` (all other rows carry zero gradient)"""
    (W0, b0), (W1, b1), (W2, b2) = c.params
    H = c.H
    xh = _bf(c.x[rows])
    a0, da0 = _act(c.act, xh @ _bf(W0).T + b0.double())
    h0 = _bf(a0)
    a1, da1 = _act(c.act, h0 @ _bf(W1).T + b1.double())
    h1 = _bf(a1 + h0 if c.res else a1)
    f = rows % H
    g = dp[rows].double()
    dH1 = g[:, None] * _bf(W2)[f]
    dZ1 = _bf(dH1 * da1)
    dH0 = dZ1 @ _bf(W1)
    if c.res:
        dH0 = dH0 + dH1
    dZ0 = _bf(dH0 * da0)
    dW2 = torch.zeros(H, H, dtype=torch.float64).index_add_(0, f, g[:, None] * h1)
    db2 = torch.zeros(H, dtype=torch.float64).index_add_(0, f, g)
    return [dZ0.T @ xh, dZ0.sum(0), dZ1.T @ h0, dZ1.sum(0), dW2, db2]


@pytest.mark.parametrize("H,act,res,d,tiles", CASES, ids=[_ids(c) for c in CASES])
def test_pipelined_chain_bit_exact_vs_serial(H, act, res, d, tiles):
    c = _setup(H, act, res, d, tiles)
    assert bool((c.dp != 0).all())
    with _bwd_pipe(1):
        pipe = _bwd(c, c.dp)
        again = _bwd(c, c.dp)
    with _bwd_pipe(0):
        serial = _bwd(c, c.dp)
    for name, p, a, s in zip(NAMES, pipe, again, serial):
        assert torch.equal(p, a), (name, "two pipelined runs differ")
        assert torch.equal(p, s), (name, "pipelined != serial", float((p - s).abs().max()))


@pytest.mark.parametrize("H,act,res,d,tiles", CASES, ids=[_ids(c) for c in CASES])
def test_pipelined_chain_tiles_match_reference(H, act, res, d, tiles):
    c = _setup(H, act, res, d, tiles)
    first = list(range(0, c.T, c.grid))                # CTA 0: the most tiles
    last = list(range(c.grid - 1, c.T, c.grid))        # last CTA: the fewest (none when T = 1)
    sel = torch.tensor(first + last, dtype=torch.int64)
    rows = (sel[:, None] * 128 + torch.arange(128)).reshape(-1)
    dp = torch.zeros(c.n)
    dp[rows] = c.dp[rows]
    dp[rows[rows % 13 == 5]] = 0.0                     # empty sets: the row gather zeroes their pooled gradient
    got = _bwd(c, dp)
    ref = _reference(c, dp, rows)
    errs = {}
    for name, a, r in zip(NAMES, got, ref):
        assert bool(torch.isfinite(a).all()), name
        errs[name] = float((a.double() - r).abs().max() / r.abs().max())
    print(f"H={H} {act} res={res} d={d} T={c.T} grid={c.grid} tiles CTA0 {first} last {last}: "
          + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for name, e in errs.items():
        assert e <= TOL[name], (name, e, TOL[name])
