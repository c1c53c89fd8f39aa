import os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "point-cloud-classifier_b200"))
import pcc_b200
from pcc_b200 import _lib
pool = sys.argv[1] if len(sys.argv) > 1 else "sum"
act = sys.argv[2] if len(sys.argv) > 2 else "relu"
res = len(sys.argv) > 3 and sys.argv[3] == "res"
B, N = 256, 1024
m = pcc_b200.DeepSets(3, [256, 256], [256], 10, act, layer_norm=False, residual_block=res, pooling=pool, precision="bf16").cuda()
x = torch.randn(B * N, 3, device="cuda"); idx = torch.arange(B, device="cuda").repeat_interleave(N)
y = (torch.rand(B, 10, device="cuda") > 0.5).float(); lf = torch.nn.BCEWithLogitsLoss()
buf = torch.zeros(4 * 4096, dtype=torch.int64, device="cuda")
for it in range(3):
    if it == 2: _lib.call("pcc_debug_set_trace", _lib.ptr(buf))
    loss = lf(m(x, idx, num_sets=B), y); m.zero_grad(set_to_none=True)
    if it == 2:
        buf.zero_()   # drop the forward kernel's events; keep the backward's
    loss.backward()
torch.cuda.synchronize(); _lib.call("pcc_debug_set_trace", None)
t = buf.cpu().numpy().reshape(4, 2048, 2)
# epilogue (role 0) events; with max pooling and two hidden layers the h_0 and h_1 / dZ_1 passes hand their slabs to the
# MMA thread as they finish (no event), and with ReLU the next tile's x is staged right after event 13
names = {0: "tile start", 1: "bufG free (acquire; max pooling, L = 3: fetched in the h0 pass)", 2: "x staged (ReLU max pooling: first tile only)",
         3: "final dZ built / final weight rows requested", 4: "final dZ stored", 5: "z0 ready", 6: "h0 pass done",
         7: "h0 handed over", 8: "dH_last ready (non-virtual rows)", 9: "z1 ready", 10: "h0 stores read (acquire)",
         11: "h1/dZ1 pass done", 12: "h1/dZ1 stores issued", 13: "h1/dZ1 stores read", 14: "dH0 (and recomputed z0) ready",
         15: "acquire done", 16: "dZ0 pass done", 17: "dZ0 stored"}
ev = [(int(t[0, i, 1]), int(t[0, i, 0])) for i in range(2048) if t[0, i, 1] != 0]
t0 = ev[0][0]; prev = None; tiles = 0
for ts, id_ in ev:
    if id_ == 0: tiles += 1
    if tiles == 2:
        print(f"{ts - t0:9d} (+{0 if prev is None else ts - prev:6d}) {names.get(id_, id_)}")
    prev = ts
print("tiles", tiles, "total", ev[-1][0] - t0)
# waits of the MMA thread (role 1) and the weight producer (role 2) inside the traced tile's window
if tiles >= 2:
    starts = [ts for ts, id_ in ev if id_ == 0]
    w0, w1 = starts[1], (starts[2] if len(starts) > 2 else ev[-1][0])
    for role, pairs in ((1, {40: "MMA: operand hand-over waits", 42: "MMA: weight slab (ring full) waits", 44: "MMA: slab hand-over waits"}),
                        (2, {30: "producer: ring slot (empty) waits"})):
        rv = [(int(t[role, i, 1]), int(t[role, i, 0])) for i in range(2048) if t[role, i, 1] != 0]
        tot = {k: [0, 0] for k in pairs}
        for (ta, ia), (tb, ib) in zip(rv, rv[1:]):
            if ia in pairs and ib == ia + 1 and ta >= w0 and tb <= w1:
                tot[ia][0] += tb - ta; tot[ia][1] += 1
        for k, name in pairs.items():
            print(f"{name:40s} {tot[k][0]:7d} cycles over {tot[k][1]} waits")
    print("tile window", w1 - w0, "cycles")
    mma = {41: "x handed over", 43: "weight slab landed", 45: "h0/dZ1 slab handed over"}
    print("MMA thread, same tile:")
    for ts, id_ in [(int(t[1, i, 1]), int(t[1, i, 0])) for i in range(2048) if t[1, i, 1] != 0]:
        if w0 <= ts <= w1 and id_ in mma:
            print(f"{ts - t0:9d} {mma[id_]}")
