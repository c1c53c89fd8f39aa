"""Secondary measurement (BASELINE config 4): GraphNet (configs/graph_net.yaml model) on kNN graphs,
k=20, N=1024 points per cloud; kNN build and train step timed separately with CUDA events.

With --aggr / --precision (one or more values each): the graphed train step of `bench.py --config graphnet`
(KnnGraphNet, kNN build inside, tanh, deepchem_style, B clouds of N points) for every (precision, aggr) arm, the arms
alternated over --rounds rounds on the same batch; then, in a separate run with the pcc_prof_* event brackets on, the
per-launch times of gnn_conv_fwd_kernel (slot 3) and gnn_agg_bwd_kernel (slot 5) of the bf16 arms.  Prints one JSON
document (also written to --out) with the card name and power limit read in the same process."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "point-cloud-classifier_b200"))
import pcc_b200
from pcc_b200 import functional as PF


def timeit(fn, steps=10, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run(B, N=1024, k=20):
    torch.manual_seed(0)
    m = pcc_b200.GraphNet(input_dim=4, hidden_dim=128, output_dim=1, activation="tanh", local_pooling="add",
                          global_pooling="mean", deepchem_style=True).cuda()
    n = B * N
    feats = torch.randn(n, 4, device="cuda")
    feats[:, 0] = torch.rand(n, device="cuda")
    memb = torch.arange(B, device="cuda").repeat_interleave(N)
    y = (torch.rand(B, 1, device="cuda") > 0.5).float()
    off = PF.segment_offsets(memb, B)
    t_knn = timeit(lambda: PF.knn(feats[:, 1:4], off, k))
    nbr, _ = PF.knn(feats[:, 1:4], off, k)
    edges = PF.knn_edges(nbr)
    lf = torch.nn.BCEWithLogitsLoss()

    def step():
        loss = lf(m(feats, memb, edges, num_graphs=B), y)
        m.zero_grad(set_to_none=True)
        loss.backward()
    t_step = timeit(step, steps=5, warmup=2)
    # the same step captured in a CUDA graph (101 launches per step: eager mode is launch bound)
    t_graph = float("nan")
    try:
        from pcc_b200.train_step import GraphedTrainStep
        gs = GraphedTrainStep(m, [feats, memb, edges], y, forward_kwargs={"num_graphs": B})
        t_graph = timeit(gs.run, steps=5, warmup=2)
    except Exception as e:  # noqa: BLE001
        print(f"  (graph capture failed: {type(e).__name__}: {e})")
    pairs = B * N * N
    print(f"GraphNet B={B:4d} N={N} k={k}: kNN {t_knn:8.3f} ms ({pairs / t_knn / 1e6:8.1f} Gpairs/s) | "
          f"train step eager {t_step:8.3f} ms, CUDA graph {t_graph:8.3f} ms = {B / t_graph * 1e3:8.0f} graphs/s, "
          f"E={edges.shape[1]}", flush=True)


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({type(e).__name__})"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def run_arms(precisions, aggrs, B, N, k, rounds, steps, warmup):
    """alternating graphed-step timings of every (precision, aggr) arm + per-kernel times of the bf16 arms"""
    from pcc_b200 import _lib
    from pcc_b200.train_step import GraphedTrainStep
    n = B * N
    g = torch.Generator(device="cuda").manual_seed(0)
    feats = torch.randn(n, 4, device="cuda", generator=g)
    feats[:, 0] = torch.rand(n, device="cuda", generator=g)
    memb = torch.arange(B, device="cuda").repeat_interleave(N)
    y = (torch.rand(B, 1, device="cuda", generator=g) > 0.5).float()
    arms = {}
    for prec in precisions:
        for aggr in aggrs:
            torch.manual_seed(0)
            m = pcc_b200.KnnGraphNet(k=k, precision=prec, input_dim=4, hidden_dim=128, output_dim=1, activation="tanh",
                                     local_pooling=aggr, global_pooling="mean", deepchem_style=True).cuda()
            m.train()
            gs = GraphedTrainStep(m, [feats, memb], y, forward_kwargs={"num_graphs": B})
            arms[f"{prec}/{aggr}"] = (m, gs)
            assert m.net.last_path == ("fused-bf16" if prec == "bf16" else "fp32"), (prec, aggr, m.net.last_path)
    times = {name: [] for name in arms}
    for _ in range(rounds):
        for name, (_, gs) in arms.items():
            times[name].append(timeit(gs.run, steps=steps, warmup=warmup))
    out = {"B": B, "N": N, "k": k, "E": n * k, "rounds": rounds, "steps_per_round": steps, "card": _card(),
           "step_ms": {name: {"median": sorted(t)[len(t) // 2], "min": min(t), "max": max(t), "all": t}
                       for name, t in times.items()}}
    # per-kernel times: eager steps with the event brackets on (not under graph capture)
    slots = {"gnn_conv_fwd_kernel": 3, "gnn_agg_bwd_kernel": 5}
    kern = {}
    lf = torch.nn.BCEWithLogitsLoss()
    for name, (m, _) in arms.items():
        if not name.startswith("bf16/"):
            continue
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            lf(m(feats, memb, num_graphs=B), y).backward()
        torch.cuda.synchronize()
        _lib.call("pcc_prof_enable", 1)
        for _ in range(steps):
            m.zero_grad(set_to_none=True)
            lf(m(feats, memb, num_graphs=B), y).backward()
        torch.cuda.synchronize()
        _lib.call("pcc_prof_enable", 0)
        row = {}
        for kname, slot in slots.items():
            t, c = ctypes.c_double(0.0), ctypes.c_int64(0)
            _lib.call("pcc_prof_read", slot, ctypes.byref(t), ctypes.byref(c))
            row[kname] = {"ms_per_launch": t.value / max(c.value, 1), "launches": c.value}
        kern[name] = row
    out["kernel_ms"] = kern
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("dense_precision", nargs="?", help='"tf32": single-TF32 node-level GEMMs (legacy table)')
    ap.add_argument("--aggr", nargs="+", help="local_pooling of the arms (add / mean / max)")
    ap.add_argument("--precision", nargs="+", help="GraphNet precision of the arms (fp32 / bf16)")
    ap.add_argument("--B", type=int, default=256)
    ap.add_argument("--N", type=int, default=1024)
    ap.add_argument("--k", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON document here")
    a = ap.parse_args()
    if a.aggr or a.precision:
        res = run_arms(a.precision or ["bf16"], a.aggr or ["add"], a.B, a.N, a.k, a.rounds, a.steps, a.warmup)
        text = json.dumps(res, indent=1)
        print(text, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(text + "\n")
        sys.exit(0)
    if a.dense_precision:
        PF.set_dense_precision(a.dense_precision)   # "tf32": single-TF32 node-level GEMMs
        print(f"dense precision: {a.dense_precision}")
    run(32)
    run(256)
    for N in (256, 4096):
        run(262144 // N, N=N)
