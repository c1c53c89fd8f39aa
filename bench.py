#!/usr/bin/env python
"""bench.py — benchmark of the B200-native point-set encoder hot path.

Metric (BASELINE.json): train samples/sec (fwd+bwd), DeepSets B=256 N=1024 per GPU.
A "step" = forward + BCEWithLogitsLoss + backward of one batch (+ gradient all-reduce when N > 1).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # headline: configs[1] (relu + max, bf16 path)
  python bench.py --config yaml|ragged|graphnet|sweep [...]       # the other BASELINE configs (see WORKLOADS)
  python bench.py --impl reference [...]                          # reference CPU path (oracle port) on the host cores
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N    # one rank per GPU (weak scaling)

Prints ONE JSON line on rank 0.  A timed window is exactly K steps between barrier + synchronize; `--repeats R` times
R windows (default 1) and reports the MEDIAN window, all windows are listed in `windows_ms`.

`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (float32): `loss`,
`logits` and `grad.<parameter name>` for every parameter (rank 0's shard).  The inputs and the initial parameters are
seeded, so two builds of the project run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "point-cloud-classifier_b200"))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_ROTATE = 32   # distinct input batches per rank (headline: 166 MB > 126 MB L2)


# ---------------------------------------------------------------------------- workloads
def _lognormal_sizes(B, seed=2):
    """SURVEY.md section 8d, C3: N_i = clamp(round(exp(N(ln 1500, 0.8^2))), 16, 4096)"""
    g = torch.Generator().manual_seed(seed)
    s = torch.exp(torch.randn(B, generator=g) * 0.8 + math.log(1500.0)).round().clamp(16, 4096)
    return [int(v) for v in s]


class DeepSetsWorkload:
    kind = "deepsets"

    def __init__(self, name, B, N, d, out, act, pool, res, ragged=False, H=256, desc=""):
        self.name, self.B, self.N, self.d, self.out, self.H, self.ragged = name, B, N, d, out, H, ragged
        self.cfg = dict(input_dim=d, phi_layers=[H, H], rho_layers=[H], output_dim=out, activation=act, layer_norm=False,
                        residual_block=res, pooling=pool)
        self.sizes = _lognormal_sizes(B) if ragged else [N] * B
        self.points = sum(self.sizes)
        self.desc = desc
        # SURVEY.md section 8(d): algorithmic FLOP per point, reference formulation, recompute not credited
        self.flop_fwd_pt = 2 * (H * d + 2 * H * H)
        self.flop_train_pt = 3 * self.flop_fwd_pt - 2 * H * d
        self.kernel_flop_pt = {"phi_pool_fwd_kernel": self.flop_fwd_pt, "phi_bwd_chain_kernel": 2 * (2 * H * H),
                               "phi_wgrad_kernel": self.flop_fwd_pt}
        self.unit_name = "sets"

    def forward_kwargs(self):
        return {"num_sets": self.B}

    def build_model(self, dev, precision):
        import pcc_b200
        return pcc_b200.DeepSets(**self.cfg, precision=precision).to(dev)

    def expected_path(self, precision):
        return "fused-bf16" if precision == "bf16" else "fp32"

    def make_batches(self, n_batches, seed, pin=True, B=None):
        """[(inputs tuple, target)] on the host, in the layout of the reference collate (utils/data.py:651-663)"""
        B = B or self.B
        sizes = self.sizes[:B] if self.ragged else [self.N] * B
        g = torch.Generator().manual_seed(seed)
        idx = torch.cat([torch.full((s,), i, dtype=torch.long) for i, s in enumerate(sizes)])
        out = []
        for _ in range(n_batches):
            x = torch.randn(sum(sizes), self.d, generator=g)
            y = (torch.rand(B, self.out, generator=g) > 0.5).float()
            ts = (x, idx, y)
            if pin:
                ts = tuple(t.pin_memory() for t in ts)
            out.append((ts[:2], ts[2]))
        return out

    # reference CPU arm: oracle port (pinned to the reference module by tests/golden)
    def cpu_state(self):
        from oracle import deepsets_oracle as O
        return O.init_state_dict(self.cfg, seed=0)

    def cpu_step(self, sd, inputs, y):
        from oracle import deepsets_oracle as O
        return O.deepsets_train_step(sd, self.cfg, inputs[0], inputs[1], y)

    def workload_text(self):
        return self.desc


class GraphNetWorkload:
    """configs[3]: configs/graph_net.yaml model on kNN graphs (k = 20) over N = 1024-point clouds.  A step = kNN graph
    build (pcc_knn) + CSR + forward + BCEWithLogitsLoss + backward."""
    kind = "graphnet"

    def __init__(self, name, B, N, k=20, hidden=128, desc=""):
        self.name, self.B, self.N, self.k, self.hidden = name, B, N, k, hidden
        self.cfg = dict(input_dim=4, hidden_dim=hidden, output_dim=1, activation="tanh", use_gat=False, gat_heads=4,
                        sag_pool=False, pool_ratio=0.5, local_pooling="add", global_pooling="mean", deepchem_style=True)
        self.points = B * N
        self.desc = desc
        C = hidden
        # SURVEY.md section 8(d), per node: fwd 2 (2*4*C + 2*C*C + C*256) FLOP, train ~3x; aggregation gather bytes
        # k*C*4 per conv and direction (conv1: C = 4), edges 16 B / edge
        self.flop_fwd_pt = 2 * (2 * 4 * C + 2 * C * C + C * 256)
        self.flop_train_pt = 3 * self.flop_fwd_pt
        self.bytes_gather_pt = 2 * (k * 4 * 4 + k * C * 4) + 2 * k * 16
        self.unit_name = "graphs"

    def forward_kwargs(self):
        return {"num_graphs": self.B}

    def build_model(self, dev, precision):
        import pcc_b200
        return pcc_b200.KnnGraphNet(k=self.k, precision=precision, **self.cfg).to(dev)

    def expected_path(self, precision):
        return None

    def make_batches(self, n_batches, seed, pin=True, B=None):
        B = B or self.B
        g = torch.Generator().manual_seed(seed)
        memb = torch.arange(B).repeat_interleave(self.N)
        out = []
        for _ in range(n_batches):
            f = torch.randn(B * self.N, 4, generator=g)          # col 0: normalised energy, cols 1:4 xyz (data.py:808-813)
            f[:, 0] = torch.rand(B * self.N, generator=g)
            y = (torch.rand(B, 1, generator=g) > 0.5).float()
            ts = (f, memb, y)
            if pin:
                ts = tuple(t.pin_memory() for t in ts)
            out.append((ts[:2], ts[2]))
        return out

    def cpu_state(self):
        from oracle import graphnet_oracle as GO
        return GO.init_state_dict(self.cfg, seed=0)

    def cpu_step(self, sd, inputs, y):
        import numpy as np
        from oracle import graphnet_oracle as GO
        from oracle import knn_oracle as KO
        f, memb = inputs
        B = int(memb.max()) + 1
        off = np.arange(B + 1, dtype=np.int64) * self.N
        nbr, _ = KO.knn_neighbours(f[:, 1:4].numpy(), off, self.k)
        edges = torch.from_numpy(KO.knn_edges(nbr))
        return GO.graphnet_train_step(sd, self.cfg, f, memb, edges, None, y)

    def workload_text(self):
        return self.desc


def make_workload(name, B=None, N=None):
    if name == "deepsets":
        return DeepSetsWorkload(name, B or 256, N or 1024, 3, 10, "relu", "max", False,
                                desc="configs[1]: DeepSets B=256 N=1024 per GPU, phi[3-256-256]+final(256) relu, max pool, "
                                     "rho[256]-10, fwd + BCEWithLogitsLoss + bwd")
    if name == "yaml":
        return DeepSetsWorkload(name, B or 256, N or 1024, 6, 1, "gelu", "mean", True,
                                desc="configs/deep_sets.yaml model (gelu + ResidualBlock + mean pool, d=6, out=1, no LayerNorm) "
                                     "at B=256 N=1024 per GPU, fwd + BCEWithLogitsLoss + bwd")
    if name == "ragged":
        return DeepSetsWorkload(name, B or 256, N or 1024, 3, 10, "relu", "sum", False, ragged=True,
                                desc="configs[2]: DeepSets variable-size sets, N_i log-normal in [16, 4096] (478 k points per "
                                     "256 sets), sum pool (sum / sqrt(n)), relu, fwd + loss + bwd")
    if name == "graphnet":
        return GraphNetWorkload(name, B or 256, N or 1024,
                                desc="configs[3]: configs/graph_net.yaml GraphNet (tanh, add aggregation, deepchem) on kNN k=20 "
                                     "graphs, N=1024 per cloud, B=256 per GPU; step = kNN build + CSR + fwd + loss + bwd")
    raise SystemExit(f"unknown --config {name}")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0))),
                "tflops_burst": float(d.get("bf16_tflops", 1650.0)),
                "hbm": float(d.get("hbm_gbs", 6650.0)), "source": "MEASURED_PEAKS.json"}
    return {"tflops": 1400.0, "tflops_burst": 1650.0, "hbm": 6650.0, "source": "B200_PROFILING.md fallback"}


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML from a background thread, ~2 ms
    period; the timed region lasts tens of milliseconds, too short for `nvidia-smi -lms`)."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop, self._thr, self._err = False, None, None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            while not self._stop:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for k, b in bits.items():
                        if r & b:
                            self.reasons.add(k)
                except Exception:
                    pass
                time.sleep(0.002)
        except Exception as e:  # NVML missing: report it, never fail the bench
            self._err = f"{type(e).__name__}: {e}"

    def start(self):
        import threading
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()

    def stop(self):
        self._stop = True
        if self._thr is not None:
            self._thr.join(timeout=2)
        out = {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
               "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if self._err:
            out["error"] = self._err
        return out


# ---------------------------------------------------------------------------- reference arm (host CPU)
def cpu_reference_rate(wl, steps, warmup, sample_units=None, budget_s=25.0):
    """The reference's own CPU path (oracle port: functional restatement of models/deep_sets.py / graph_net.py +
    wrapper.py:38 loss, pinned to the reference by tests/golden) on the box's host cores, all threads.
    One step = fwd + loss + bwd of `sample_units` sets / graphs of the workload (default: the FULL per-GPU batch)."""
    torch.set_num_threads(os.cpu_count() or 1)
    units = sample_units or wl.B
    sd = wl.cpu_state()
    (inputs, y), = wl.make_batches(1, seed=1, pin=False, B=units)
    times = []
    t_begin = time.perf_counter()
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        wl.cpu_step(sd, inputs, y)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        if time.perf_counter() - t_begin > budget_s and len(times) >= 2:
            break
    ms = statistics.median(times) * 1e3
    pts = inputs[0].shape[0]
    return {"value": units / ms * 1e3, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{len(times)} steps of fwd+loss+bwd on {units} {wl.unit_name} ({pts} points, "
                      f"{'the full per-GPU batch' if units == wl.B else 'a sample'} of the same workload), median",
            "ms_per_step": ms, "steps": len(times), "units": units}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = make_workload(args.config if args.config != "sweep" else "deepsets")
    # the full 256-set batch per step (same config as the CUDA arm); GraphNet's numpy kNN oracle is O(N^2): 32 graphs
    units = None if wl.kind == "deepsets" else 32
    cb = cpu_reference_rate(wl, args.steps, min(args.warmup, 3), sample_units=units, budget_s=150.0)
    line = {"impl": "reference", "metric": metric_name(wl), "value": cb["value"],
            "unit": "samples/s", "n_gpus": args.gpus, "steps": cb["steps"], "warmup": min(args.warmup, 3),
            "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl.workload_text(), "name": wl.name, "units_per_gpu": cb["units"],
                       "points_per_gpu": wl.points if cb["units"] == wl.B else cb["units"] * wl.N, "device": "host CPU",
                       "precision_mode": "fp32"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def metric_name(wl):
    if wl.name == "deepsets":
        return "train samples/sec (fwd+bwd), DeepSets B=256 N=1024"
    return f"train samples/sec (fwd+bwd), {wl.name} B={wl.B} N={wl.N}"


# ---------------------------------------------------------------------------- comparators (single GPU, rank 0)
def eager_gpu_baseline(wl, dev, steps=5, warmup=2):
    """The reference's "existing GPU path": its algorithm as stock PyTorch eager ops on the same B200 (oracle port
    moved to cuda:0, fp32, TF32 off — the port runs at the reference module's speed, DESIGN.md section 2)."""
    if wl.kind != "deepsets":
        return eager_gpu_baseline_graph(wl, dev, steps, warmup)
    from oracle import deepsets_oracle as O
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        sd = {k: v.to(dev) for k, v in wl.cpu_state().items()}
        (inputs, y), = wl.make_batches(1, seed=3, pin=False)
        x, idx, y = inputs[0].to(dev), inputs[1].to(dev), y.to(dev)
        for _ in range(warmup):
            O.deepsets_train_step(sd, wl.cfg, x, idx, y)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            O.deepsets_train_step(sd, wl.cfg, x, idx, y)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return {"value": wl.B / ms * 1e3, "unit": "samples/s", "ms_per_step": ms, "steps": steps,
            "what": "reference algorithm as stock PyTorch eager ops on cuda:0 (oracle port, fp32, TF32 off): cuBLAS sgemm + "
                    "B-iteration pooling loop + counts.tolist() sync, same batch shape"}


def eager_gpu_baseline_graph(wl, dev, steps=5, warmup=2):
    """GraphNet: the reference algorithm as stock PyTorch eager ops on cuda:0 (oracle port: index_add scatter for GraphConv,
    torch BatchNorm arithmetic, fp32, TF32 off).  The kNN graph is built once OUTSIDE the timed region (the reference builds
    its edges offline, utils/data.py:847-929), so this arm times less work than the step it is compared with."""
    from oracle import graphnet_oracle as GO
    import pcc_b200
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        sd = {k: v.to(dev) for k, v in wl.cpu_state().items()}
        (inputs, y), = wl.make_batches(1, seed=3, pin=False)
        f, memb, y = inputs[0].to(dev), inputs[1].to(dev), y.to(dev)
        edges, _ = pcc_b200.knn_graph(f, memb, wl.k, num_graphs=wl.B)
        for _ in range(warmup):
            GO.graphnet_train_step(sd, wl.cfg, f, memb, edges, None, y)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            GO.graphnet_train_step(sd, wl.cfg, f, memb, edges, None, y)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
    except Exception as e:   # the arm is a comparator, not the product: report instead of failing the bench line
        return {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return {"value": wl.B / ms * 1e3, "unit": "samples/s", "ms_per_step": ms, "steps": steps,
            "what": "reference GraphNet algorithm as stock PyTorch eager ops on cuda:0 (oracle port, fp32, TF32 off), kNN edge list "
                    "prebuilt outside the timed region"}


def wrapper_loop_e2e(wl, dev, precision, steps=20, warmup=5):
    """The literal training-loop sequence of the reference (models/wrapper.py:51-74) on the drop-in module: pageable
    host tensors `.to(device)`, model(*inputs), optimizer.zero_grad(), BCEWithLogitsLoss, loss.backward(), torch AdamW
    step, loss.item() — eager launches, no CUDA graph, no fused loss / optimizer.  Wall-clock timed."""
    if wl.kind != "deepsets":
        return None
    model = wl.build_model(dev, precision)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)          # wrapper.py:33
    criterion = torch.nn.BCEWithLogitsLoss()                       # wrapper.py:38
    batches = wl.make_batches(4, seed=5, pin=False)
    model.train()

    def one(i):
        inputs, y = batches[i % len(batches)]
        inputs = [t.to(dev) for t in inputs if t is not None]      # wrapper.py:54
        y = y.to(dev)                                              # wrapper.py:55
        logits = model(*inputs)                                    # wrapper.py:58
        opt.zero_grad()                                            # wrapper.py:61
        loss = criterion(logits, y)                                # wrapper.py:64
        loss.backward()                                            # wrapper.py:67
        opt.step()                                                 # wrapper.py:70
        return loss.item() + loss.item()                           # wrapper.py:73-74 (two host reads)
    for i in range(warmup):
        one(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        one(warmup + i)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) / steps * 1e3
    return {"value": wl.B / ms * 1e3, "unit": "samples/s", "ms_per_step": ms, "steps": steps, "precision_mode": precision,
            "what": "wrapper.py:51-74 sequence on pcc_b200.DeepSets: pageable .to(device), eager forward, torch AdamW step, "
                    "loss.item() x2 per step (wall clock, includes the optimizer)"}


# ---------------------------------------------------------------------------- this repo
def run_ours(args):
    import ctypes as C
    import torch.distributed as dist
    from pcc_b200 import _lib
    from pcc_b200.train_step import GraphedTrainStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (sm_100a); there is no CPU fallback. Use --impl reference for the CPU arm.")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    def log(msg):
        if rank == 0:
            print(f"[bench] {msg}", file=sys.stderr, flush=True)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        log(f"process group up: world {world}")
    _lib.call("pcc_check_device", local)

    if args.config == "sweep":
        return run_sweep(args, dev, rank, world, log)
    wl = make_workload(args.config, args.batch, args.points)
    torch.manual_seed(0)
    model = wl.build_model(dev, args.precision)
    n_rot = N_ROTATE if wl.kind == "deepsets" else 8
    host = wl.make_batches(n_rot, seed=1000 + rank)
    devb = [(tuple(t.to(dev) for t in ins), y.to(dev)) for ins, y in host]
    kw = wl.forward_kwargs()

    def build(use_graph, allreduce=None):
        step = GraphedTrainStep(model, devb[0][0], devb[0][1], forward_kwargs=kw,
                                allreduce=(world > 1) if allreduce is None else allreduce, use_graph=use_graph)
        # a replay refills the gradient tensors allocated while its graph was captured; building the next step points
        # the parameters' .grad elsewhere, so each captured step keeps its own
        step.grads = {n: p.grad for n, p in model.named_parameters()} if step.graph is not None else None
        return step
    try:
        gs = build(not args.no_graph)
        graphed = not args.no_graph
    except Exception as e:  # graph capture unavailable (e.g. NCCL capture) -> eager launches
        log(f"CUDA graph capture failed ({type(e).__name__}: {e}); running eager")
        gs = build(False)
        graphed = False
    exp = wl.expected_path(args.precision)
    assert exp is None or model.last_path == exp, (model.last_path, exp)
    log(f"train step built (cuda graph: {graphed})")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, repeats):
        """`repeats` windows of exactly `steps` steps, each bracketed by barrier + synchronize, CUDA-event timed, max
        over ranks per window; returns (median ms per step, [ms per step of every window])"""
        for i in range(warmup):
            fn(i)
        wins, it = [], warmup
        for _ in range(repeats):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn(it)
                it += 1
            e1.record()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            wins.append(float(ms.item()) / steps)
        return statistics.median(wins), wins

    W = max(args.warmup, 3)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # Both timed loops feed the captured step the same way, like a prefetching input pipeline: two captured steps
    # (GraphedTrainStep instances over the same model) own one set of static input buffers each; while step i
    # computes out of slot i%2, the copy stream moves batch i+1 straight into the other slot's static buffers.
    #   value: the rotating batches are already resident in HBM (device -> device copies);
    #   e2e:   they sit in pinned host memory (H2D inside the timed region) and the loss of every step is copied
    #          back to pinned memory on a third stream and read by the host one step later (wrapper.py:73).
    copy_stream = torch.cuda.Stream()
    d2h_stream = torch.cuda.Stream()
    slots = [gs, build(graphed)]
    last_run = {}

    def make_feed(batches, readback):
        staged_ev = [torch.cuda.Event() for _ in range(2)]
        free_ev = [torch.cuda.Event() for _ in range(2)]
        loss_host = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ev = [torch.cuda.Event() for _ in range(2)]
        state = {"primed": False, "seen": 0}

        def enqueue_copy(i):
            b, slot = batches[i % n_rot], i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(free_ev[slot])          # the step that consumed this slot has finished with it
                slots[slot].load(b[0], b[1])                   # batch -> the slot's static device buffers
                staged_ev[slot].record(copy_stream)

        def step(i):
            main = torch.cuda.current_stream()
            if not state["primed"]:
                for ev in free_ev:
                    ev.record(main)
                enqueue_copy(i)
                state["primed"] = True
            slot = i % 2
            main.wait_event(staged_ev[slot])
            loss = slots[slot].run()
            last_run["step"] = slots[slot]
            free_ev[slot].record(main)
            enqueue_copy(i + 1)                                # overlaps with this step's compute
            if readback:
                with torch.cuda.stream(d2h_stream):            # off the compute stream: the next replay does not
                    d2h_stream.wait_event(free_ev[slot])       # queue behind a copy-engine round trip
                    loss_host[slot].copy_(loss.detach(), non_blocking=True)
                    loss_ev[slot].record(d2h_stream)
                if state["seen"] > 0:
                    loss_ev[1 - slot].synchronize()            # host reads the previous step's loss
                    _ = float(loss_host[1 - slot])
            state["seen"] += 1
        return step

    # ---- value: inputs resident in HBM when the timed region starts
    ms_dev, wins_dev = timed(make_feed(devb, False), args.steps, W, args.repeats)
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_run["step"], model)
    # ---- e2e: pinned host buffers -> H2D inside the timed region, loss read back every step
    ms_e2e, wins_e2e = timed(make_feed(host, True), args.steps, W, args.repeats)
    log(f"timing done: {ms_dev:.4f} ms/step device-resident, {ms_e2e:.4f} ms/step e2e")
    clocks = sampler.stop() if rank == 0 else None

    # ---- N > 1: every rank must hold bitwise identical averaged gradients after a step
    grad_identical = None
    if world > 1:
        flat = torch.cat([p.grad.detach().reshape(-1).double() for p in model.parameters() if p.grad is not None])
        chk = torch.stack([flat.sum(), flat.abs().sum()])
        allc = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        grad_identical = all(bool(torch.equal(c, allc[0])) for c in allc)
        assert grad_identical, "averaged gradients differ between ranks"

    # ---- per-kernel durations (CUDA events inside the library, eager launches of the same step)
    eager = GraphedTrainStep(model, devb[0][0], devb[0][1], forward_kwargs=kw, allreduce=False, use_graph=False, warmup=2)
    _lib.call("pcc_launch_count", 1)
    eager.step(devb[1][0], devb[1][1])
    torch.cuda.synchronize()
    launches = int(_lib.call("pcc_launch_count", 1))
    _lib.call("pcc_prof_enable", 1)
    ksteps = min(args.steps, 20)
    for i in range(ksteps):
        eager.step(devb[i % n_rot][0], devb[i % n_rot][1])
    torch.cuda.synchronize()
    _lib.call("pcc_prof_enable", 0)
    kern = {}
    for slot, name in enumerate(PROF_SLOTS):
        ms_tot, cnt = C.c_double(0), C.c_int64(0)
        _lib.call("pcc_prof_read", slot, C.byref(ms_tot), C.byref(cnt))
        if cnt.value:
            kern[name] = ms_tot.value / cnt.value
    barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    pts = wl.points
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):   # dram bytes per launch from the committed `ncu --set full` capture (tools/summarize_profile.py)
        traffic = json.load(open(tpath)).get("kernels", {})
    roof = None
    if wl.kind == "deepsets":
        kd = {k: v for k, v in kern.items() if k in wl.kernel_flop_pt}
        if kd:
            dom = max(kd, key=kd.get)
            ach = wl.kernel_flop_pt[dom] * pts / (kd[dom] * 1e-3) / 1e12
            roof = {"bound": "tensor", "kernel": KERNEL_SYMBOL.get(dom, dom) if wl.name == "deepsets" else dom,
                    "achieved": ach, "peak": peaks["tflops_burst"], "unit": "TFLOP/s", "frac": ach / peaks["tflops_burst"],
                    "frac_of_sustained": ach / peaks["tflops"],
                    "traffic": traffic.get(dom), "traffic_unit": "dram bytes per launch (ncu --set full, profiles/ncu_traffic.json)",
                    "peak_source": peaks["source"] + ": bf16_tflops (burst: the kernel is timed alone with CUDA events)",
                    "kernel_ms": {k: round(v, 4) for k, v in kern.items()},
                    "algorithmic_flop_per_point": wl.kernel_flop_pt[dom]}
    else:
        kd = {k: v for k, v in kern.items() if k.startswith("gnn_")}
        if kd:
            dom = max(kd, key=kd.get)
            table = GRAPH_KERNEL_BYTES_PT(wl)
            nbytes = table.get(dom, (0, 0))[0] * pts
            ach = nbytes / (kd[dom] * 1e-3) / 1e9
            per_kernel = {k: {"ms": round(v, 4), "dram_bytes_per_node": table[k][0], "gathered_l2_bytes_per_node": table[k][1],
                              "hbm_frac": round(table[k][0] * pts / (v * 1e-3) / 1e9 / peaks["hbm"], 3),
                              "l2_gather_GBps": round(table[k][1] * pts / (v * 1e-3) / 1e9, 1)}
                          for k, v in kd.items() if k in table}
            roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": ach / peaks["hbm"], "traffic": traffic.get(dom),
                    "traffic_unit": "dram bytes per launch (ncu --set full, profiles/ncu_traffic.json)",
                    "peak_source": peaks["source"] + ": hbm_gbs",
                    "kernel_ms": {k: round(v, 4) for k, v in kern.items()},
                    "algorithmic_bytes_per_node": table.get(dom, (0, 0))[0],
                    "kernels": per_kernel,
                    "note": "algorithmic bytes = what must cross HBM (every tensor once; ncu's dram bytes agree).  The two gather "
                            "kernels additionally pull k bf16 neighbour rows per node out of L2 (gathered_l2_bytes_per_node, the "
                            "67 MB tensor stays in the 126 MB L2) and are bound by that delivery rate, not by HBM: their HBM "
                            "fraction is low by construction; gnn_conv_bwd_kernel is the streaming, HBM-bound one"}
    step_tf = wl.flop_train_pt * pts / (ms_dev * 1e-3) / 1e12
    extras = {}
    if world == 1 and not args.no_baselines:
        units = None if wl.kind == "deepsets" else 8
        cb = cpu_reference_rate(wl, 8, 1, sample_units=units, budget_s=25.0)
        extras["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        extras["eager_gpu_baseline"] = eager_gpu_baseline(wl, dev)
        extras["e2e_wrapper"] = wrapper_loop_e2e(wl, dev, args.precision)
        if wl.kind == "deepsets" and args.precision == "bf16":   # the fp32-parity mode of the same step (rtol 1e-4 path)
            m32 = wl.build_model(dev, "fp32")
            g32 = GraphedTrainStep(m32, devb[0][0], devb[0][1], forward_kwargs=kw, allreduce=False)
            for _ in range(2):
                g32.run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                g32.run()
            e1.record()
            torch.cuda.synchronize()
            ms32 = e0.elapsed_time(e1) / 5
            extras["fp32_mode"] = {"value": wl.B / ms32 * 1e3, "unit": "samples/s", "ms_per_step": ms32,
                                   "what": "same step with precision='fp32' (3xTF32 mma.sync layer-wise kernels, rtol 1e-4 parity mode)"}
    else:
        extras["cpu_baseline"] = None
    h2d = sum(t.numel() * t.element_size() for t in host[0][0]) + host[0][1].numel() * host[0][1].element_size()
    line = {
        "metric": metric_name(wl), "value": world * wl.B / ms_dev * 1e3,
        "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": W, "ms_per_step": ms_dev,
        "repeats": args.repeats, "windows_ms": [round(w, 5) for w in wins_dev],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": wl.workload_text() +
                   ((" + gradient all-reduce (own one-shot kernel over NVLink peer memory, inside the graph)"
                     if gs.peer is not None else " + NCCL gradient all-reduce") if world > 1 else ""),
                   "name": wl.name, "units_per_gpu": wl.B, "points_per_gpu": pts, "cuda_graph": graphed,
                   "l2": f"inputs rotate over {n_rot} distinct batches per rank and every step streams far more than the "
                         "126 MB L2 through the staged operands / activations",
                   "parallelism": f"dp{world}", "precision_mode": args.precision,
                   "timing": f"median of {args.repeats} windows of {args.steps} steps (CUDA events, max over ranks per window)"},
        "e2e": {"value": world * wl.B / ms_e2e * 1e3, "unit": "samples/s", "ms_per_step": ms_e2e,
                "windows_ms": [round(w, 5) for w in wins_e2e],
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "api": "GraphedTrainStep.load/run, two captured slots fed alternately from pinned host inputs (H2D on a copy "
                       "stream, one step ahead) + per-step loss read-back on a third stream; the device-resident value uses "
                       "the same feed with device-to-device copies"},
        "gpu_launches": launches * args.steps * args.repeats,
        "gpu_launches_per_step": launches,
        "roofline": roof,
        "roofline_step": {"bound": "tensor", "achieved": step_tf, "peak": peaks["tflops"], "unit": "TFLOP/s",
                          "frac": step_tf / peaks["tflops"], "algorithmic_flop_per_point": wl.flop_train_pt,
                          "note": "reference-formulation FLOPs over the whole step against the sustained peak; for max pooling "
                                  "the backward physically runs on the B*H argmax rows only (DESIGN.md section 4), so this "
                                  "overstates tensor-pipe utilisation — `roofline` (forward kernel) is the honest figure"},
        "grad_checksum_identical_on_all_ranks": grad_identical,
        "clocks": clocks,
    }
    line.update(extras)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, step, model):
    """loss, logits and parameter gradients of the last run of `step` -> out_dir/<name>.npy (float32)"""
    import numpy as np
    grads = step.grads if step.grads is not None else {n: p.grad for n, p in model.named_parameters()}
    arrays = {"loss": step.loss, "logits": step.logits}
    arrays.update((f"grad.{n}", g) for n, g in grads.items() if g is not None)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


PROF_SLOTS = ("phi_pool_fwd_kernel", "phi_bwd_chain_kernel", "phi_wgrad_kernel", "gnn_conv_fwd_kernel",
              "gnn_conv_bwd_kernel", "gnn_agg_bwd_kernel", "knn_tiled_kernel", "gnn_fc1_bwd_kernel")
KERNEL_SYMBOL = {"phi_pool_fwd_kernel": "phi_pool_fwd_pair_kernel"}   # H = 256 + max pooling runs the CTA-pair variant


def GRAPH_KERNEL_BYTES_PT(wl):
    """per node: (bytes that must cross HBM, bytes gathered out of L2) of the fused bf16 kernels (DESIGN.md section 4b).
    Activations h and the gradient tensors between the backward kernels are bf16 (2 B / channel), pre-activations fp32."""
    k, Cc = wl.k, wl.hidden
    return {"gnn_conv_fwd_kernel": (Cc * 2 + Cc * 2 + Cc * 4 + k * 4, k * Cc * 2),      # h in (once), agg out, z out, ids | rows
            "gnn_conv_bwd_kernel": (Cc * 2 + Cc * 4 + 2 * Cc * 2 + 2 * Cc * 2, 0),     # dh, z, agg, h in; dagg, droot out
            "gnn_agg_bwd_kernel": (Cc * 2 + 2 * Cc * 2 + Cc * 4 + k * 4, k * Cc * 2),   # dagg (once), droot in / dh out, z1, ids | rows
            "gnn_fc1_bwd_kernel": (Cc * 2 + Cc * 4 + Cc * 2, 0)}                         # h2, z2 in; dh2 out


# ---------------------------------------------------------------------------- configs[4]: point-count sweep
def run_sweep(args, dev, rank, world, log):
    """N = 256 .. 16384 at constant points per GPU and step (B = 262144 / N), DeepSets (relu + max and relu + sum)
    and GraphNet (kNN k=20), CUDA-graph train step; CPU column = oracle port on the host cores on a bounded sample."""
    import torch.distributed as dist
    from pcc_b200.train_step import GraphedTrainStep
    total = 262144
    rows = []
    for model_name in ("deepsets", "deepsets_sum", "graphnet"):
        for N in (256, 512, 1024, 2048, 4096, 8192, 16384):
            B = total // N
            if model_name == "graphnet":
                wl = GraphNetWorkload("graphnet", B, N)
            else:
                wl = DeepSetsWorkload("deepsets", B, N, 3, 10, "relu", "max" if model_name == "deepsets" else "sum", False)
            torch.manual_seed(0)
            model = wl.build_model(dev, args.precision)
            (ins, y), = wl.make_batches(1, seed=7 + rank, pin=False)
            ins, y = tuple(t.to(dev) for t in ins), y.to(dev)
            gs = GraphedTrainStep(model, ins, y, forward_kwargs=wl.forward_kwargs(), allreduce=world > 1)
            for _ in range(3):
                gs.run()
            wins = []
            for _ in range(3):
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    gs.run()
                e1.record()
                torch.cuda.synchronize()
                ms = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
                if world > 1:
                    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
                wins.append(float(ms))
            ms = statistics.median(wins)
            row = {"model": model_name, "N": N, "B_per_gpu": B, "ms_per_step": round(ms, 4),
                   "samples_per_s": world * B / ms * 1e3, "Mpoints_per_s": world * total / ms / 1e3}
            if rank == 0 and world == 1 and not args.no_baselines:
                units = max(2, (32768 if model_name != "graphnet" else 8192) // N)
                cb = cpu_reference_rate(wl, 2, 1, sample_units=min(units, B), budget_s=20.0)
                row["cpu_samples_per_s"] = cb["value"]
                row["cpu_sample"] = cb["sample"]
                row["cpu_cores"] = cb["cores"]
            rows.append(row)
            log(json.dumps(row))
            if gs.peer is not None:
                gs.peer.close()
            del gs, model
            torch.cuda.empty_cache()
    if rank == 0:
        head = next(r for r in rows if r["model"] == "deepsets" and r["N"] == 1024)
        line = {"metric": "train samples/sec (fwd+bwd), point-count sweep N=256..16384 at 262144 points per GPU and step",
                "value": head["samples_per_s"], "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": 3,
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
                "config": {"workload": "configs[4]: point-count scaling sweep, DeepSets (relu+max, relu+sum) and GraphNet (kNN k=20); "
                                       "`value` is the DeepSets relu+max N=1024 row", "name": "sweep", "parallelism": f"dp{world}"},
                "sweep": rows}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=1, help="timed windows of --steps steps; the median is reported")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="deepsets", choices=["deepsets", "yaml", "ragged", "graphnet", "sweep"])
    ap.add_argument("--batch", type=int, default=None, help="sets / graphs per GPU (default 256)")
    ap.add_argument("--points", type=int, default=None, help="points per set / cloud (default 1024)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-baselines", action="store_true", help="skip the CPU / eager-GPU / wrapper-loop comparator legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, logits and gradients of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config == "sweep"):
        ap.error("--dump-outputs needs --impl ours and a single-workload --config")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
