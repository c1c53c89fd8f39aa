"""GPU: `bench.py --dump-outputs` writes what its last timed step computed.  The test regenerates that step's seeded
batch and the seeded initial parameters, runs the same train step eagerly on the drop-in module and compares loss,
logits and every parameter gradient with the dumped arrays."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


@pytest.mark.timeout(600)
def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    # N > H so that max pooling takes the argmax-row backward of the headline configuration
    B, N, steps, warmup = 8, 512, 3, 3
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
           "--batch", str(B), "--points", str(N), "--no-baselines", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=540, cwd=tmp_path)
    assert r.returncode == 0, r.stdout[-2000:] + "\n" + r.stderr[-3000:]

    import bench
    wl = bench.make_workload("deepsets", B, N)
    torch.manual_seed(0)
    model = wl.build_model("cuda", "bf16")
    # the timed steps follow `warmup` untimed ones, step i consumes rotating batch i (rank 0 seeds its batches with 1000)
    (x, idx), y = wl.make_batches(bench.N_ROTATE, seed=1000, pin=False)[warmup + steps - 1]
    logits = model(x.cuda(), idx.cuda(), **wl.forward_kwargs())
    loss = torch.nn.BCEWithLogitsLoss()(logits, y.cuda())
    loss.backward()
    torch.cuda.synchronize()

    names = [n for n, _ in model.named_parameters()]
    assert sorted(os.listdir(out)) == sorted(["loss.npy", "logits.npy"] + [f"grad.{n}.npy" for n in names])
    dumped = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype == np.float32 for a in dumped.values())
    assert abs(float(dumped["loss"]) - float(loss)) < 1e-5 * abs(float(loss))
    torch.testing.assert_close(torch.from_numpy(dumped["logits"]), logits.detach().cpu(), rtol=1e-4, atol=1e-5)
    for n, p in model.named_parameters():
        assert dumped[f"grad.{n}"].shape == tuple(p.shape), n
        assert rel_l2(torch.from_numpy(dumped[f"grad.{n}"]), p.grad) < 1e-3, n
