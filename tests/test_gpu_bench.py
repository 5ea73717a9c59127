"""GPU: bench.py runs exactly --steps timed steps and --dump-outputs writes what the last one computed."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _targets(workload, n):
    """The label matrix bench.py trains on (both workloads are seeded)."""
    sys.path.insert(0, ROOT)
    from chromegcn_b200 import synthetic
    if workload == "c1":
        return synthetic.make_features("chr22", n, 128, 103)["target"].numpy()
    gen = torch.Generator().manual_seed(100)               # rank 0's rows, drawn in bench.run_stress's order
    torch.randn(n, 128, generator=gen), torch.randn(n, 128, generator=gen)
    return (torch.rand(n, 103, generator=gen) < 0.05).float().numpy()


@pytest.mark.parametrize("workload,graph,extra", [("c1", "chr22", []), ("st", "st", ["--st-rows", "20000", "--st-pairs", "100000"])])
@pytest.mark.parametrize("steps", [1, 2])
def test_dump_outputs_of_the_last_step(tmp_path, workload, graph, extra, steps):
    out_dir = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", str(steps), "--warmup", "3",
                        "--no-cpu-baseline", "--no-gpu-baseline", "--no-e2e", "--no-roofline", "--dump-outputs", str(out_dir)] + extra,
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps
    files = {os.path.basename(p)[:-4]: np.load(p) for p in glob.glob(str(out_dir / "*.npy"))}
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert sum(os.path.getsize(p) for p in glob.glob(str(out_dir / "*.npy"))) <= 64 << 20
    probs = files["probs." + graph].astype(np.float64)
    assert probs.shape == (20000, 103) and np.all((probs >= 0) & (probs <= 1))       # graphs this small are written whole
    # the dumped loss is the last step's own BCE over these probabilities, not a sum over the warm-up and timed passes
    t = _targets(workload, probs.shape[0])
    p = np.clip(probs, 1e-7, 1 - 1e-7)
    bce = float(-(t * np.log(p) + (1 - t) * np.log(1 - p)).mean())
    loss = files["loss." + graph]
    assert loss.shape == (1,) and abs(float(loss[0]) - bce) <= 1e-3 * bce, (float(loss[0]), bce)
    assert files["model.GC1.weight"].shape == (128, 128) and files["model.out.weight"].shape == (103, 128)
    # num_batches_tracked counts every train-mode forward: 2 strands x (3 warm-up + the timed) steps
    assert files["model.batch_norm.num_batches_tracked"] == 2 * (3 + steps)
