"""bench.py end to end at a small size: it times exactly --steps steps and --dump-outputs writes what the timed path
returned, which must be the oracle's forward on the same seeded inputs and weights."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from distegnn_b200 import synth
from oracle import fastegnn_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_bench_steps_and_dumped_outputs(tmp_path):
    n, steps = 20_000, 2
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--nodes", str(n), "--steps", str(steps), "--warmup", "1",
           "--no-cpu-baseline", "--no-e2e", "--no-train", "--dump-outputs", str(tmp_path)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["value"] > 0
    assert sorted(os.listdir(tmp_path)) == ["node_loc.npy", "virtual_loc.npy"]
    out, X = np.load(tmp_path / "node_loc.npy"), np.load(tmp_path / "virtual_loc.npy")
    assert out.dtype == np.float32 and X.dtype == np.float32

    w = synth.WORKLOADS["synth1m"]
    host = synth.make_partitions(w, n_nodes=n, seed=0)[0]
    with torch.no_grad():
        ref, refX = orc.forward(bench.make_state_dict(w), **host, normalize=w.normalize)
    assert out.shape == tuple(ref.shape) and X.shape == tuple(refX.shape)
    err = float(np.abs(out - ref.numpy()).max())
    disp = float((ref - host["node_loc"]).abs().max())
    assert err <= 1e-5 * max(1.0, float(ref.abs().max())) and err <= 1e-4 * disp, (err, disp)
    assert float(np.abs(X - refX.numpy()).max()) <= 1e-5 * max(1.0, float(refX.abs().max()))
