"""GPU: `bench.py --dump-outputs DIR` writes what the last timed step computed, the same from run to run, and `--steps K` times K
steps in every leg."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "mutag", "--headline-only", "--no-cpu-baseline",
                          "--steps", str(steps), "--warmup", "3", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def test_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    line1, d1 = _bench(tmp_path / "a", 1)
    _, d1_again = _bench(tmp_path / "b", 1)
    line3, d3 = _bench(tmp_path / "c", 3)
    assert line1["steps"] == line1["e2e"]["steps"] == 1 and line3["steps"] == line3["e2e"]["steps"] == 3
    assert {"loss", "output", "grad.fs.wh", "grad.rho.wo", "param.fs.wh", "param.rho.wo"} <= set(d1) and set(d1) == set(d3)
    assert all(a.dtype == np.float32 for a in d1.values()) and sum(a.nbytes for a in d1.values()) <= 64 << 20
    assert d1["output"].shape == (4337, 1) and np.isfinite(d1["loss"])
    y = bench.make_graph_workload(seed=0).y                  # the labels of the timed batch (rank 0)
    for d in (d1, d3):                                       # loss and output come from the same (last timed) forward
        want = torch.nn.functional.binary_cross_entropy_with_logits(torch.from_numpy(d["output"]).double().flatten(), y.double())
        assert abs(float(d["loss"]) - float(want)) < 1e-5 * max(1.0, abs(float(want))), (float(d["loss"]), float(want))
    for k, a in d1.items():                                  # same seeded inputs: the same results up to summation order
        assert a.shape == d1_again[k].shape and np.allclose(a, d1_again[k], rtol=1e-4, atol=1e-6), k
    for k in ("param.fs.wh", "output", "loss"):              # two more timed steps: moved weights, hence another forward
        assert not np.array_equal(d1[k], d3[k]), k
