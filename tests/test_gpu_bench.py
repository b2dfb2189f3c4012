"""bench.py --dump-outputs: what the last timed step computed, written so that two builds can be compared
output for output.  Runs bench.py on a small graph in subprocesses (one JSON line each)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def bench(tmp_path, out, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--nodes", "20000", "--raw-edges", "200000", "--feat", "32", "--no-cpu-baseline", "--no-epoch-metric",
           "--no-ssl-metric", "--cache-dir", str(tmp_path / "cache"), "--dump-outputs", str(tmp_path / out)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps
    d = tmp_path / out
    assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 64_000_000
    return {f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))}


def test_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    a = bench(tmp_path, "a", 2)             # generates and caches the graph
    b = bench(tmp_path, "b", 2)             # same arguments, graph from the cache
    c = bench(tmp_path, "c", 3)             # one more timed step: the dropout stream moves on
    assert {"loss", "get_em_0", "get_em_1"} <= set(a) and any(k.startswith("grad.") for k in a)
    assert set(a) == set(b) == set(c)
    for k, v in a.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), k
        assert v.shape == b[k].shape == c[k].shape, k
        scale = max(float(np.abs(v).max()), 1e-30)
        np.testing.assert_allclose(b[k], v, rtol=1e-4, atol=1e-5 * scale, err_msg=k)
    assert a["get_em_0"].shape[0] == 20000          # the whole graph fits the byte budget at this size
    assert not np.allclose(c["get_em_1"], a["get_em_1"])
    # the dumped embedding and loss belong to the same step: bench's loss is sum(get_em[1] * R), R the seeded
    # loss weights (rows of one 64K-row block of the stream with seed 99 * 1_000_003, D = 64)
    g = torch.Generator().manual_seed(99 * 1_000_003)
    R = torch.randn(65536, 64, generator=g)[:20000].double().numpy()
    for run in (a, b, c):
        terms = run["get_em_1"].astype(np.float64) * R
        assert abs(terms.sum() - float(run["loss"][0])) <= 1e-5 * np.abs(terms).sum()
