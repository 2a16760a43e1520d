"""bench.py --dump-outputs: what the timed path computed in its last step, written so that two builds run with the same
arguments can be compared output for output."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.conftest import ROOT


def _bench(monkeypatch):
    # bench.py sets this on import (setdefault); setting it first makes that a no-op, and the test's end restores it
    monkeypatch.setenv("CUDA_DEVICE_MAX_CONNECTIONS", os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS", "32"))
    spec = importlib.util.spec_from_file_location("bench_main", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_dump_outputs_layout_and_sample(tmp_path, monkeypatch):
    bm = _bench(monkeypatch)
    B, R = 8, 3
    u0 = [torch.arange(2 * B, dtype=torch.float64).reshape(2, B) + 100 * q for q in range(R)]
    st = [torch.full((B,), q, dtype=torch.int32) for q in range(R)]
    bm.dump_outputs(str(tmp_path / "all"), [0, 2], B, dict(u0=u0, status=st))
    p = np.load(tmp_path / "all" / "problem.npy"); u = np.load(tmp_path / "all" / "u0.npy"); s = np.load(tmp_path / "all" / "status.npy")
    assert p.dtype == u.dtype == s.dtype == np.float64
    np.testing.assert_array_equal(p, np.r_[0:B, 2 * B:3 * B])
    np.testing.assert_array_equal(u, np.concatenate([u0[0].numpy(), u0[2].numpy()], axis=1))
    np.testing.assert_array_equal(s, np.r_[np.zeros(B), np.full(B, 2.0)])
    # above the cap: the same seeded sample of columns every time, taken from every array alike
    monkeypatch.setattr(bm, "DUMP_MAX_PROBLEMS", 5)
    for d in ("a", "b"):
        bm.dump_outputs(str(tmp_path / d), [0, 1, 2], B, dict(u0=u0, status=st))
    pa = np.load(tmp_path / "a" / "problem.npy"); ua = np.load(tmp_path / "a" / "u0.npy")
    assert pa.shape == (5,) and ua.shape == (2, 5) and np.all(np.diff(pa) > 0)
    np.testing.assert_array_equal(pa, np.load(tmp_path / "b" / "problem.npy"))
    q, i = (pa // B).astype(int), (pa % B).astype(int)
    np.testing.assert_array_equal(ua, np.stack([u0[a][:, b].numpy() for a, b in zip(q, i)], axis=1))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "status.npy"), q.astype(np.float64))


@pytest.mark.gpu
def test_bench_dump_is_reproducible_and_steps_are_timed(tmp_path):
    """Two runs with the same inputs but a different number of timed steps and streams dump the same results, and the
    timed region launches in proportion to --steps.  (--max-ctas is fixed: by default it follows the stream count, and
    with fewer CTAs than the batch needs every solve also launches the queue-order kernel.)"""
    base = [sys.executable, os.path.join(ROOT, "bench.py"), "--batch", "512", "--sets", "4", "--batches-per-step", "8",
            "--max-ctas", "16", "--warmup", "3", "--no-extras", "--no-cpu-baseline", "--e2e-inflight", "4"]
    lines, dumps = [], []
    for k, (steps, streams) in enumerate(((1, 2), (2, 8))):
        d = tmp_path / str(k)
        r = subprocess.run(base + ["--steps", str(steps), "--streams", str(streams), "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        lines.append(json.loads(r.stdout.strip().splitlines()[-1]))
        dumps.append({f[:-4]: np.load(d / f) for f in os.listdir(d)})
    assert [ln["steps"] for ln in lines] == [1, 2]
    assert lines[0]["gpu_launches"] > 0 and lines[1]["gpu_launches"] == 2 * lines[0]["gpu_launches"]
    a, b = dumps
    assert sorted(a) == ["coeffs", "iters", "kkt", "obj", "pred", "problem", "state", "status", "u0"]
    assert a["problem"].shape == (4 * 512,) and a["u0"].shape == (2, 4 * 512) and a["pred"].shape == (60, 4 * 512)
    assert (a["status"] == 1).mean() >= 0.99
    for name in a:
        assert a[name].dtype == np.float64
        np.testing.assert_array_equal(a[name], b[name], err_msg=name)
