"""bench.py on the GPU: --steps sets the number of timed steps, and --dump-outputs writes a seeded sample of what the last
timed step computed — the same files from run to run, equal to an independent stable sort of the generated input."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS = 300_000


def _bench(workload, steps, out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--rows", str(ROWS),
                        "--steps", str(steps), "--warmup", "1", "--quick", "--no-e2e", "--no-cpu-baseline", "--no-groupby",
                        "--dump-outputs", out_dir], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def _words(path):
    """float64 [k, 2w] of 32-bit halves -> uint64 [k, w]."""
    return np.ascontiguousarray(np.load(path).astype(np.uint32)).view(np.uint64)


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["sort", "pipeline"])
def test_steps_and_dumped_outputs(workload):
    import torch
    with tempfile.TemporaryDirectory() as a, tempfile.TemporaryDirectory() as b:
        one, three = _bench(workload, 1, a), _bench(workload, 3, b)
        assert one["steps"] == 1 and three["steps"] == 3
        assert three["gpu_launches"] == 3 * one["gpu_launches"] > 0
        names = sorted(os.listdir(a))
        assert names == sorted(os.listdir(b))
        assert "sorted_rows.npy" in names and ("groups.npy" in names) == (workload == "pipeline")
        total = 0
        for f in names:
            x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
            assert x.dtype == np.float64 and np.array_equal(x, y), f
            total += x.nbytes
        assert total <= 64 << 20

        import bench
        rows = bench.gen_rows_device(ROWS, torch.device("cuda", 0), 0, workload).view(torch.int64).view(ROWS, 8).cpu().numpy()
        keys = rows[:, 0].view(np.uint64)
        want = rows[np.argsort(keys, kind="stable")].view(np.uint64)
        idx = np.load(os.path.join(a, "sorted_rows_index.npy")).astype(np.int64)
        assert len(idx) == min(ROWS, 1 << 18) and (np.diff(idx) > 0).all()
        assert np.array_equal(_words(os.path.join(a, "sorted_rows.npy")), want[idx])
        if workload == "pipeline":
            uk, inv, cnt = np.unique(keys, return_inverse=True, return_counts=True)
            sums = np.bincount(inv, weights=rows[:, 1].astype(np.float64))
            gidx = np.load(os.path.join(a, "groups_index.npy")).astype(np.int64)
            g = _words(os.path.join(a, "groups.npy")).view(np.int64)
            assert np.array_equal(g[:, 0].view(np.uint64), uk[gidx]) and np.array_equal(g[:, 2], cnt[gidx])
            assert np.array_equal(g[:, 1].astype(np.float64), sums[gidx])
