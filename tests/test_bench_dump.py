"""bench.py --dump-outputs: what the timed commit returned, written as float64 .npy files that compare two builds output for
output.  The dumped root is the golden root of the bench input (tests/golden/bench_roots.json), and every dumped row with its
Merkle path opens against that root."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOG_ROWS = 16  # the smallest size with a golden root
GOLDEN = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_roots.json")))["roots"][f"log_rows={LOG_ROWS},seed=0xB200"]


def bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr


def test_reference_arm_dumps_its_root(tmp_path):
    line = bench("--impl", "reference", "--log-rows", str(LOG_ROWS), "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path))
    root = np.load(tmp_path / "commit_root.npy")
    assert root.dtype == np.float64 and root.tolist() == line["root"] == GOLDEN


@pytest.mark.gpu
def test_dump_is_what_the_last_timed_commit_returned(tmp_path, oracle):
    line = bench("--log-rows", str(LOG_ROWS), "--steps", "2", "--warmup", "1", "--no-prove", "--no-cpu-baseline", "--no-e2e",
                 "--dump-outputs", str(tmp_path))
    assert line["steps"] == 2
    d = {n[:-4]: np.load(tmp_path / n) for n in os.listdir(tmp_path)}
    assert set(d) == {"commit_root", "opened_row_index", "opened_rows", "opening_paths"}
    assert all(a.dtype == np.float64 for a in d.values()) and sum(a.nbytes for a in d.values()) <= 64 << 20
    assert d["commit_root"].tolist() == line["root"] == GOLDEN
    leaves = 2 << LOG_ROWS
    idx = d["opened_row_index"].astype(np.int64)
    assert len(idx) == 2048 and len(set(idx.tolist())) == len(idx) and 0 <= idx.min() and idx.max() < leaves
    assert d["opened_rows"].shape == (len(idx), 256) and d["opening_paths"].shape == (len(idx), LOG_ROWS + 1, 8)
    root = d["commit_root"].astype(np.uint32)
    for i, row, path in zip(idx, d["opened_rows"].astype(np.uint32), d["opening_paths"].astype(np.uint32)):
        assert oracle.verify_batch(root, [(leaves, 256)], int(i), [row], path), i
