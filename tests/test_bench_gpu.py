"""bench.py on the GPU (-m gpu): --dump-outputs writes what the last timed step returned, and that is the oracle's
answer for the batch that step scanned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from ahocorasick_rs_b200 import workloads as W
from oracle import Oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_last_timed_steps_result(tmp_path):
    n, steps = 3000, 4   # config 2 alternates two batches: step 3, the last, scans batch 1 (haystacks n .. 2n - 1)
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
    p = subprocess.run([sys.executable, "bench.py", "--steps", str(steps), "--warmup", "3", "--haystacks", str(n), "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=900, env=env)
    assert p.returncode == 0, p.stderr[-3000:]
    assert json.loads(p.stdout)["steps"] == steps
    pats, data, offs = W.config2(n, first_index=n)
    total, counts, rec = Oracle([q.encode() for q in pats], "Standard").scan_batch(data, offs, codepoints=True)
    assert sorted(os.listdir(tmp_path)) == ["match_offsets.npy", "matches.npy", "total.npy"]
    got = {k: np.load(tmp_path / f"{k}.npy") for k in ("matches", "match_offsets", "total")}
    assert all(v.dtype == np.float64 for v in got.values())
    assert total > 0 and int(got["total"]) == total
    assert np.array_equal(got["matches"], rec)
    assert np.array_equal(got["match_offsets"], np.concatenate([[0], np.cumsum(counts, dtype=np.int64)]))
