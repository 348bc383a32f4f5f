"""bench.py's stdout contract, as far as a machine without a GPU can check it: the result is ONE JSON line on the
process's stdout, whatever libraries write to file descriptor 1 (NCCL's version banner did), and the reference arm
(the oracle port on the host cores) produces the line the driver expects."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_result_line_is_alone_on_stdout():
    code = ("import os, bench\n"
            "bench.claim_stdout()\n"
            "os.write(1, b'NCCL version 0.0.0\\n')\n"      # a library writing to fd 1 behind Python's back
            "print('chatter')\n"
            "bench.emit({'metric': 'm', 'value': 1.5})\n")
    p = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr
    assert json.loads(p.stdout) == {"metric": "m", "value": 1.5}       # exactly one line, and it parses
    assert "NCCL version" in p.stderr and "chatter" in p.stderr


def test_reference_arm_line():
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    p = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0", "--scale", "0.02"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = p.stdout.strip().splitlines()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["higher_is_better"] is True
    assert d["metric"] == "haystack_GB_per_s_scanned_find_matches_as_indexes" and d["unit"] == "GB/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_exact_below_the_limit_and_a_seeded_sample_above(tmp_path):
    import bench
    rng = np.random.default_rng(1)
    m = rng.integers(0, 1 << 32, size=(5000, 4), dtype=np.uint64).astype(np.uint32)   # rows as the scan returns them
    arrays = {"matches": m, "match_offsets": np.arange(1001, dtype=np.int64) * 5, "total": np.array(5000)}
    bench.write_outputs(tmp_path / "a", arrays)
    assert sorted(os.listdir(tmp_path / "a")) == ["match_offsets.npy", "matches.npy", "total.npy"]
    for k, v in arrays.items():
        got = np.load(tmp_path / "a" / f"{k}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, v)
    # above the limit: the large array keeps the same rows on every call, in order; the small ones stay whole; the
    # files stay within the limit
    limit = 100_000
    for d in ("b", "c"):
        bench.write_outputs(tmp_path / d, arrays, limit=limit)
    files = sorted(os.listdir(tmp_path / "b"))
    assert files == ["match_offsets.npy", "matches.npy", "matches_rows.npy", "total.npy"]
    assert sum(os.path.getsize(tmp_path / "b" / f) for f in files) <= limit
    for f in files:
        assert np.array_equal(np.load(tmp_path / "b" / f), np.load(tmp_path / "c" / f))
    rows = np.load(tmp_path / "b" / "matches_rows.npy").astype(np.int64)
    assert len(rows) > 2000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "b" / "matches.npy"), m[rows])
    assert np.array_equal(np.load(tmp_path / "b" / "match_offsets.npy"), arrays["match_offsets"])
    # a later dump below the limit into the same directory leaves no stale row numbers behind
    bench.write_outputs(tmp_path / "b", arrays)
    assert sorted(os.listdir(tmp_path / "b")) == ["match_offsets.npy", "matches.npy", "total.npy"]


def test_steps_below_one_and_dump_on_the_reference_arm_are_refused():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        p = subprocess.run([sys.executable, "bench.py"] + extra, cwd=ROOT, capture_output=True, text=True, timeout=120)
        assert p.returncode == 2 and p.stdout == "", p.stderr


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       cwd=ROOT, capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""
