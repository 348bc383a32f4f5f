#!/usr/bin/env python
"""bench.py -- haystack GB/s scanned (+ matches/s) for find_matches_as_indexes on the BASELINE.json workloads.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|3|4|5] [--dump-outputs DIR]

--config (default 2, the configuration BASELINE.json's metric is quoted on at one GPU):
  2  benchmarks/names.txt patterns (4 244), Implementation.DFA, 100k x 4 KiB synthetic UTF-8 haystacks, AhoCorasick
     (code point indexes), MatchKind.Standard                                              409.6 MB per GPU and step
  3  10k token patterns, MatchKind.LeftmostLongest, 1M x 256 B log lines, BytesAhoCorasick   256 MB per GPU and step
  4  100k patterns of 5-8 letters, Implementation.ContiguousNFA, ONE 4 GiB haystack, overlapping=True
  5  50k patterns of 5-12 letters, 2M x 4 KiB haystacks = 8 GiB per GPU and step (64 GiB on 8 GPUs), MatchKind.Standard

One "step" = one pass of the hot path over one device-resident batch (always larger than L2).  `value` is
device-resident throughput (CUDA events on the launching stream, max over ranks); `e2e` is the same work through the
public host-buffer API (scan_host: pinned host memory in, host arrays out, H2D/D2H inside the timed region).  After the
timed region the result of one batch is compared with the CPU oracle ("verified").  `--impl reference` times the
reference's CPU path: the Rust crate cannot be built in this image, so that arm runs the C oracle port (oracle/) on all
host cores and says so in cpu_baseline.kind = "port".

`--dump-outputs DIR` writes what the last timed step returned (rank 0's match list, match offsets and total; with several
GPUs also the gathered list) as DIR/<name>.npy in float64.  The inputs are seeded, so two builds run with the same
arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

METRIC = "haystack_GB_per_s_scanned_find_matches_as_indexes"
HAY_BYTES = 4096

CONFIGS = {
    2: dict(name="config2", kind="Standard", overlapping=False, codepoints=True,
            workload="config2: benchmarks/names.txt patterns (4244, Implementation.DFA, MatchKind.Standard), 100k x 4 KiB synthetic UTF-8 "
                     "haystacks, AhoCorasick (code point indexes)"),
    3: dict(name="config3", kind="LeftmostLongest", overlapping=False, codepoints=False,
            workload="config3: 10k token patterns (length 4-16 over [a-z0-9_./:-]), MatchKind.LeftmostLongest, 1M x 256 B log lines, "
                     "BytesAhoCorasick (byte offsets)"),
    4: dict(name="config4", kind="Standard", overlapping=True, codepoints=False,
            workload="config4: 100k patterns (length 5-8 over a-z), Implementation.ContiguousNFA, ONE 4 GiB haystack of uniform a-z, "
                     "overlapping=True, BytesAhoCorasick (64-bit offsets)"),
    5: dict(name="config5", kind="Standard", overlapping=False, codepoints=False,
            workload="config5: 50k patterns (length 5-12 over a-z), MatchKind.Standard, 2M x 4 KiB uniform a-z haystacks = 8 GiB per GPU "
                     "(64 GiB on 8 GPUs), BytesAhoCorasick"),
}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile(prefix="clocks_", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = [float(r[1]) for r in rows]
            out["samples"] = len(rows)
            if sm:
                out["sm_mhz"] = float(np.median(sm))
                out["sm_max_mhz"] = float(rows[0][2])
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for i, nm in enumerate(names):
                    if any("Active" in r[5 + i] and "Not" not in r[5 + i] for r in rows):
                        out["reasons"].append(nm)
            os.unlink(self.path)
        except Exception:
            pass
        return out


def usable_cores() -> int:
    """Host threads this process may really run: the affinity mask, cut down to the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


# ------------------------------------------------------------------------------------------------ host-side samples
def host_sample(cfg: int, n_units: int, rank: int = 0, first: int = 0):
    """A host copy of the config's workload at a bounded size: (patterns as bytes, data u8, offsets i64).
    n_units = haystacks (configs 2, 3, 5) or bytes (config 4)."""
    from ahocorasick_rs_b200 import workloads as W
    if cfg == 2:
        pats, data, offs = W.config2(n_units, HAY_BYTES, first_index=first)
        return [p.encode() for p in pats], data, offs
    if cfg == 3:
        pats, data, offs = W.config3(n_patterns=10_000, n_lines=n_units, seed=3 + rank)
        return pats, data, offs
    if cfg == 4:
        pats, data = W.config4(n_patterns=100_000, hay_bytes=n_units)
        return pats, data, np.array([0, len(data)], dtype=np.int64)
    pats, data, offs = W.config5(n_patterns=50_000, n_haystacks=n_units, hay_bytes=HAY_BYTES, shard=rank)
    return pats, data, offs


def cpu_port(cfg: int, pats, data, offs, steps: int, warmup: int, threads: int):
    """The oracle port (dense DFA, one contiguous shard of haystacks -- or, for one big haystack, one call -- per host
    thread).  -> (GB/s, matches/s, seconds per step)."""
    from oracle import Oracle
    c = CONFIGS[cfg]
    orc = Oracle(pats, c["kind"])
    if len(offs) - 1 < threads:
        # one haystack: cut it into `threads` haystacks that overlap by nothing (a bounded-sample throughput figure,
        # not a result: matches across the cuts are lost, the bytes scanned are the same)
        cuts = np.linspace(offs[0], offs[-1], threads + 1).astype(np.int64)
        offs = cuts
    if warmup:
        orc.time_batch(data, offs, overlapping=c["overlapping"], codepoints=c["codepoints"], nthreads=threads, reps=warmup)
    t0 = time.perf_counter()
    matches = orc.time_batch(data, offs, overlapping=c["overlapping"], codepoints=c["codepoints"], nthreads=threads, reps=steps)
    dt = time.perf_counter() - t0
    return steps * float(offs[-1] - offs[0]) / dt / 1e9, matches / dt, dt / steps


CPU_SAMPLE_UNITS = {2: 100_000, 3: 400_000, 4: 256 << 20, 5: 32_768}   # haystacks (bytes for config 4) per CPU step


def run_reference(args, rank):
    """--impl reference: the reference's CPU path (oracle port), rank 0 only."""
    if rank != 0:
        return
    cfg = args.config
    pats, data, offs = host_sample(cfg, CPU_SAMPLE_UNITS[cfg])
    threads = usable_cores()
    gbs, mps, sec = cpu_port(cfg, pats, data, offs, steps=args.steps, warmup=max(args.warmup, 1), threads=threads)
    sample = (f"each step = {(offs[-1] - offs[0]) / 1e6:.1f} MB of the {CONFIGS[cfg]['name']} workload ({len(offs) - 1} haystacks), "
              f"{threads} host threads, one contiguous shard per thread, all steps inside one thread launch")
    line = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": CONFIGS[cfg]["workload"],
                   "reference_arm": "C oracle port of the reference's CPU path (Rust aho-corasick 1.1.4 cannot be built here: no rustc/cargo)"},
        "matches_per_s": mps,
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def make_dense(pats, data, offs, seed=7):
    """The dense-match variant: pattern number (j mod n) written at every 64th byte of every haystack, where that
    overwrites ASCII bytes only (keeps the text valid UTF-8) and fits inside the haystack."""
    data = data.copy()
    lens = np.array([len(p) for p in pats])
    maxlen = int(lens.max())
    blob = np.zeros((len(pats), maxlen), dtype=np.uint8)
    for i, p in enumerate(pats):
        blob[i, : len(p)] = np.frombuffer(p, dtype=np.uint8)
    n = len(offs) - 1
    hay_len = int(offs[1] - offs[0])
    assert np.all(np.diff(offs) == hay_len), "dense variant: equal-length haystacks"
    rows = data.reshape(n, hay_len)
    j = 0
    for at in range(32, hay_len - maxlen, 64):
        pid = (np.arange(n) + j) % len(pats)
        ok = (rows[:, at:at + maxlen] < 0x80).all(axis=1) & (rows[:, at - 1] < 0x80) & (rows[:, at + maxlen] < 0x80) if at + maxlen < hay_len else np.zeros(n, bool)
        for ln in np.unique(lens):
            sel = ok & (lens[pid] == ln)
            if sel.any():
                rows[sel, at:at + ln] = blob[pid[sel], :ln]
        j += 1
    return data


# ------------------------------------------------------------------------------------------------ device workloads
def device_random_lowercase(torch, dev, n_bytes: int, seed: int):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    out = torch.empty(n_bytes, dtype=torch.uint8, device=dev)
    step = 1 << 28
    for a in range(0, n_bytes, step):
        b = min(a + step, n_bytes)
        out[a:b] = torch.randint(97, 123, (b - a,), dtype=torch.uint8, device=dev, generator=g)
    return out


_RESULT_OUT = None   # the process's real stdout, once claim_stdout() has pointed fd 1 at stderr


def claim_stdout():
    """stdout carries ONE JSON line.  Libraries write to fd 1 behind Python's back (NCCL prints "NCCL version ..." there
    at every debug level but NONE), so fd 1 is pointed at stderr for the whole run and the result line goes to a
    duplicate of the original descriptor."""
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _RESULT_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_BYTES = 64_000_000   # --dump-outputs writes at most this much, .npy headers included


def write_outputs(out_dir, arrays, limit=DUMP_BYTES, seed=0):
    """--dump-outputs: each array as out_dir/<name>.npy in float64 (the values are integers below 2^53, so exact).
    Smallest first, each array gets an equal share of the `limit` bytes not yet written; one larger than its share
    keeps a sample of its rows, drawn with a fixed seed and kept in order, and out_dir/<name>_rows.npy holds the
    numbers of the rows kept.  Two builds that computed the same lists write the same files."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    room = limit - 512 * len(arrays)   # (.npy headers)
    for i, name in enumerate(sorted(arrays, key=lambda k: (arrays[k].size, k))):
        a = arrays[name]
        share = room // (len(arrays) - i)
        rows_path = os.path.join(out_dir, name + "_rows.npy")
        if a.size * 8 > share and a.ndim:
            keep = share // (8 * (a.size // a.shape[0] + 1))   # a kept row costs its values and its row number
            rows = np.sort(np.random.default_rng(seed).choice(a.shape[0], size=keep, replace=False))
            a = a[rows]
            np.save(rows_path, rows.astype(np.float64))
            room -= 8 * keep
        elif os.path.exists(rows_path):
            os.remove(rows_path)   # left by an earlier, sampled dump into the same directory
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))
        room -= 8 * a.size


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--dense", action="store_true", help="configs 2 and 3: the dense-match variant (a pattern written every 64 bytes: ~1 match per 64 B), "
                                                           "to expose the output path (SURVEY.md 8d)")
    ap.add_argument("--scale", type=float, default=1.0, help=argparse.SUPPRESS)       # shrink the workload (development only)
    ap.add_argument("--haystacks", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--no-cpu-baseline", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-verify", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--segment-bytes", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--kernel", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--hot-rows", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--table", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results (match list, per-haystack match "
                                                           "offsets, total; on rank 0, and the gathered list with several GPUs) "
                                                           "as DIR/<name>.npy in float64, at most 64 MB in all (a seeded sample of rows beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm counts matches, it keeps no match list")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    claim_stdout()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist

    from ahocorasick_rs_b200 import AhoCorasick, BytesAhoCorasick, Implementation, MatchKind, _capi
    from ahocorasick_rs_b200.sharding import MatchListGather, decode_gathered, gather_match_lists

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    L = _capi.lib()
    if args.segment_bytes or args.hot_rows or args.table or args.kernel:
        _capi.set_tuning(args.kernel, args.hot_rows, args.segment_bytes, args.table)
    cfg = args.config
    C = CONFIGS[cfg]
    ovl, cp = C["overlapping"], C["codepoints"]
    kind = MatchKind[C["kind"]]

    # ---- the workload on this rank (weak scaling: every rank its own batch of the full per-GPU size) ----------------
    host_batches = []   # host copies (configs 2, 3): for the end-to-end leg and the oracle check
    if cfg == 2:
        n_hay = args.haystacks or int(100_000 * args.scale)
        for b in range(2):  # two different batches alternate
            pats, data, offs = host_sample(2, n_hay, first=(rank * 2 + b) * n_hay)
            if args.dense:
                data = make_dense(pats, data, offs)
            host_batches.append((data, offs))
        ac = AhoCorasick([p.decode() for p in pats], implementation=Implementation.DFA)
        d_batches = [(torch.from_numpy(d).to(dev), torch.from_numpy(o).to(dev)) for d, o in host_batches]
    elif cfg == 3:
        n_hay = args.haystacks or int(1_000_000 * args.scale)
        pats, data, offs = host_sample(3, n_hay, rank=rank)
        if args.dense:
            data = make_dense(pats, data, offs)
        host_batches.append((data, offs))
        ac = BytesAhoCorasick(pats, kind)
        d_batches = [(torch.from_numpy(data).to(dev), torch.from_numpy(offs).to(dev))]
    elif cfg == 4:
        from ahocorasick_rs_b200 import workloads as W
        n_hay = 1
        n_bytes = int((1 << 32) * args.scale)
        pats = W.random_lowercase_patterns(100_000, 5, 8, 4)
        ac = BytesAhoCorasick(pats, kind, implementation=Implementation.ContiguousNFA)
        d = device_random_lowercase(torch, dev, n_bytes, 1004 + rank)
        d_batches = [(d, torch.tensor([0, n_bytes], dtype=torch.int64, device=dev))]
    else:
        from ahocorasick_rs_b200 import workloads as W
        n_hay = args.haystacks or int((1 << 21) * args.scale)
        pats = W.random_lowercase_patterns(50_000, 5, 12, 5)
        ac = BytesAhoCorasick(pats, kind)
        d = device_random_lowercase(torch, dev, n_hay * HAY_BYTES, 1005 + rank)
        d_batches = [(d, torch.arange(n_hay + 1, dtype=torch.int64, device=dev) * HAY_BYTES)]
    bytes_per_step = int(d_batches[0][0].numel())
    big = bytes_per_step > ac._ac.WINDOW_BYTES   # scanned as several calls by the host layer (32-bit offsets per call)

    # capacities from one synchronous scan per batch
    results0 = []
    for b, (d, o) in enumerate(d_batches):
        m, mo, total = ac.scan_device(d, o, ovl)
        results0.append((m.clone() if b == 0 else None, mo.clone() if b == 0 else None, int(total)))
    totals = [r[2] for r in results0]
    cap = max(1 << 16, int(max(totals) * 1.25) + 1024)
    scan_stats = dict(ac._ac.last_stats)

    SLOTS = 4   # workspaces / exchanges in flight (multi-GPU: the gather of step i overlaps the scans of steps i+1 .. i+3)

    def step(i):
        d, o = d_batches[i % len(d_batches)]
        if big:
            return ac.scan_device(d, o, ovl)                         # windows / runs of whole haystacks, synchronous
        return ac.scan_device(d, o, ovl, capacity=cap, sync=False, ws_slot=i % SLOTS)

    # ---- device-resident throughput ------------------------------------------------
    for i in range(max(args.warmup, SLOTS)):   # (every workspace slot is allocated and has run before the timed region)
        step(i)
    torch.cuda.synchronize()
    gather = None
    if world > 1 and not big:
        gather_cap = max(4096, -(-2 * max(totals) // 4096) * 4096)  # rows per rank in the match-list gather
        gather = MatchListGather(gather_cap, dev, slots=SLOTS)
        for i in range(max(args.warmup, 10)):  # warm the exchange too (communicator set-up, buffers)
            o_, _, t_ = step(i)
            gather(o_, t_, (rank * 2 + (i & 1)) * n_hay, slot=i % SLOTS)
        gather.finish()
    def big_gather(out):
        rows = out.to(torch.int32) if (out.dtype != torch.int32 and bytes_per_step // max(n_hay, 1) < (1 << 31) and n_hay * world < (1 << 31)) else out
        return gather_match_lists(rows, rank * n_hay)   # exact sizes, two collectives (the lists are tens of MB here)

    if world > 1 and big:
        for i in range(max(args.warmup, 3)):   # warm the exchange too: communicator set-up, the kept buffers, the allocator's blocks
            gathered = big_gather(step(i)[0])
        gathered = None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    L.acb_timing_enable(1)
    launches0 = L.acb_launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    host_t0 = time.perf_counter()
    gathered = None
    for i in range(args.steps):
        out, moffs, tot = step(i)
        if world > 1:
            # the only exchange of the path: gather the per-shard match lists
            if gather is not None:
                gathered = gather(out, tot, (rank * 2 + (i & 1)) * n_hay, slot=i % SLOTS)   # fixed-size blocks, side stream, no host round trip
            else:
                gathered = big_gather(out)
    if gather is not None:
        gather.finish()  # the exchanges ran on a side stream: the timed region ends when the last one has
    ev1.record()
    host_enqueue_ms = (time.perf_counter() - host_t0) * 1e3 / max(args.steps, 1)
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        # now, before a later scan reuses the last step's workspace slot
        if big:
            matches, total = out, tot
        else:
            status = tot.tolist()   # sync=False: the device status, read as scan_device reads it when it synchronises
            total = status[0]
            assert status[1] or total == status[4] == 0, "the last timed step's match list did not fit its capacity"
            matches = out[:total]
        dump = {"matches": matches, "match_offsets": moffs, "total": np.array(total)}
        if world > 1:
            dump["gathered_matches"] = decode_gathered(gathered) if gather is not None else gathered
        for k, v in dump.items():
            if isinstance(v, torch.Tensor):
                v = v.cpu().numpy()
                dump[k] = v.view(np.uint32) if v.dtype == np.int32 else v
        write_outputs(args.dump_outputs, dump)
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    launches = int(L.acb_launch_count() - launches0)
    kms, kn = ctypes.c_double(0), ctypes.c_uint64(0)
    L.acb_timing_read(ctypes.byref(kms), ctypes.byref(kn))
    L.acb_timing_enable(0)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    matches_per_step = sum(totals) / len(totals)

    # ---- what was timed is what the reference computes: compare with the oracle -------------------------
    verified = None
    if not args.no_verify:
        from oracle import Oracle
        threads = usable_cores()
        orc = Oracle(pats if cfg != 2 else [p.encode() if isinstance(p, str) else p for p in pats], C["kind"])
        m0, mo0, t0 = results0[0]
        if cfg in (2, 3):
            data, offs = host_batches[0]
            et, ecounts, erec = orc.scan_batch(data, offs, overlapping=ovl, codepoints=cp)
            got = m0.cpu().numpy().view(np.uint32)
            assert t0 == et and np.array_equal(got, erec), "GPU result differs from the oracle"
            assert np.array_equal(np.diff(mo0.cpu().numpy()), ecounts.astype(np.int64))
            verified = {"against": "oracle, one whole batch", "bytes": int(offs[-1]), "matches": int(et)}
            if gathered is not None and gather is not None:
                # the last step's gathered lists, decoded after the timed region: rank r's block must be rank r's result
                glob = decode_gathered(gathered)
                last = (args.steps - 1) & 1
                mine = glob[glob[:, 0] >= (rank * 2 + last) * n_hay][: totals[last]].cpu().numpy().view(np.uint32).copy()
                mine[:, 0] -= (rank * 2 + last) * n_hay
                exp = got if last == 0 else orc.scan_batch(*host_batches[1], overlapping=ovl, codepoints=cp)[2]
                assert np.array_equal(mine, exp), "gathered match list differs from the oracle"
                verified["gathered"] = "rank-0 block of the last step's NCCL gather equals the oracle's list"
        else:
            d, o = d_batches[0]
            got = m0.cpu().numpy().astype(np.int64) if m0.dtype != torch.int32 else m0.cpu().numpy().view(np.uint32).astype(np.int64)
            checked = 0
            if cfg == 4:
                spans = [(0, min(96 << 20, bytes_per_step))]
                cut = ac._ac.WINDOW_BYTES - max(ac._ac.max_pattern_len - 1, 0)
                if bytes_per_step > cut + (16 << 20):
                    spans.append((cut - (16 << 20), cut + (16 << 20)))   # across the host layer's window cut
                for a, b in spans:
                    sl = d[a:b].cpu().numpy()
                    et, _, erec = orc.scan_batch(sl, np.array([0, b - a], dtype=np.int64), overlapping=True)
                    sel = got[(got[:, 2] >= a) & (got[:, 3] <= b)]
                    exp = erec.astype(np.int64)
                    exp[:, 2] += a
                    exp[:, 3] += a
                    assert np.array_equal(sel, exp), f"GPU result differs from the oracle in bytes [{a}, {b})"
                    checked += int(et)
                verified = {"against": "oracle, byte ranges " + ", ".join(f"[{a}, {b})" for a, b in spans), "matches": checked}
            else:
                nh = min(n_hay, 32_768)
                sl = d[: nh * HAY_BYTES].cpu().numpy()
                oo = np.arange(nh + 1, dtype=np.int64) * HAY_BYTES
                et, ecounts, erec = orc.scan_batch(sl, oo, overlapping=False)
                sel = got[got[:, 0] < nh]
                assert np.array_equal(sel, erec.astype(np.int64)), "GPU result differs from the oracle"
                assert np.array_equal(np.diff(mo0.cpu().numpy())[:nh], ecounts.astype(np.int64))
                verified = {"against": f"oracle, first {nh} haystacks", "bytes": nh * HAY_BYTES, "matches": int(et)}

    # ---- end to end through the public host API (rank-local): pinned host memory in, host arrays out ---------------
    if cfg in (2, 3):
        e2e_in = [(torch.from_numpy(d).pin_memory(), o) for d, o in host_batches]
    else:
        nb = min(bytes_per_step, 1 << 30)
        nb -= nb % HAY_BYTES
        hbuf = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
        hbuf.copy_(d_batches[0][0][:nb])
        e2e_in = [(hbuf, np.array([0, nb], dtype=np.int64) if cfg == 4 else np.arange(nb // HAY_BYTES + 1, dtype=np.int64) * HAY_BYTES)]
    e2e_bytes = int(e2e_in[0][0].numel())

    def e2e_step(i):
        hd, ho = e2e_in[i % len(e2e_in)]
        return ac.scan_host(hd, ho, ovl)     # H2D (pipelined), scan, D2H of the match list

    e2e_steps = max(3, min(args.steps, 10))
    for i in range(2):
        e2e_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    d2h = 0
    for i in range(e2e_steps):
        m, mo = e2e_step(i)
        d2h += m.nbytes + mo.nbytes
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    total_bytes = bytes_per_step * args.steps * world
    value = total_bytes / (ms_max * 1e-3) / 1e9
    # algorithmic bytes of the scan kernel(s) of one step: haystack bytes + int64 offsets + 16 B per match (24 B with 64-bit offsets)
    rec_bytes = 24 if cfg == 4 else 16
    alg_bytes = bytes_per_step + 8 * (n_hay + 1) + rec_bytes * matches_per_step
    k_ms = kms.value / max(args.steps, 1)      # scan kernel time per step (a step above 2 GiB is several launches)
    lps = max(kn.value / max(args.steps, 1), 1.0)   # scan kernel launches per step
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    engine = scan_stats.get("engine")
    kernel_name = "sieve_scan_kernel" if engine == "sieve" else ("scan_global_kernel" if scan_stats.get("global_table") else "scan_staged_kernel")
    traffic, traffic_src = None, None
    tj = os.path.join(ROOT, "profiles", f"r02_{C['name']}_scan_kernel.json")
    if os.path.exists(tj) and args.scale == 1.0 and not args.haystacks:
        with open(tj) as f:
            tjv = json.load(f)
        if tjv.get("kernel") == kernel_name:
            traffic, traffic_src = tjv["dram_traffic_bytes_per_launch"], f"profiles/r02_{C['name']}_scan_kernel.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum)"
    line = {
        "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": C["workload"] + (" -- DENSE variant: a pattern written every 64 bytes" if args.dense else ""), "haystacks_per_gpu": n_hay, "bytes_per_gpu_per_step": bytes_per_step,
                   "l2": f"inputs ({bytes_per_step / 1e6:.1f} MB per batch{', two batches alternating' if len(d_batches) > 1 else ''}) are larger than L2; no flush needed",
                   "multi_gpu": "one process per GPU, batch sharded by haystack index, tables replicated; per step one gather of the match lists (NCCL)"},
        "matches_per_s": matches_per_step * args.steps * world / (ms_max * 1e-3),
        "matches_per_step_per_gpu": matches_per_step,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel": kernel_name,
                     "kernel_ms": k_ms / lps, "kernel_ms_per_step": k_ms, "kernel_launches_per_step": lps,
                     "algorithmic_bytes_per_launch": alg_bytes / lps},
        "e2e": {"value": e2e_bytes * e2e_steps * world / e2e_s / 1e9, "unit": "GB/s",
                "h2d_bytes_per_step": e2e_bytes + 8 * (len(e2e_in[0][1])), "d2h_bytes_per_step": d2h // e2e_steps,
                "steps": e2e_steps, "bytes_per_step": e2e_bytes,
                "api": "scan_host: pinned host bytes in (chunked H2D overlapped with the scan), host numpy arrays out"},
        "gpu_launches": launches,
        "scan_stats": scan_stats,
        "verified": verified,
        "host_enqueue_ms_per_step": host_enqueue_ms,
        "clocks": clocks,
    }
    if not args.no_cpu_baseline:
        units = CPU_SAMPLE_UNITS[cfg]
        if cfg in (2, 3) and units >= n_hay:
            spats, sdata, soffs = (pats if cfg != 2 else [p.encode() if isinstance(p, str) else p for p in pats]), host_batches[0][0], host_batches[0][1]
        else:
            spats, sdata, soffs = host_sample(cfg, units)
        threads = usable_cores()
        _, _, one = cpu_port(cfg, spats, sdata, soffs, steps=1, warmup=1, threads=threads)
        reps = int(max(1, min(2000, 12.0 / max(one, 1e-4))))
        gbs, mps, _ = cpu_port(cfg, spats, sdata, soffs, steps=reps, warmup=0, threads=threads)
        line["cpu_baseline"] = {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "port", "matches_per_s": mps,
                                "sample": f"{(soffs[-1] - soffs[0]) / 1e6:.1f} MB of the same workload ({len(soffs) - 1} haystacks) x {reps} passes inside one thread launch, "
                                          f"{threads} threads, one contiguous shard per thread"}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
