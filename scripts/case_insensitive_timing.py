"""Cost of ASCII case-insensitive matching, device-resident, at the BASELINE sizes of configs 2, 3 and 5.

For every config the case-sensitive and the case-insensitive automaton scan the SAME data (config 2: the text with half
of its letters re-cased; configs 3 and 5: as generated, plus the same re-casing), alternately, with each engine the
auto choice can take (the table walker where the profile picks it, and the sieve).  On re-cased text the
case-sensitive automaton finds far fewer matches, so a third variant isolates the fold: the case-sensitive automaton of
the folded patterns on the folded text does exactly the case-insensitive scan's work without folding.  Per variant: kernel time (the
library's CUDA events around the scan kernel), step time (CUDA events around whole scan_device calls), GB/s over the
step, and the match count.  Every case-insensitive result is checked against the oracle on the folded inputs (config 5:
on its first 65 536 haystacks, and whole against the case-sensitive scan of the folded text).

    python scripts/case_insensitive_timing.py [--steps N] [--rounds R] [--only 2,3,5]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from ahocorasick_rs_b200 import AhoCorasick, BytesAhoCorasick, Implementation, MatchKind, _capi, workloads as W
from oracle import Oracle


def fold_np(a):
    return np.where((a >= 0x41) & (a <= 0x5A), a | 0x20, a).astype(np.uint8)


def ascii_lower(p: str) -> str:
    return "".join(c.lower() if "A" <= c <= "Z" else c for c in p)  # (str.lower would also lower non-ASCII letters)


def fold_dev(t):
    return torch.where((t >= 0x41) & (t <= 0x5A), t | 0x20, t)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # (the numbers are still printed; the card's limits are then unknown)
        q = f"unknown ({e})"
    return f"{name}, power limit / max SM clock: {q}"


def time_variant(ac, d, o, engine, steps, cap):
    """-> (kernel ms per step, step ms, total matches).  Buffers above one call's 2 GiB are scanned in runs of whole
    haystacks by the host layer, synchronously (as bench.py does): the kernel time is then the sum over the runs."""
    big = d.numel() > ac._ac.WINDOW_BYTES
    _capi.set_tuning(5 if engine == "sieve" else 0)
    try:
        L = _capi.lib()

        def step(i):
            if big:
                return ac.scan_device(d, o)
            return ac.scan_device(d, o, capacity=cap, sync=False, ws_slot=i % 2)

        for i in range(3):
            step(i)
        torch.cuda.synchronize()
        L.acb_timing_enable(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            _, _, tot = step(i)
        e1.record()
        torch.cuda.synchronize()
        kms, kn = C.c_double(0), C.c_uint64(0)
        L.acb_timing_read(C.byref(kms), C.byref(kn))
        L.acb_timing_enable(0)
        if big:
            total = int(tot)
        else:
            status = tot.tolist()
            assert status[1], "capacity too small"
            total = int(status[0])
        return kms.value / steps, e0.elapsed_time(e1) / steps, total
    finally:
        _capi.set_tuning(0)


def engine_of(ac, d, o, engine):
    _capi.set_tuning(5 if engine == "sieve" else 0)
    try:
        m, mo, t = ac.scan_device(d, o)
        return ac._ac.last_stats.get("engine"), m.clone(), mo.clone(), int(t)
    finally:
        _capi.set_tuning(0)


def check_rows(got, rec, what):
    got = got.cpu().numpy().astype(np.int64) & 0xFFFFFFFF   # int32 rows (one call) or int64 rows (runs of calls)
    ok = got.shape == rec.shape and np.array_equal(got, rec.astype(np.int64))
    print(f"  check {what}: {'ok' if ok else 'MISMATCH'} ({rec.shape[0]} matches)", flush=True)
    assert ok


def run_config(name, make_ac, d, o, nbytes, steps, rounds, oracle_check):
    # the third variant does the same work as the case-insensitive one (same matches, same survivors) without the fold:
    # the case-sensitive automaton of the folded patterns on the folded text
    acs = {"case-sensitive": (make_ac(False, False), d), "case-insensitive": (make_ac(True, False), d),
           "fold(P) on fold(H)": (make_ac(False, True), fold_dev(d))}
    engines = []
    for eng in ("auto", "sieve"):
        picked, m, mo, t = engine_of(acs["case-insensitive"][0], d, o, eng)
        if eng == "sieve" or picked != "sieve":
            engines.append((eng, picked))
        if eng == "auto":
            oracle_check(m, mo, t)
    print(f"{name}: {nbytes / 1e6:.1f} MB per step; engines {engines}", flush=True)
    res = {}
    for r in range(rounds):  # alternate the variants: drift of the shared machine falls on all of them alike
        for eng, picked in engines:
            for ci_name, (ac, dv) in acs.items():
                t0 = engine_of(ac, dv, o, eng)[3]
                cap = max(1 << 20, int(t0 * 1.25) + 1024)
                res.setdefault((eng, picked, ci_name), []).append(time_variant(ac, dv, o, eng, steps, cap))
    for (eng, picked, ci_name), v in res.items():
        k = sorted(x[0] for x in v)[len(v) // 2]
        s = sorted(x[1] for x in v)[len(v) // 2]
        print(f"  {picked:6s} {ci_name:18s} kernel {k:8.3f} ms  step {s:8.3f} ms  {nbytes / s / 1e6:8.1f} GB/s  "
              f"{v[0][2]:>10d} matches  (kernel ms per round: {' '.join(f'{x[0]:.3f}' for x in v)})", flush=True)
    for eng, picked in engines:
        med = {v: sorted(x[0] for x in res[(eng, picked, v)])[rounds // 2] for v in acs}
        print(f"  {picked}: case-insensitive kernel time / case-sensitive = {med['case-insensitive'] / med['case-sensitive']:.3f}, "
              f"/ fold(P) on fold(H) (the fold alone) = {med['case-insensitive'] / med['fold(P) on fold(H)']:.3f}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", default="2,3,5")
    args = ap.parse_args()
    only = {int(x) for x in args.only.split(",")}
    torch.cuda.set_device(0)
    print(f"card: {card()}", flush=True)
    t_start = time.time()

    if 2 in only:
        pats, data, offs = W.config2(100_000)
        data = W.recase(data, 0.5, 20)
        pb = [p.encode() for p in pats]
        d, o = torch.from_numpy(data).cuda(), torch.from_numpy(offs).cuda()

        def check2(m, mo, t):
            total, counts, rec = Oracle([fold_np(np.frombuffer(p, dtype=np.uint8)).tobytes() for p in pb], "Standard").scan_batch(
                fold_np(data), offs, codepoints=True)
            assert t == total
            check_rows(m, rec, "config 2 vs oracle(fold(P), fold(H))")

        run_config("config 2 (4244 names, Standard, code points, 100k x 4 KiB, half the letters re-cased)",
                   lambda ci, f: AhoCorasick([ascii_lower(p) if f else p for p in pats], implementation=Implementation.DFA, ascii_case_insensitive=ci),
                   d, o, data.size, args.steps, args.rounds, check2)
        del d, o, data

    if 3 in only:
        pats, data, offs = W.config3(n_patterns=10_000, n_lines=1_000_000)
        data = W.recase(data, 0.5, 30)
        d, o = torch.from_numpy(data).cuda(), torch.from_numpy(offs).cuda()

        def check3(m, mo, t):
            total, counts, rec = Oracle([fold_np(np.frombuffer(p, dtype=np.uint8)).tobytes() for p in pats], "LeftmostLongest").scan_batch(
                fold_np(data), offs)
            assert t == total
            check_rows(m, rec, "config 3 vs oracle(fold(P), fold(H))")

        run_config("config 3 (10k tokens, LeftmostLongest, 1M x 256 B, half the letters re-cased)",
                   lambda ci, f: BytesAhoCorasick([p.lower() if f else p for p in pats], MatchKind.LeftmostLongest, ascii_case_insensitive=ci),
                   d, o, data.size, args.steps, args.rounds, check3)
        del d, o, data

    if 5 in only:
        pats = W.random_lowercase_patterns(50_000, 5, 12, 5)
        n_hay, hb = 1 << 21, 4096
        g = torch.Generator(device="cuda").manual_seed(1005)
        d = torch.randint(97, 123, (n_hay * hb,), dtype=torch.uint8, device="cuda", generator=g)
        d ^= (torch.randint(0, 2, d.shape, dtype=torch.uint8, device="cuda", generator=g) << 5)  # half the letters upper case
        o = torch.arange(n_hay + 1, dtype=torch.int64, device="cuda") * hb

        def check5(m, mo, t):
            cs = BytesAhoCorasick(pats)
            fm, fmo, ft = cs.scan_device(fold_dev(d), o)
            assert ft == t and torch.equal(fm, m) and torch.equal(fmo, mo)
            print(f"  check config 5 vs the case-sensitive scan of the folded text: ok ({t} matches)", flush=True)
            k = 65_536
            sub = d[: k * hb].cpu().numpy()
            total, counts, rec = Oracle(pats, "Standard").scan_batch(fold_np(sub), np.arange(k + 1, dtype=np.int64) * hb)
            check_rows(m[: int(mo[k].item())], rec, f"config 5, first {k} haystacks, vs oracle(fold(P), fold(H))")

        run_config("config 5 (50k patterns a-z, Standard, 2M x 4 KiB = 8 GiB, half the letters upper case)",
                   lambda ci, f: BytesAhoCorasick([p.lower() if f else p for p in pats], ascii_case_insensitive=ci), d, o, d.numel(), args.steps, args.rounds, check5)
    print(f"done in {time.time() - t_start:.0f} s", flush=True)


if __name__ == "__main__":
    main()
