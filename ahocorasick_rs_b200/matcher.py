"""Host-side mirror of the reference's Python API on top of the C ABI.

Reference being mirrored: /root/reference/src/lib.rs (PyO3 classes
``AhoCorasick`` 29-33/134-273, ``BytesAhoCorasick`` 360-435, enums 91-128) and
pysrc/ahocorasick_rs/ahocorasick_rs.pyi.  Same names, argument meaning and
error behaviour; the scan itself runs in the sm_100a kernels behind
include/acb200.h.  There is no CPU fallback: without the CUDA library or a
CUDA device every search raises.

Additions next to the drop-in methods (the reference API is one haystack per
call): ``find_matches_as_indexes_batch`` and ``scan_device`` for batches that
are already device resident.
"""
from __future__ import annotations

import ctypes as C
import enum
import threading
from typing import Iterable, Optional, Sequence

import numpy as np

from . import _capi


class MatchKind(enum.Enum):
    """reference: src/lib.rs:92-98"""
    Standard = 0
    LeftmostFirst = 1
    LeftmostLongest = 2


class Implementation(enum.Enum):
    """reference: src/lib.rs:111-118.  Here, as there, a table-format choice that never changes results
    (tests/test_ac.py:22-56): DFA = the dense transition table (walked by the staged / L2 kernels when the data
    suits them), the two NFA values = the compact sieve image (filters + reverse trie, csrc/sieve.h); None = the
    library decides from a profile of the data."""
    NoncontiguousNFA = 0
    ContiguousNFA = 1
    DFA = 2


_TRACE = bool(__import__("os").environ.get("ACB200_TRACE"))


def _torch():
    import torch
    return torch


def _require_cuda():
    torch = _torch()
    if not torch.cuda.is_available():
        raise RuntimeError("ahocorasick_rs_b200 needs a CUDA device: the scan has no CPU fallback")
    return torch


def _count_cont(x) -> int:
    """UTF-8 continuation bytes (10xxxxxx) in a uint8 numpy array or torch tensor."""
    return int(((x & 0xC0) == 0x80).sum())


def scan_in_windows(scan_window, hay, window_bytes: int, halo: int, codepoints: bool):
    """An OVERLAPPING search over one haystack too large for one call, as independent windows that share `halo` =
    max_pattern_len - 1 bytes (what ends at a position depends on no more than that).  scan_window(window) returns the
    window's matches as int64 rows (haystack, pattern, start, end), window-relative, byte offsets or code point indexes,
    sorted by end.  Every window keeps the matches that END beyond the bytes it shares with its predecessor (those were
    reported, whole, by the predecessor) -- a suffix of its sorted rows --, rebased to the haystack.  `hay` is a uint8
    numpy array or torch tensor; returns the list of per-window row blocks, in order (concatenated they are in the
    reference's order)."""
    total_len = len(hay)
    step = window_bytes - halo
    if step <= 0:
        raise ValueError("window smaller than the longest pattern")
    parts = []
    cont_before = 0  # continuation bytes before the window start (code point indexes)
    w0 = 0
    while w0 < total_len:
        w1 = min(w0 + window_bytes, total_len)
        window = hay[w0:w1]
        part = scan_window(window)
        if w0 > 0 and part.shape[0]:
            cut = halo
            if codepoints:
                # the same cut in code points: ends are character boundaries, so "byte end > halo" is "code point
                # end > code points that start before byte `halo`" -- minus one when a character straddles that
                # byte (its end is beyond the shared bytes although no new character starts in between)
                cut = halo - _count_cont(window[:halo])
                if halo < len(window) and (int(window[halo]) & 0xC0) == 0x80:
                    cut -= 1
            ends = part[:, 3]
            if hasattr(ends, "contiguous"):   # torch: the rows are sorted by end, the kept ones are a suffix
                import torch
                k0 = int(torch.searchsorted(ends.contiguous(), torch.tensor([cut], dtype=ends.dtype, device=ends.device), right=True).item())
            else:
                k0 = int(np.searchsorted(ends, cut, side="right"))
            part = part[k0:]
        base = (w0 - cont_before) if codepoints else w0
        if base:
            part[:, 2] += base
            part[:, 3] += base
        parts.append(part)
        if w1 == total_len:
            break
        if codepoints:
            nxt = w0 + step
            for a in range(w0, nxt, 1 << 28):  # count in slices: the mask is a temporary of the slice's size
                cont_before += _count_cont(hay[a:min(a + (1 << 28), nxt)])
        w0 += step
    return parts


class _Automaton:
    """Owns the host automaton handle, its device image and a growable device
    workspace.  Shared by both public classes."""

    def __init__(self, pattern_bytes: Sequence[bytes], matchkind: MatchKind, implementation: Optional[Implementation],
                 ascii_case_insensitive: bool = False):
        L = _capi.lib()
        n = len(pattern_bytes)
        offs = np.zeros(n + 1, dtype=np.uint64)
        if n:
            np.cumsum(np.fromiter((len(p) for p in pattern_bytes), dtype=np.uint64, count=n), out=offs[1:])
        blob = np.frombuffer(b"".join(pattern_bytes) or b"\0", dtype=np.uint8)
        h = C.c_void_p()
        impl = -1 if implementation is None else implementation.value
        flags = _capi.ACB_ASCII_CASE_INSENSITIVE if ascii_case_insensitive else 0
        rc = L.acb_build_ex(blob.ctypes.data, offs.ctypes.data, n, matchkind.value, impl, flags, C.byref(h))
        if rc != _capi.ACB_OK:
            raise ValueError(_capi.last_error())
        self._h = h
        self._L = L
        self.matchkind = matchkind
        self.implementation = implementation
        self.ascii_case_insensitive = bool(ascii_case_insensitive)
        self.n_patterns = n
        self.num_states = int(L.acb_num_states(h))
        self.num_columns = int(L.acb_num_columns(h))
        self.max_pattern_len = int(L.acb_max_pattern_len(h))
        self._images = {}      # device index -> uint8 tensor
        self._sieves = {}      # device index -> (uint8 tensor, SieveDesc)
        self._hot = {}         # device index -> dict(tensor, rows, reprofile, calls, backoff)
        self._ws = {}          # (device index, slot) -> dict of tensors
        self._small = {}       # device index -> the small-call context
        self.last_stats = {}
        self._lock = threading.Lock()
        self._host_lock = threading.RLock()   # host-buffer calls: staging buffer + workspaces until the results are on the host

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._L.acb_free(h)
            self._h = None

    # ---- device residency ---------------------------------------------------
    def image(self, device):
        """The flat tables on `device` (uploaded once, then cached)."""
        torch = _require_cuda()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        img = self._images.get(idx)
        if img is None:
            nbytes = int(self._L.acb_image_bytes(self._h))
            host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
            rc = self._L.acb_image_write(self._h, host.data_ptr(), nbytes)
            if rc != _capi.ACB_OK:
                raise RuntimeError(_capi.last_error())
            img = host.to(torch.device("cuda", idx), non_blocking=False)
            self._images[idx] = img
        return img

    # ---- the sieve image (position-parallel scan: Bloom filter in shared memory + reverse trie in HBM/L2) ----
    ENGINE = __import__("os").environ.get("ACB200_ENGINE", "auto")   # "auto" | "sieve" | "table": kernel family (see scan_device)
    AUTO_PROFILE_BYTES = 4 << 20     # "auto": inputs below this never pay for the profiling pass
    SIEVE_SMEM_RESERVE = int(__import__("os").environ.get("ACB200_SIEVE_RESERVE_KB", "46")) * 1024   # 24 warps x (one ring slot of text + two queues); barrier
    SIEVE_W_MAX = 0                  # 0 = the builder chooses the primary window

    def sieve(self, device):
        """(device tensor, SieveDesc) of the sieve image on `device`, built and uploaded once."""
        torch = _require_cuda()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        ent = self._sieves.get(idx)
        if ent is None:
            props = torch.cuda.get_device_properties(idx)
            smem = int(getattr(props, "shared_memory_per_block_optin", 227 * 1024))
            nbytes = int(self._L.acb_sieve_build(self._h, max(4096, smem - self.SIEVE_SMEM_RESERVE), self.SIEVE_W_MAX))
            if nbytes == 0:
                raise RuntimeError(_capi.last_error())
            host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
            if self._L.acb_sieve_write(self._h, host.data_ptr(), nbytes) != _capi.ACB_OK:
                raise RuntimeError(_capi.last_error())
            desc = _capi.SieveDesc()
            if self._L.acb_sieve_describe(host.data_ptr(), C.byref(desc)) != _capi.ACB_OK:
                raise RuntimeError(_capi.last_error())
            ent = (host.to(torch.device("cuda", idx)), desc)
            self._sieves[idx] = ent
        return ent

    # ---- the hot image (rows kept in shared memory), chosen from a sample of the data ----
    HOT_TABLE_BYTES = 40 * 1024   # with 32 warps of staging buffers next to it, this is what fits on chip
    HOT_COVERAGE_MIN = 0.99       # share of sampled state visits the hot rows must cover for the shared-memory kernel to be used

    def _max_hot_rows(self):
        return max(2, min(4096, self.HOT_TABLE_BYTES // (2 * self.num_columns) - 1))

    def _upload_hot(self, idx, visits_host):
        torch = _torch()
        rows = self._max_hot_rows()
        nbytes = int(self._L.acb_hot_bytes(self._h, rows))
        host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        vp = visits_host.ctypes.data if visits_host is not None else None
        rc = self._L.acb_hot_build(self._h, vp, rows, host.data_ptr(), nbytes)
        if rc != _capi.ACB_OK:
            raise RuntimeError(_capi.last_error())
        desc = _capi.HotDesc()
        if self._L.acb_hot_describe(host.data_ptr(), C.byref(desc)) != _capi.ACB_OK:
            raise RuntimeError(_capi.last_error())
        return host.to(torch.device("cuda", idx)), desc

    def hot(self, device, data=None, offsets=None, overlapping=False):
        """The hot image on `device`.  Built from a profile of (data, offsets) the
        first time this automaton scans on the device, and again -- with
        exponential back-off -- when the kernel reports that the fast path keeps
        falling out of the hot set (the data changed character)."""
        torch = _torch()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        st = self._hot.get(idx)
        need = st is None or st["reprofile"]
        if need and data is not None and data.numel() > 0 and offsets is not None and offsets.numel() > 1:
            img = self.image(device)
            visits = torch.empty(self.num_states, dtype=torch.int32, device=device)
            stream = torch.cuda.current_stream(device).cuda_stream
            n = offsets.numel() - 1
            rc = self._L.acb_profile(self._h, img.data_ptr(), data.data_ptr(), offsets.data_ptr(), n, data.numel(),
                                     int(bool(overlapping)), visits.data_ptr(), stream)
            if rc != _capi.ACB_OK:
                raise RuntimeError(_capi.last_error())
            vh = visits.cpu().numpy().view(np.uint32)
            t, rows = self._upload_hot(idx, vh)
            # How much of the sampled scan the hot rows cover.  Every byte outside them costs the staged kernel a
            # detour through the exact scanner while 31 lanes wait; below ~99 % the segment kernel that reads the
            # table from global memory / L2 is faster (dense automata on random text: BASELINE configs 4 and 5).
            total_visits = int(vh.sum(dtype=np.uint64))
            if total_visits > 0 and rows.rows < self.num_states:
                top = np.partition(vh, len(vh) - rows.rows)[len(vh) - rows.rows:]
                coverage = float(top.sum(dtype=np.uint64)) / total_visits
            else:
                coverage = 1.0
            rows.reserved = 1 if coverage < self.HOT_COVERAGE_MIN else 0
            backoff = (st["backoff"] * 2) if st else 1
            st = {"tensor": t, "rows": rows, "reprofile": False, "calls": 0, "backoff": backoff, "coverage": coverage}
            self._hot[idx] = st
        elif st is None:
            t, rows = self._upload_hot(idx, None)
            st = {"tensor": t, "rows": rows, "reprofile": True, "calls": 0, "backoff": 1, "coverage": 1.0}
            self._hot[idx] = st
        return st

    def _note_trap_stats(self, st, groups: int, traps: int):
        st["calls"] += 1
        if st["rows"].reserved & 1:
            return  # scanning from global memory: the hot rows are not in use
        if groups > 4096 and traps * 10 > groups and st["calls"] >= st["backoff"]:
            st["reprofile"] = True
            st["calls"] = 0

    def _plan(self, data, n_haystacks: int):
        plan = _capi.Plan()
        rc = self._L.acb_plan_scan(self._h, data.data_ptr(), data.numel(), n_haystacks, C.byref(plan))
        if rc != _capi.ACB_OK:
            raise RuntimeError(_capi.last_error())
        return plan

    def _workspace(self, device, plan, n_haystacks: int, capacity: int, slot: int = 0):
        torch = _torch()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        key = (idx, slot)   # (the host pipeline alternates between two workspaces)
        ws = self._ws.get(key)
        need = (ws is None or ws["n_units"] < plan.n_units or ws["n_segments"] < plan.n_segments or
                ws["scratch"].numel() < plan.scratch_words or ws["n_haystacks"] < n_haystacks or ws["capacity"] < capacity)
        if need:
            n_units = max(plan.n_units, ws["n_units"] if ws else 0, 1)
            n_seg = max(plan.n_segments, ws["n_segments"] if ws else 0, 1)
            n_hay = max(n_haystacks, ws["n_haystacks"] if ws else 0, 1)
            n_scr = max(plan.scratch_words, ws["scratch"].numel() if ws else 0, 16)
            cap = max(capacity, ws["capacity"] if ws else 0, 1024)
            dev = torch.device("cuda", idx)
            ws = {
                "n_units": n_units, "n_segments": n_seg, "n_haystacks": n_hay, "capacity": cap,
                "raw": torch.empty((cap, 4), dtype=torch.int32, device=dev),
                "raw_seq": torch.empty(cap, dtype=torch.int32, device=dev),
                "raw_unit": torch.empty(cap, dtype=torch.int32, device=dev),
                "raw_aux": torch.empty(cap, dtype=torch.int32, device=dev),
                "unit_counts": torch.empty(n_units, dtype=torch.int32, device=dev),
                "unit_offsets": torch.empty(n_units + 1, dtype=torch.int64, device=dev),
                "seg_info": torch.empty((n_seg, 8), dtype=torch.int32, device=dev),
                "scratch": torch.zeros(n_scr, dtype=torch.int64, device=dev),  # zeroed: its head holds the kernels' counters
                "total": torch.zeros(8, dtype=torch.int64, device=dev),
                "out": torch.empty((cap, 4), dtype=torch.int32, device=dev),
                "match_offsets": torch.empty(n_hay + 1, dtype=torch.int64, device=dev),
            }
            self._ws[key] = ws
        return ws

    def _ws_struct(self, ws):
        s = _capi.Workspace()
        s.dev_raw = ws["raw"].data_ptr()
        s.dev_raw_seq = ws["raw_seq"].data_ptr()
        s.dev_raw_unit = ws["raw_unit"].data_ptr()
        s.dev_raw_aux = ws["raw_aux"].data_ptr()
        s.raw_capacity = ws["capacity"]
        s.dev_unit_counts = ws["unit_counts"].data_ptr()
        s.dev_unit_offsets = ws["unit_offsets"].data_ptr()
        s.dev_seg_info = ws["seg_info"].data_ptr()
        s.dev_scratch = ws["scratch"].data_ptr()
        s.dev_total = ws["total"].data_ptr()
        s.dev_out = ws["out"].data_ptr()
        s.out_capacity = ws["capacity"]
        s.dev_match_offsets = ws["match_offsets"].data_ptr()
        return s

    def check_overlapping(self, overlapping):
        # reference: the iterator is refused before any byte is read (src/lib.rs:52-54, 36-39)
        if overlapping and overlapping != 2 and self.matchkind != MatchKind.Standard:
            raise ValueError(f"match kind {self.matchkind.name} does not support overlapping searches")

    # ---- scans ------------------------------------------------------------------
    def scan_device(self, data, offsets, overlapping=False, codepoints=False, capacity: Optional[int] = None,
                    sync: bool = True, ws_slot: int = 0):
        """Scan a device-resident batch.  data: uint8 CUDA tensor, offsets: int64
        CUDA tensor (n+1).  One haystack of any size is simply n = 1.  Returns
        (matches, match_offsets, total): matches is an int32 CUDA tensor
        (total, 4) = (haystack, pattern, start, end) in the reference's order,
        match_offsets (n+1) brackets each haystack's rows.  With sync=False the
        call returns right after enqueueing (total is the 8-entry device status
        tensor and matches the whole capacity-sized buffer).

        The returned tensors are VIEWS of this automaton's workspace `ws_slot` on the
        device: they are valid until the next scan that uses the same slot (copy them,
        or use scan_host / the find_* methods, when several threads share one automaton)."""
        torch = _require_cuda()
        self.check_overlapping(overlapping)
        dev = data.device
        n = offsets.numel() - 1
        if data.numel() > self.WINDOW_BYTES:
            if not sync:
                raise ValueError(f"buffers above {self.WINDOW_BYTES} bytes are scanned in windows: sync=False is not available")
            return self._scan_device_windows(data, offsets, overlapping, codepoints)
        img = self.image(dev)
        cap = capacity or max(1024, n * 2)
        stream = torch.cuda.current_stream(dev).cuda_stream
        # which kernel family: the position-parallel sieve (default) or the table walkers (forced by the tuning knob,
        # or ENGINE = "table").  Results are identical; only the device images a scan needs differ.
        forced = _capi.current_kernel()
        with self._lock, torch.cuda.device(dev):
            # Which kernel family.  Results are identical; only speed and the device images a scan needs differ.
            #   table  the automaton walkers: best when the scan lives in a few hundred states that fit in shared memory
            #          (sparse matches in text) -- the profile of the data says so (hot-row coverage);
            #   sieve  the position-parallel filter + exact verification: everything else (dense pattern sets, whose
            #          states live in L2), and small inputs, where the profiling pass would cost more than the scan.
            hot = None
            if overlapping == 2 or forced == 5 or (forced == 0 and self.ENGINE == "sieve"):
                use_sieve = True
            elif forced in (1, 2, 3, 4) or self.ENGINE == "table":
                use_sieve = False
            elif self.implementation in (Implementation.ContiguousNFA, Implementation.NoncontiguousNFA):
                use_sieve = True   # the caller asked for a compact (non-DFA) table format: that is the sieve image
            else:
                use_sieve = data.numel() < self.AUTO_PROFILE_BYTES and self._hot.get(dev.index if dev.index is not None else torch.cuda.current_device()) is None
                if not use_sieve:
                    hot = self.hot(dev, data, offsets, overlapping)
                    use_sieve = bool(hot["rows"].reserved & 1)
            if use_sieve:
                sieve_t, sieve_d = self.sieve(dev)
                hot = None
            elif hot is None:
                hot = self.hot(dev, data, offsets, overlapping)
            plan = self._plan(data, n)
            while True:
                ws = self._workspace(dev, plan, n, cap, ws_slot)
                st = self._ws_struct(ws)
                rc = self._L.acb_scan_batch(self._h, img.data_ptr(),
                                            hot["tensor"].data_ptr() if hot else None, C.byref(hot["rows"]) if hot else None,
                                            sieve_t.data_ptr() if use_sieve else None,
                                            data.data_ptr(), offsets.data_ptr(), n, data.numel(),
                                            2 if overlapping == 2 else int(bool(overlapping)), int(bool(codepoints)), C.byref(plan), C.byref(st), stream)
                if rc != _capi.ACB_OK:
                    err = _capi.last_error()
                    ws["scratch"][:8].zero_()   # a scan that failed half way may have left its counters dirty
                    raise (ValueError if rc == _capi.ACB_EUNSUPPORTED else RuntimeError)(err)
                if not sync:
                    return ws["out"], ws["match_offsets"][: n + 1], ws["total"]
                tot = ws["total"].tolist()
                total, complete, raw_total = tot[0], tot[1], tot[4]
                if hot:
                    self._note_trap_stats(hot, tot[2], tot[3])
                    self.last_stats = {"engine": "table", "groups": tot[2], "traps": tot[3], "repairs": tot[5], "segments": plan.n_segments,
                                       "hot_rows": hot["rows"].rows, "hot_rows128": hot["rows"].rows128,
                                       "hot_visited": hot["rows"].visited, "hot_coverage": round(hot.get("coverage", 1.0), 5),
                                       "global_table": bool(hot["rows"].reserved & 1),
                                       "segment_bytes": plan.segment_bytes, "lane_stride": plan.lane_stride}
                else:
                    self.last_stats = {"engine": "sieve", "window": sieve_d.window, "last_level": sieve_d.last_level,
                                       "probes": sieve_d.probes, "bloom_bytes": sieve_d.bloom_bytes, "nodes": sieve_d.nodes,
                                       "keys": sieve_d.keys, "filter_entries": sieve_d.filter_entries,
                                       "task_bytes": plan.task_bytes, "list_records": raw_total}
                if complete or (total == 0 and raw_total == 0):
                    return ws["out"][:total], ws["match_offsets"][: n + 1], total
                cap = max(total, raw_total) + max(total, raw_total) // 8 + 16

    # One kernel call addresses its buffer with 32-bit offsets.  Larger inputs are cut up here: a batch into
    # runs of whole haystacks, a single haystack above the limit into overlapping windows.
    WINDOW_BYTES = (1 << 31) - (1 << 16)   # (below 2^31: every offset of one call is a non-negative int32)

    def _scan_device_windows(self, data, offsets, overlapping, codepoints):
        """scan_device for buffers above WINDOW_BYTES.  Same results, as int64 tensors
        (offsets no longer fit 32 bits): (matches (k, 4) int64, match_offsets (n + 1) int64, total).
        Everything stays on the device; the host only learns where the runs of whole haystacks end."""
        torch = _require_cuda()
        dev = data.device
        n = offsets.numel() - 1
        limit = self.WINDOW_BYTES
        parts = []          # (k, 4) int64 tensors in haystack order
        mo = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        lens = offsets[1:] - offsets[:-1]
        oversized = bool((lens > limit).any().item()) if n else False
        base_count = 0
        h = 0
        while h < n:
            start = int(offsets[h].item())
            if oversized and int(lens[h].item()) > limit:
                part = self._scan_one_large(data[start:start + int(lens[h].item())], overlapping, codepoints)
                part[:, 0] = h
                parts.append(part)
                base_count += int(part.shape[0])
                mo[h + 1] = base_count
                h += 1
                continue
            # the longest run of whole haystacks that fits one call (and stops before an oversized one)
            h1 = int(torch.searchsorted(offsets, torch.tensor([start + limit], dtype=torch.int64, device=dev), right=True).item()) - 1
            h1 = max(h + 1, min(h1, n))
            if oversized:
                big = torch.nonzero(lens[h:h1] > limit)
                if big.numel():
                    h1 = h + int(big[0].item())
            end = int(offsets[h1].item())
            sub_offs = offsets[h:h1 + 1] - start
            _t0 = __import__("time").perf_counter() if _TRACE else 0
            m, mo_run, total = self.scan_device(data[start:end], sub_offs, overlapping, codepoints)
            _t1 = __import__("time").perf_counter() if _TRACE else 0
            part = m.to(torch.int64)
            if h:
                part[:, 0] += h
            parts.append(part)
            mo[h + 1:h1 + 1] = mo_run[1:h1 - h + 1].to(torch.int64) + base_count
            base_count += int(total)
            if _TRACE:
                torch.cuda.synchronize()
                print(f"[trace] run haystacks {h}..{h1} ({end - start} B): scan_device {(_t1 - _t0) * 1e3:.2f} ms, post {(__import__('time').perf_counter() - _t1) * 1e3:.2f} ms, total {total}", flush=True)
            h = h1
        out = torch.cat(parts, dim=0) if len(parts) != 1 else parts[0]
        if not parts:
            out = torch.zeros((0, 4), dtype=torch.int64, device=dev)
        return out, mo, int(out.shape[0])

    def _scan_one_large(self, hay, overlapping, codepoints):
        """One haystack above WINDOW_BYTES (BASELINE config 4: one 4 GiB haystack, overlapping).  The OVERLAPPING list
        is exact window by window: windows that share max_pattern_len - 1 bytes are independent (what ends at a position
        depends on no more than that), each keeps the matches that END beyond the shared bytes.  A non-overlapping
        search restarts at every match end, which chains the windows to each other: its result is SELECTED from the
        overlapping list afterwards (acb_select_non_overlapping; SURVEY.md 8c), for all three match kinds."""
        torch = _require_cuda()
        dev = hay.device

        def scan_window(window):
            one = torch.tensor([0, window.numel()], dtype=torch.int64, device=dev)
            m, _, _ = self._scan_overlapping_list(window, one, codepoints)
            return m.to(torch.int64)

        parts = scan_in_windows(scan_window, hay, self.WINDOW_BYTES, max(self.max_pattern_len - 1, 0), codepoints)
        rows = torch.cat(parts, dim=0) if parts else torch.zeros((0, 4), dtype=torch.int64, device=dev)
        if overlapping or rows.shape[0] == 0:
            return rows
        rows = rows.contiguous()
        out = torch.empty_like(rows)
        count = torch.zeros(1, dtype=torch.int64, device=dev)
        rc = self._L.acb_select_non_overlapping(self._h, rows.data_ptr(), rows.shape[0], out.data_ptr(), count.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream)
        if rc != _capi.ACB_OK:
            raise RuntimeError(_capi.last_error())
        return out[: int(count.item())]

    def _scan_overlapping_list(self, data, offsets, codepoints):
        """The overlapping match list whatever the automaton's match kind: the sieve's structures do not depend on the
        kind (overlapping = 2 is the library-internal form of the request; the public overlapping=True on a leftmost
        automaton stays an error, like the reference's)."""
        return self.scan_device(data, offsets, 2, codepoints)

    # ---- host-resident input (the reference's situation: src/lib.rs:229-249, 422-434 take host str / buffers) ----
    HOST_CHUNK_BYTES = 1 << 30     # inputs up to this size go in one piece (the scan is ~100x faster than PCIe: nothing to hide);
                                   # larger ones in runs of this size: copy of run i+1 || scan of run i || results of run i-1
    _staging = None                # grow-only pinned staging buffer for inputs that are not pinned already

    def _pinned(self, nbytes: int):
        torch = _torch()
        st = self._staging
        if st is None or st.numel() < nbytes:
            st = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8, pin_memory=True)
            self._staging = st
        return st

    def scan_host(self, data, offsets, overlapping: bool = False, codepoints: bool = False, chunk_bytes: Optional[int] = None):
        """Scan a batch that lives in HOST memory: data = 1-D uint8 (numpy array or CPU torch tensor; pinned memory
        makes the copies asynchronous), offsets = int64 (n + 1).  Returns host numpy arrays
        (matches (k, 4) uint32 -- int64 when a window path was needed --, match_offsets (n + 1) int64).

        Large inputs are cut into runs of whole haystacks of about `chunk_bytes`: the host->device copy of run i+1
        (copy stream, second device buffer) overlaps the scan of run i, whose results are copied back while run i+1
        is scanned (two workspaces).  The whole call holds the automaton's lock, so threads sharing one automaton
        are serialised here instead of corrupting each other's workspace."""
        torch = _require_cuda()
        self.check_overlapping(overlapping)
        if isinstance(data, np.ndarray):
            hdata = torch.from_numpy(data) if data.flags.writeable else torch.from_numpy(data.copy())
        else:
            hdata = data
        offs = offsets.numpy() if hasattr(offsets, "numpy") else np.asarray(offsets)
        offs = np.ascontiguousarray(offs, dtype=np.int64)
        n = len(offs) - 1
        total_bytes = int(offs[-1] - offs[0]) if n > 0 else 0
        dev = torch.device("cuda", torch.cuda.current_device())
        chunk = int(chunk_bytes or self.HOST_CHUNK_BYTES)
        with self._host_lock:
            if n <= 0 or total_bytes <= chunk or int(np.max(np.diff(offs))) > self.WINDOW_BYTES:
                # one shot (small input), or the oversized-haystack window path
                lo, hi = (int(offs[0]), int(offs[-1])) if n > 0 else (0, 0)
                d_data = hdata[lo:hi].to(dev, non_blocking=True)
                d_offs = torch.from_numpy(offs - lo).to(dev, non_blocking=True)
                m, moffs, _ = self.scan_device(d_data, d_offs, overlapping, codepoints)
                m = m.cpu().numpy()
                return (m.view(np.uint32) if m.dtype == np.int32 else m), moffs.cpu().numpy().astype(np.int64)
            # runs of whole haystacks
            cuts = [0]
            while cuts[-1] < n:
                h0 = cuts[-1]
                h1 = int(np.searchsorted(offs, offs[h0] + chunk, side="right")) - 1
                cuts.append(min(max(h1, h0 + 1), n))
            runs = list(zip(cuts[:-1], cuts[1:]))
            max_bytes = max(int(offs[b] - offs[a]) for a, b in runs)
            max_hay = max(b - a for a, b in runs)
            dbuf = [torch.empty(max_bytes, dtype=torch.uint8, device=dev) for _ in range(2)]
            doff = [torch.empty(max_hay + 1, dtype=torch.int64, device=dev) for _ in range(2)]
            hoff = [torch.empty(max_hay + 1, dtype=torch.int64, pin_memory=True) for _ in range(2)]
            main = torch.cuda.current_stream(dev)
            copier = torch.cuda.Stream(device=dev)
            scanned = [None, None]
            parts, counts = [], np.zeros(n, dtype=np.int64)
            cap = max(4096, 2 * max_hay)

            def collect(job):
                slot, a, b, nbytes, out, mo, tot = job
                t = tot.tolist()            # waits for that run's scan only
                total, complete, raw_total = t[0], t[1], t[4]
                if not (complete or (total == 0 and raw_total == 0)):
                    # rare: the run had more matches than room; redo it with what it needs
                    m, mo2, total = self.scan_device(dbuf[slot][:nbytes], doff[slot][: b - a + 1], overlapping, codepoints,
                                                     capacity=max(total, raw_total) + max(total, raw_total) // 8 + 16, ws_slot=slot)
                    out, mo = m, mo2
                part = np.empty((total, 4), dtype=np.uint32)
                if total:
                    torch.from_numpy(part.view(np.int32)).copy_(out[:total])   # one D2H copy straight into the result array
                    if a:
                        part[:, 0] += a
                parts.append(part)
                run_mo = np.empty(b - a + 1, dtype=np.int64)
                torch.from_numpy(run_mo).copy_(mo[: b - a + 1])
                counts[a:b] = np.diff(run_mo)

            pending = None
            for i, (a, b) in enumerate(runs):
                slot = i & 1
                nbytes = int(offs[b] - offs[a])
                with torch.cuda.stream(copier):
                    if scanned[slot] is not None:
                        copier.wait_event(scanned[slot])   # the scan that read this device buffer two runs ago
                    dbuf[slot][:nbytes].copy_(hdata[int(offs[a]):int(offs[b])], non_blocking=True)
                    hoff[slot][: b - a + 1].copy_(torch.from_numpy(offs[a:b + 1] - offs[a]))
                    doff[slot][: b - a + 1].copy_(hoff[slot][: b - a + 1], non_blocking=True)
                    copied = torch.cuda.Event()
                    copied.record(copier)
                main.wait_event(copied)
                if pending is not None and pending[0] == slot:
                    collect(pending)        # (never: slots alternate) keeps the workspace of this slot free
                    pending = None
                out, mo, tot = self.scan_device(dbuf[slot][:nbytes], doff[slot][: b - a + 1], overlapping, codepoints,
                                                capacity=cap, sync=False, ws_slot=slot)
                ev = torch.cuda.Event()
                ev.record(main)
                scanned[slot] = ev
                job = (slot, a, b, nbytes, out, mo, tot)
                if pending is not None:
                    collect(pending)        # D2H of the previous run while this one is being scanned
                pending = job
            collect(pending)
            m = np.concatenate(parts, axis=0) if parts else np.zeros((0, 4), dtype=np.uint32)
            mo = np.zeros(n + 1, dtype=np.int64)
            np.cumsum(counts, out=mo[1:])
            return m, mo

    # ---- one small haystack per call: the reference's own usage (benchmarks/test_comparison.py:119-122) ----
    SMALL_CALL_BYTES = 256 << 10   # up to here a single-haystack call takes the lean path below
    SMALL_CALL_ROWS = 64           # matches copied back with the status words in ONE transfer (more: a second copy)

    def _small_ctx(self, dev):
        """Everything a small call needs, allocated once per device: pinned and device input buffers (offsets first,
        then the bytes), a workspace whose status words and output rows are adjacent (one D2H copy fetches both), its
        ctypes description, the sieve image."""
        torch = _torch()
        idx = dev.index
        ctx = self._small.get(idx)
        if ctx is None:
            cap_b = self.SMALL_CALL_BYTES
            sieve_t, sieve_d = self.sieve(dev)
            img = self.image(dev)
            h_in = torch.zeros(16 + cap_b + 16, dtype=torch.uint8, pin_memory=True)
            d_in = torch.zeros(16 + cap_b + 16, dtype=torch.uint8, device=dev)
            plan = _capi.Plan()
            if self._L.acb_plan_scan(self._h, d_in.data_ptr() + 16, cap_b, 1, C.byref(plan)) != _capi.ACB_OK:
                raise RuntimeError(_capi.last_error())
            cap = 4096
            n_units = int(plan.n_units) + 8
            res = torch.zeros(8 + 2 * cap, dtype=torch.int64, device=dev)
            ws = {
                "n_units": n_units, "n_segments": int(plan.n_segments) + 4, "n_haystacks": 1, "capacity": cap,
                "raw": torch.empty((cap, 4), dtype=torch.int32, device=dev),
                "raw_seq": torch.empty(cap, dtype=torch.int32, device=dev),
                "raw_unit": torch.empty(cap, dtype=torch.int32, device=dev),
                "raw_aux": torch.empty(cap, dtype=torch.int32, device=dev),
                "unit_counts": torch.empty(n_units, dtype=torch.int32, device=dev),
                "unit_offsets": torch.empty(n_units + 1, dtype=torch.int64, device=dev),
                "seg_info": torch.empty((int(plan.n_segments) + 4, 8), dtype=torch.int32, device=dev),
                "scratch": torch.zeros(int(plan.scratch_words) + 64, dtype=torch.int64, device=dev),
                "total": res[:8], "out": res[8:].view(torch.int32).view(cap, 4),
                "match_offsets": torch.empty(2, dtype=torch.int64, device=dev),
            }
            ctx = {"h_in": h_in, "d_in": d_in, "hv": h_in.numpy(), "res": res, "ws": ws, "st": self._ws_struct(ws),
                   "h_res": torch.zeros(8 + 2 * self.SMALL_CALL_ROWS, dtype=torch.int64, pin_memory=True),
                   "sieve": sieve_t, "img": img, "plan": plan, "max_scratch": int(plan.scratch_words) + 64, "max_units": n_units}
            ctx["hr"] = ctx["h_res"].numpy()
            self._small[idx] = ctx
        return ctx

    def _small_call(self, hay, overlapping: bool, codepoints: bool):
        """One haystack of at most SMALL_CALL_BYTES (a bytes-like object): one H2D copy, scan + epilogue, one D2H copy of
        (status, first rows), one synchronisation.  -> uint32 (k, 4) host array."""
        torch = _require_cuda()
        dev = torch.device("cuda", torch.cuda.current_device())
        n = len(hay)
        with self._host_lock:
            ctx = self._small_ctx(dev)
            hv = ctx["hv"]
            hv[:16].view(np.int64)[:] = (0, n)
            if n:
                hv[16:16 + n] = np.frombuffer(hay, dtype=np.uint8)
            d_in = ctx["d_in"]
            d_in[:16 + n].copy_(ctx["h_in"][:16 + n], non_blocking=True)
            plan = ctx["plan"]
            base = d_in.data_ptr()
            if self._L.acb_plan_scan(self._h, base + 16, n, 1, C.byref(plan)) != _capi.ACB_OK:
                raise RuntimeError(_capi.last_error())
            if plan.scratch_words > ctx["max_scratch"] or plan.n_units > ctx["max_units"]:
                return None   # (a tuning knob changed the plan beyond what was allocated: let the general path do it)
            stream = torch.cuda.current_stream(dev)
            rc = self._L.acb_scan_batch(self._h, ctx["img"].data_ptr(), None, None, ctx["sieve"].data_ptr(), base + 16, base, 1, n,
                                        int(bool(overlapping)), int(bool(codepoints)), C.byref(plan), C.byref(ctx["st"]), stream.cuda_stream)
            if rc != _capi.ACB_OK:
                err = _capi.last_error()
                ctx["ws"]["scratch"][:8].zero_()   # a scan that failed half way may have left its counters dirty
                raise (ValueError if rc == _capi.ACB_EUNSUPPORTED else RuntimeError)(err)
            ctx["h_res"].copy_(ctx["res"][: ctx["h_res"].numel()], non_blocking=True)
            stream.synchronize()
            hr = ctx["hr"]
            total, complete = int(hr[0]), int(hr[1])
            if not complete:
                return None   # more matches than the small workspace holds: the general path sizes one
            if total <= self.SMALL_CALL_ROWS:
                return hr[8:8 + 2 * total].view(np.uint32).reshape(total, 4).copy()
            return ctx["ws"]["out"][:total].cpu().numpy().view(np.uint32)

    def scan_host_batch(self, chunks: Sequence[bytes], overlapping: bool, codepoints: bool):
        """Host buffers (bytes-like objects, one per haystack) in, host numpy out: (matches uint32 (k,4),
        match_offsets int64 (n+1)).  The haystacks are gathered into this automaton's pinned staging buffer
        (for a single haystack: one copy straight out of the caller's buffer), then scan_host takes over."""
        torch = _require_cuda()
        self.check_overlapping(overlapping)
        n = len(chunks)
        if n == 1 and len(chunks[0]) <= self.SMALL_CALL_BYTES and _capi.current_kernel() in (0, 5) and self.ENGINE != "table":
            m = self._small_call(chunks[0], overlapping, codepoints)
            if m is not None:
                return m, np.array([0, m.shape[0]], dtype=np.int64)
        lens = np.fromiter((len(c) for c in chunks), dtype=np.int64, count=n)
        offs = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lens, out=offs[1:])
        total_bytes = int(offs[-1])
        with self._host_lock:
            host = self._pinned(total_bytes)
            hv = host.numpy()
            if n == 1:
                hv[:total_bytes] = np.frombuffer(chunks[0], dtype=np.uint8)
            elif total_bytes:
                hv[:total_bytes] = np.frombuffer(b"".join(chunks), dtype=np.uint8)  # one C-speed concatenation, one copy into pinned memory
            return self.scan_host(host[:total_bytes], offs, overlapping, codepoints)


def _as_buffer_bytes(obj) -> bytes:
    """reference PyBufferBytes::try_from (src/lib.rs:281-302): 1-D, C-contiguous u8 buffer."""
    if isinstance(obj, str):
        raise TypeError("a bytes-like object is required, not 'str'")
    try:
        mv = memoryview(obj)
    except TypeError as e:
        raise TypeError(str(e)) from None
    if mv.ndim > 1:
        raise TypeError("Only one-dimensional sequences are supported")
    if not mv.c_contiguous:
        raise TypeError("Must be a contiguous sequence of bytes")
    if mv.itemsize != 1 or mv.format not in ("B", "b", "c"):
        raise BufferError("buffer contents are not compatible with u8")
    # zero-copy like the reference's PyBufferBytes (src/lib.rs:304-340): the caller's memory is read in place (one copy,
    # into the pinned staging buffer the H2D transfer starts from); as there, the caller must not mutate it meanwhile
    return obj if isinstance(obj, bytes) else (mv if mv.format == "B" else mv.cast("B"))


def _check_ascii_case_insensitive(value):
    if not isinstance(value, bool):
        raise TypeError("ascii_case_insensitive must be a bool")


def _tuples(m: np.ndarray):
    return list(zip(m[:, 1].tolist(), m[:, 2].tolist(), m[:, 3].tolist()))


class AhoCorasick:
    """Search for multiple pattern strings against a haystack string
    (reference: src/lib.rs:15-33, 134-273).

    * ``patterns``: any iterable of non-empty ``str``.
    * ``matchkind``: ``MatchKind.Standard`` (default), ``LeftmostFirst`` or ``LeftmostLongest``.
    * ``store_patterns``: keep references to the patterns to speed up
      ``find_matches_as_strings``; ``None`` = store iff total length <= 4096 code points.
    * ``implementation``: ``Implementation`` hint or ``None``.
    * ``ascii_case_insensitive`` (keyword only): an ASCII letter in a pattern matches either case of that letter in
      the haystack (the crate's ``AhoCorasickBuilder::ascii_case_insensitive``); every other character must match
      exactly, so ``"é"`` does not match ``"É"``.  Indexes stay code point indexes of the haystack as given.
    """

    def __init__(self, patterns: Iterable[str], matchkind: MatchKind = MatchKind.Standard,
                 store_patterns: Optional[bool] = None, implementation: Optional[Implementation] = None, *,
                 ascii_case_insensitive: bool = False):
        if not isinstance(matchkind, MatchKind):
            raise TypeError("matchkind must be a MatchKind")
        if implementation is not None and not isinstance(implementation, Implementation):
            raise TypeError("implementation must be an Implementation or None")
        _check_ascii_case_insensitive(ascii_case_insensitive)
        it = iter(patterns)  # TypeError for non-iterables, like try_iter()? at src/lib.rs:147
        strs = []
        encoded = []
        total = 0
        decide = store_patterns is None
        store = True if decide else bool(store_patterns)
        for p in it:
            if not isinstance(p, str):
                raise TypeError(f"'{type(p).__name__}' object cannot be converted to 'PyString'")
            if p == "":
                raise ValueError("You passed in an empty string as a pattern")
            try:
                b = p.encode("utf-8")
            except UnicodeEncodeError:
                break  # reference quirk: a pattern that is not valid UTF-8 silently ends ingestion (src/lib.rs:200-203)
            if decide and store:
                total += len(p)
                if total > 4096:
                    store = False
                    strs = []
            if store:
                strs.append(p)
            encoded.append(b)
        self._patterns = strs if store else None
        self._ac = _Automaton(encoded, matchkind, implementation, ascii_case_insensitive)

    def find_matches_as_indexes(self, haystack: str, overlapping: bool = False):
        """-> list of (pattern index, start, end) in code points (src/lib.rs:229-249)."""
        if not isinstance(haystack, str):
            raise TypeError("argument 'haystack': 'str' expected")
        self._ac.check_overlapping(overlapping)
        m, _ = self._ac.scan_host_batch([haystack.encode("utf-8")], overlapping, codepoints=True)
        return _tuples(m)

    def find_matches_as_strings(self, haystack: str, overlapping: bool = False):
        """-> list of matched patterns (src/lib.rs:253-272).

        With ``ascii_case_insensitive`` the list holds the matched text OF THE HAYSTACK (``"Hello"`` for the pattern
        ``"hello"``), never the stored pattern, whatever ``store_patterns`` says."""
        if not isinstance(haystack, str):
            raise TypeError("argument 'haystack': 'str' expected")
        self._ac.check_overlapping(overlapping)
        m, _ = self._ac.scan_host_batch([haystack.encode("utf-8")], overlapping, codepoints=True)
        if self._patterns is not None and not self._ac.ascii_case_insensitive:
            pats = self._patterns
            return [pats[i] for i in m[:, 1].tolist()]
        return [haystack[s:e] for s, e in zip(m[:, 2].tolist(), m[:, 3].tolist())]

    # ---- additions: batches ------------------------------------------------------
    def find_matches_as_indexes_batch(self, haystacks: Sequence[str], overlapping: bool = False):
        """One list of (pattern, start, end) per haystack, each exactly what
        ``find_matches_as_indexes`` returns for it."""
        self._ac.check_overlapping(overlapping)
        m, offs = self._ac.scan_host_batch([h.encode("utf-8") for h in haystacks], overlapping, codepoints=True)
        t = _tuples(m)
        return [t[offs[i]:offs[i + 1]] for i in range(len(haystacks))]

    def scan_device(self, data, offsets, overlapping: bool = False, **kw):
        """Device-resident UTF-8 batch -> (matches, match_offsets, total); code point indexes."""
        return self._ac.scan_device(data, offsets, overlapping, codepoints=True, **kw)

    def scan_host(self, data, offsets, overlapping: bool = False, **kw):
        """Host-resident UTF-8 batch (uint8 array + int64 offsets) -> host arrays (matches (k, 4), match_offsets (n + 1));
        code point indexes.  Copies and scans are pipelined (see _Automaton.scan_host)."""
        return self._ac.scan_host(data, offsets, overlapping, codepoints=True, **kw)


class BytesAhoCorasick:
    """Search for multiple pattern bytes against a bytes-like haystack
    (reference: src/lib.rs:342-363, 366-435).  No references to the patterns are kept.

    ``ascii_case_insensitive`` (keyword only): an ASCII letter in a pattern matches either case of that letter in the
    haystack; every other byte, 0x80-0xff included, must match exactly."""

    def __init__(self, patterns: Iterable, matchkind: MatchKind = MatchKind.Standard,
                 implementation: Optional[Implementation] = None, *, ascii_case_insensitive: bool = False):
        if not isinstance(matchkind, MatchKind):
            raise TypeError("matchkind must be a MatchKind")
        if implementation is not None and not isinstance(implementation, Implementation):
            raise TypeError("implementation must be an Implementation or None")
        _check_ascii_case_insensitive(ascii_case_insensitive)
        encoded = []
        for p in iter(patterns):
            b = _as_buffer_bytes(p)
            if len(b) == 0:
                raise ValueError("You passed in an empty pattern")
            encoded.append(b)
        self._ac = _Automaton(encoded, matchkind, implementation, ascii_case_insensitive)

    def find_matches_as_indexes(self, haystack, overlapping: bool = False):
        """-> list of (pattern index, start, end) in byte offsets (src/lib.rs:422-434)."""
        hay = _as_buffer_bytes(haystack)
        self._ac.check_overlapping(overlapping)
        m, _ = self._ac.scan_host_batch([hay], overlapping, codepoints=False)
        return _tuples(m)

    def find_matches_as_indexes_batch(self, haystacks: Sequence, overlapping: bool = False):
        self._ac.check_overlapping(overlapping)
        m, offs = self._ac.scan_host_batch([_as_buffer_bytes(h) for h in haystacks], overlapping, codepoints=False)
        t = _tuples(m)
        return [t[offs[i]:offs[i + 1]] for i in range(len(haystacks))]

    def scan_device(self, data, offsets, overlapping: bool = False, **kw):
        """Device-resident batch -> (matches, match_offsets, total); byte offsets."""
        return self._ac.scan_device(data, offsets, overlapping, codepoints=False, **kw)

    def scan_host(self, data, offsets, overlapping: bool = False, **kw):
        """Host-resident batch (uint8 array + int64 offsets) -> host arrays (matches (k, 4), match_offsets (n + 1));
        byte offsets.  Copies and scans are pipelined (see _Automaton.scan_host)."""
        return self._ac.scan_host(data, offsets, overlapping, codepoints=False, **kw)
