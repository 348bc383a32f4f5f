"""Test infrastructure for ASCII case-insensitive matching (acb_build_ex with ACB_ASCII_CASE_INSENSITIVE).

Two independent statements of the semantics, and the product's images as the interpreters read them:

* ``CrateReference`` -- the crate's construction (``AhoCorasickBuilder::ascii_case_insensitive(true)``) restated in
  plain Python: whenever the trie gets a NEW edge on an ASCII letter, the same state gets the edge on the opposite case
  of that letter, to the same child; failure links breadth first (a child reached by both cases is visited once) with
  the leftmost "dead state" rule; the find / find_overlapping loops of oracle/ac_oracle.c on that NFA.  Nothing is
  ever folded.  Slow: small inputs only.
* ``FoldedOracle`` -- the C oracle of the folded patterns run on the folded haystack, original pattern ids: the
  statement the product's implementation follows, fast enough for full-size batches.
* ``CiImage`` / ``CiSieveImage`` -- tests/image_interp.py's and tests/sieve_interp.py's interpreters on images built
  with the flag; the sieve interpreter folds the text the way the FOLD kernel does.
"""
from __future__ import annotations

import struct
from collections import deque

import numpy as np

from ahocorasick_rs_b200 import _capi
from oracle import Oracle
from tests import image_interp as ii
from tests import sieve_interp as si

KIND_IDS = {"Standard": 0, "LeftmostFirst": 1, "LeftmostLongest": 2}


def fold(b: bytes) -> bytes:
    """sieve.h ascii_fold on every byte: A-Z -> a-z, every other byte as it is"""
    return bytes(x | 0x20 if 0x41 <= x <= 0x5A else x for x in b)


def fold_array(a):
    a = np.asarray(a, dtype=np.uint8)
    return np.where((a >= 0x41) & (a <= 0x5A), a | np.uint8(0x20), a).astype(np.uint8)


def fold_str(s: str) -> str:
    return "".join(c.lower() if "A" <= c <= "Z" else c for c in s)


def _kind(kind):
    return KIND_IDS[kind] if isinstance(kind, str) else int(getattr(kind, "value", kind))


def _code_points(raw: bytes):
    b2c, cp = [None] * (len(raw) + 1), 0
    for i, x in enumerate(raw):
        if (x & 0xC0) != 0x80:
            b2c[i] = cp
            cp += 1
    b2c[len(raw)] = cp
    return b2c


# ---------------------------------------------------------------- the crate's construction, in Python
DEAD, FAIL, START = 0, 1, 2


class CrateReference:
    def __init__(self, patterns, kind=0, ascii_case_insensitive=True):
        self.kind = _kind(kind)
        pats = [bytes(p) for p in patterns]
        self.pat_len = [len(p) for p in pats]
        self.edges = [{}, {}, {}]
        self.fail = [START, START, START]
        self.matches = [[], [], []]
        for pid, p in enumerate(pats):
            assert p, "empty pattern"
            prev, dropped = START, False
            for b in p:
                # leftmost-first: an earlier pattern that is a proper prefix of this one always wins
                if self.kind == 1 and self.matches[prev]:
                    dropped = True
                    break
                nx = self.edges[prev].get(b)
                if nx is None:
                    nx = len(self.edges)
                    self.edges.append({})
                    self.fail.append(START)
                    self.matches.append([])
                    self.edges[prev][b] = nx
                    if ascii_case_insensitive and 0x61 <= (b | 0x20) <= 0x7A:
                        self.edges[prev][b ^ 0x20] = nx  # the opposite case, to the same child
                prev = nx
            if not dropped:
                self.matches[prev].append(pid)
        leftmost = self.kind != 0
        queue, seen = deque(), set()
        for b, c in sorted(self.edges[START].items()):
            if c not in seen:
                seen.add(c)
                queue.append(c)
                self.fail[c] = DEAD if (leftmost and self.matches[c]) else START
        while queue:
            s = queue.popleft()
            for b, c in sorted(self.edges[s].items()):
                if c in seen:
                    continue
                seen.add(c)
                queue.append(c)
                if leftmost and self.matches[c]:
                    self.fail[c] = DEAD
                    continue
                f = self.fail[s]
                while self._goto(f, b) == FAIL:
                    f = self.fail[f]
                f = self._goto(f, b)
                self.fail[c] = f
                self.matches[c] = self.matches[c] + self.matches[f]

    def _goto(self, s, b):
        if s == DEAD:
            return DEAD
        n = self.edges[s].get(b)
        if n is not None:
            return n
        return START if s == START else FAIL

    def _next(self, s, b):
        while True:
            n = self._goto(s, b)
            if n != FAIL:
                return n
            s = self.fail[s]

    def find(self, haystack: bytes, overlapping=False):
        """-> [(pid, start, end)] byte offsets, in the reference's iteration order"""
        hay, out = bytes(haystack), []
        if overlapping:
            assert self.kind == 0
            sid = START
            for at, b in enumerate(hay):
                sid = self._next(sid, b)
                out += [(pid, at + 1 - self.pat_len[pid], at + 1) for pid in self.matches[sid]]
            return out
        start = 0
        while start <= len(hay):
            sid, best = START, None
            for at in range(start, len(hay)):
                sid = self._next(sid, hay[at])
                if sid == DEAD:
                    break
                if self.matches[sid]:
                    best = (self.matches[sid][0], at + 1)
                    if self.kind == 0:
                        break
            if best is None:
                return out
            pid, end = best
            out.append((pid, end - self.pat_len[pid], end))
            start = end

    def find_str(self, haystack: str, overlapping=False):
        raw = haystack.encode("utf-8")
        b2c = _code_points(raw)
        return [(p, b2c[s], b2c[e]) for (p, s, e) in self.find(raw, overlapping)]


# ---------------------------------------------------------------- the fold statement, through the C oracle
class FoldedOracle:
    """Oracle(fold(P), kind) on fold(H): the same interface as oracle.Oracle for the calls the tests make."""

    def __init__(self, patterns, kind=0):
        self._o = Oracle([fold(bytes(p)) for p in patterns], kind)

    def find(self, haystack: bytes, overlapping=False):
        return self._o.find(fold(bytes(haystack)), overlapping)

    def find_str(self, haystack: str, overlapping=False):
        return self._o.find_str(fold_str(haystack), overlapping)

    def scan_batch(self, data, offsets, overlapping=False, codepoints=False, **kw):
        return self._o.scan_batch(fold_array(data), offsets, overlapping=overlapping, codepoints=codepoints, **kw)


# ---------------------------------------------------------------- the interpreters on case-insensitive images
class _BuildCaseInsensitive:
    """The library as an interpreter's constructor sees it: acb_build builds with ACB_ASCII_CASE_INSENSITIVE
    (acb_build_ex); every other entry point is the library's own."""

    def __init__(self, lib):
        self._lib = lib

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def acb_build(self, blob, offsets, n, kind, implementation, out):
        return self._lib.acb_build_ex(blob, offsets, n, kind, implementation, _capi.ACB_ASCII_CASE_INSENSITIVE, out)


class _CapiBuildingCaseInsensitive:
    def lib(self):
        return _BuildCaseInsensitive(_capi.lib())

    def __getattr__(self, name):
        return getattr(_capi, name)


def _construct(module, cls, obj, *args, **kw):
    """cls.__init__(obj, ...) with the interpreter module's library binding building case-insensitively"""
    saved = module._capi
    module._capi = _CapiBuildingCaseInsensitive()
    try:
        cls.__init__(obj, *args, **kw)
    finally:
        module._capi = saved
    obj._L = _capi.lib()


class CiImage(ii.Image):
    """The dense image built with the flag (ImageHeader.flags is word 11 of the header)."""

    def __init__(self, patterns, kind=0, implementation=-1):
        _construct(ii, ii.Image, self, patterns, kind, implementation)
        self.flags = struct.unpack_from("<I", self.raw.tobytes(), 44)[0]


class CiSieveImage(si.SieveImage):
    """The sieve image built with the flag (SieveHeader.flags is word 14); the scan reads folded text, as the FOLD
    kernel does."""

    def __init__(self, patterns, kind=0, bloom_bytes_max=200 * 1024, w_max=0):
        _construct(si, si.SieveImage, self, patterns, kind, bloom_bytes_max, w_max)
        self.flags = struct.unpack_from("<I", self.raw.tobytes(), 56)[0]

    def overlapping(self, data, offs):
        return super().overlapping(fold_array(data), offs)


def sieve_flags(image: si.SieveImage) -> int:
    return struct.unpack_from("<I", image.raw.tobytes(), 56)[0]


def image_flags(image: ii.Image) -> int:
    return struct.unpack_from("<I", image.raw.tobytes(), 44)[0]
