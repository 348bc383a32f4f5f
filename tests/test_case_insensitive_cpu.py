"""CPU tests of ASCII case-insensitive matching (acb_build_ex with ACB_ASCII_CASE_INSENSITIVE).

The semantics: results(P, H, ci) == results(fold(P), fold(H)) with the ORIGINAL pattern ids, lengths and positions,
fold = A-Z -> a-z, every other byte as it is.  Three independent statements of it are checked against each other --
the crate's construction restated in Python (opposite-case trie edges, nothing folded: tests/case_insensitive_ref.py),
the oracle on folded inputs, and the brute-force specification on folded inputs -- and then the product's images,
through the image and sieve interpreters, on the UNFOLDED haystacks."""
import ctypes as C
import struct

import numpy as np
import pytest

from oracle import Oracle
from tests import image_interp as ii
from tests.case_insensitive_ref import CiImage, CiSieveImage, CrateReference, FoldedOracle, fold, image_flags, sieve_flags
from tests.sieve_interp import SieveImage, scan
from tests.spec_bruteforce import spec_find
from ahocorasick_rs_b200 import AhoCorasick, BytesAhoCorasick, MatchKind, _capi, workloads as W

KINDS = ["Standard", "LeftmostFirst", "LeftmostLongest"]
# the fold's edges: '@' 'A' 'Z' '[' '`' 'a' 'z' '{', and high bytes whose low seven bits look like letters
BOUNDARY = b"@AZ[`az{" + bytes([0xC1, 0xE1, 0xFA])


def random_case(rng, alphabet, n_pat, lo, hi, n_hay, max_hay):
    al = np.frombuffer(alphabet, dtype=np.uint8)
    pats = [bytes(al[rng.integers(0, len(al), size=int(rng.integers(lo, hi + 1)))]) for _ in range(n_pat)]
    pats += [p.swapcase() for p in pats[:3]]  # patterns that differ only in case: distinct ids
    lens = rng.integers(0, max_hay + 1, size=n_hay)
    data = al[rng.integers(0, len(al), size=int(lens.sum()))].astype(np.uint8)
    offs = np.zeros(n_hay + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    return pats, data, offs


def oracle_rows(orc, data, offs, overlapping):
    _, _, rec = orc.scan_batch(np.asarray(data, dtype=np.uint8), np.asarray(offs, dtype=np.int64), overlapping=overlapping)
    return [tuple(int(x) for x in r) for r in rec]


# ---------------------------------------------------------------- the semantics, three ways
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("alphabet", [b"aAbB", BOUNDARY, b"aAzZ@[`{", b"xyXY\xc1\xe1"])
def test_oracle_semantics(kind, alphabet):
    rng = np.random.default_rng(len(alphabet) * 7 + KINDS.index(kind))
    for rep in range(6):
        pats, data, _ = random_case(rng, alphabet, 10, 1, 4, 1, 0)
        hay = bytes(np.frombuffer(alphabet, dtype=np.uint8)[rng.integers(0, len(alphabet), size=300)])
        ci = CrateReference(pats, kind)
        fp, fh = [fold(p) for p in pats], fold(hay)
        for overlapping in ([False, True] if kind == "Standard" else [False]):
            got = ci.find(hay, overlapping)
            assert got == Oracle(fp, kind).find(fh, overlapping)
            assert got == FoldedOracle(pats, kind).find(hay, overlapping)
            assert got == spec_find(fp, fh, kind, overlapping)
            # the Python restatement of the crate's construction, case-sensitive, is the C oracle
            assert CrateReference(pats, kind, ascii_case_insensitive=False).find(hay, overlapping) == Oracle(pats, kind).find(hay, overlapping)
    # nothing outside A-Z / a-z is folded
    assert CrateReference([b"\xc1"], "Standard").find(b"\xe1\xc1") == [(0, 1, 2)]
    assert CrateReference([b"@"], "Standard").find(b"`@") == [(0, 1, 2)]


def test_case_only_duplicates():
    pats = [b"abc", b"ABC", b"aBc", b"bc"]
    hay = b"xAbC"
    for ref in (CrateReference, FoldedOracle):
        assert ref(pats, "Standard").find(hay, True) == [(0, 1, 4), (1, 1, 4), (2, 1, 4), (3, 2, 4)]
        assert ref(pats, "LeftmostFirst").find(hay) == [(0, 1, 4)]
        assert ref(pats, "LeftmostLongest").find(hay) == [(0, 1, 4)]


# ---------------------------------------------------------------- the images
def test_sieve_image_is_the_image_of_the_folded_patterns():
    rng = np.random.default_rng(3)
    for alphabet, lo, hi in ((b"aAbBcC", 2, 9), (BOUNDARY, 1, 5), (b"Hello, World", 5, 14)):
        pats, _, _ = random_case(rng, alphabet, 60, lo, hi, 1, 0)
        ci = CiSieveImage(pats, 0)
        cs = SieveImage([fold(p) for p in pats], 0)
        assert ci.flags == _capi.ACB_ASCII_CASE_INSENSITIVE and sieve_flags(cs) == 0
        a, b = ci.raw.copy(), cs.raw.copy()
        a[14 * 4:15 * 4] = 0  # SieveHeader.flags
        assert np.array_equal(a, b)


def test_dense_image_folds_its_columns():
    rng = np.random.default_rng(4)
    for alphabet in (b"aAbBcC", BOUNDARY, b"ab01", b"0123"):
        pats, _, _ = random_case(rng, alphabet, 40, 1, 6, 1, 0)
        for kind in range(3):
            ci = CiImage(pats, kind)
            cs = ii.Image([fold(p) for p in pats], kind)
            assert ci.flags == 1 and image_flags(cs) == 0
            # the same states and match lists; the same transition for every byte (the column layouts may differ: the
            # folded list alone may take the arithmetic column map)
            assert ci.n_states == cs.n_states and np.array_equal(ci.match_off, cs.match_off)
            assert np.array_equal(ci.match_pid, cs.match_pid)
            for b in range(256):
                assert np.array_equal(ci.trans[:, ci.col(b)], cs.trans[:, cs.col(fold(bytes([b]))[0])])
            if any(x in b"abcdefghijklmnopqrstuvwxyz" for p in pats for x in fold(p)):
                assert ci.col_mode == 1  # the arithmetic column map cannot fold
                for b in range(0x41, 0x5B):
                    assert ci.colmap[b] == ci.colmap[b | 0x20]


def test_byte_indexed_table_folds():
    im = CiImage([b"Hello", b"hELP", b"World", b"wor", b"~x"], 0)
    n = im._L.acb_hot_bytes(im._h, 40)
    buf = np.zeros(n, dtype=np.uint8)
    assert im._L.acb_hot_build(im._h, None, 40, buf.ctypes.data, n) == 0
    magic, rows, n_cols, n_states, o_t, o_h2f, o_f2h, total, rows128, visited, o_t128 = struct.unpack_from("<4I4Q2IQ", buf.tobytes()[:64])
    assert rows128 == rows > 0
    t = buf[o_t:o_t + 2 * (rows + 1) * n_cols].view(np.uint16).reshape(rows + 1, n_cols) // (2 * n_cols)
    t128 = buf[o_t128:o_t128 + 2 * (rows128 + 1) * 128].view(np.uint16).reshape(rows128 + 1, 128) // 256
    for b in range(128):
        assert np.array_equal(t128[:, b], t[:, im.col(b)])
        assert np.array_equal(t128[:, b], t128[:, fold(bytes([b]))[0]])


# ---------------------------------------------------------------- the scans' logic on unfolded text
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_image_interpreter_matches_oracle(kind):
    rng = np.random.default_rng(50 + kind)
    for alphabet in (b"aAbB", BOUNDARY):
        pats, data, offs = random_case(rng, alphabet, 12, 1, 5, 8, 200)
        im = CiImage(pats, kind)
        orc = FoldedOracle(pats, kind)
        for overlapping in ([False, True] if kind == 0 else [False]):
            exp = oracle_rows(orc, data, offs, overlapping)
            crate = CrateReference(pats, kind)
            assert exp == [(h, p, s, e) for h in range(len(offs) - 1)
                           for (p, s, e) in crate.find(bytes(data[offs[h]:offs[h + 1]]), overlapping)]
            assert ii.emulate_plain(im, data, offs, overlapping) == exp
            for H in (3, 40):
                assert ii.emulate_scan(im, data, offs, overlapping, H=H, base_addr=5, segment_bytes=64) == exp


def test_image_interpreter_code_points():
    pats = ["Straße", "É", "é", "ÄBC", "abc"]
    text = "STRAßE straße StraSSe É é ÄbC äbc ABC" * 3
    bp = [p.encode() for p in pats]
    im = CiImage(bp, 0)
    raw = text.encode()
    exp = CrateReference(bp, 0).find_str(text, True)
    assert exp == FoldedOracle(bp, 0).find_str(text, True)
    assert ii.find(im, raw, True, cp=True) == exp
    assert ii.find_staged(im, raw, True, cp=True, H=5, segment_bytes=64) == exp
    assert [text[s:e] for (_, s, e) in exp][:4] == ["STRAßE", "straße", "É", "é"]


@pytest.mark.parametrize("w_max", [1, 2, 3, 4, 5, 6, 7, 8])
def test_sieve_interpreter_matches_oracle(w_max):
    rng = np.random.default_rng(90 + w_max)
    pats, data, offs = random_case(rng, b"aAbB@[`{", 50, 8, 12, 6, 200)
    img = CiSieveImage(pats, 0, w_max=w_max)
    assert img.W == w_max
    for kind in (0, 1, 2):
        img.kind = kind  # the image does not depend on the kind: only the selection does
        orc = FoldedOracle(pats, kind)
        for overlapping in ([False, True] if kind == 0 else [False]):
            assert scan(img, data, offs, overlapping) == oracle_rows(orc, data, offs, overlapping)


# ---------------------------------------------------------------- the C ABI and the Python surface
def test_build_ex_flags():
    L = _capi.lib()
    blob = np.frombuffer(b"abBc", dtype=np.uint8)
    offs = np.array([0, 2, 4], dtype=np.uint64)
    for flags in (0, _capi.ACB_ASCII_CASE_INSENSITIVE):
        h = C.c_void_p()
        assert L.acb_build_ex(blob.ctypes.data, offs.ctypes.data, 2, 0, -1, flags, C.byref(h)) == _capi.ACB_OK
        assert L.acb_build_flags(h) == flags
        L.acb_free(h)
    h = C.c_void_p()
    assert L.acb_build(blob.ctypes.data, offs.ctypes.data, 2, 0, -1, C.byref(h)) == _capi.ACB_OK
    assert L.acb_build_flags(h) == 0
    L.acb_free(h)
    for bad in (2, 0x80000000, 3):
        h = C.c_void_p()
        assert L.acb_build_ex(blob.ctypes.data, offs.ctypes.data, 2, 0, -1, bad, C.byref(h)) == _capi.ACB_EINVAL
        assert "flag" in _capi.last_error()


def test_python_keyword():
    assert AhoCorasick(["Hello"], ascii_case_insensitive=True)._ac.ascii_case_insensitive
    assert not AhoCorasick(["Hello"])._ac.ascii_case_insensitive
    assert BytesAhoCorasick([b"Hello"], ascii_case_insensitive=True)._ac.ascii_case_insensitive
    for bad in (1, 0, "yes", None):
        with pytest.raises(TypeError):
            AhoCorasick(["Hello"], ascii_case_insensitive=bad)
        with pytest.raises(TypeError):
            BytesAhoCorasick([b"Hello"], ascii_case_insensitive=bad)
    with pytest.raises(TypeError):  # keyword only: not a fifth / fourth positional argument
        AhoCorasick(["Hello"], MatchKind.Standard, None, None, True)
    with pytest.raises(TypeError):
        BytesAhoCorasick([b"Hello"], MatchKind.Standard, None, True)


def test_recase():
    data = np.frombuffer(b"Hello, World! @[`{ az AZ \xc3\xa1\xc1\xe1" * 50, dtype=np.uint8)
    r = W.recase(data, 0.5, 1)
    assert fold(r.tobytes()) == fold(data.tobytes()) and r.tobytes() != data.tobytes()
    assert np.array_equal(r, W.recase(data, 0.5, 1))  # seeded
    assert W.recase(data, 1.0, 0).tobytes() == data.tobytes().swapcase()
    assert W.recase(data, 0.0, 0).tobytes() == data.tobytes()
