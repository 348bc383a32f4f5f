"""GPU tests (-m gpu) of ASCII case-insensitive matching: every kernel family against the oracle of the folded patterns
on the folded haystack (FoldedOracle), and where inputs are small enough also against the crate's construction
restated in Python (CrateReference: opposite-case trie edges, nothing folded), on haystacks whose letters have been
re-cased at random.  The sieve's text fold (SWAR, four bytes per word) is exercised with every byte value at every
offset of a 16-byte chunk, for every primary window size."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from ahocorasick_rs_b200 import AhoCorasick, BytesAhoCorasick, Implementation, MatchKind, _capi, workloads as W
from tests.case_insensitive_ref import CrateReference, FoldedOracle

KINDS = [MatchKind.Standard, MatchKind.LeftmostFirst, MatchKind.LeftmostLongest]


def set_kernel(kernel=0, hot_rows=0, segment_bytes=0, table=0):
    _capi.set_tuning(kernel, hot_rows, segment_bytes, table)


@pytest.fixture(params=["sieve", "sieve-small-tasks", "staged-compact-table", "staged-byte-table-tiny", "plain",
                        "global-small-segments", "staged-two-per-lane-tiny"])
def kernel(request):
    set_kernel(*{
        "sieve": (5,),                            # position-parallel filter + exact verification (the FOLD variant)
        "sieve-small-tasks": (5, 0, 512),         # one 512-byte window per task: the edge loads everywhere
        "staged-compact-table": (2, 0, 0, 1),     # hot rows in shared memory, column-indexed (colmap folds)
        "staged-byte-table-tiny": (2, 7, 256, 2), # byte-indexed table (built through colmap), 7 rows, 256-byte segments
        "plain": (1,),                            # one thread per haystack, table in global memory
        "global-small-segments": (4, 0, 128),     # segments from global memory, repair everywhere
        "staged-two-per-lane-tiny": (3, 6, 128, 1),
    }[request.param])
    yield request.param
    set_kernel(0)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def check_batch(pats_bytes, kind, data, offs, overlapping=False, codepoints=False, implementation=None):
    orc = FoldedOracle(pats_bytes, kind.name)
    total, counts, rec = orc.scan_batch(data, offs, overlapping=overlapping, codepoints=codepoints)
    if codepoints:
        ac = AhoCorasick([p.decode() for p in pats_bytes], kind, implementation=implementation, ascii_case_insensitive=True)
    else:
        ac = BytesAhoCorasick(pats_bytes, kind, implementation=implementation, ascii_case_insensitive=True)
    m, moffs, gtotal = ac.scan_device(dev(data), dev(offs), overlapping)
    assert gtotal == total
    assert np.array_equal(np.diff(moffs.cpu().numpy()), counts.astype(np.int64))
    assert np.array_equal(m.cpu().numpy().view(np.uint32), rec)
    return total


@pytest.mark.parametrize("kind", KINDS, ids=lambda k: k.name)
def test_ragged_small_alphabet(kind, kernel):
    rng = np.random.default_rng(41)
    al = np.frombuffer(b"aAbBcC", dtype=np.uint8)
    pats = sorted({bytes(al[rng.integers(0, 6, size=rng.integers(1, 6))]) for _ in range(40)})
    pats += [p.swapcase() for p in pats[:3]] + pats[:2]  # case-only and exact duplicates: distinct ids
    data, offs = W.ragged(3000, 300, b"aAbBcC@[`{", seed=42)
    n = check_batch(pats, kind, data, offs)
    assert n > 1000
    if kind == MatchKind.Standard:
        check_batch(pats, kind, data, offs, overlapping=True)


@pytest.mark.parametrize("kind", KINDS, ids=lambda k: k.name)
def test_config2_shape_recased(kind, kernel):
    pats, data, offs = W.config2(1500)
    n = check_batch([p.encode() for p in pats], kind, W.recase(data, 0.5, 2), offs, codepoints=True,
                    implementation=Implementation.DFA)
    assert n > 50


@pytest.mark.parametrize("kind", KINDS, ids=lambda k: k.name)
def test_config3_shape_recased(kind, kernel):
    pats, data, offs = W.config3(n_patterns=2000, n_lines=4000)
    n = check_batch(pats, kind, W.recase(data, 0.5, 3), offs)
    assert n > 1000


def test_config5_shape_recased(kernel):
    pats, data, offs = W.config5(n_patterns=20000, n_haystacks=512, hay_bytes=4096)
    check_batch(pats, MatchKind.Standard, W.recase(data, 0.5, 5), offs)


# ---------------------------------------------------------------- the sieve's fold: every byte at every chunk offset
BLOCKS = [bytes(np.roll(np.arange(256, dtype=np.uint8), -o)) for o in range(16)]  # byte v at offsets (v - o) % 16


@pytest.mark.parametrize("w", [1, 2, 3, 4, 5, 6, 7, 8])
def test_sieve_fold_every_byte_every_offset(w):
    # patterns at the fold's boundaries, at least 8 bytes long so that w decides the primary window
    pats = [b"@abcdefg", b"`ABCDEFG", b"xyz[\\]^_", b"TUVWXYZ{", b"stuvwxyz", b"\xc0\xc1\xc2\xc3\xc4\xc5\xc6\xc7",
            b"\xe0\xe1\xe2\xe3\xe4\xe5\xe6\xe7", b"\xe1\xe2\xe3\xe4\xe5\xe6\xe7\xe8", b"?@ABCDEFGH", b"YZ[\\]^_`abcd"]
    rng = np.random.default_rng(70 + w)
    hays = []
    for o in range(16):
        block = BLOCKS[o]
        hays.append(block + W.recase(np.frombuffer(block, dtype=np.uint8), 0.5, o).tobytes())
        hays.append(block[o:o + 37])  # short haystacks: a task edge in nearly every window
    data = np.frombuffer(b"".join(hays), dtype=np.uint8)
    offs = np.zeros(len(hays) + 1, dtype=np.int64)
    np.cumsum([len(h) for h in hays], out=offs[1:])
    for segment in (0, 512):
        set_kernel(5, 0, segment)
        try:
            for kind in KINDS:
                orc = FoldedOracle(pats, kind.name)
                ac = BytesAhoCorasick(pats, kind, ascii_case_insensitive=True)
                ac._ac.SIEVE_W_MAX = w
                for shift in (0, 3):  # a buffer that does not start on the task grid
                    buf = np.concatenate([rng.integers(0, 256, size=shift).astype(np.uint8), data])
                    for overlapping in ([False, True] if kind == MatchKind.Standard else [False]):
                        total, counts, rec = orc.scan_batch(data, offs, overlapping=overlapping)
                        m, mo, t = ac.scan_device(dev(buf), dev(offs + shift), overlapping)
                        assert ac._ac.last_stats["window"] == w
                        assert t == total and np.array_equal(m.cpu().numpy().view(np.uint32), rec), (kind, overlapping, shift)
                if kind == MatchKind.Standard:
                    assert total > 16 * 8
        finally:
            set_kernel(0)


# ---------------------------------------------------------------- the str API, the host paths, the windows
@pytest.mark.parametrize("store_patterns", [True, False])
def test_str_api_on_non_ascii_text(store_patterns):
    pats = ["straße", "É", "é", "ÄBC", "hello", "wORLD"]
    text = "HELLO Straße STRASSE É é ÄbC äbc Wörld World ☃hello☃ " * 20
    ac = AhoCorasick(pats, store_patterns=store_patterns, ascii_case_insensitive=True)
    exp = CrateReference([p.encode() for p in pats], "Standard").find_str(text, True)
    assert ac.find_matches_as_indexes(text, overlapping=True) == exp
    strs = ac.find_matches_as_strings(text, overlapping=True)
    assert strs == [text[s:e] for (_, s, e) in exp]
    assert strs[:5] == ["HELLO", "Straße", "É", "é", "ÄbC"]  # the haystack's text, not the stored pattern
    lf = AhoCorasick(pats, MatchKind.LeftmostFirst, store_patterns=store_patterns, ascii_case_insensitive=True)
    assert lf.find_matches_as_strings("xHeLLo World") == ["HeLLo", "World"]
    assert lf.find_matches_as_indexes("☃HeLLo") == [(4, 1, 6)]


def test_small_call_host_runs_and_windows(monkeypatch):
    from ahocorasick_rs_b200 import matcher
    rng = np.random.default_rng(51)
    pats = sorted({bytes(rng.integers(97, 101, size=rng.integers(2, 9)).astype(np.uint8)) for _ in range(200)})
    # (a) the small-call path: one haystack per call
    for kind in KINDS:
        orc, crate = FoldedOracle(pats, kind.name), CrateReference(pats, kind.name)
        ac = BytesAhoCorasick(pats, kind, ascii_case_insensitive=True)
        for n in (0, 1, 7, 1000, 100_000):
            hay = W.recase(rng.integers(97, 101, size=n).astype(np.uint8), 0.5, n).tobytes()
            got = ac.find_matches_as_indexes(hay)
            assert got == orc.find(hay)
            if n <= 1000:
                assert got == crate.find(hay)
    # (b) scan_host in several runs
    data, offs = W.ragged(400, 3000, b"abcdABCD", seed=52)
    for kind in KINDS:
        orc = FoldedOracle(pats, kind.name)
        total, counts, rec = orc.scan_batch(data, offs)
        ac = BytesAhoCorasick(pats, kind, ascii_case_insensitive=True)
        hm, hmo = ac.scan_host(data, offs, chunk_bytes=100_000)
        assert np.array_equal(hm, rec) and np.array_equal(np.diff(hmo), counts.astype(np.int64))
        # (c) the windows / runs path of buffers above one call's range
        monkeypatch.setattr(matcher._Automaton, "WINDOW_BYTES", 50_000)
        m1, o1, t1 = ac.scan_device(dev(data), dev(offs))
        monkeypatch.undo()
        assert t1 == total and np.array_equal(m1.cpu().numpy(), rec.astype(np.int64))
    hay = W.recase(rng.integers(97, 101, size=400_000).astype(np.uint8), 0.5, 9)
    ac = BytesAhoCorasick(pats, ascii_case_insensitive=True)
    monkeypatch.setattr(matcher._Automaton, "WINDOW_BYTES", 30_001)
    got = ac.find_matches_as_indexes(hay.tobytes(), overlapping=True)
    non = {kind: BytesAhoCorasick(pats, kind, ascii_case_insensitive=True).find_matches_as_indexes(hay.tobytes()) for kind in KINDS}
    monkeypatch.undo()
    assert got == FoldedOracle(pats, "Standard").find(hay.tobytes(), overlapping=True)
    for kind in KINDS:
        assert non[kind] == FoldedOracle(pats, kind.name).find(hay.tobytes()), kind


@pytest.mark.parametrize("engine", ["auto", "sieve"])
def test_config2_full_size_recased_vs_oracle(engine):
    pats, data, offs = W.config2(100_000)
    data = W.recase(data, 0.5, 20)
    pb = [p.encode() for p in pats]
    total, counts, rec = FoldedOracle(pb, "Standard").scan_batch(data, offs, codepoints=True)
    set_kernel(5 if engine == "sieve" else 0)
    try:
        ac = AhoCorasick(pats, implementation=Implementation.DFA, ascii_case_insensitive=True)
        m, mo, t = ac.scan_device(dev(data), dev(offs))
        assert t == total and total > 7000
        assert np.array_equal(m.cpu().numpy().view(np.uint32), rec)
        assert np.array_equal(np.diff(mo.cpu().numpy()), counts.astype(np.int64))
    finally:
        set_kernel(0)
