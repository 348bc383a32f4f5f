"""Synthetic inputs for the BASELINE.json configs (SURVEY.md 8d), seeded and
scalable.  Used by bench.py (full size) and the parity tests (scaled down).
Everything is generated on the host with numpy; nothing here reads
/root/reference (the two data fixtures it needs are committed under
ahocorasick_rs_b200/data/ by tests/golden/make_fixtures.py)."""
from __future__ import annotations

import os

import numpy as np

_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")   # the two input-data fixtures of config 2


def patterns_long():
    """PATTERNS_LONG of the reference benchmark (benchmarks/test_comparison.py:16-18): 4 244 names, 221 duplicates."""
    with open(os.path.join(_GOLDEN, "patterns_long.txt")) as f:
        return [line.strip() for line in f if line.strip()]


def haystack_template() -> str:
    with open(os.path.join(_GOLDEN, "haystack_template.txt"), encoding="utf-8") as f:
        return f.read()


def _csr(chunks):
    lens = np.fromiter((len(c) for c in chunks), dtype=np.int64, count=len(chunks))
    offs = np.zeros(len(chunks) + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    return np.frombuffer(b"".join(chunks), dtype=np.uint8), offs


def config1():
    """C1: README quickstart patterns, one 1 024-byte ASCII haystack (README.md:30-31 sentence repeated)."""
    sentence = "this is my first hello world. hello! "
    hay = (sentence * 40)[:1024]
    return ["hello", "world", "fish"], hay


def config2(n_haystacks=100_000, hay_bytes=4096, first_index=0):
    """C2: names patterns; haystack i = the benchmark's template line formatted with
    (PATTERNS_LONG[i % 4244] if i % 90 == 0 else "notaperson", i)
    (benchmarks/test_comparison.py:22-31), repeated to >= hay_bytes UTF-8 bytes, cut at a
    char boundary and space-padded to exactly hay_bytes.  Returns (patterns, data u8, offsets i64)."""
    pats = patterns_long()
    tmpl = haystack_template()
    out = np.full((n_haystacks, hay_bytes), 0x20, dtype=np.uint8)
    for r in range(n_haystacks):
        i = first_index + r
        name = pats[i % len(pats)] if i % 90 == 0 else "notaperson"
        line = tmpl.format(name, i).encode("utf-8")
        reps = -(-hay_bytes // len(line))
        buf = (line * reps)[: hay_bytes + 4]
        cut = hay_bytes
        while cut > 0 and (buf[cut] & 0xC0) == 0x80:  # never split a UTF-8 sequence
            cut -= 1
        out[r, :cut] = np.frombuffer(buf[:cut], dtype=np.uint8)
    offs = np.arange(n_haystacks + 1, dtype=np.int64) * hay_bytes
    return pats, out.reshape(-1), offs


_TOKEN_ALPHABET = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz0123456789_./:-", dtype=np.uint8)


def config3(n_patterns=10_000, n_lines=1_000_000, line_bytes=256, seed=3):
    """C3: distinct tokens, length U[4,16] over [a-z0-9_./:-]; log lines
    "<ts> <LEVEL> host<k> <tokens...>", 5 % of tokens drawn from the pattern set,
    space-padded to line_bytes.  Returns (patterns as bytes, data, offsets)."""
    rng = np.random.default_rng(seed)
    pats = set()
    while len(pats) < n_patterns:
        ln = int(rng.integers(4, 17))
        pats.add(bytes(_TOKEN_ALPHABET[rng.integers(0, len(_TOKEN_ALPHABET), size=ln)]))
    pats = sorted(pats)
    rng.shuffle(pats)
    levels = [b"INFO", b"WARN", b"ERROR", b"DEBUG"]
    out = np.full((n_lines, line_bytes), 0x20, dtype=np.uint8)
    # draw all randomness in bulk, assemble per line
    n_tok = 24
    tok_len = rng.integers(3, 13, size=(n_lines, n_tok))
    tok_is_pat = rng.random((n_lines, n_tok)) < 0.05
    tok_pat = rng.integers(0, n_patterns, size=(n_lines, n_tok))
    tok_chars = _TOKEN_ALPHABET[rng.integers(0, len(_TOKEN_ALPHABET), size=(n_lines, n_tok, 12))]
    lvl = rng.integers(0, 4, size=n_lines)
    host = rng.integers(0, 512, size=n_lines)
    for r in range(n_lines):
        parts = [b"2026-09-24T05:%02d:%02d.%03dZ" % (r // 60000 % 60, r // 1000 % 60, r % 1000), levels[lvl[r]],
                 b"host%d" % host[r]]
        used = sum(len(p) for p in parts) + len(parts)
        for t in range(n_tok):
            tok = pats[tok_pat[r, t]] if tok_is_pat[r, t] else bytes(tok_chars[r, t, : tok_len[r, t]])
            if used + len(tok) + 1 > line_bytes:
                break
            parts.append(tok)
            used += len(tok) + 1
        line = b" ".join(parts)
        out[r, : len(line)] = np.frombuffer(line, dtype=np.uint8)
    offs = np.arange(n_lines + 1, dtype=np.int64) * line_bytes
    return pats, out.reshape(-1), offs


def random_lowercase_patterns(n, lo, hi, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(lo, hi + 1, size=n)
    chars = rng.integers(97, 123, size=int(lens.sum()), dtype=np.uint8).astype(np.uint8)
    offs = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    raw = chars.tobytes()
    return [raw[offs[i]:offs[i + 1]] for i in range(n)]


def config4(n_patterns=100_000, hay_bytes=1 << 32, seed=4):
    """C4: n_patterns patterns, length U[5,8] over a-z (duplicates allowed); ONE haystack,
    i.i.d. uniform a-z.  Returns (patterns as bytes, data)."""
    pats = random_lowercase_patterns(n_patterns, 5, 8, seed)
    rng = np.random.default_rng(seed + 1000)
    data = rng.integers(97, 123, size=hay_bytes, dtype=np.uint8).astype(np.uint8)
    return pats, data


def config5(n_patterns=50_000, n_haystacks=16_777_216, hay_bytes=4096, seed=5, shard=0):
    """C5: n_patterns patterns, length U[5,12] over a-z; a batch of uniform a-z haystacks
    (one shard of it: the seed is offset by `shard`).  Returns (patterns, data, offsets)."""
    pats = random_lowercase_patterns(n_patterns, 5, 12, seed)
    rng = np.random.default_rng(seed + 1000 + shard)
    data = rng.integers(97, 123, size=n_haystacks * hay_bytes, dtype=np.uint8).astype(np.uint8)
    offs = np.arange(n_haystacks + 1, dtype=np.int64) * hay_bytes
    return pats, data, offs


def recase(data, frac=0.5, seed=0):
    """A copy of `data` (uint8) in which a seeded fraction `frac` of the ASCII letters has the other case: the input
    of the case-insensitive tests and timings (the matches of a case-insensitive automaton do not change).  Works in
    slices of 64 MiB so that a full-size batch needs no more than twice its own size."""
    data = np.asarray(data, dtype=np.uint8)
    out = np.empty_like(data)
    rng = np.random.default_rng(seed)
    flat_in, flat_out = data.reshape(-1), out.reshape(-1)
    thresh = int(round(frac * 65536))
    step = 64 << 20
    for a in range(0, flat_in.size, step):
        x = flat_in[a:a + step]
        letter = ((x | np.uint8(0x20)) - np.uint8(0x61)) < 26   # uint8 arithmetic: bytes below 'a' wrap above 26
        flip = letter & (rng.integers(0, 65536, size=x.size, dtype=np.uint16) < thresh)
        flat_out[a:a + step] = x ^ (flip.astype(np.uint8) << np.uint8(5))
    return out


def ragged(n_haystacks=1000, max_len=700, alphabet=b"abc", seed=7, empty_frac=0.05):
    """Ragged batch with empty haystacks, for edge-case parity."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, max_len + 1, size=n_haystacks)
    lens[rng.random(n_haystacks) < empty_frac] = 0
    al = np.frombuffer(alphabet, dtype=np.uint8)
    data = al[rng.integers(0, len(al), size=int(lens.sum()))]
    offs = np.zeros(n_haystacks + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    return data.astype(np.uint8), offs
