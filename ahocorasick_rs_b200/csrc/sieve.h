// sieve.h -- the "sieve" image: a position-parallel form of the matcher.
//
// The dense-table kernels (scan_staged / scan_global) walk an automaton: one
// DEPENDENT table load per haystack byte.  That chain is what bounds them (41 %
// of HBM bandwidth on lock-step text, 2 % on dense pattern sets whose states live
// in L2).  The sieve turns the problem around, using the fact that the set of
// patterns ending at a position depends only on the bytes before it
// (SURVEY.md App. B.1):
//
//   1. every byte position e is tested INDEPENDENTLY: the W bytes ending at e are
//      hashed and looked up in a sparse bitmap of the patterns' W-byte suffixes that
//      lives in shared memory (the "primary" filter: one bit per suffix, one probe) --
//      no chain, one shared-memory load per byte;
//   2. the few survivors are checked against a second, denser Bloom filter on chip
//      that holds the W-byte suffixes again (other hash functions), the longer
//      suffixes as far as its bit budget goes, and a mark for every complete
//      pattern: they walk back towards the pattern start through it, so that on
//      sparse pattern sets (names in text) almost nothing but true matches leaves
//      the SM;
//   3. what is left is verified EXACTLY against a reverse trie in global memory /
//      L2: a hash table maps the W-byte suffix to its trie node, the walk continues
//      byte by byte towards the pattern start, and the deepest terminal node on
//      the path names every pattern that ends at e, longest first (a link chain
//      through the shorter ones) -- the reference's order at one end position.
//
// That yields the OVERLAPPING match list (reference: try_find_overlapping_iter,
// src/lib.rs:52-54) in its exact order.  The non-overlapping lists of all three
// match kinds (try_find_iter, src/lib.rs:58-60) are a greedy selection from it
// (SURVEY.md 8c: "among occurrences with start >= s pick the minimum of ..."),
// done per haystack by the epilogue.  Nothing here depends on the match kind.
//
// The functions below are shared by the host builder (sieve.cpp) and the kernel
// (scan_sieve.cuh): both sides must hash identically.
#pragma once
#include <cstdint>
#include <vector>

#if defined(__CUDACC__)
#define ACB_HD __host__ __device__ __forceinline__
#else
#define ACB_HD inline
#endif

namespace acb {

constexpr uint32_t kSieveMagic = 0x32424341u;  // "ACB2"
constexpr uint32_t kSieveMaxW = 8;             // the primary window: W = min(shortest pattern, 8) bytes at most
constexpr uint32_t kSieveMaxLevel = 16;        // deepest suffix length the on-chip filter may hold (the kernel keeps 16 bytes of history on chip)
constexpr uint32_t kSieveNoNode = 0xffffffffu;
// geometry of the scan kernel's shared memory that the builder sizes the filters against (scan_sieve.cuh asserts both)
constexpr uint32_t kSieveScanWarps = 24;       // warps per CTA
constexpr uint32_t kSieveRingSlotBytes = 576;  // one window of text in a warp's ring

// ---- hashing --------------------------------------------------------------------------------
// A window of d bytes ending at position e is identified by a 32-bit value x_d:
//   x_W   = lo' + hi' * kMixHi   with (hi:lo) the 8 bytes ending at e, little endian (the byte at e-1 is the top
//           byte of lo), cut down to the newest W bytes: W <= 4: lo' = lo >> 8(4-W), hi' = 0;
//           W > 4: lo' = lo, hi' = hi >> 8(8-W);
//   x_d+1 = step(x_d, byte at e-d-1).
constexpr uint32_t kMixHi = 0x9E3779B1u;
constexpr uint32_t kMulA = 0x85EBCA6Bu;   // the primary bitmap's probe (fast path)
constexpr uint32_t kMulB = 0xC2B2AE35u;   // secondary filter, first probe
constexpr uint32_t kMulC = 0x27D4EB2Fu;   // secondary filter, second probe
constexpr uint32_t kSaltTerm = 0x5BD1E995u;  // x ^ kSaltTerm: "a complete pattern of this length ends here"
constexpr uint32_t kMulSlot = 0x7FEB352Du;   // hash table slot

// from the cut-down words (lo', hi'): what the hash table stores as a slot's key
ACB_HD uint32_t sieve_x_packed(uint32_t lo_cut, uint32_t hi_cut) { return lo_cut + hi_cut * kMixHi; }
ACB_HD uint32_t sieve_x(uint32_t lo, uint32_t hi, uint32_t W) {
    if (W <= 4) return lo >> (8u * (4u - W));
    return lo + (hi >> (8u * (8u - W))) * kMixHi;
}
ACB_HD uint32_t sieve_step(uint32_t x, uint32_t byte) {
    x = (x + byte + 1u) * kMixHi;
    return x ^ (x >> 15);
}
// probe i of x in a filter of n_words 32-bit words: the word comes from the top bits of the product, the bit from its low bits
ACB_HD uint32_t sieve_mulhi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
ACB_HD uint32_t sieve_probe_word(uint32_t p, uint32_t n_words) { return sieve_mulhi(p, n_words); }
ACB_HD uint32_t sieve_probe_bit(uint32_t p) { return p & 31u; }

// ---- ASCII case folding ---------------------------------------------------------------------
// Built with kAsciiCaseInsensitive, the image holds the FOLDED patterns and the scan folds the text before it hashes or
// compares a byte: an ASCII upper-case letter (0x41-0x5A) becomes its lower-case form (| 0x20), every other byte --
// bytes >= 0x80 included, so no UTF-8 sequence changes -- stays as it is.
constexpr uint32_t kAsciiCaseInsensitive = 1u;  // = ACB_ASCII_CASE_INSENSITIVE (include/acb200.h)
ACB_HD uint32_t ascii_fold(uint32_t b) { return b - 0x41u < 26u ? (b | 0x20u) : b; }
// the same for the four bytes of a word: a byte is upper case when its top bit is clear and its low seven bits are
// >= 0x41 (t + 0x3f carries into bit 7) and not >= 0x5b (t + 0x25 does not); no sum carries into the next byte
ACB_HD uint32_t ascii_fold4(uint32_t w) {
    const uint32_t t = w & 0x7f7f7f7fu;
    const uint32_t upper = (t + 0x3f3f3f3fu) & ~(t + 0x25252525u) & ~w & 0x80808080u;
    return w | (upper >> 2);
}

// ---- the image ------------------------------------------------------------------------------
// All offsets are bytes from the start of the image, 16-byte aligned.
struct SieveHeader {
    uint32_t magic;
    uint32_t W;            // primary window, 1..8 bytes (<= shortest pattern)
    uint32_t last_level;   // deepest suffix length present in the filter (W <= last_level <= 16)
    uint32_t n_probes;     // probes per key in the secondary filter (1..2)
    uint32_t bloom_words;  // 32-bit words of both filters together: [primary: prim_words][secondary: bloom_words - prim_words]
    uint32_t ht_mask;      // hash table slots - 1 (a power of two)
    uint32_t n_nodes;
    uint32_t n_pids;
    uint32_t max_pat_len;
    uint32_t min_pat_len;
    uint32_t n_keys;       // distinct W-byte suffixes
    uint32_t n_filter_entries;
    uint32_t prim_words;   // the primary bitmap: ONE bit per W-byte suffix, kept sparse (the fast path tests only this)
    uint32_t term_levels;  // bit d: some pattern is exactly d bytes long (d <= 16): only those levels carry end marks
    uint32_t flags;        // kAsciiCaseInsensitive: built from the folded patterns, the scan folds the text
    uint32_t pad2;
    uint64_t off_bloom;    // u32[bloom_words]
    uint64_t off_ht;       // SieveSlot[ht_mask + 1]
    uint64_t off_node_a;   // SieveNodeA[n_nodes]
    uint64_t off_node_b;   // SieveNodeB[n_nodes]
    uint64_t off_pids;     // u32[n_pids]: the patterns ending at each terminal node, ascending id
    uint64_t total_bytes;
};

// hash table: W-byte suffix -> reverse-trie node of depth W
struct SieveSlot {
    uint32_t key_lo, key_hi;  // the window's bytes (as sieve_x sees them: lo', hi'), exact
    uint32_t node;            // kSieveNoNode = empty
    uint32_t pad;
};

// Reverse trie, nodes of depth >= W, children of a node contiguous and sorted by byte.
// A node at depth d stands for a d-byte string s; a pattern ENDS at position e with this node on its path when the d
// bytes before e are s.  Its children prepend one more byte (the byte at e-d-1).
struct SieveNodeA {           // what the walk reads
    uint32_t first_kid;
    uint32_t meta;            // bits 0-7: the byte this node prepends to its parent's string; 8-16: number of children; 17: terminal
};
struct SieveNodeB {           // what the emission reads
    uint32_t own_off, own_cnt;  // pids[own_off .. own_off + own_cnt): patterns equal to this node's string
    uint32_t term_link;         // nearest terminal proper ancestor (a shorter pattern ending at the same position), kSieveNoNode = none
    uint32_t depth;             // = pattern length of the own patterns
    uint32_t chain_cnt;         // own_cnt summed along the term_link chain from here: matches reported when this is the deepest terminal
    uint32_t pad0, pad1, pad2;
};
constexpr uint32_t kNodeTerminal = 1u << 17;

struct Automaton;
// Builds the sieve image for the automaton's patterns.  bloom_bytes_max: the shared memory the filters may take when the
// scan keeps one window of text per warp on chip (the builder may use less, to leave room for a deeper ring: sieve.cpp).
// w_max: cap on the primary window (0 = automatic).  flags: kAsciiCaseInsensitive or 0.
uint64_t sieve_image_build(const uint8_t *blob, const uint64_t *offsets, uint64_t n, uint32_t bloom_bytes_max, uint32_t w_max,
                           uint32_t flags, std::vector<uint8_t> &out);

}  // namespace acb
