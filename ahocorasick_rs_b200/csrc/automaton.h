// automaton.h -- host-side automaton and the flat device image the kernels read.
//
// Stands in for what AhoCorasickBuilder::build returns at
// /root/reference/src/lib.rs:186-215 and 401-406 (the crate's NFA/DFA), laid
// out for HBM rather than for a CPU cache: see DESIGN.md "Data layout".
#pragma once
#include <cstdint>
#include <mutex>
#include <string>
#include <vector>

namespace acb {

constexpr uint32_t kDead = 0;  // absorbing; only reachable under leftmost kinds
constexpr uint32_t kRoot = 1;  // unanchored start state
constexpr uint32_t kMatchFlag = 0x80000000u;  // set on a transition entry whose target is a match state
constexpr uint32_t kStateMask = 0x7fffffffu;

enum ColMode : uint32_t {
    kColRange = 0,  // column = min(byte - lo, ncols - 1) (unsigned): no table lookup per byte
    kColClass = 1,  // column = colmap[byte]
};

// Header of the device image.  Copied by value into kernel parameters; the
// offsets are byte offsets from the start of the image.
struct ImageHeader {
    uint32_t magic;
    uint32_t version;
    uint32_t match_kind;
    uint32_t col_mode;
    uint32_t n_states;      // including kDead and kRoot
    uint32_t n_cols;        // row width, in entries
    uint32_t col_lo;        // kColRange: first byte that has its own column
    uint32_t n_patterns;
    uint32_t max_pat_len;
    uint32_t min_pat_len;
    uint32_t n_hot_eligible; // states are BFS ordered; rows [0, n_hot_eligible) may be cached on chip
    uint32_t flags;          // kAsciiCaseInsensitive (sieve.h): the trie holds the folded patterns, colmap folds the text
    uint64_t off_colmap;     // u8[256]
    uint64_t off_trans;      // u32[n_states * n_cols]: next state | kMatchFlag
    uint64_t off_match_off;  // u32[n_states + 1]
    uint64_t off_match_pid;  // u32[match_off[n_states]]: own patterns first (ascending id), then suffixes, longest first
    uint64_t off_pat_len;    // u32[n_patterns] bytes
    uint64_t off_pat_cplen;  // u32[n_patterns] code points (non-continuation bytes)
    uint64_t total_bytes;
};

constexpr uint32_t kImageMagic = 0x30424341u;  // "ACB0"

// The hot image: the part of the automaton the staged kernel keeps in shared
// memory.  Rows are ordered hottest first (by sampled visit counts, the root
// always first, then shallow states as filler), so a kernel that can only fit
// H' < n_rows rows takes a prefix.  Table entries are the BYTE OFFSET of the next
// state's row inside the table (hot index * n_cols * 2, so one add forms the
// shared-memory address); n_rows * n_cols * 2 = the trap row.
struct HotHeader {
    uint32_t magic;
    uint32_t n_rows;    // H
    uint32_t n_cols;
    uint32_t n_states;
    uint64_t off_table;     // u16[(H + 1) * n_cols]; row H (the trap row) maps everything to itself
    uint64_t off_hot2full;  // u32[H + 1]
    uint64_t off_full2hot;  // u16[n_states]; 0xffff = not hot
    uint64_t total_bytes;
    // ASCII variant of the table (only when no pattern uses a byte >= 0x7f): the first n_rows128 hot
    // rows again, 128 entries wide and indexed by the raw byte, so the scan needs no byte -> column
    // arithmetic at all on text without high bytes.  0 rows = not available.
    uint32_t n_rows128;
    uint32_t n_visited;     // rows that the profile actually saw (the rest is filler)
    uint64_t off_table128;  // u16[(n_rows128 + 1) * 128]; entries are row byte offsets (index * 256)
};
constexpr uint32_t kAsciiCols = 128;
constexpr uint32_t kHotMagic = 0x31424341u;  // "ACB1"
constexpr uint16_t kNotHot = 0xffffu;

struct Automaton {
    ImageHeader hdr{};
    std::vector<uint8_t> image;  // header + tables, ready to copy to the device
    int implementation = -1;
    // the patterns themselves (the sieve image is built from them on demand: sieve.h)
    std::vector<uint8_t> pat_blob;
    std::vector<uint64_t> pat_offs;
    std::mutex sieve_mutex;
    std::vector<uint8_t> sieve;       // built by acb_sieve_build
    uint32_t sieve_bloom_max = 0, sieve_w_max = 0;
};

// Builds the automaton; throws std::runtime_error with a message on failure.  flags: kAsciiCaseInsensitive or 0.
Automaton *build_automaton(const uint8_t *blob, const uint64_t *offsets, uint64_t n, int match_kind,
                           int implementation, uint32_t flags);

// Size of / builder for the hot image with at most max_rows rows.  visits may be
// null (no profile yet: breadth-first prefix) or n_states sampled visit counts.
uint64_t hot_image_bytes(const Automaton &a, uint32_t max_rows);
void build_hot_image(const Automaton &a, const uint32_t *visits, uint32_t max_rows, uint8_t *dst);

}  // namespace acb
