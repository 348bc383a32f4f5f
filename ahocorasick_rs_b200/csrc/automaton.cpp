// automaton.cpp -- host-side construction of the matcher and its device image.
//
// Reference behaviour being reproduced (not its code): the crate call at
// /root/reference/src/lib.rs:186-215 / 401-406 builds trie + failure links and
// then a DFA or NFA; match semantics per MatchKind are documented in
// README.md:86-161 and pinned by tests/test_ac.py:196-292.  This builder goes
// straight to a breadth-first-numbered dense table: shallow (hot) states get
// the lowest ids so a prefix of the table can live in shared memory, and match
// information rides on the transition entries so the scan never has to look a
// state up just to learn it is uninteresting.
#include "automaton.h"

#include <algorithm>
#include <cstring>
#include <stdexcept>
#include <thread>

#include "sieve.h"  // ascii_fold: the one fold the builders and the sieve kernel share

namespace acb {
namespace {

struct TrieBuilder {
    // temporary trie in creation order; node 0 is the root
    std::vector<std::vector<std::pair<uint8_t, uint32_t>>> kids;
    std::vector<uint32_t> own_head, own_tail;  // per node: list of pattern ids ending here
    std::vector<uint32_t> own_next;            // per pattern
    uint32_t root_kid[256];

    static constexpr uint32_t kNone = 0xffffffffu;

    TrieBuilder() {
        std::fill(root_kid, root_kid + 256, kNone);
        new_node();
    }
    uint32_t new_node() {
        kids.emplace_back();
        own_head.push_back(kNone);
        own_tail.push_back(kNone);
        return static_cast<uint32_t>(kids.size() - 1);
    }
    uint32_t child(uint32_t s, uint8_t b) const {
        if (s == 0) return root_kid[b];
        for (const auto &kv : kids[s])
            if (kv.first == b) return kv.second;
        return kNone;
    }
    uint32_t add_child(uint32_t s, uint8_t b) {
        uint32_t c = new_node();
        kids[s].emplace_back(b, c);
        if (s == 0) root_kid[b] = c;
        return c;
    }
};

inline uint64_t align16(uint64_t x) { return (x + 15) & ~uint64_t(15); }

}  // namespace

Automaton *build_automaton(const uint8_t *blob, const uint64_t *offsets, uint64_t n, int match_kind,
                           int implementation, uint32_t flags) {
    if (match_kind < 0 || match_kind > 2) throw std::runtime_error("unknown match kind");
    if (n >= 0x7fffffffull) throw std::runtime_error("too many patterns: pattern ids must fit in 31 bits");
    const bool leftmost = match_kind != 0;
    const bool leftmost_first = match_kind == 1;
    // case-insensitive: the trie holds the folded patterns and the column map sends both cases of a letter to one
    // column, so the scan kernels see folded text without folding anything themselves
    const bool fold = (flags & kAsciiCaseInsensitive) != 0;

    // ---- 1. trie -----------------------------------------------------------
    TrieBuilder tb;
    tb.own_next.assign(n, TrieBuilder::kNone);
    std::vector<uint32_t> pat_len(n), pat_cplen(n);
    bool used[256] = {false};
    uint32_t max_len = 0, min_len = 0xffffffffu;
    for (uint64_t i = 0; i < n; i++) {
        const uint8_t *p = blob + offsets[i];
        const uint64_t len = offsets[i + 1] - offsets[i];
        if (len == 0) throw std::runtime_error("empty pattern at index " + std::to_string(i));
        if (len > 0x7fffffffull) throw std::runtime_error("pattern too long");
        pat_len[i] = static_cast<uint32_t>(len);
        uint32_t cps = 0;
        for (uint64_t k = 0; k < len; k++) cps += (p[k] & 0xC0) != 0x80;
        pat_cplen[i] = cps;
        max_len = std::max(max_len, pat_len[i]);
        min_len = std::min(min_len, pat_len[i]);
        uint32_t s = 0;
        bool shadowed = false;
        for (uint64_t k = 0; k < len; k++) {
            // LeftmostFirst: an earlier pattern that is a proper prefix of this
            // one always beats it, so it can never be reported.
            if (leftmost_first && tb.own_head[s] != TrieBuilder::kNone) {
                shadowed = true;
                break;
            }
            const uint8_t b = fold ? static_cast<uint8_t>(ascii_fold(p[k])) : p[k];
            used[b] = true;
            uint32_t c = tb.child(s, b);
            if (c == TrieBuilder::kNone) c = tb.add_child(s, b);
            s = c;
        }
        if (shadowed) continue;
        if (tb.own_tail[s] == TrieBuilder::kNone)
            tb.own_head[s] = static_cast<uint32_t>(i);
        else
            tb.own_next[tb.own_tail[s]] = static_cast<uint32_t>(i);
        tb.own_tail[s] = static_cast<uint32_t>(i);
    }
    if (n == 0) min_len = 0;
    const uint64_t n_nodes = tb.kids.size();
    if (n_nodes + 1 >= 0x7fffffffull) throw std::runtime_error("too many states: state ids must fit in 31 bits");
    const uint32_t n_states = static_cast<uint32_t>(n_nodes + 1);  // + kDead

    // ---- 2. breadth-first renumbering: kDead=0, kRoot=1, then by depth -------
    // In this order the children of a state are contiguous and a state's
    // failure target always has a smaller id.
    std::vector<uint32_t> order;  // new id - 1 -> temp node
    order.reserve(n_nodes);
    std::vector<uint32_t> new_id(n_nodes);
    std::vector<uint32_t> first_kid(n_states + 1, 0), parent(n_states, 0);
    std::vector<uint8_t> in_byte(n_states, 0);
    order.push_back(0);
    new_id[0] = kRoot;
    for (size_t q = 0; q < order.size(); q++) {
        const uint32_t t = order[q];
        auto &kv = tb.kids[t];
        std::sort(kv.begin(), kv.end());
        first_kid[new_id[t]] = static_cast<uint32_t>(order.size() + 1);
        for (const auto &e : kv) {
            const uint32_t id = static_cast<uint32_t>(order.size() + 1);
            new_id[e.second] = id;
            parent[id] = new_id[t];
            in_byte[id] = e.first;
            order.push_back(e.second);
        }
    }
    first_kid[0] = first_kid[kRoot];  // kDead has no children: empty range ends where root's begins
    first_kid[n_states] = n_states;
    // n_kids(s) = first_kid[s+1] - first_kid[s] holds because ranges are laid out in id order
    auto kid_of = [&](uint32_t s, uint8_t b) -> uint32_t {
        for (uint32_t c = first_kid[s], e = first_kid[s + 1]; c < e; c++)
            if (in_byte[c] == b) return c;
        return 0;  // none (0 is never a child)
    };

    // ---- 3. failure links + match lists --------------------------------------
    std::vector<uint32_t> fail(n_states, kRoot);
    std::vector<uint32_t> own_cnt(n_states, 0);
    for (uint32_t s = kRoot; s < n_states; s++) {
        uint32_t c = 0;
        for (uint32_t p = tb.own_head[order[s - 1]]; p != TrieBuilder::kNone; p = tb.own_next[p]) c++;
        own_cnt[s] = c;
    }
    fail[kDead] = kDead;
    fail[kRoot] = kRoot;
    for (uint32_t s = kRoot + 1; s < n_states; s++) {
        if (leftmost && own_cnt[s]) {
            // A pattern ends exactly here.  Under leftmost semantics nothing that
            // starts later may be found through this state or below it.
            fail[s] = kDead;
            continue;
        }
        const uint32_t par = parent[s];
        if (par == kRoot) {
            fail[s] = kRoot;
            continue;
        }
        uint32_t f = fail[par];
        const uint8_t b = in_byte[s];
        uint32_t t = 0;
        for (;;) {
            if (f == kDead) break;  // t stays kDead
            t = kid_of(f, b);
            if (t) break;
            if (f == kRoot) {
                t = kRoot;
                break;
            }
            f = fail[f];
        }
        fail[s] = t;
    }
    std::vector<uint32_t> match_off(n_states + 1, 0);
    {
        // list(s) = patterns ending exactly at s (ascending id), then list(fail(s)):
        // the reference's order within one end position (longest first, then id)
        std::vector<uint32_t> cnt(n_states, 0);
        uint64_t run = 0;
        for (uint32_t s = kRoot; s < n_states; s++) {
            uint64_t c = own_cnt[s];
            if (s > kRoot && !(leftmost && own_cnt[s])) c += cnt[fail[s]];
            cnt[s] = static_cast<uint32_t>(c);
            match_off[s] = static_cast<uint32_t>(run);
            run += c;
            if (run > 0x7fffffffull) throw std::runtime_error("match lists too large");
        }
        match_off[n_states] = static_cast<uint32_t>(run);
    }
    std::vector<uint32_t> match_pid(match_off[n_states]);
    for (uint32_t s = kRoot; s < n_states; s++) {
        uint32_t w = match_off[s];
        for (uint32_t p = tb.own_head[order[s - 1]]; p != TrieBuilder::kNone; p = tb.own_next[p]) match_pid[w++] = p;
        if (s > kRoot && !(leftmost && own_cnt[s])) {
            const uint32_t f = fail[s];
            for (uint32_t k = match_off[f]; k < match_off[f + 1]; k++) match_pid[w++] = match_pid[k];
        }
    }

    // ---- 4. byte -> column map -------------------------------------------------
    uint32_t lo = 256, hi = 0, n_used = 0;
    for (uint32_t b = 0; b < 256; b++)
        if (used[b]) {
            lo = std::min(lo, b);
            hi = b;
            n_used++;
        }
    if (n_used == 0) lo = hi = 0;
    const uint32_t class_cols = n_used + 1;    // column 0 = every byte no pattern uses
    const uint32_t range_cols = hi - lo + 2;   // last column = every byte outside [lo, hi]
    // kColRange computes the column arithmetically in the kernels: it cannot send 'A' to the column of 'a', so a
    // case-insensitive automaton whose patterns hold a letter takes the class map
    bool letters = false;
    for (uint32_t b = 'a'; b <= 'z'; b++) letters |= used[b];
    uint32_t col_mode, n_cols;
    uint8_t colmap[256];
    if (range_cols * 4 <= class_cols * 5 && range_cols <= 256 && !(fold && letters)) {
        col_mode = kColRange;
        n_cols = range_cols;
        for (uint32_t b = 0; b < 256; b++) colmap[b] = static_cast<uint8_t>(std::min(b - lo, n_cols - 1));  // unsigned wrap for b < lo
    } else {
        col_mode = kColClass;
        n_cols = class_cols;
        if (n_cols > 256) {  // all 256 byte values used: no "other" column needed
            n_cols = 256;
            for (uint32_t b = 0; b < 256; b++) colmap[b] = static_cast<uint8_t>(b);
        } else {
            uint32_t next = 1;
            for (uint32_t b = 0; b < 256; b++) colmap[b] = used[b] ? static_cast<uint8_t>(next++) : 0;
        }
        if (fold)
            for (uint32_t b = 'A'; b <= 'Z'; b++) colmap[b] = colmap[b | 0x20u];
    }

    // ---- 5. image ---------------------------------------------------------------
    const uint64_t trans_bytes = uint64_t(n_states) * n_cols * 4;
    if (trans_bytes > (uint64_t(48) << 30))
        throw std::runtime_error("transition table would need " + std::to_string(trans_bytes >> 20) + " MiB");
    auto *A = new Automaton();
    A->implementation = implementation;
    A->pat_offs.assign(offsets, offsets + n + 1);
    if (n && offsets[n]) A->pat_blob.assign(blob, blob + offsets[n]);
    ImageHeader &h = A->hdr;
    h.magic = kImageMagic;
    h.version = 1;
    h.match_kind = static_cast<uint32_t>(match_kind);
    h.col_mode = col_mode;
    h.n_states = n_states;
    h.n_cols = n_cols;
    h.col_lo = lo;
    h.n_patterns = static_cast<uint32_t>(n);
    h.max_pat_len = max_len;
    h.min_pat_len = min_len;
    h.n_hot_eligible = n_states;
    h.flags = flags & kAsciiCaseInsensitive;
    uint64_t off = align16(sizeof(ImageHeader));
    h.off_colmap = off;
    off = align16(off + 256);
    h.off_trans = off;
    off = align16(off + trans_bytes);
    h.off_match_off = off;
    off = align16(off + uint64_t(n_states + 1) * 4);
    h.off_match_pid = off;
    off = align16(off + uint64_t(match_pid.size()) * 4 + 4);
    h.off_pat_len = off;
    off = align16(off + n * 4 + 4);
    h.off_pat_cplen = off;
    off = align16(off + n * 4 + 4);
    h.total_bytes = off;
    try {
        A->image.assign(off, 0);
    } catch (const std::bad_alloc &) {
        delete A;
        throw std::runtime_error("out of host memory for the device image");
    }
    uint8_t *img = A->image.data();
    std::memcpy(img, &h, sizeof(h));
    std::memcpy(img + h.off_colmap, colmap, 256);
    std::memcpy(img + h.off_match_off, match_off.data(), uint64_t(n_states + 1) * 4);
    if (!match_pid.empty()) std::memcpy(img + h.off_match_pid, match_pid.data(), match_pid.size() * 4);
    if (n) {
        std::memcpy(img + h.off_pat_len, pat_len.data(), n * 4);
        std::memcpy(img + h.off_pat_cplen, pat_cplen.data(), n * 4);
    }
    // dense rows, in id order: a row starts as a copy of its failure target's row
    // (already final, smaller id) and then takes the state's own trie edges
    uint32_t *T = reinterpret_cast<uint32_t *>(img + h.off_trans);
    auto entry = [&](uint32_t t) -> uint32_t {
        return t | ((match_off[t + 1] != match_off[t]) ? kMatchFlag : 0u);
    };
    for (uint32_t c = 0; c < n_cols; c++) T[uint64_t(kRoot) * n_cols + c] = entry(kRoot);  // kDead row stays all kDead
    auto fill_rows = [&](uint32_t lo, uint32_t hi) {
        for (uint32_t s = lo; s < hi; s++) {
            uint32_t *row = T + uint64_t(s) * n_cols;
            if (s != kRoot) std::memcpy(row, T + uint64_t(fail[s]) * n_cols, uint64_t(n_cols) * 4);
            for (uint32_t c = first_kid[s], e = first_kid[s + 1]; c < e; c++) row[colmap[in_byte[c]]] = entry(c);
        }
    };
    // A row needs its failure target's row, which is strictly shallower: the rows of ONE trie level are independent of
    // each other, so each level (contiguous in the breadth-first numbering) is filled by several threads.
    std::vector<uint32_t> level_start;  // first state of each depth, then n_states
    {
        std::vector<uint32_t> depth(n_states, 0);
        level_start.push_back(kRoot);
        for (uint32_t s = kRoot + 1; s < n_states; s++) {
            depth[s] = depth[parent[s]] + 1;
            if (depth[s] != depth[s - 1]) level_start.push_back(s);
        }
        level_start.push_back(n_states);
    }
    const unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    for (size_t lv = 0; lv + 1 < level_start.size(); lv++) {
        const uint32_t lo = level_start[lv], hi = level_start[lv + 1];
        const uint64_t cells = uint64_t(hi - lo) * n_cols;
        const unsigned nt = cells < (1u << 18) ? 1u : hw;
        if (nt == 1) {
            fill_rows(lo, hi);
            continue;
        }
        std::vector<std::thread> pool;
        const uint32_t per = (hi - lo + nt - 1) / nt;
        for (unsigned t = 0; t < nt; t++) {
            const uint32_t a = lo + t * per, b = std::min(hi, a + per);
            if (a < b) pool.emplace_back(fill_rows, a, b);
        }
        for (auto &th : pool) th.join();
    }
    return A;
}

static uint32_t hot_rows_for(const Automaton &a, uint32_t max_rows) {
    uint32_t H = max_rows;
    if (H > a.hdr.n_states - 1) H = a.hdr.n_states - 1;  // kDead is never hot
    // entries are u16 BYTE offsets of rows (hot index * row bytes), so the trap row must start below 64 KiB
    const uint32_t by_offset = 65535u / (a.hdr.n_cols * 2u);
    if (H > by_offset) H = by_offset;
    if (H < 1) H = 1;
    return H;
}

// ASCII table: available when every byte >= 0x7f falls in the "no pattern uses it" column
static uint32_t ascii_rows_for(const Automaton &a, uint32_t H) {
    const uint8_t *colmap = a.image.data() + a.hdr.off_colmap;
    const uint8_t other = colmap[255];
    for (uint32_t b = 127; b < 256; b++)
        if (colmap[b] != other) return 0;
    // column `other` must really be the shared one: no trie edge uses it
    if (a.hdr.col_mode == kColRange ? other != a.hdr.n_cols - 1 : other != 0) return 0;
    return H < 255 ? H : 255;  // the trap row starts at 255 * 256 < 64 KiB
}

uint64_t hot_image_bytes(const Automaton &a, uint32_t max_rows) {
    const uint32_t H = hot_rows_for(a, max_rows);
    uint64_t off = align16(sizeof(HotHeader));
    off = align16(off + uint64_t(H + 1) * a.hdr.n_cols * 2);
    off = align16(off + uint64_t(H + 1) * 4);
    off = align16(off + uint64_t(a.hdr.n_states) * 2);
    off = align16(off + uint64_t(ascii_rows_for(a, H) + 1) * kAsciiCols * 2);
    return off;
}

void build_hot_image(const Automaton &a, const uint32_t *visits, uint32_t max_rows, uint8_t *dst) {
    const ImageHeader &ih = a.hdr;
    const uint32_t H = hot_rows_for(a, max_rows);
    const uint32_t n_cols = ih.n_cols, n_states = ih.n_states;
    HotHeader hh{};
    hh.magic = kHotMagic;
    hh.n_rows = H;
    hh.n_cols = n_cols;
    hh.n_states = n_states;
    uint64_t off = align16(sizeof(HotHeader));
    hh.off_table = off;
    off = align16(off + uint64_t(H + 1) * n_cols * 2);
    hh.off_hot2full = off;
    off = align16(off + uint64_t(H + 1) * 4);
    hh.off_full2hot = off;
    off = align16(off + uint64_t(n_states) * 2);
    const uint32_t H128 = ascii_rows_for(a, H);
    hh.n_rows128 = H128;
    hh.off_table128 = off;
    off = align16(off + uint64_t(H128 + 1) * kAsciiCols * 2);
    hh.total_bytes = off;
    std::memset(dst, 0, off);
    uint16_t *table = reinterpret_cast<uint16_t *>(dst + hh.off_table);
    uint32_t *hot2full = reinterpret_cast<uint32_t *>(dst + hh.off_hot2full);
    uint16_t *full2hot = reinterpret_cast<uint16_t *>(dst + hh.off_full2hot);
    for (uint32_t s = 0; s < n_states; s++) full2hot[s] = kNotHot;

    // choose the rows: root, then sampled states by visit count, then shallow states
    uint32_t n = 0;
    auto take = [&](uint32_t s) {
        if (n < H && s != kDead && full2hot[s] == kNotHot) {
            full2hot[s] = static_cast<uint16_t>(n);
            hot2full[n++] = s;
        }
    };
    take(kRoot);
    uint32_t n_visited = 1;
    if (visits) {
        std::vector<uint32_t> seen;
        for (uint32_t s = kRoot; s < n_states; s++)
            if (visits[s]) seen.push_back(s);
        n_visited = static_cast<uint32_t>(seen.size()) + (visits[kRoot] ? 0 : 1);
        const size_t keep = std::min<size_t>(seen.size(), H);
        std::partial_sort(seen.begin(), seen.begin() + keep, seen.end(), [&](uint32_t x, uint32_t y) {
            return visits[x] != visits[y] ? visits[x] > visits[y] : x < y;
        });
        for (size_t i = 0; i < keep; i++) take(seen[i]);
    }
    for (uint32_t s = kRoot; s < n_states && n < H; s++) take(s);
    // n == H here because H <= n_states - 1

    const uint32_t *T = reinterpret_cast<const uint32_t *>(a.image.data() + ih.off_trans);
    const uint32_t row_bytes = n_cols * 2;
    for (uint32_t h = 0; h < H; h++) {
        const uint32_t *row = T + uint64_t(hot2full[h]) * n_cols;
        uint16_t *out = table + uint64_t(h) * n_cols;
        for (uint32_t c = 0; c < n_cols; c++) {
            const uint32_t e = row[c], t = e & kStateMask;
            uint32_t v = H;
            if (!(e & kMatchFlag) && t != kDead && full2hot[t] != kNotHot) v = full2hot[t];
            out[c] = static_cast<uint16_t>(v * row_bytes);
        }
    }
    for (uint32_t c = 0; c < n_cols; c++) table[uint64_t(H) * n_cols + c] = static_cast<uint16_t>(H * row_bytes);
    hot2full[H] = kDead;

    if (H128) {
        // the same rows, indexed by the raw byte (bytes >= 128 are clamped to column 127 by the scan,
        // which is the "no pattern uses it" column by construction)
        uint16_t *t128 = reinterpret_cast<uint16_t *>(dst + hh.off_table128);
        const uint8_t *colmap = a.image.data() + ih.off_colmap;
        for (uint32_t h = 0; h < H128; h++) {
            const uint32_t *row = T + uint64_t(hot2full[h]) * n_cols;
            for (uint32_t b = 0; b < kAsciiCols; b++) {
                const uint32_t e = row[colmap[b]], t = e & kStateMask;
                uint32_t v = H128;
                if (!(e & kMatchFlag) && t != kDead && full2hot[t] < H128) v = full2hot[t];
                t128[uint64_t(h) * kAsciiCols + b] = static_cast<uint16_t>(v * kAsciiCols * 2);
            }
        }
        for (uint32_t b = 0; b < kAsciiCols; b++) t128[uint64_t(H128) * kAsciiCols + b] = static_cast<uint16_t>(H128 * kAsciiCols * 2);
    }
    hh.n_visited = n_visited > H ? H : n_visited;
    std::memcpy(dst, &hh, sizeof(hh));
}

}  // namespace acb
