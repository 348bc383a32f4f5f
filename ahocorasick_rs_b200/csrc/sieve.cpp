// sieve.cpp -- host-side construction of the sieve image (sieve.h): Bloom filter
// over pattern suffixes, hash table W-byte suffix -> reverse-trie node, the
// reverse trie itself.  Stands, like automaton.cpp, for the builder call at
// /root/reference/src/lib.rs:186-215 / 401-406; the layout is this repo's own.
#include "sieve.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <stdexcept>
#include <unordered_map>
#include <unordered_set>
#include <vector>

namespace acb {
namespace {

inline uint64_t align16(uint64_t x) { return (x + 15) & ~uint64_t(15); }

// the newest W bytes of a string ending at p + len, as the kernel sees them in its (hi:lo) window registers
inline void pack_tail(const uint8_t *p, uint64_t len, uint32_t W, uint32_t &lo, uint32_t &hi) {
    lo = hi = 0;
    if (W <= 4) {
        for (uint32_t i = 0; i < W; i++) lo |= uint32_t(p[len - W + i]) << (8 * i);
    } else {
        for (uint32_t i = 0; i < 4; i++) lo |= uint32_t(p[len - 4 + i]) << (8 * i);
        for (uint32_t i = 0; i < W - 4; i++) hi |= uint32_t(p[len - W + i]) << (8 * i);
    }
}

struct TNode {
    std::vector<std::pair<uint8_t, uint32_t>> kids;
    std::vector<uint32_t> own;
    uint32_t depth = 0;
    uint32_t x = 0;  // window hash of the node's string
};

// the filters live back to back in one array: words [base, base + n_words)
void filter_insert(std::vector<uint32_t> &bits, uint32_t base, uint32_t n_words, uint32_t x, const uint32_t *muls, uint32_t n_probes) {
    for (uint32_t i = 0; i < n_probes; i++) {
        const uint32_t p = x * muls[i];
        bits[base + sieve_probe_word(p, n_words)] |= 1u << sieve_probe_bit(p);
    }
}

}  // namespace

uint64_t sieve_image_build(const uint8_t *blob, const uint64_t *offsets, uint64_t n, uint32_t bloom_bytes_max, uint32_t w_max,
                           uint32_t flags, std::vector<uint8_t> &out) {
    // case-insensitive: everything below is built from the folded patterns (the image equals the case-sensitive image
    // of the folded pattern list but for the flag)
    std::vector<uint8_t> folded;
    if (flags & kAsciiCaseInsensitive) {
        folded.assign(blob, blob + (n ? offsets[n] : 0));
        for (auto &b : folded) b = (uint8_t)ascii_fold(b);
        blob = folded.data();
    }
    uint32_t min_len = 0xffffffffu, max_len = 0;
    bool used[256] = {false};
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t len = offsets[i + 1] - offsets[i];
        if (len == 0) throw std::runtime_error("empty pattern at index " + std::to_string(i));
        if (len > 0x7fffffffull) throw std::runtime_error("pattern too long");
        min_len = std::min<uint32_t>(min_len, (uint32_t)len);
        max_len = std::max<uint32_t>(max_len, (uint32_t)len);
        for (uint64_t k = 0; k < len; k++) used[blob[offsets[i] + k]] = true;
    }
    if (n == 0) min_len = max_len = 0;
    uint32_t sigma = 0;
    for (int b = 0; b < 256; b++) sigma += used[b];

    // ---- the primary window ------------------------------------------------------------------
    // As short as possible (the fast path hashes one 32-bit word up to W = 4, two beyond), but selective: the share of
    // all sigma^w strings that are some pattern's w-byte suffix estimates how often random text passes the filter.
    uint32_t W = 1;
    if (n) {
        const uint32_t w_hi = std::min<uint32_t>(min_len, kSieveMaxW);
        if (w_max) {
            W = std::min(w_hi, w_max);
        } else {
            // Up to 4 bytes the fast path hashes one word; 5..8 cost it three more instructions per byte but cut the
            // survivors (on text, 4-byte suffixes of a few thousand names pass 3 % of the positions, 5-byte ones 1 %).
            W = std::min<uint32_t>(w_hi, n > 256 ? 5 : 4);
            for (; W < w_hi; W++) {
                std::unordered_set<uint64_t> seen;
                for (uint64_t i = 0; i < n; i++) {
                    uint32_t lo, hi;
                    pack_tail(blob + offsets[i], offsets[i + 1] - offsets[i], W, lo, hi);
                    seen.insert((uint64_t(hi) << 32) | lo);
                }
                const double space = std::pow((double)std::max<uint32_t>(sigma, 2), (double)W);
                if (W >= 5 && (double)seen.size() <= 0.02 * space) break;
                if (W < 5 && (double)seen.size() <= 0.002 * space) break;
            }
        }
        if (W < 1) W = 1;
    }

    // ---- reverse trie of everything beyond the window ------------------------------------------
    std::vector<TNode> nodes;
    std::unordered_map<uint64_t, uint32_t> root_of;
    std::vector<uint64_t> root_key;
    root_of.reserve(n * 2 + 16);
    for (uint64_t i = 0; i < n; i++) {
        const uint8_t *p = blob + offsets[i];
        const uint64_t len = offsets[i + 1] - offsets[i];
        uint32_t lo, hi;
        pack_tail(p, len, W, lo, hi);
        const uint64_t key = (uint64_t(hi) << 32) | lo;
        auto it = root_of.find(key);
        uint32_t v;
        if (it == root_of.end()) {
            v = (uint32_t)nodes.size();
            nodes.emplace_back();
            nodes[v].depth = W;
            nodes[v].x = sieve_x_packed(lo, hi);
            root_of.emplace(key, v);
            root_key.push_back(key);
        } else {
            v = it->second;
        }
        for (uint64_t j = len - W; j-- > 0;) {
            const uint8_t b = p[j];
            uint32_t c = kSieveNoNode;
            for (const auto &kv : nodes[v].kids)
                if (kv.first == b) {
                    c = kv.second;
                    break;
                }
            if (c == kSieveNoNode) {
                c = (uint32_t)nodes.size();
                nodes.emplace_back();
                nodes[c].depth = nodes[v].depth + 1;
                nodes[c].x = sieve_step(nodes[v].x, b);
                nodes[v].kids.emplace_back(b, c);
            }
            v = c;
        }
        nodes[v].own.push_back((uint32_t)i);
        if (nodes.size() >= 0x7fffffffull) throw std::runtime_error("too many trie nodes");
    }
    const uint32_t n_nodes = (uint32_t)nodes.size();
    const uint32_t n_keys = (uint32_t)root_key.size();

    // breadth-first numbering: the roots keep their creation order, children are contiguous and sorted by byte
    std::vector<uint32_t> order;  // new id -> old id
    std::vector<uint32_t> new_id(n_nodes), parent_new(n_nodes, kSieveNoNode), first_kid(n_nodes, 0);
    std::vector<uint8_t> in_byte(n_nodes, 0);
    order.reserve(n_nodes);
    for (uint32_t r = 0; r < n_keys; r++) {
        const uint32_t old = root_of[root_key[r]];
        new_id[old] = (uint32_t)order.size();
        order.push_back(old);
    }
    for (size_t q = 0; q < order.size(); q++) {
        TNode &t = nodes[order[q]];
        std::sort(t.kids.begin(), t.kids.end());
        first_kid[q] = (uint32_t)order.size();
        for (const auto &kv : t.kids) {
            const uint32_t id = (uint32_t)order.size();
            new_id[kv.second] = id;
            parent_new[id] = (uint32_t)q;
            in_byte[id] = kv.first;
            order.push_back(kv.second);
        }
    }

    // ---- how deep the on-chip filter goes --------------------------------------------------------
    // entries(L) = nodes of depth <= L (suffix present) + terminal nodes of depth <= L (pattern complete)
    const uint32_t level_cap = std::min<uint32_t>(kSieveMaxLevel, std::max<uint32_t>(max_len, W));
    std::vector<uint64_t> per_level(kSieveMaxLevel + 2, 0);
    std::vector<uint64_t> terms_at(kSieveMaxLevel + 2, 0);
    for (uint32_t v = 0; v < n_nodes; v++) {
        const TNode &t = nodes[order[v]];
        if (t.depth <= level_cap) {
            per_level[t.depth] += 1 + (t.own.empty() ? 0 : 1);
            terms_at[t.depth] += t.own.empty() ? 0 : 1;
        }
    }
    if (bloom_bytes_max < 1024) bloom_bytes_max = 1024;
    // ---- filters against text ring ---------------------------------------------------------------
    // bloom_bytes_max is what the filters may take when each warp of the scan keeps ONE window of text on chip.  A warp
    // has to finish the survivors of a window before that window's slot in its ring is overwritten, so with a ring of one
    // stage 1 runs after every window that has a survivor, however few lanes that fills; with a ring of r it waits
    // for 32 of them (or r windows).  A deeper ring costs kSieveScanWarps x kSieveRingSlotBytes of filter per extra
    // window, i.e. a denser primary bitmap and more chance survivors.  Stage-1 rounds per window are about
    // max(chance survivors / 32, 1 / r): take a deeper ring while that drops by a quarter or more.  (Dense pattern sets
    // keep the ring of one -- their rounds are full anyway; a few thousand patterns get 4 or 8 windows.)  The kernel
    // launch sizes the ring from the shared memory the filters leave, so nothing else has to know.
    {
        auto rounds = [&](uint32_t r, uint64_t bytes) {
            uint64_t pb = std::min<uint64_t>(uint64_t(n_keys) * 256, bytes * 8 * 7 / 10);
            pb = std::max<uint64_t>(pb, 4096);
            const double chance = 512.0 * double(n_keys) / double(pb);
            return std::max(chance / 32.0, 1.0 / double(r));
        };
        double best = rounds(1, bloom_bytes_max);
        uint32_t budget = bloom_bytes_max;
        for (uint32_t r = 2; r <= 8; r *= 2) {
            const uint64_t extra = uint64_t(kSieveScanWarps) * (r - 1) * kSieveRingSlotBytes;
            if (uint64_t(bloom_bytes_max) < extra + 16384) break;
            const double c = rounds(r, bloom_bytes_max - extra);
            if (c > 0.75 * best) break;
            best = c;
            budget = (uint32_t)(bloom_bytes_max - extra);
        }
        bloom_bytes_max = budget;
    }
    const uint64_t max_bits = uint64_t(bloom_bytes_max) * 8;
    // The primary bitmap (one bit per W-byte suffix, the only thing the fast path looks at) is kept sparse -- its fill
    // is the share of text positions that need a second look -- but never takes more than 70 % of the budget.
    uint64_t prim_bits = uint64_t(n_keys) * 256;
    if (prim_bits > max_bits * 7 / 10) prim_bits = max_bits * 7 / 10;
    if (prim_bits < 4096) prim_bits = 4096;
    const uint32_t prim_words = (uint32_t)(((prim_bits + 31) / 32 + 3) & ~uint64_t(3));
    const uint64_t sec_max_bits = max_bits > uint64_t(prim_words) * 32 + 4096 ? max_bits - uint64_t(prim_words) * 32 : 4096;
    // The secondary filter goes as deep as it can hold at >= 12 bits per entry.
    uint32_t last_level = W;
    uint64_t entries = per_level[W];
    for (uint32_t L = W + 1; L <= level_cap; L++) {
        if ((entries + per_level[L]) * 12 > sec_max_bits) break;
        entries += per_level[L];
        last_level = L;
    }
    if (max_len > last_level) entries -= terms_at[last_level];  // those end marks are not stored (see below)
    uint64_t bits = entries * 16;
    if (bits > sec_max_bits) bits = sec_max_bits;
    if (bits < 4096) bits = 4096;
    const uint32_t sec_words = (uint32_t)(((bits + 31) / 32 + 3) & ~uint64_t(3));
    const double bpe = entries ? double(sec_words) * 32.0 / double(entries) : 1e9;
    const uint32_t n_probes = bpe >= 3.0 ? 2 : 1;
    const uint32_t bloom_words = prim_words + sec_words;  // a multiple of 16 bytes (one bulk copy)
    std::vector<uint32_t> bloom(bloom_words, 0);
    const uint32_t mul_prim[1] = {kMulA}, mul_sec[2] = {kMulB, kMulC};
    for (uint32_t v = 0; v < n_nodes; v++) {
        const TNode &t = nodes[order[v]];
        if (t.depth > last_level) continue;
        if (t.depth == W) filter_insert(bloom, 0, prim_words, t.x, mul_prim, 1);
        filter_insert(bloom, prim_words, sec_words, t.x, mul_sec, n_probes);
        // (at the last level, when longer patterns exist, every survivor goes to the exact check anyway: no end marks)
        if (!t.own.empty() && !(t.depth == last_level && max_len > last_level))
            filter_insert(bloom, prim_words, sec_words, t.x ^ kSaltTerm, mul_sec, n_probes);
    }

    // ---- hash table: window -> root node ------------------------------------------------------------
    uint32_t ht_size = 16;
    while (ht_size < 2 * uint64_t(n_keys)) ht_size <<= 1;
    std::vector<SieveSlot> ht(ht_size, SieveSlot{0, 0, kSieveNoNode, 0});
    for (uint32_t r = 0; r < n_keys; r++) {
        const uint32_t lo = (uint32_t)root_key[r], hi = (uint32_t)(root_key[r] >> 32);
        const uint32_t x = nodes[order[r]].x;
        uint32_t s = sieve_mulhi(x * kMulSlot, ht_size);
        while (ht[s].node != kSieveNoNode) s = (s + 1) & (ht_size - 1);
        ht[s] = SieveSlot{lo, hi, r, 0};
    }

    // ---- nodes ------------------------------------------------------------------------------------------
    std::vector<SieveNodeA> na(std::max<uint32_t>(n_nodes, 1));
    std::vector<SieveNodeB> nb(std::max<uint32_t>(n_nodes, 1));
    std::vector<uint32_t> pids;
    pids.reserve(n);
    for (uint32_t v = 0; v < n_nodes; v++) {
        const TNode &t = nodes[order[v]];
        const uint32_t nk = (uint32_t)t.kids.size();
        na[v].first_kid = first_kid[v];
        na[v].meta = uint32_t(in_byte[v]) | (nk << 8) | (t.own.empty() ? 0u : kNodeTerminal);
        SieveNodeB b{};
        b.own_off = (uint32_t)pids.size();
        b.own_cnt = (uint32_t)t.own.size();
        for (uint32_t pid : t.own) pids.push_back(pid);
        b.depth = t.depth;
        const uint32_t par = parent_new[v];
        b.term_link = kSieveNoNode;
        if (par != kSieveNoNode) b.term_link = nb[par].own_cnt ? par : nb[par].term_link;
        uint64_t chain = b.own_cnt;
        if (b.term_link != kSieveNoNode) chain += nb[b.term_link].chain_cnt;
        if (chain > 0x7fffffffull) throw std::runtime_error("match lists too large");
        b.chain_cnt = (uint32_t)chain;
        nb[v] = b;
    }

    // ---- image ------------------------------------------------------------------------------------------------
    SieveHeader h{};
    h.magic = kSieveMagic;
    h.W = W;
    h.last_level = last_level;
    h.n_probes = n_probes;
    h.bloom_words = bloom_words;
    h.ht_mask = ht_size - 1;
    h.n_nodes = n_nodes;
    h.n_pids = (uint32_t)pids.size();
    h.max_pat_len = max_len;
    h.min_pat_len = min_len;
    h.n_keys = n_keys;
    h.n_filter_entries = (uint32_t)std::min<uint64_t>(entries, 0xffffffffull);
    h.prim_words = prim_words;
    h.flags = flags & kAsciiCaseInsensitive;
    for (uint32_t d = 1; d <= kSieveMaxLevel; d++)
        if (d <= level_cap && terms_at[d]) h.term_levels |= 1u << d;
    uint64_t off = align16(sizeof(SieveHeader));
    h.off_bloom = off;
    off = align16(off + uint64_t(bloom_words) * 4);
    h.off_ht = off;
    off = align16(off + uint64_t(ht_size) * sizeof(SieveSlot));
    h.off_node_a = off;
    off = align16(off + uint64_t(na.size()) * sizeof(SieveNodeA));
    h.off_node_b = off;
    off = align16(off + uint64_t(nb.size()) * sizeof(SieveNodeB));
    h.off_pids = off;
    off = align16(off + uint64_t(pids.size()) * 4 + 16);
    h.total_bytes = off;
    out.assign(off, 0);
    uint8_t *img = out.data();
    std::memcpy(img, &h, sizeof(h));
    std::memcpy(img + h.off_bloom, bloom.data(), uint64_t(bloom_words) * 4);
    std::memcpy(img + h.off_ht, ht.data(), uint64_t(ht_size) * sizeof(SieveSlot));
    std::memcpy(img + h.off_node_a, na.data(), uint64_t(na.size()) * sizeof(SieveNodeA));
    std::memcpy(img + h.off_node_b, nb.data(), uint64_t(nb.size()) * sizeof(SieveNodeB));
    if (!pids.empty()) std::memcpy(img + h.off_pids, pids.data(), pids.size() * 4);
    return off;
}

}  // namespace acb
