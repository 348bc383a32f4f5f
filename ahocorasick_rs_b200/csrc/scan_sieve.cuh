// scan_sieve.cuh -- the position-parallel scan (see sieve.h for the idea and the image).
//
// One persistent CTA per SM, 24 warps.  Dynamic shared memory:
//   [ primary bitmap | secondary Bloom filter : bloom_words x u32 ]   one TMA bulk copy (cp.async.bulk + mbarrier)
//   [ mbarrier ]
//   [ per warp: R x (16 B history | 512 B window) | 16 B pad ]   the "stash": a ring of the last R windows of text the
//        warp looked at, for the few positions that survive the first probe (their hash is recomputed from here, the
//        on-chip walk reads older bytes from here); a window is written only when it has survivors
//   [ per warp: two queues of 64 entries ]   survivors of the first probe waiting for stage 1 (positions: their text is
//        in the ring), survivors of stage 1 waiting for stage 2 (position + key: they need nothing from the ring): the
//        later stages run 32 positions at a time (one per lane) whatever window they came from
//
// Work: the byte stream is cut into TASKS of task_bytes (a multiple of 512) on a grid anchored at a 512-byte aligned
// address; warps claim tasks from an atomic counter and walk them in 512-byte WINDOWS: lane l holds bytes
// [16 l, 16 l + 16) of the window in registers (one coalesced LDG.128 per lane; the next window's load is in flight
// while this one is scanned).
//
// Per window:
//   fast path   for each of its 16 bytes a lane forms the W-byte window ending there (funnel shifts over its own words and
//               the two words before them, which come from the neighbouring lane), hashes it (one IMAD; two for W > 4)
//               and tests ONE bit of the filter: IMAD.HI (word) + LEA + LDS + SHF (bit) + SHF (collect).  No chain,
//               no branch: 16 independent probes per lane.
//   queueing    survivors (a few % of positions) are appended, in stream order, to the warp's first queue (ballot /
//               prefix sums over the lanes' hit masks).
//   stage 1     whenever 32 positions are waiting (or their text is about to leave the ring): one position per lane --
//               the hash is recomputed from the stash, the second filter is probed, then the on-chip walk towards the
//               pattern start through the deeper filter levels.  What is left goes to the second queue.
//   stage 2     the same way, 32 at a time: hash table -> reverse-trie walk in global memory / L2 -> the deepest terminal
//               node = every pattern ending there; matches are written with ONE atomicAdd per round (warp-aggregated
//               reservation; ranks by shuffle prefix sums), each tagged with (task, rank in task) so that the epilogue
//               can place it without a sort.  Both queues are first-in first-out, so matches leave in stream order.
//   The queueing and the two stages exist once in the code: a service loop after every window decides which runs.
//
// Output of this kernel = the OVERLAPPING match list.  sieve_epilogue_kernel (capi.cu) orders it and, for the
// non-overlapping searches, selects from it per haystack.
#pragma once
#include "scan_staged.cuh"
#include "sieve.h"

namespace acb {

#ifndef ACB_SIEVE_WARPS
#define ACB_SIEVE_WARPS 24
#endif
constexpr int kSieveWarps = ACB_SIEVE_WARPS;   // 768 threads: 85 registers per thread (with 32 warps the window loop rematerialised half its state)
constexpr int kSieveThreads = kSieveWarps * 32;
constexpr uint32_t kWin = 512;                       // bytes per warp window
constexpr uint32_t kSlotText = 16 + kWin;            // one ring slot: 16 bytes of history, then the window,
constexpr uint32_t kSlotBytes = kSlotText + 48;      // then (code points) continuation bytes per 16-byte chunk (32 x u8) and before the window (u32)
static_assert(kSieveWarps != 24 || (kSieveScanWarps == 24 && kSieveRingSlotBytes == kSlotBytes), "sieve.h: the builder's copy of the kernel geometry");
constexpr uint32_t kQueueCap = 64;                   // positions per queue (a round takes 32; at most 32 arrive at a time)
constexpr uint32_t kRingMax = 8;
constexpr uint32_t kQ2Entry = 16;                    // second queue: position, key (2 words), code point count
// per warp: ring | pad | first queue (positions) | second queue
__host__ __device__ constexpr uint32_t sieve_warp_bytes(uint32_t ring, bool cp) { return ring * kSlotBytes + 16 + kQueueCap * 4u + kQueueCap * kQ2Entry; }
__host__ __device__ constexpr uint32_t sieve_smem_bytes(uint32_t filter_bytes, uint32_t ring, bool cp) {
    return filter_bytes + 16 + kSieveWarps * sieve_warp_bytes(ring, cp);
}

struct DevSieve {
    const uint32_t *bloom;
    const SieveSlot *ht;
    const SieveNodeA *na;
    const SieveNodeB *nb;
    const uint32_t *pids;
    uint32_t W, last_level, n_probes, bloom_words, prim_words, ht_size, max_pat_len, term_levels;
};

struct SievePlan {
    int64_t origin;      // stream position of task 0's start (<= 0; dev_bytes + origin is 512-byte aligned)
    int64_t n_tasks;
    uint64_t buf_bytes;  // length of the byte buffer (loads stay inside [0, buf_bytes))
    uint64_t avg_len;    // hint for the first haystack lookup of a task
    uint32_t task_bytes;
    uint32_t ring;       // windows of text each warp keeps in shared memory (1..kRingMax)
};

__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};\n" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t lds32v(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(v) : "r"(addr));
    return v;
}
// (hi:lo) >> (s & 31), low word
__device__ __forceinline__ uint32_t shf_r_wrap(uint32_t lo, uint32_t hi, uint32_t s) {
    uint32_t d;
    asm("shf.r.wrap.b32 %0, %1, %2, %3;\n" : "=r"(d) : "r"(lo), "r"(hi), "r"(s));
    return d;
}

// 16 bytes at stream position q, zero outside [vlo, vhi) (the stream, clipped to the buffer)
__device__ __forceinline__ uint4 load_chunk(const uint8_t *bytes, int64_t q, int64_t vlo, int64_t vhi) {
    if (q >= vlo && q + 16 <= vhi) return __ldg(reinterpret_cast<const uint4 *>(bytes + q));
    uint32_t w[4] = {0, 0, 0, 0};
    if (q + 16 > vlo && q < vhi) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const int64_t p = q + k;
            if (p >= vlo && p < vhi) w[k >> 2] |= (uint32_t)__ldg(bytes + p) << (8 * (k & 3));
        }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// continuation bytes among the first nbytes (0..16) of the 16-byte chunk at shared address a
__device__ __forceinline__ uint32_t cont_prefix(uint32_t a, uint32_t nbytes) {
    uint32_t n = 0;
#pragma unroll
    for (int w = 0; w < 4; w++) {
        const uint32_t v = lds32v(a + 4 * w);
        const int left = (int)nbytes - 4 * w;
        const uint32_t mask = left >= 4 ? 0xffffffffu : (left <= 0 ? 0u : ((1u << (8 * left)) - 1u));
        n += __popc(v & ~(v << 1) & 0x80808080u & mask);
    }
    return n;
}

__device__ __forceinline__ uint32_t warp_excl_scan(uint32_t v, uint32_t lane, uint32_t *total) {
    uint32_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= (uint32_t)d) x += y;
    }
    *total = __shfl_sync(0xffffffffu, x, 31);
    return x - v;
}

// WC: 0 = W < 4 (the window word is shifted down), 1 = W == 4, 2 = W in 6..8 (two words), 3 = W == 5 (a word and a byte)
// FOLD: the image was built case-insensitively (sieve.h, kAsciiCaseInsensitive): text is folded where it enters registers
// -- the carry before the task's first window and every window as it becomes the current one (ascii_fold4, 4 bytes per
// instruction group) -- and the one byte per step stage 2 reads from global memory.  Everything else (the fast path, the
// ring and its history, stage 1, the code point counts) then sees folded bytes; the fold never touches a byte >= 0x80.
//
// Positions inside a task are 32-bit offsets from the task's start (`rel`); the 64-bit stream position is t_lo + rel.
template <bool CP, int WC, bool FOLD>
__global__ void __launch_bounds__(kSieveThreads, 1)
sieve_scan_kernel(DevSieve sv, Batch B, SievePlan P, Sink out, uint32_t *task_cont, uint32_t *hay_cont, unsigned int *task_counter) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t bloom_s = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t bloom_bytes = sv.bloom_words * 4;
    const uint32_t bar_s = bloom_s + bloom_bytes;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t R = P.ring;  // a power of two
    uint32_t ring_s = bar_s + 16 + warp * sieve_warp_bytes(R, CP);
    asm volatile("" : "+r"(ring_s));  // (kept in a register: left alone, the compiler recomputes it from the thread id at every use)
    const uint32_t ring_end = ring_s + R * kSlotBytes;
    const uint32_t q1_s = ring_end + 16, q2_s = q1_s + kQueueCap * 4u;
    const uint32_t n_words = sv.prim_words;              // the primary bitmap (fast path)
    const uint32_t sec_s = bloom_s + sv.prim_words * 4;  // the secondary filter
    const uint32_t sec_words = sv.bloom_words - sv.prim_words;

    // ---- prologue: the filters ----------------------------------------------------------------
    if (threadIdx.x == 0) {
        mbar_init(bar_s, 1);
        mbar_expect_tx(bar_s, bloom_bytes);
        tma_bulk_g2s(bloom_s, sv.bloom, bloom_bytes, bar_s);
    }
    // the pad behind the ring stays zero (a key read may touch one aligned word past the last slot)
    if (lane < 4) asm volatile("st.shared.u32 [%0], %1;\n" ::"r"(ring_s + R * kSlotBytes + lane * 4), "r"(0u) : "memory");
    __syncthreads();
    mbar_wait(bar_s, 0);

    const int64_t stream_lo = __ldg(B.offsets), stream_hi = __ldg(B.offsets + B.n_haystacks);
    // bytes that may be read: the stream, inside the buffer
    const int64_t vlo = max(stream_lo, (int64_t)0), vhi = min(stream_hi, (int64_t)P.buf_bytes);
    const uint32_t W = sv.W;
    const uint32_t sh_lo = 8u * (4u - min(W, 4u)), sh_hi = 8u * (8u - max(W, 4u));
    const uint32_t T = P.task_bytes;

    auto sec_bit = [&](uint32_t p) -> uint32_t {
        const uint32_t word = lds32v(sec_s + __umulhi(p, sec_words) * 4u);
        return (word >> (p & 31u)) & 1u;
    };
    auto sec_has = [&](uint32_t x) -> bool { return sec_bit(x * kMulB) && (sv.n_probes < 2 || sec_bit(x * kMulC)); };
    // shared address of the byte at task-relative position rel (its window must still be in the ring)
    auto text_s = [&](uint32_t rel) -> uint32_t { return ring_s + ((rel >> 9) & (R - 1)) * kSlotBytes + 16 + (rel & (kWin - 1)); };
    // the 8 bytes ending at rel (inclusive), from the stash: (lo', hi') as the filters key them
    auto stash_key = [&](uint32_t rel, uint32_t &klo, uint32_t &khi) {
        const uint32_t a = text_s(rel) - 7;  // the slot's 16 bytes of history cover the reach
        const uint32_t j = a & ~3u, r = (a & 3u) * 8u;
        const uint32_t w0 = lds32v(j), w1 = lds32v(j + 4), w2 = lds32v(j + 8);
        const uint32_t hi = shf_r_wrap(w0, w1, r), lo = shf_r_wrap(w1, w2, r);
        klo = W <= 4 ? lo >> sh_lo : lo;
        khi = W <= 4 ? 0u : hi >> sh_hi;
    };
    auto q1_store = [&](uint32_t i, uint32_t rel) { asm volatile("st.shared.u32 [%0], %1;\n" ::"r"(q1_s + i * 4u), "r"(rel) : "memory"); };
    // code points: where a ring slot keeps the continuation bytes of its window per 16-byte chunk (32 x u8), and before it (u32)
    auto slot_s = [&](uint32_t rel) -> uint32_t { return ring_s + ((rel >> 9) & (R - 1)) * kSlotBytes; };
    // continuation bytes of the task before the END of the candidate at rel (its window is in the ring)
    auto cont_upto_end = [&](uint32_t rel) -> uint32_t {
        const uint32_t sl = slot_s(rel), L = (rel & (kWin - 1)) >> 4, k = rel & 15u;
        uint32_t n = lds32v(sl + kSlotText + 32);
#pragma unroll
        for (int w = 0; w < 8; w++) {
            const int left = (int)L - 4 * w;  // chunks of this word that lie before chunk L
            const uint32_t mask = left >= 4 ? 0xffffffffu : (left <= 0 ? 0u : ((1u << (8 * left)) - 1u));
            n = __dp4a(lds32v(sl + kSlotText + 4 * w) & mask, 0x01010101u, n);
        }
        return n + cont_prefix(sl + 16 + 16 * L, k + 1);
    };

    unsigned int claimed = 0;
    if (lane == 0) claimed = atomicAdd(task_counter, 1u);
    for (;;) {
        const unsigned int task = __shfl_sync(0xffffffffu, claimed, 0);
        if ((int64_t)task >= P.n_tasks) break;
        if (lane == 0) claimed = atomicAdd(task_counter, 1u);  // the next one: its round trip overlaps this task
        const int64_t t_lo = P.origin + (int64_t)task * T;
        if (t_lo >= vhi || t_lo + (int64_t)T <= vlo) {
            if (lane == 0) {
                out.unit_counts[task] = 0;
                if (CP) task_cont[task] = 0;
            }
            continue;
        }
        // the task's part of the stream, [lo_r, hi_r) relative to t_lo; positions (= index of a window's LAST byte) from
        // plo_r on can end a match: the W-byte window must lie inside the stream
        const uint32_t lo_r = (uint32_t)max(vlo - t_lo, (int64_t)0), hi_r = (uint32_t)min(vhi - t_lo, (int64_t)T);
        const uint32_t plo_r = (uint32_t)max((int64_t)lo_r, vlo + (int64_t)W - 1 - t_lo);
        const uint8_t *tptr = B.bytes + t_lo;  // (may point before the buffer: only [lo_r, hi_r) is ever dereferenced)
        const uint32_t wfirst = lo_r & ~(kWin - 1), wlast = (hi_r - 1) & ~(kWin - 1);
        auto load16 = [&](uint32_t rel) -> uint4 {  // 16 bytes at rel (may be "negative": the history before the task)
            const int64_t q = t_lo + (int64_t)(int32_t)rel;
            return load_chunk(B.bytes, q, vlo, vhi);
        };

        // ---- haystack bookkeeping: lane l caches the start of haystack hb + l, relative to the task (saturated) ----
        int64_t hb;
        {
            const int64_t lo = t_lo + lo_r;
            int64_t h = P.avg_len ? (int64_t)((uint64_t)(lo - stream_lo) / P.avg_len) : 0;
            if (h >= B.n_haystacks) h = B.n_haystacks - 1;
            if (!(__ldg(B.offsets + h) <= lo && lo < __ldg(B.offsets + h + 1))) h = find_haystack(B, lo);
            hb = h;
        }
        auto load_offc = [&](int64_t base) -> int32_t {
            const int64_t idx = base + lane;
            if (idx > B.n_haystacks) return 0x7fffffff;
            const int64_t d = __ldg(B.offsets + idx) - t_lo;
            return (int32_t)max(min(d, (int64_t)0x7ffffffe), (int64_t)-0x7fffffff);
        };
        int32_t offc = load_offc(hb);
        int32_t next_start = __shfl_sync(0xffffffffu, offc, 1);  // start of haystack hb + 1
        // Haystack containing the byte at rel, and its start (relative).  The shuffles are executed by the whole warp (rel
        // may differ per lane).  Positions before the cached range (queued in an earlier window) walk back from it; a
        // window with more than 31 haystack starts (haystacks of a few bytes) falls back to a search.
        auto hay_of = [&](uint32_t rel, int32_t &hs) -> int64_t {
            const int32_t p = (int32_t)rel;
            uint32_t l = 0;
#pragma unroll
            for (int step = 16; step >= 1; step >>= 1) {
                const uint32_t c = l + step;
                const int32_t v = __shfl_sync(0xffffffffu, offc, c & 31);
                if (c < 32 && v <= p) l = c;
            }
            hs = __shfl_sync(0xffffffffu, offc, l);
            int64_t h = hb + l;
            if (hs > p) {
                // before the cache: the haystack is a few entries back
                const int64_t pa = t_lo + p;
                int64_t step = 1, below = hb;
                while (below > 0 && __ldg(B.offsets + below) > pa) {
                    below = max(below - step, (int64_t)0);
                    step <<= 1;
                }
                h = below;
                while (h + 1 < B.n_haystacks && __ldg(B.offsets + h + 1) <= pa) h++;  // last haystack that starts at or before p
                hs = (int32_t)max(__ldg(B.offsets + h) - t_lo, (int64_t)-0x7fffffff);
            } else if (l == 31 && h + 1 < B.n_haystacks && __ldg(B.offsets + h + 1) <= t_lo + p) {
                h = find_haystack(B, t_lo + p);
                hs = (int32_t)max(__ldg(B.offsets + h) - t_lo, (int64_t)-0x7fffffff);
            }
            return h;
        };

        uint32_t n_emitted = 0, q1n = 0, q2n = 0;
        uint32_t q1_head = 0;  // window index of the first queue's first entry (valid while the queue is not empty)
        uint32_t cp_before = 0;             // code points: continuation bytes of the task before the current window
        uint32_t wrel = wfirst;

        // ---- stage 2: exact verification of the first (up to) 32 positions of the second queue ----
        auto round2 = [&]() {
            const uint32_t n = min(q2n, 32u);
            const bool active = lane < n;
            uint4 ent2 = make_uint4(0, 0, 0, 0);  // position, key (2 words), continuation bytes before the end
            if (active) ent2 = lds128(q2_s + lane * kQ2Entry);
            const uint32_t rel = ent2.x, aux = ent2.w;
            int32_t hs;
            const int64_t h = hay_of(active ? rel : max(wrel, lo_r), hs);
            uint32_t best = kSieveNoNode, cnt = 0;
            if (active && (int32_t)rel - (int32_t)(W - 1) >= hs) {
                const uint32_t klo = ent2.y, khi = ent2.z;
                const uint32_t x = klo + khi * kMixHi;
                uint32_t s = __umulhi(x * kMulSlot, sv.ht_size);
                uint32_t v = kSieveNoNode;
                for (;;) {
                    const uint4 ent = __ldg(reinterpret_cast<const uint4 *>(sv.ht + s));
                    if (ent.z == kSieveNoNode) break;
                    if (ent.x == klo && ent.y == khi) {
                        v = ent.z;
                        break;
                    }
                    s = (s + 1) & (sv.ht_size - 1);
                }
                // walk towards the pattern start: node v = the d bytes that end at rel
                uint32_t d = W;
                uint2 na = make_uint2(0, 0);
                if (v != kSieveNoNode) na = __ldg(reinterpret_cast<const uint2 *>(sv.na + v));
                while (v != kSieveNoNode) {
                    if (na.y & kNodeTerminal) best = v;
                    const uint32_t nk = (na.y >> 8) & 0x1ffu;
                    if (nk == 0 || (int32_t)rel - (int32_t)d < hs) break;  // no longer pattern, or it would start before the haystack
                    uint32_t b = __ldg(tptr + ((int64_t)(int32_t)rel - (int64_t)d));
                    if (FOLD) b = ascii_fold(b);
                    uint32_t c = kSieveNoNode;
                    uint2 nc = make_uint2(0, 0);
                    if (nk <= 8) {
                        for (uint32_t t = 0; t < nk; t++) {
                            const uint2 cand = __ldg(reinterpret_cast<const uint2 *>(sv.na + na.x + t));
                            const uint32_t cb = cand.y & 0xffu;
                            if (cb >= b) {
                                if (cb == b) {
                                    c = na.x + t;
                                    nc = cand;
                                }
                                break;
                            }
                        }
                    } else {
                        uint32_t l0 = 0, l1 = nk;  // first child with byte >= b
                        while (l0 < l1) {
                            const uint32_t mid = (l0 + l1) >> 1;
                            if ((__ldg(&sv.na[na.x + mid].meta) & 0xffu) < b)
                                l0 = mid + 1;
                            else
                                l1 = mid;
                        }
                        if (l0 < nk) {
                            const uint2 cand = __ldg(reinterpret_cast<const uint2 *>(sv.na + na.x + l0));
                            if ((cand.y & 0xffu) == b) {
                                c = na.x + l0;
                                nc = cand;
                            }
                        }
                    }
                    v = c;
                    na = nc;
                    d++;
                }
                if (best != kSieveNoNode) cnt = __ldg(&sv.nb[best].chain_cnt);
            }
            const uint32_t hits = __ballot_sync(0xffffffffu, cnt != 0);
            if (hits) {
                uint32_t total;
                const uint32_t exc = warp_excl_scan(cnt, lane, &total);
                unsigned long long rbase = 0;
                if (lane == 0) rbase = atomicAdd(out.raw_total, (unsigned long long)total);
                rbase = __shfl_sync(0xffffffffu, rbase, 0);
                if (cnt) {
                    unsigned long long idx = rbase + exc;
                    uint32_t seq = n_emitted + exc;
                    const uint32_t end_rel = (uint32_t)((int32_t)rel + 1 - hs);
                    for (uint32_t u = best; u != kSieveNoNode;) {
                        const uint4 nb = __ldg(reinterpret_cast<const uint4 *>(sv.nb + u));  // own_off, own_cnt, term_link, depth
                        for (uint32_t t = 0; t < nb.y; t++, idx++, seq++) {
                            if (idx < out.cap) {
                                const uint32_t pid = __ldg(sv.pids + nb.x + t);
                                reinterpret_cast<uint4 *>(out.raw)[idx] = make_uint4((uint32_t)h, pid, end_rel - nb.w, end_rel);
                                out.raw_seq[idx] = seq;
                                out.raw_unit[idx] = task;
                                if (CP) out.raw_aux[idx] = aux;
                            }
                        }
                        u = nb.z;
                    }
                }
                n_emitted += total;
            }
            // pop the round
            uint4 keep = make_uint4(0, 0, 0, 0);
            const bool mv = 32 + lane < q2n;
            if (mv) keep = lds128(q2_s + (32 + lane) * kQ2Entry);
            __syncwarp();
            if (mv) sts128(q2_s + lane * kQ2Entry, keep);
            q2n -= n;
            __syncwarp();
        };

        // ---- stage 1: second filter and the on-chip walk for the first (up to) 32 positions of the first queue ----
        auto round1 = [&]() {  // (the caller has made room for 32 survivors in the second queue)
            const uint32_t n = min(q1n, 32u);
            const bool active = lane < n;
            uint32_t rel = 0, klo = 0, khi = 0;
            bool go = false;
            if (active) {
                rel = lds32v(q1_s + lane * 4u);
                stash_key(rel, klo, khi);
                uint32_t x = klo + khi * kMixHi;
                if (sec_has(x)) {
                    const uint32_t ta = text_s(rel);
                    uint32_t d = W;
                    for (;;) {
                        if (d >= sv.last_level && sv.max_pat_len > sv.last_level) {
                            go = true;  // patterns longer than this are not on chip (nor are this level's end marks)
                            break;
                        }
                        if (((sv.term_levels >> d) & 1u) && sec_has(x ^ kSaltTerm)) {
                            go = true;  // a pattern of length d may end here
                            break;
                        }
                        if (d >= sv.last_level) break;
                        const uint32_t b = lds8(ta - d);  // the byte before the d-byte suffix
                        x = sieve_step(x, b);
                        d++;
                        if (!sec_has(x)) break;
                    }
                }
            }
            const uint32_t surv = __ballot_sync(0xffffffffu, go);
            if (surv) {
                // survivors take their key (and, code points, their count) along: stage 2 needs nothing from the ring
                if (go) sts128(q2_s + (q2n + __popc(surv & ((1u << lane) - 1u))) * kQ2Entry, make_uint4(rel, klo, khi, CP ? cont_upto_end(rel) : 0u));
                q2n += __popc(surv);
            }
            // pop the round
            uint32_t keep = 0;
            const bool mv = 32 + lane < q1n;
            if (mv) keep = lds32v(q1_s + (32 + lane) * 4u);
            __syncwarp();
            if (mv) q1_store(lane, keep);
            q1n -= n;
            q1_head = __shfl_sync(0xffffffffu, keep, 0) >> 9;
            __syncwarp();
        };

        // case-insensitive: the text as the image expects it (the next window is folded when it becomes the current one,
        // not at its load: the load stays in flight while this window is scanned)
        auto fold16 = [&](uint4 v) -> uint4 {
            if (FOLD) v = make_uint4(ascii_fold4(v.x), ascii_fold4(v.y), ascii_fold4(v.z), ascii_fold4(v.w));
            return v;
        };
        uint32_t carry_z = 0, carry_w = 0;
        {
            const uint4 c = fold16(load16(wrel - 16));
            carry_z = c.z;
            carry_w = c.w;
            if (lane == 0) sts128(text_s(wrel) - 16, c);
        }
        uint4 cur = fold16(load16(wrel + 16 * lane));
        uint4 nxt = make_uint4(0, 0, 0, 0);
        uint32_t cur_slot = slot_s(wrel);  // the ring slot of the current window

        for (;; wrel += kWin) {
            if (wrel + kWin <= wlast) {
                // the next window (a window takes a warp a few microseconds: one load in flight per lane covers the latency);
                // whole windows inside the stream (all but a task's edges) take the direct load
                if (wrel + kWin >= lo_r && wrel + 2 * kWin <= hi_r)
                    nxt = __ldg(reinterpret_cast<const uint4 *>(tptr + (wrel + kWin + 16 * lane)));
                else
                    nxt = load16(wrel + kWin + 16 * lane);
            }
            // ---- fast path: first filter probe for the 16 positions of this lane ----
            uint32_t pz = __shfl_up_sync(0xffffffffu, cur.z, 1), pw = __shfl_up_sync(0xffffffffu, cur.w, 1);
            if (lane == 0) {
                pz = carry_z;
                pw = carry_w;
            }
            const uint32_t a[6] = {pz, pw, cur.x, cur.y, cur.z, cur.w};
            uint32_t acc = 0;
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const int j = 2 + (k >> 2), r = k & 3;
                const uint32_t wlo = r == 3 ? a[j] : __funnelshift_r(a[j - 1], a[j], 8 * (r + 1));
                uint32_t x;
                if (WC == 3) {
                    // W == 5: the one byte before the 4-byte window, picked straight out of its word
                    x = wlo + __byte_perm(a[1 + (k >> 2)], 0u, 0x4440u | (uint32_t)r) * kMixHi;
                } else if (WC == 2) {
                    const uint32_t whi = r == 3 ? a[j - 1] : __funnelshift_r(a[j - 2], a[j - 1], 8 * (r + 1));
                    x = wlo + (whi >> sh_hi) * kMixHi;
                } else if (WC == 1) {
                    x = wlo;
                } else {
                    x = wlo >> sh_lo;
                }
                const uint32_t p = x * kMulA;
                const uint32_t word = lds32(bloom_s + __umulhi(p, n_words) * 4u);
                acc = __funnelshift_r(acc, shf_r_wrap(word, 0u, p), 1);  // bit (p & 31) of the word -> top of acc
            }
            uint32_t m1 = acc >> 16;
            // positions outside [plo_r, hi_r) cannot end a match (first and last window of the task only)
            if (wrel < plo_r || wrel + kWin > hi_r) {
                const int32_t q = (int32_t)(wrel + 16 * lane);
                const int from = min(max((int32_t)plo_r - q, 0), 16), to = min(max((int32_t)hi_r - q, 0), 16);
                m1 &= ((1u << to) - 1u) & ~((1u << from) - 1u);
            }
            const uint32_t wend = min(wrel + kWin, hi_r);  // one past the last stream byte of this window
            // does the cached range still start at the haystack that holds this window's first byte?
            if (next_start <= (int32_t)wrel) {
                const int32_t first = (int32_t)max(wrel, lo_r);
                const uint32_t ahead = __popc(__ballot_sync(0xffffffffu, offc <= first));
                hb = ahead == 32 ? find_haystack(B, t_lo + first) : hb + ahead - 1;
                offc = load_offc(hb);
                next_start = __shfl_sync(0xffffffffu, offc, 1);
            }
            uint32_t wc = 0;  // code points: continuation bytes in this lane's chunk
            bool starts_inside = false, wany = false;
            if (CP) {
                const bool high = ((cur.x | cur.y | cur.z | cur.w) & 0x80808080u) != 0;
                if (high) wc = cont_bytes(cur.x) + cont_bytes(cur.y) + cont_bytes(cur.z) + cont_bytes(cur.w);
                wany = __any_sync(0xffffffffu, high);
                // haystacks that START in this window record how many continuation bytes the task has seen before them
                starts_inside = next_start < (int32_t)wend || __shfl_sync(0xffffffffu, offc, 0) >= (int32_t)max(wrel, lo_r);
            }
            const bool any = __any_sync(0xffffffffu, m1 != 0);
            uint32_t tot1 = 0, ex1 = 0;  // survivors of the first probe in this window, and in the lanes before this one
            if (any || starts_inside) {
                const uint32_t sl = cur_slot;
                sts128(sl + 16 + 16 * lane, cur);
                if (CP) {
                    asm volatile("st.shared.u8 [%0], %1;\n" ::"r"(sl + kSlotText + lane), "r"(wc) : "memory");
                    if (lane == 0) asm volatile("st.shared.u32 [%0], %1;\n" ::"r"(sl + kSlotText + 32), "r"(cp_before) : "memory");
                }
                __syncwarp();
                if (CP && starts_inside) {
                    uint32_t exw = 0, wtot = 0;
                    if (wany) exw = warp_excl_scan(wc, lane, &wtot);
                    // continuation bytes in [lo_r, pos) for pos in [wrel, wrel + 512]; executed by the whole warp
                    auto cont_before = [&](uint32_t pos) -> uint32_t {
                        const uint32_t rl = pos - wrel;
                        const uint32_t L = min(rl >> 4, 31u);
                        const uint32_t ex = __shfl_sync(0xffffffffu, exw, L);
                        if (wtot == 0) return cp_before;  // (an ASCII window: nothing to add)
                        return cp_before + ex + cont_prefix(sl + 16 + 16 * L, rl - 16 * L);
                    };
                    for (;;) {
                        const bool mine = offc >= (int32_t)max(wrel, lo_r) && offc < (int32_t)wend && hb + lane < B.n_haystacks;
                        const uint32_t c = cont_before(mine ? (uint32_t)offc : wrel);
                        if (mine) hay_cont[hb + lane] = c;
                        // more than 32 starts in one window: move the cache on and repeat
                        if (__shfl_sync(0xffffffffu, offc, 31) >= (int32_t)wend || hb + 31 >= B.n_haystacks) break;
                        hb += 31;
                        offc = load_offc(hb);
                        next_start = __shfl_sync(0xffffffffu, offc, 1);
                    }
                }
                if (any) ex1 = warp_excl_scan(__popc(m1), lane, &tot1);
            }
            if (CP && wany) cp_before += __reduce_add_sync(0xffffffffu, wc);
            // ---- queue this window's survivors, in stream order (a lane's go behind those of the lanes before it), and
            // run the later stages: ONE instance of each in the code (they are large; four inlined copies of them cost more
            // in instruction fetch than the calls they saved).  A window with more survivors than the first queue has room
            // for is pushed in pieces.  Stage 1 runs when 32 positions wait, or when their text is about to leave the
            // ring; the last window of the task drains both queues.
            {
                const bool last = wrel >= wlast;
                const uint32_t next_w = (wrel >> 9) + 1;
                uint32_t base = 0;
                for (;;) {
                    const uint32_t take = min(tot1 - base, kQueueCap - q1n);
                    if (take) {
                        if (q1n == 0) q1_head = wrel >> 9;
                        uint32_t g = ex1 - base;  // rank of this lane's first survivor in this piece (wraps below 0 for those already pushed)
                        uint32_t at = q1_s + (q1n + g) * 4u;
                        const uint32_t pos0 = wrel + 16 * lane - 1;
                        for (uint32_t m = m1; m; m &= m - 1, g++, at += 4)
                            if (g < take) asm volatile("st.shared.u32 [%0], %1;\n" ::"r"(at), "r"(pos0 + (uint32_t)__ffs(m)) : "memory");
                        q1n += take;
                        base += take;
                        __syncwarp();
                    }
                    const bool drain = last && base >= tot1;
                    for (;;) {
                        const bool do2 = q2n > 32 || (drain && q1n == 0 && q2n != 0);
                        const bool do1 = q1n >= 32 || (q1n != 0 && (drain || q1_head + R <= next_w));
                        if (do2)
                            round2();
                        else if (do1)
                            round1();
                        else
                            break;
                    }
                    if (base >= tot1) break;
                }
                if (last) break;
            }
            __syncwarp();  // every lane is done with the slot before its history is replaced
            cur_slot += kSlotBytes;
            if (cur_slot == ring_end) cur_slot = ring_s;
            if (lane == 31) sts128(cur_slot, cur);  // the next window's history
            carry_z = __shfl_sync(0xffffffffu, cur.z, 31);
            carry_w = __shfl_sync(0xffffffffu, cur.w, 31);
            cur = nxt;
            if (FOLD) cur = fold16(cur);
        }
        if (lane == 0) out.unit_counts[task] = n_emitted;
        if (CP && lane == 0) task_cont[task] = cp_before;
        __syncwarp();
    }
}

}  // namespace acb
