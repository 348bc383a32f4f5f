// capi.cu -- the C ABI (include/acb200.h): planning, kernel dispatch, ordering passes.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include <cooperative_groups.h>

#include "repair.cuh"
#include "scan_staged.cuh"
#include "scan_global.cuh"
#include "scan_sieve.cuh"

namespace acb {

// ---------------------------------------------------------------------------
// plain kernel: the exact scanner over whole haystacks, table in global memory
// (units = haystacks; used when no hot image is given, and as the cross-check
// of the staged + repair path in the tests)
// ---------------------------------------------------------------------------
template <int MODE, bool CP>
__global__ void __launch_bounds__(128) scan_plain_kernel(DevImage im, Batch B, Sink out) {
    for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h < B.n_haystacks; h += (int64_t)gridDim.x * blockDim.x) {
        const int64_t hs = B.offsets[h], he = B.offsets[h + 1];
        PieceCtx c;
        c.base = B.bytes + hs;
        c.at = 0;
        c.stop = c.limit = (uint32_t)(he - hs);
        c.emit_from = 0;
        c.state = kRoot;
        c.have = 0;
        c.last_pid = c.last_end = 0;
        c.hay = (uint32_t)h;
        c.hay_delta = 0;
        c.unit = (uint32_t)h;
        c.nemit = 0;
        c.cp_pos = 0;
        c.cp_cont = 0;
        exact_scan<MODE, CP>(c, im, out, false, 0, HotMap{nullptr, 0});
        out.unit_counts[h] = c.nemit;
    }
}

// ---------------------------------------------------------------------------
// profile kernel: walks a sample of the input through the dense table and
// counts state visits; the host ranks states by these counts to choose the rows
// the staged kernel keeps in shared memory (automaton.cpp: build_hot_image)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
profile_kernel(DevImage im, Batch B, uint32_t *visits, int64_t n_samples, uint32_t max_bytes, int restart_on_match) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_samples) return;
    // sample i reads max_bytes at stream position lo + i * (len / n_samples), staying inside one haystack
    const int64_t lo = B.offsets[0], hi = B.offsets[B.n_haystacks];
    if (hi <= lo) return;
    const int64_t p0 = lo + ((hi - lo) / n_samples) * i;
    const int64_t h = find_haystack(B, p0);
    const uint8_t *p = B.bytes + p0;
    uint64_t len = (uint64_t)(B.offsets[h + 1] - p0);
    if (len > max_bytes) len = max_bytes;
    uint32_t s = kRoot;
    for (uint64_t k = 0; k < len; k++) {
        const uint32_t e = __ldg(im.trans + (size_t)s * im.n_cols + __ldg(im.colmap + __ldg(p + k)));
        s = e & kStateMask;
        if (s == kDead || (restart_on_match && (e & kMatchFlag))) s = kRoot;
        atomicAdd(visits + s, 1u);
    }
}

// ---------------------------------------------------------------------------
// exclusive prefix sum u32[n] (strided) -> u64[n+1]: building blocks of the epilogue kernel's phases 1 and 2
// ---------------------------------------------------------------------------
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ __forceinline__ unsigned long long block_exclusive_scan(unsigned long long v, unsigned long long *total) {
    __shared__ unsigned long long warp_sums[kScanThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = lane < kScanThreads / 32 ? warp_sums[lane] : 0;
#pragma unroll
        for (int d = 1; d < kScanThreads / 32; d <<= 1) {
            unsigned long long y = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += y;
        }
        if (lane < kScanThreads / 32) warp_sums[lane] = w;
    }
    __syncthreads();
    const unsigned long long before = warp ? warp_sums[warp - 1] : 0;
    *total = warp_sums[kScanThreads / 32 - 1];
    __syncthreads();
    return before + x - v;
}

// item i = in[i * stride] (+ in[i * stride + 1] when PAIR: the two slots of a segment) for i in [0, n); one tile.
// dense != null: the items are also written there, packed (a strided source is read only once that way).
template <bool PAIR>
__device__ __forceinline__ unsigned long long scan_item(const uint32_t *in, uint32_t stride, uint64_t i) {
    if (PAIR) {
        const uint2 v = *reinterpret_cast<const uint2 *>(in + i * stride);
        return (unsigned long long)v.x + v.y;
    }
    return in[i * stride];
}

template <bool PAIR>
__device__ __forceinline__ void tile_sum_body(const uint32_t *in, uint32_t stride, uint64_t n, unsigned long long *tile_sums, uint64_t tile,
                                              uint32_t *dense) {
    const uint64_t base = tile * kScanTile + (uint64_t)threadIdx.x * kScanItems;
    unsigned long long v = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; i++)
        if (base + i < n) {
            const unsigned long long x = scan_item<PAIR>(in, stride, base + i);
            if (dense) dense[base + i] = (uint32_t)x;
            v += x;
        }
    unsigned long long total;
    block_exclusive_scan(v, &total);
    if (threadIdx.x == 0) tile_sums[tile] = total;
}

// sum of tile_sums[0 .. tile): every block works out the start of its own tile (a few hundred values at most for a
// batch, a few thousand for a multi-gigabyte buffer) instead of waiting for one block to scan them all
__device__ __forceinline__ unsigned long long tile_prefix(const unsigned long long *tile_sums, uint64_t tile) {
    unsigned long long v = 0;
    for (uint64_t i = threadIdx.x; i < tile; i += kScanThreads) v += tile_sums[i];
    unsigned long long total;
    block_exclusive_scan(v, &total);
    return total;
}

template <bool PAIR>
__device__ __forceinline__ void tile_apply_body(const uint32_t *in, uint32_t stride, uint64_t n, const unsigned long long *tile_sums,
                                                unsigned long long *out, uint64_t tile) {
    const unsigned long long tile_start = tile_prefix(tile_sums, tile);
    const uint64_t base = tile * kScanTile + (uint64_t)threadIdx.x * kScanItems;
    unsigned long long vals[kScanItems], v = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; i++) {
        vals[i] = base + i < n ? scan_item<PAIR>(in, stride, base + i) : 0;
        v += vals[i];
    }
    unsigned long long total;
    unsigned long long run = tile_start + block_exclusive_scan(v, &total);
#pragma unroll
    for (int i = 0; i < kScanItems; i++) {
        if (base + i < n) out[base + i] = run;
        run += vals[i];
        if (base + i + 1 == n) out[n] = run;
    }
}

// ---------------------------------------------------------------------------
// final placement: raw match i of unit u with rank r goes to unit_offsets[u] + r
// (segments: minus the matches the repair pass superseded); code point fix-up
// ---------------------------------------------------------------------------
struct OrderArgs {
    const acb_match *raw;
    const uint32_t *raw_seq, *raw_unit, *raw_aux;
    unsigned long long raw_cap;
    const unsigned long long *raw_total;
    const unsigned long long *unit_offsets;  // segments: one entry per SEGMENT (slot 0 first, then slot 1); else per unit
    const uint32_t *unit_counts;
    const SegInfo *seg_info;             // null: units are haystacks (plain kernel)
    const unsigned long long *cont_cum;  // exclusive prefix sum of SegInfo.cont_tail (code points + segments)
    const int64_t *hay_offsets;
    const uint32_t *pat_cplen;
    int64_t origin;
    uint32_t seg_bytes;
    int codepoints;
    acb_match *out;
    unsigned long long out_cap;
};

__device__ __forceinline__ void order_body(const OrderArgs &A) {
    unsigned long long n = *A.raw_total;
    if (n > A.raw_cap) n = A.raw_cap;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t u = A.raw_unit[i];
        uint32_t seq = A.raw_seq[i];
        if (A.seg_info && (u & 1u)) {
            const uint32_t drop = A.seg_info[u >> 1].drop;
            if (seq < drop) continue;  // superseded by the repair pass
            seq -= drop;
        }
        // a segment's slot-1 matches (the scan kernel's) come after its slot-0 matches (the repair pass's)
        const unsigned long long dst =
            A.seg_info ? A.unit_offsets[u >> 1] + ((u & 1u) ? A.unit_counts[u & ~1u] : 0u) + seq : A.unit_offsets[u] + seq;
        if (dst >= A.out_cap) continue;
        uint4 r = reinterpret_cast<const uint4 *>(A.raw)[i];  // haystack, pattern, start, end (bytes)
        if (A.codepoints) {
            unsigned long long cont = A.raw_aux[i];  // continuation bytes from the counting origin to the match end
            if (A.seg_info) {
                const int64_t j = u >> 1;
                const int64_t hs = A.hay_offsets[r.x];
                if (hs < A.origin + j * (int64_t)A.seg_bytes) {
                    // the match's haystack began in an earlier segment: add what those segments counted
                    const int64_t j0 = (hs - A.origin) / (int64_t)A.seg_bytes;
                    cont += A.cont_cum[j] - A.cont_cum[j0];
                }
            }
            const uint32_t end_cp = r.w - (uint32_t)cont;
            r.w = end_cp;
            r.z = end_cp - A.pat_cplen[r.y];
        }
        reinterpret_cast<uint4 *>(A.out)[dst] = r;
    }
}

// The head of dev_scratch: counters the kernels accumulate into.  Zero when a workspace is first used (the caller
// allocates it zeroed) and zero again after every scan (the epilogue's last phase resets them).
constexpr int kAccQueue = 0;    // u32 task counter of the staged kernel | u32 "some speculated segment start was wrong"
constexpr int kAccRaw = 2;      // raw matches emitted (also the allocation cursor of the raw buffer)
constexpr int kAccGroups = 3;   // 16-byte groups in the stream
constexpr int kAccTraps = 4;    // times a lane left the hot table
constexpr int kAccRepairs = 5;  // segment boundaries repaired
constexpr int kAccWords = 8;

// per-haystack CSR offsets into the ordered output (binary search per haystack) + the totals
__device__ __forceinline__ void
match_offsets_body(const acb_match *out, const unsigned long long *unit_offsets, uint64_t n_units, unsigned long long *totals,
                   unsigned long long *acc, unsigned long long raw_cap, unsigned long long out_cap, int64_t n_haystacks,
                   unsigned long long *match_offsets) {
    const unsigned long long total = unit_offsets[n_units];
    const unsigned long long avail = total < out_cap ? total : out_cap;
    for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h <= n_haystacks; h += (int64_t)gridDim.x * blockDim.x) {
        unsigned long long lo = 0, hi = avail;  // first index whose haystack >= h
        while (lo < hi) {
            const unsigned long long mid = (lo + hi) >> 1;
            if ((int64_t)out[mid].haystack < h)
                lo = mid + 1;
            else
                hi = mid;
        }
        match_offsets[h] = (h == n_haystacks) ? total : lo;
        if (h == 0) {
            // publish the totals, and leave the workspace's counters at zero for the next scan (nothing else
            // touches them in this phase): a scan needs no clearing launch in front of it
            const unsigned long long raw_total = acc[kAccRaw];
            totals[0] = total;
            totals[1] = (raw_total <= raw_cap && total <= out_cap) ? 1 : 0;  // complete?
            totals[2] = acc[kAccGroups];
            totals[3] = acc[kAccTraps];
            totals[4] = raw_total;
            totals[5] = acc[kAccRepairs];
            totals[6] = totals[7] = 0;
            acc[kAccRaw] = acc[kAccGroups] = acc[kAccTraps] = acc[kAccRepairs] = 0;
            acc[kAccQueue] = 0;  // the scan kernel's task queue (low word) and the repair flag (high word)
        }
    }
}

// ---------------------------------------------------------------------------
// everything after the scan in ONE cooperative kernel (grid-wide barriers
// between the phases): repair -> prefix sums -> ordered output -> per-haystack
// offsets.  (As ten separate launches this cost more than the work they do.)
// ---------------------------------------------------------------------------
struct EpilogueArgs {
    DevImage im;
    Batch B;
    SegPlan P;
    Sink out;
    SegInfo *seg_info;
    unsigned long long *totals, *acc;
    const uint32_t *unit_counts;
    uint64_t n_units;
    unsigned long long *tile_sums, *unit_offsets;
    const uint32_t *cont_tail;  // null: no code point prefix needed
    uint64_t n_segments;
    unsigned long long *cont_tiles, *cont_cum;
    uint32_t *cont_dense;  // packed copy of SegInfo.cont_tail
    OrderArgs order;
    unsigned long long *match_offsets;
    unsigned int *need_repair;  // zeroed with the totals; set when a speculated segment start was wrong
    int do_repair;
};

template <int MODE, bool CP>
__global__ void __launch_bounds__(kScanThreads) epilogue_kernel(EpilogueArgs E) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    // segments: one scan item per segment (its two slots summed); plain kernel: one per haystack
    const bool pairs = E.order.seg_info != nullptr;
    const uint64_t n_items = pairs ? E.n_units / 2 : E.n_units;
    const uint64_t tiles = (n_items + kScanTile - 1) / kScanTile;
    const uint64_t ctiles = E.cont_tail ? (E.n_segments + kScanTile - 1) / kScanTile : 0;
    auto sums = [&]() {
        // (one tile space for both arrays, so that different blocks take the count tiles and the tail tiles)
        for (uint64_t tt = blockIdx.x; tt < tiles + ctiles; tt += gridDim.x) {
            if (tt >= tiles)  // SegInfo.cont_tail sits at a 32-byte stride: read it once, keep a packed copy for the second pass
                tile_sum_body<false>(E.cont_tail, 8, E.n_segments, E.cont_tiles, tt - tiles, E.cont_dense);
            else if (pairs)
                tile_sum_body<true>(E.unit_counts, 2, n_items, E.tile_sums, tt, nullptr);
            else
                tile_sum_body<false>(E.unit_counts, 1, n_items, E.tile_sums, tt, nullptr);
        }
    };
    // phase 1: tile sums of the counts as the scan kernel left them, and -- non-overlapping searches -- the check of
    // every speculated segment start against the state its predecessor ended in (repair.cuh has the same rule)
    if (E.do_repair) {
        unsigned int dirty = 0;
        for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x + 1; k < E.n_segments; k += (uint64_t)gridDim.x * blockDim.x) {
            const uint32_t spec = E.seg_info[k].spec_state;
            if (spec == kNoState) continue;  // the segment starts with a haystack (or outside all of them)
            const uint4 prev = *reinterpret_cast<const uint4 *>(E.seg_info + k - 1);  // spec, end_state, end_over, head_count
            dirty |= (prev.z != 0 || prev.y != spec) ? 1u : 0u;
        }
        if (__any_sync(0xffffffffu, dirty) && (threadIdx.x & 31) == 0) atomicOr(E.need_repair, 1u);
    }
    sums();
    grid.sync();
    if (E.do_repair && *reinterpret_cast<volatile unsigned int *>(E.need_repair)) {
        // rare: some guess was wrong.  Redo those places exactly, then count again.
        repair_body<MODE, CP>(E.im, E.B, E.P, E.out, E.seg_info, E.acc + kAccRepairs);
        grid.sync();
        sums();
        grid.sync();
    }
    // phase 2: exclusive prefix sums (every block derives its tile's start from the tile sums)
    for (uint64_t tt = blockIdx.x; tt < tiles + ctiles; tt += gridDim.x) {
        if (tt >= tiles)
            tile_apply_body<false>(E.cont_dense, 1, E.n_segments, E.cont_tiles, E.cont_cum, tt - tiles);
        else if (pairs)
            tile_apply_body<true>(E.unit_counts, 2, n_items, E.tile_sums, E.unit_offsets, tt);
        else
            tile_apply_body<false>(E.unit_counts, 1, n_items, E.tile_sums, E.unit_offsets, tt);
    }
    grid.sync();
    // phase 3: ordered output; phase 4: per-haystack offsets into it
    order_body(E.order);
    grid.sync();
    match_offsets_body(E.order.out, E.unit_offsets, n_items, E.totals, E.acc, E.order.raw_cap, E.order.out_cap, E.B.n_haystacks,
                       E.match_offsets);
}


// ---------------------------------------------------------------------------
// Epilogue of the sieve scan (scan_sieve.cuh).  The scan leaves the OVERLAPPING
// match list as raw records tagged (task, rank in task); tasks are in stream
// order, so the ordered list needs prefix sums and one placement pass, no sort.
// Non-overlapping searches then SELECT from that list, per haystack (SURVEY.md
// 8c: "among occurrences with start >= s pick the minimum of (end, start, pid) /
// (start, pid) / (start, -end, pid)"; the list is sorted by (end, start, pid)),
// and the selected records are packed.  One cooperative launch.
// ---------------------------------------------------------------------------
struct SieveEpiArgs {
    Batch B;
    uint32_t *unit_counts;               // [n_tasks] from the scan; later [n_haystacks] selected per haystack
    uint64_t n_tasks;
    unsigned long long *tile_sums, *unit_offsets;  // unit_offsets: [n_tasks + 1]; later [n_haystacks] first record of each haystack
    const uint32_t *cont_tail;           // [n_tasks] (code points): continuation bytes in each task
    const uint32_t *hay_cont;            // [n_haystacks] (code points): continuation bytes between the start of the task a haystack starts in and the haystack
    unsigned long long *cont_tiles, *cont_cum;
    const acb_match *raw;
    const uint32_t *raw_seq, *raw_unit, *raw_aux;
    unsigned long long raw_cap;
    acb_match *ordered;                  // the overlapping list, ordered (overlapping search: the output buffer)
    acb_match *final_out;                // non-overlapping: the output buffer
    unsigned long long out_cap;
    const uint32_t *pat_cplen;
    int64_t origin;
    uint32_t task_bytes;
    uint32_t max_pat_len;
    int longest;                         // kModeLeftmost: 1 = LeftmostLongest, 0 = LeftmostFirst
    unsigned long long *totals, *acc, *match_offsets;
};

// index of the first record of `list[0 .. n)` whose haystack is >= h
__device__ __forceinline__ unsigned long long first_of_haystack(const acb_match *list, unsigned long long n, int64_t h) {
    unsigned long long lo = 0, hi = n;
    while (lo < hi) {
        const unsigned long long mid = (lo + hi) >> 1;
        if ((int64_t)list[mid].haystack < h)
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo;
}

// The reference's non-overlapping iteration over ONE haystack, as a selection from its overlapping list r[0 .. n)
// (sorted by end, start, pattern).  The selected records are packed to the front; returns how many.
template <int MODE>
__device__ __forceinline__ uint32_t select_non_overlapping(acb_match *r, unsigned long long n, uint32_t max_len, int longest) {
    unsigned long long w = 0;
    uint32_t s = 0;  // the search restarts here (the end of the previous match)
    if (MODE == kModeStandard) {
        // the first occurrence, in list order, that starts at or after s
        for (unsigned long long i = 0; i < n; i++) {
            const uint4 m = reinterpret_cast<const uint4 *>(r)[i];
            if (m.z >= s) {
                reinterpret_cast<uint4 *>(r)[w++] = m;
                s = m.w;
            }
        }
        return (uint32_t)w;
    }
    unsigned long long i = 0;
    while (i < n) {
        bool have = false;
        uint4 best = make_uint4(0, 0, 0, 0);
        for (unsigned long long j = i; j < n; j++) {
            const uint4 m = reinterpret_cast<const uint4 *>(r)[j];
            if (have && m.w > best.z + max_len) break;  // everything from here on starts after `best` does
            if (m.z < s) continue;
            bool better = !have || m.z < best.z;
            if (have && m.z == best.z) better = longest ? (m.w > best.w || (m.w == best.w && m.y < best.y)) : (m.y < best.y);
            if (better) {
                best = m;
                have = true;
            }
        }
        if (!have) break;
        reinterpret_cast<uint4 *>(r)[w++] = best;  // w <= i: only records that can no longer be chosen are overwritten
        s = best.w;
        while (i < n && r[i].end <= s) i++;
    }
    return (uint32_t)w;
}

template <int MODE, bool CP>
__global__ void __launch_bounds__(kScanThreads) sieve_epilogue_kernel(SieveEpiArgs E) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    const uint64_t tiles = (E.n_tasks + kScanTile - 1) / kScanTile;
    const uint64_t ctiles = CP ? tiles : 0;
    // phase 1 + 2: where each task's matches go (and, code points, the continuation bytes before each task)
    for (uint64_t tt = blockIdx.x; tt < tiles + ctiles; tt += gridDim.x) {
        if (tt >= tiles)
            tile_sum_body<false>(E.cont_tail, 1, E.n_tasks, E.cont_tiles, tt - tiles, nullptr);
        else
            tile_sum_body<false>(E.unit_counts, 1, E.n_tasks, E.tile_sums, tt, nullptr);
    }
    grid.sync();
    for (uint64_t tt = blockIdx.x; tt < tiles + ctiles; tt += gridDim.x) {
        if (tt >= tiles)
            tile_apply_body<false>(E.cont_tail, 1, E.n_tasks, E.cont_tiles, E.cont_cum, tt - tiles);
        else
            tile_apply_body<false>(E.unit_counts, 1, E.n_tasks, E.tile_sums, E.unit_offsets, tt);
    }
    grid.sync();
    // phase 3: the ordered overlapping list
    {
        unsigned long long n = E.acc[kAccRaw];
        if (n > E.raw_cap) n = E.raw_cap;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
             i += (unsigned long long)gridDim.x * blockDim.x) {
            const uint32_t u = E.raw_unit[i];
            const unsigned long long dst = E.unit_offsets[u] + E.raw_seq[i];
            if (dst >= E.out_cap) continue;
            uint4 r = reinterpret_cast<const uint4 *>(E.raw)[i];  // haystack, pattern, start, end (bytes)
            if (CP) {
                // continuation bytes between the haystack's start and the match's end: both counts are relative to
                // the start of the task they were taken in, cont_cum carries them to a common origin
                const int64_t hs = E.B.offsets[r.x];
                const int64_t u0 = (hs - E.origin) / (int64_t)E.task_bytes;
                const unsigned long long cont = (E.cont_cum[u] + E.raw_aux[i]) - (E.cont_cum[u0] + E.hay_cont[r.x]);
                const uint32_t end_cp = r.w - (uint32_t)cont;
                r.w = end_cp;
                r.z = end_cp - E.pat_cplen[r.y];
            }
            reinterpret_cast<uint4 *>(E.ordered)[dst] = r;
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            E.totals[6] = E.unit_offsets[E.n_tasks];
            E.totals[7] = E.acc[kAccRaw];
        }
        if (MODE != kModeOverlap) {
            // the per-haystack selection counts start at zero (the task counts in this array were consumed by phase 2)
            for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h < E.B.n_haystacks; h += (int64_t)gridDim.x * blockDim.x) E.unit_counts[h] = 0;
        }
    }
    grid.sync();
    // (from here on unit_counts / unit_offsets are per HAYSTACK: the task-level values have been consumed)
    const unsigned long long list_total = E.totals[6];
    const unsigned long long avail = list_total < E.out_cap ? list_total : E.out_cap;
    if (list_total > E.out_cap || E.totals[7] > E.raw_cap) {
        // The buffers were too small: the ordered list has holes (stale records): nothing may be read from it, not even
        // the haystack ids for the per-haystack offsets.
        // Report how much room is needed; the caller retries.  (Every block takes this branch: totals[6..7] were
        // published before the barrier and nobody writes them again.)
        for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h <= E.B.n_haystacks; h += (int64_t)gridDim.x * blockDim.x) E.match_offsets[h] = 0;
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            const unsigned long long raw_total = E.totals[7];
            E.totals[0] = list_total;
            E.totals[1] = 0;
            E.totals[2] = E.totals[3] = E.totals[5] = 0;
            E.totals[4] = raw_total > list_total ? raw_total : list_total;
            E.acc[kAccRaw] = E.acc[kAccGroups] = E.acc[kAccTraps] = E.acc[kAccRepairs] = 0;
            E.acc[kAccQueue] = 0;
        }
        return;
    }
    if (MODE == kModeOverlap) {
        // per-haystack offsets into the list: the first record of every haystack is found where the haystack id changes
        // (one pass over the records; the haystacks in between, which have no matches, get the same offset)
        const int64_t nh = E.B.n_haystacks;
        if (avail == 0) {
            for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h <= nh; h += (int64_t)gridDim.x * blockDim.x) E.match_offsets[h] = h == nh ? list_total : 0;
        } else {
            for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < avail; i += (unsigned long long)gridDim.x * blockDim.x) {
                const int64_t hc = (int64_t)E.ordered[i].haystack, hp = i ? (int64_t)E.ordered[i - 1].haystack : -1;
                for (int64_t h = hp + 1; h <= hc; h++) E.match_offsets[h] = i;
                if (i + 1 == avail)
                    for (int64_t h = hc + 1; h <= nh; h++) E.match_offsets[h] = h == nh ? list_total : avail;
            }
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            const unsigned long long raw_total = E.acc[kAccRaw];
            E.totals[0] = list_total;
            E.totals[1] = (raw_total <= E.raw_cap && list_total <= E.out_cap) ? 1 : 0;
            E.totals[2] = E.totals[3] = E.totals[5] = 0;
            E.totals[4] = raw_total > list_total ? raw_total : list_total;
            E.totals[7] = 0;
            E.acc[kAccRaw] = E.acc[kAccGroups] = E.acc[kAccTraps] = E.acc[kAccRepairs] = 0;
            E.acc[kAccQueue] = 0;
        }
        return;
    }
    // phase 4: per haystack, select the non-overlapping matches and pack them to the front of the haystack's stretch.
    // A haystack's stretch starts where the haystack id changes: the thread that sees the change owns it.  (Haystacks
    // without matches keep the zero count written in phase 3.)
    const uint64_t n_hay = (uint64_t)E.B.n_haystacks;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < avail; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t hc = E.ordered[i].haystack;
        if (i && E.ordered[i - 1].haystack == hc) continue;
        unsigned long long hi = i + 1;
        while (hi < avail && E.ordered[hi].haystack == hc) hi++;
        E.unit_offsets[hc] = i;
        E.unit_counts[hc] = select_non_overlapping<MODE>(E.ordered + i, hi - i, E.max_pat_len, E.longest);
    }
    grid.sync();
    // phase 5 + 6: per-haystack offsets into the output
    const uint64_t htiles = (n_hay + kScanTile - 1) / kScanTile;
    for (uint64_t tt = blockIdx.x; tt < htiles; tt += gridDim.x) tile_sum_body<false>(E.unit_counts, 1, n_hay, E.tile_sums, tt, nullptr);
    grid.sync();
    for (uint64_t tt = blockIdx.x; tt < htiles; tt += gridDim.x) tile_apply_body<false>(E.unit_counts, 1, n_hay, E.tile_sums, E.match_offsets, tt);
    grid.sync();
    // phase 7: pack
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < avail; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint4 r = reinterpret_cast<const uint4 *>(E.ordered)[i];
        const unsigned long long k = i - E.unit_offsets[r.x];
        if (k < E.unit_counts[r.x]) {
            const unsigned long long dst = E.match_offsets[r.x] + k;
            if (dst < E.out_cap) reinterpret_cast<uint4 *>(E.final_out)[dst] = r;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const unsigned long long raw_total = E.acc[kAccRaw];
        const unsigned long long total = n_hay ? E.match_offsets[n_hay] : 0;
        E.totals[0] = total;
        E.totals[1] = (raw_total <= E.raw_cap && list_total <= E.out_cap) ? 1 : 0;
        E.totals[2] = E.totals[3] = E.totals[5] = 0;
        E.totals[4] = raw_total > list_total ? raw_total : list_total;  // room the overlapping list needs
        E.totals[7] = 0;
        E.acc[kAccRaw] = E.acc[kAccGroups] = E.acc[kAccTraps] = E.acc[kAccRepairs] = 0;
        E.acc[kAccQueue] = 0;
    }
}

// ---------------------------------------------------------------------------
// Multi-GPU: the block a rank contributes to the gather of the match lists --
// row 0 = (count, haystack base, complete flag, 0), then its first `cap`
// matches -- assembled by ONE launch straight from a scan's output buffers.
// ---------------------------------------------------------------------------
__global__ void pack_gather_block_kernel(const unsigned long long *totals, const acb_match *out, uint32_t hay_base, unsigned long long cap,
                                         uint4 *block) {
    const unsigned long long total = totals[0];
    const unsigned long long n = total < cap ? total : cap;
    if (blockIdx.x == 0 && threadIdx.x == 0)
        block[0] = make_uint4((uint32_t)(total > 0xffffffffull ? 0xffffffffull : total), hay_base, (uint32_t)totals[1], 0u);
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x)
        block[1 + i] = reinterpret_cast<const uint4 *>(out)[i];
}

// ---------------------------------------------------------------------------
// The non-overlapping selection (select_non_overlapping above) for ONE haystack whose overlapping list was
// assembled by the caller from several scans (a haystack above one call's 32-bit range): rows of four int64
// (haystack, pattern, start, end), sorted by (end, start, pattern).  One thread: the selection is a chain.
// ---------------------------------------------------------------------------
__global__ void select_rows_kernel(const long long *rows, unsigned long long n, int mode, int longest, long long max_len, long long *out,
                                   unsigned long long *count) {
    if (blockIdx.x || threadIdx.x) return;
    unsigned long long w = 0;
    long long s = 0;
    auto put = [&](unsigned long long j) {
        for (int c = 0; c < 4; c++) out[4 * w + c] = rows[4 * j + c];
        w++;
    };
    if (mode == kModeStandard) {
        for (unsigned long long i = 0; i < n; i++)
            if (rows[4 * i + 2] >= s) {
                s = rows[4 * i + 3];
                put(i);
            }
    } else {
        unsigned long long i = 0;
        while (i < n) {
            bool have = false;
            unsigned long long best = 0;
            for (unsigned long long j = i; j < n; j++) {
                const long long st = rows[4 * j + 2], en = rows[4 * j + 3], pid = rows[4 * j + 1];
                if (have && en > rows[4 * best + 2] + max_len) break;
                if (st < s) continue;
                bool better = !have || st < rows[4 * best + 2];
                if (have && st == rows[4 * best + 2])
                    better = longest ? (en > rows[4 * best + 3] || (en == rows[4 * best + 3] && pid < rows[4 * best + 1])) : (pid < rows[4 * best + 1]);
                if (better) {
                    best = j;
                    have = true;
                }
            }
            if (!have) break;
            s = rows[4 * best + 3];
            put(best);
            while (i < n && rows[4 * i + 3] <= s) i++;
        }
    }
    *count = w;
}

// when the input is empty: nothing ran, publish zeros
__global__ void zero_outputs_kernel(unsigned long long *unit_offsets, unsigned long long *match_offsets, int64_t n_haystacks,
                                    unsigned long long *totals) {
    if (blockIdx.x == 0 && threadIdx.x < 8) totals[threadIdx.x] = threadIdx.x == 1 ? 1 : 0;  // no matches, complete
    for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h <= n_haystacks; h += (int64_t)gridDim.x * blockDim.x) match_offsets[h] = 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) unit_offsets[0] = 0;
}

}  // namespace acb

// ===========================================================================
// C ABI
// ===========================================================================
using namespace acb;

struct acb_automaton {
    Automaton *impl;
};

// Per-thread state only: the last error, the tuning knobs and the optional kernel timing belong to the calling
// thread (two automata scanned from two threads do not see each other's settings); the launch counter is atomic.
static thread_local std::string g_err;
static std::atomic<unsigned long long> g_launches{0};
static thread_local acb_tuning g_tuning = {0, 0, 0, 0};  // kernel, hot_rows, segment_bytes, table

// optional device timing of the dominant (scan) kernel, for bench.py's roofline
static thread_local bool g_timing = false;
static thread_local std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_timing_events;

static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

#define CUDA_OK(expr)                                                                                   \
    do {                                                                                                \
        cudaError_t e_ = (expr);                                                                        \
        if (e_ != cudaSuccess) return fail(ACB_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); \
    } while (0)

extern "C" {

const char *acb_last_error(void) { return g_err.c_str(); }
const char *acb_version(void) { return "acb200 0.2 (sm_100a)"; }
uint64_t acb_launch_count(void) { return g_launches.load(); }

int acb_timing_enable(int on) {
    g_timing = on != 0;
    return ACB_OK;
}

int acb_timing_read(double *total_ms, uint64_t *n_scans) {
    double tot = 0;
    uint64_t n = 0;
    for (auto &p : g_timing_events) {
        float ms = 0;
        CUDA_OK(cudaEventSynchronize(p.second));
        CUDA_OK(cudaEventElapsedTime(&ms, p.first, p.second));
        tot += ms;
        n++;
        cudaEventDestroy(p.first);
        cudaEventDestroy(p.second);
    }
    g_timing_events.clear();
    if (total_ms) *total_ms = tot;
    if (n_scans) *n_scans = n;
    return ACB_OK;
}

int acb_set_tuning(const acb_tuning *t) {
    if (!t) return fail(ACB_EINVAL, "null tuning");
    g_tuning = *t;
    return ACB_OK;
}

int acb_build_ex(const uint8_t *blob, const uint64_t *offsets, uint64_t n, int match_kind, int implementation, uint32_t flags,
                 acb_automaton **out) {
    if (!out || !offsets || (!blob && n && offsets[n] != 0)) return fail(ACB_EINVAL, "null argument");
    if (implementation < -1 || implementation > 2) return fail(ACB_EINVAL, "unknown implementation");
    if (flags & ~uint32_t(ACB_ASCII_CASE_INSENSITIVE)) return fail(ACB_EINVAL, "unknown build flags");
    try {
        Automaton *impl = build_automaton(blob, offsets, n, match_kind, implementation, flags);
        *out = new acb_automaton{impl};
        return ACB_OK;
    } catch (const std::exception &e) {
        return fail(ACB_EBUILD, e.what());
    }
}

int acb_build(const uint8_t *blob, const uint64_t *offsets, uint64_t n, int match_kind, int implementation,
              acb_automaton **out) {
    return acb_build_ex(blob, offsets, n, match_kind, implementation, 0u, out);
}

uint32_t acb_build_flags(const acb_automaton *a) { return a->impl->hdr.flags; }

void acb_free(acb_automaton *a) {
    if (!a) return;
    delete a->impl;
    delete a;
}

uint64_t acb_num_patterns(const acb_automaton *a) { return a->impl->hdr.n_patterns; }
uint64_t acb_num_states(const acb_automaton *a) { return a->impl->hdr.n_states; }
uint32_t acb_num_columns(const acb_automaton *a) { return a->impl->hdr.n_cols; }
uint32_t acb_max_pattern_len(const acb_automaton *a) { return a->impl->hdr.max_pat_len; }
uint32_t acb_min_pattern_len(const acb_automaton *a) { return a->impl->hdr.min_pat_len; }
int acb_match_kind(const acb_automaton *a) { return (int)a->impl->hdr.match_kind; }
uint64_t acb_image_bytes(const acb_automaton *a) { return a->impl->hdr.total_bytes; }

int acb_image_write(const acb_automaton *a, void *host_dst, uint64_t dst_bytes) {
    if (!a || !host_dst) return fail(ACB_EINVAL, "null argument");
    if (dst_bytes < a->impl->hdr.total_bytes) return fail(ACB_ECAPACITY, "image buffer too small");
    std::memcpy(host_dst, a->impl->image.data(), a->impl->hdr.total_bytes);
    return ACB_OK;
}

uint64_t acb_hot_bytes(const acb_automaton *a, uint32_t max_rows) { return hot_image_bytes(*a->impl, max_rows); }

int acb_hot_build(const acb_automaton *a, const uint32_t *host_visits, uint32_t max_rows, void *host_dst, uint64_t dst_bytes) {
    if (!a || !host_dst) return fail(ACB_EINVAL, "null argument");
    if (dst_bytes < hot_image_bytes(*a->impl, max_rows)) return fail(ACB_ECAPACITY, "hot image buffer too small");
    build_hot_image(*a->impl, host_visits, max_rows, static_cast<uint8_t *>(host_dst));
    return ACB_OK;
}

uint32_t acb_hot_rows(const void *host_hot) {
    const HotHeader *h = static_cast<const HotHeader *>(host_hot);
    return (h && h->magic == kHotMagic) ? h->n_rows : 0;
}

int acb_hot_describe(const void *host_hot, acb_hot_desc *desc) {
    const HotHeader *h = static_cast<const HotHeader *>(host_hot);
    if (!h || !desc || h->magic != kHotMagic) return fail(ACB_EINVAL, "not a hot image");
    desc->rows = h->n_rows;
    desc->rows128 = h->n_rows128;
    desc->visited = h->n_visited;
    desc->reserved = 0;
    return ACB_OK;
}

uint64_t acb_sieve_build(acb_automaton *a, uint32_t bloom_bytes_max, uint32_t w_max) {
    if (!a) {
        fail(ACB_EINVAL, "null argument");
        return 0;
    }
    Automaton &A = *a->impl;
    std::lock_guard<std::mutex> lock(A.sieve_mutex);
    if (A.sieve.empty() || A.sieve_bloom_max != bloom_bytes_max || A.sieve_w_max != w_max) {
        try {
            sieve_image_build(A.pat_blob.data(), A.pat_offs.data(), A.hdr.n_patterns, bloom_bytes_max, w_max, A.hdr.flags, A.sieve);
            A.sieve_bloom_max = bloom_bytes_max;
            A.sieve_w_max = w_max;
        } catch (const std::exception &e) {
            A.sieve.clear();
            fail(ACB_EBUILD, e.what());
            return 0;
        }
    }
    return A.sieve.size();
}

int acb_sieve_write(acb_automaton *a, void *host_dst, uint64_t dst_bytes) {
    if (!a || !host_dst) return fail(ACB_EINVAL, "null argument");
    Automaton &A = *a->impl;
    std::lock_guard<std::mutex> lock(A.sieve_mutex);
    if (A.sieve.empty()) return fail(ACB_EINVAL, "acb_sieve_build has not been called");
    if (dst_bytes < A.sieve.size()) return fail(ACB_ECAPACITY, "sieve image buffer too small");
    std::memcpy(host_dst, A.sieve.data(), A.sieve.size());
    return ACB_OK;
}

int acb_sieve_describe(const void *host_sieve, acb_sieve_desc *d) {
    const SieveHeader *h = static_cast<const SieveHeader *>(host_sieve);
    if (!h || !d || h->magic != kSieveMagic) return fail(ACB_EINVAL, "not a sieve image");
    d->window = h->W;
    d->last_level = h->last_level;
    d->probes = h->n_probes;
    d->bloom_bytes = h->bloom_words * 4;
    d->nodes = h->n_nodes;
    d->keys = h->n_keys;
    d->filter_entries = h->n_filter_entries;
    d->table_slots = h->ht_mask + 1;
    return ACB_OK;
}

// tasks of the sieve kernel: a multiple of 512 bytes (tuning.segment_bytes when the sieve kernel is forced, else 16 KiB)
static uint32_t sieve_task_bytes() {
    uint32_t t = (g_tuning.kernel == 5 && g_tuning.segment_bytes > 0) ? (uint32_t)g_tuning.segment_bytes : 16384u;
    t = (t + 511u) & ~511u;
    return t < 512u ? 512u : t;
}

int acb_plan_scan(const acb_automaton *a, const void *dev_bytes, uint64_t total_bytes, uint64_t n_haystacks, acb_plan *plan) {
    if (!a || !plan) return fail(ACB_EINVAL, "null argument");
    const uint32_t L = a->impl->hdr.max_pat_len;
    // the warm-up must cover a whole longest pattern so that the guessed state equals the true one
    // whenever the true scanner did not restart inside it
    uint32_t warm = (L + 15u) & ~15u;
    if (warm < 16) warm = 16;
    uint32_t seg = g_tuning.segment_bytes > 0 ? (uint32_t)g_tuning.segment_bytes : 1024u;
    if (seg < 8 * warm) seg = 8 * warm;
    seg = (seg + 63u) & ~63u;
    const uint64_t mis = reinterpret_cast<uintptr_t>(dev_bytes) & 63u;  // segment 0 starts at the 64-byte aligned address before the buffer
    plan->segment_bytes = seg;
    plan->warm_bytes = warm;
    plan->n_segments = (total_bytes + mis + seg - 1) / seg;
    uint64_t stride = 1;
    if (n_haystacks > 1) {
        const uint64_t avg = total_bytes / n_haystacks;
        stride = (avg + seg / 2) / seg;
        if (stride < 1) stride = 1;
        if (stride > 65536) stride = 65536;
    }
    plan->lane_stride = (uint32_t)stride;
    // the sieve kernel's tasks: a grid anchored at the 512-byte aligned address at or before the buffer
    plan->task_bytes = sieve_task_bytes();
    const uint64_t mis512 = reinterpret_cast<uintptr_t>(dev_bytes) & 511u;
    const uint64_t n_tasks = (total_bytes + mis512 + plan->task_bytes - 1) / plan->task_bytes;
    const uint64_t seg_units = 2 * plan->n_segments;
    plan->n_units = seg_units > n_haystacks ? seg_units : n_haystacks;
    if (plan->n_units < n_tasks) plan->n_units = n_tasks;
    if (plan->n_units < 1) plan->n_units = 1;
    const uint64_t tiles = (plan->n_units + kScanTile - 1) / kScanTile;
    const uint64_t per_piece = plan->n_segments > n_tasks ? plan->n_segments : n_tasks;  // segments or tasks, whichever kernel runs
    // [0..7] counters (kAcc* in capi.cu) | unit tile sums | cont tile sums | cont_cum (pieces + 1) | packed cont tails (u32)
    plan->scratch_words = 8 + (tiles + 1) + (tiles + 1) + (per_piece + 2) + (per_piece / 2 + 2);
    return ACB_OK;
}

}  // extern "C"

namespace {

struct DeviceInfo {
    int device = -1;
    int sms = 0;
    int max_smem_optin = 0;
};

int device_info(DeviceInfo &d) {
    static thread_local DeviceInfo cache;
    int dev;
    CUDA_OK(cudaGetDevice(&dev));
    if (cache.device != dev) {
        cache.device = dev;
        CUDA_OK(cudaDeviceGetAttribute(&cache.sms, cudaDevAttrMultiProcessorCount, dev));
        CUDA_OK(cudaDeviceGetAttribute(&cache.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    }
    d = cache;
    return ACB_OK;
}

DevImage make_view(const ImageHeader &h, const void *dev_image) {
    const uint8_t *b = static_cast<const uint8_t *>(dev_image);
    DevImage im;
    im.colmap = b + h.off_colmap;
    im.trans = reinterpret_cast<const uint32_t *>(b + h.off_trans);
    im.match_off = reinterpret_cast<const uint32_t *>(b + h.off_match_off);
    im.match_pid = reinterpret_cast<const uint32_t *>(b + h.off_match_pid);
    im.pat_len = reinterpret_cast<const uint32_t *>(b + h.off_pat_len);
    im.pat_cplen = reinterpret_cast<const uint32_t *>(b + h.off_pat_cplen);
    im.n_cols = h.n_cols;
    im.col_lo = h.col_lo;
    im.n_states = h.n_states;
    im.col_mode = h.col_mode;
    return im;
}

// dev_hot points at a device copy of a hot image; hot_rows is its row count (the
// host knows it: acb_hot_rows on the host copy), because the header lives on the device
int make_hot_view(const acb_automaton *a, const void *dev_hot, const acb_hot_desc &desc, DevHot &v) {
    const ImageHeader &ih = a->impl->hdr;
    const uint32_t hot_rows = desc.rows;
    if (hot_rows < 1 || (uint64_t)hot_rows * ih.n_cols * 2 > 65535 || desc.rows128 > 255)
        return fail(ACB_EINVAL, "bad hot image description");
    auto align16 = [](uint64_t x) { return (x + 15) & ~uint64_t(15); };
    const uint8_t *b = static_cast<const uint8_t *>(dev_hot);
    uint64_t off = align16(sizeof(HotHeader));
    v.table = reinterpret_cast<const uint16_t *>(b + off);
    off = align16(off + uint64_t(hot_rows + 1) * ih.n_cols * 2);
    v.hot2full = reinterpret_cast<const uint32_t *>(b + off);
    off = align16(off + uint64_t(hot_rows + 1) * 4);
    v.full2hot = reinterpret_cast<const uint16_t *>(b + off);
    v.n_rows = hot_rows;
    off = align16(off + uint64_t(ih.n_states) * 2);
    v.table128 = reinterpret_cast<const uint16_t *>(b + off);
    v.n_rows128 = desc.rows128;
    return ACB_OK;
}

template <int MODE, bool CP>
int launch_plain(const DevImage &im, const Batch &B, const Sink &out, const DeviceInfo &d, cudaStream_t st) {
    const int threads = 128;
    int64_t blocks = (B.n_haystacks + threads - 1) / threads;
    const int64_t cap = (int64_t)d.sms * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    scan_plain_kernel<MODE, CP><<<(unsigned)blocks, threads, 0, st>>>(im, B, out);
    g_launches++;
    return ACB_OK;
}

template <int MODE, bool CP, int COLMODE, int V>
int launch_staged(const DevImage &im, const DevHot &hot, const Batch &B, const SegPlan &P, const Sink &out, SegInfo *seg_info,
                  const DeviceInfo &d, unsigned int *task_counter, unsigned long long *trap_stats, cudaStream_t st) {
    auto kern = scan_staged_kernel<MODE, CP, COLMODE, V>;
    constexpr int kWarpsMax = V == 1 ? kMaxWarps : kMaxWarps2;
    const uint64_t q = P.lane_stride;
    const uint64_t tasks = ((uint64_t)P.n_segments + 32 * V * q - 1) / (32 * V * q) * q;
    const int ctas = d.sms;
    int warps = (int)((tasks + ctas - 1) / ctas);
    if (warps < 4) warps = 4;
    // as many warps as fit: the scan is a chain of dependent shared-memory loads per lane, more warps hide more of
    // it (measured 26 -> 32 warps: 170 -> 164 us); balancing the last round of tasks instead was not better
    if (warps > kWarpsMax) warps = kWarpsMax;
    const uint32_t row_bytes = COLMODE == kColAscii ? kAsciiCols * 2 : im.n_cols * 2;
    const uint32_t stage_bytes = (uint32_t)warps * V * (2 * kStageBytes + kMetaBytes);
    const uint32_t budget = (uint32_t)d.max_smem_optin;
    if (budget < stage_bytes + kStageOffset + 3 * (row_bytes + 4) + 256) return fail(ACB_ECUDA, "not enough shared memory for the staged kernel");
    uint32_t rows = (budget - stage_bytes - kStageOffset - 256) / (row_bytes + 4);  // includes the trap row; +4: the row's hot2full entry
    // table entries are 16-bit shared-memory ADDRESSES: the table (it starts dynamic shared memory) must end below 64 KB
    if (rows > (60u * 1024u) / row_bytes) rows = (60u * 1024u) / row_bytes;
    if (COLMODE == kColAscii) rows -= 1;                                        // ... and the guard row behind it
    uint32_t H = rows - 1;
    const uint32_t have = COLMODE == kColAscii ? hot.n_rows128 : hot.n_rows;
    if (H > have) H = have;
    if (g_tuning.hot_rows > 0 && (uint32_t)g_tuning.hot_rows < H) H = (uint32_t)g_tuning.hot_rows;
    if (H < 1) return fail(ACB_ECUDA, "rows too wide for the staged kernel");
    const uint32_t hot_bytes = (((H + 1 + (COLMODE == kColAscii ? 1 : 0)) * row_bytes) + 127u) & ~127u;
    const uint32_t smem = hot_bytes + kStageOffset + (((H + 1) * 4 + 127u) & ~127u) + stage_bytes;
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget));
    kern<<<ctas, warps * 32, smem, st>>>(im, hot, B, P, out, seg_info, H, hot_bytes, task_counter, trap_stats);
    g_launches++;
    return ACB_OK;
}

// how many 128-wide rows fit next to the staging buffers of a full CTA
uint32_t ascii_rows_that_fit(const DeviceInfo &d) {
    const uint32_t stage_bytes = (uint32_t)kMaxWarps * (2 * kStageBytes + kMetaBytes);
    const uint32_t budget = (uint32_t)d.max_smem_optin;
    if (budget < stage_bytes + kStageOffset + 128 + 2 * kAsciiCols * 2) return 0;
    uint32_t rows = (budget - stage_bytes - kStageOffset - 256) / (kAsciiCols * 2 + 4);
    if (rows > (60u * 1024u) / (kAsciiCols * 2)) rows = (60u * 1024u) / (kAsciiCols * 2);  // 16-bit row addresses
    return rows - 2;  // minus the trap row and the guard row
}

template <int MODE, bool CP>
int launch_staged_cols(const ImageHeader &h, const DevImage &im, const DevHot &hot, const Batch &B, const SegPlan &P, const Sink &out,
                       SegInfo *seg_info, const DeviceInfo &d, unsigned int *task_counter, unsigned long long *trap_stats,
                       cudaStream_t st, bool ascii, int per_lane) {
#define ACB_GO(COLS)                                                                                                        \
    (per_lane == 2 ? launch_staged<MODE, CP, COLS, 2>(im, hot, B, P, out, seg_info, d, task_counter, trap_stats, st)      \
                   : launch_staged<MODE, CP, COLS, 1>(im, hot, B, P, out, seg_info, d, task_counter, trap_stats, st))
    if (ascii) return ACB_GO(kColAscii);
    if (h.col_mode == kColRange) return ACB_GO(kColRange);
    return ACB_GO(kColClass);
#undef ACB_GO
}

template <int MODE, bool CP>
int launch_global(const DevImage &im, const Batch &B, const SegPlan &P, const Sink &out, SegInfo *seg_info, const DeviceInfo &d,
                  cudaStream_t st) {
    int64_t blocks = (P.n_segments + 255) / 256;
    const int64_t cap = (int64_t)d.sms * 64;  // grid-stride beyond that
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    scan_global_kernel<MODE, CP><<<(unsigned)blocks, 256, 0, st>>>(im, B, P, out, seg_info);
    g_launches++;
    return ACB_OK;
}

inline int epilogue_blocks_per_sm(int max_bps, uint64_t n_units) {
    static const int forced = [] {
        const char *e = std::getenv("ACB200_EPILOGUE_BPS");
        return e ? std::atoi(e) : 0;
    }();
    (void)n_units;
    int b = forced > 0 ? forced : max_bps;  // (one block per SM was measured: 214 vs 197 us per config-2 step -- more blocks win)
    return b > max_bps ? max_bps : (b < 1 ? 1 : b);
}

template <int MODE, bool CP>
int launch_epilogue(EpilogueArgs &E, const DeviceInfo &d, cudaStream_t st) {
    auto kern = epilogue_kernel<MODE, CP>;
    static thread_local int blocks_per_sm[3][2] = {{0, 0}, {0, 0}, {0, 0}};
    static thread_local int cached_device = -1;  // the occupancy answer belongs to a device
    if (cached_device != d.device) {
        for (auto &row : blocks_per_sm) row[0] = row[1] = 0;
        cached_device = d.device;
    }
    int &bps = blocks_per_sm[MODE][CP ? 1 : 0];
    if (bps == 0) {
        CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, kScanThreads, 0));
        if (bps < 1) return fail(ACB_ECUDA, "epilogue kernel does not fit on an SM");
        if (bps > 4) bps = 4;
    }
    void *args[] = {&E};
    const int use_bps = epilogue_blocks_per_sm(bps, E.n_units);
    CUDA_OK(cudaLaunchCooperativeKernel(reinterpret_cast<void *>(kern), dim3(d.sms * use_bps), dim3(kScanThreads), args, 0, st));
    g_launches++;
    return ACB_OK;
}


DevSieve make_sieve_view(const SieveHeader &h, const void *dev_sieve) {
    const uint8_t *b = static_cast<const uint8_t *>(dev_sieve);
    DevSieve v;
    v.bloom = reinterpret_cast<const uint32_t *>(b + h.off_bloom);
    v.ht = reinterpret_cast<const SieveSlot *>(b + h.off_ht);
    v.na = reinterpret_cast<const SieveNodeA *>(b + h.off_node_a);
    v.nb = reinterpret_cast<const SieveNodeB *>(b + h.off_node_b);
    v.pids = reinterpret_cast<const uint32_t *>(b + h.off_pids);
    v.W = h.W;
    v.last_level = h.last_level;
    v.n_probes = h.n_probes;
    v.bloom_words = h.bloom_words;
    v.prim_words = h.prim_words;
    v.ht_size = h.ht_mask + 1;
    v.max_pat_len = h.max_pat_len;
    v.term_levels = h.term_levels;
    return v;
}

template <bool CP>
int launch_sieve(const DevSieve &sv, bool fold, const Batch &B, SievePlan &P, const Sink &out, uint32_t *task_cont, uint32_t *hay_cont,
                 unsigned int *task_counter, const DeviceInfo &d, cudaStream_t st) {
    // as many windows of text per warp as fit next to the filters (a power of two): the more, the fuller the rounds of
    // the later stages when survivors are rare
    const uint32_t filter_bytes = sv.bloom_words * 4;
    uint32_t ring = kRingMax;
    while (ring > 1 && sieve_smem_bytes(filter_bytes, ring, CP) > (uint32_t)d.max_smem_optin) ring >>= 1;
    const uint32_t smem = sieve_smem_bytes(filter_bytes, ring, CP);
    if (smem > (uint32_t)d.max_smem_optin) return fail(ACB_ECUDA, "the sieve's filters do not fit in shared memory (rebuild them with a smaller bloom_bytes_max)");
    P.ring = ring;
    // (a case-insensitive image: the kernel variant that folds the text as it loads it)
#define ACB_SIEVE_GO(WC)                                                                                  \
    do {                                                                                                  \
        auto kern = fold ? sieve_scan_kernel<CP, WC, true> : sieve_scan_kernel<CP, WC, false>;            \
        CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, d.max_smem_optin)); \
        kern<<<d.sms, kSieveThreads, smem, st>>>(sv, B, P, out, task_cont, hay_cont, task_counter);       \
    } while (0)
    if (sv.W < 4)
        ACB_SIEVE_GO(0);
    else if (sv.W == 4)
        ACB_SIEVE_GO(1);
    else if (sv.W == 5)
        ACB_SIEVE_GO(3);
    else
        ACB_SIEVE_GO(2);
#undef ACB_SIEVE_GO
    g_launches++;
    return ACB_OK;
}

template <int MODE, bool CP>
int launch_sieve_epilogue(SieveEpiArgs &E, const DeviceInfo &d, cudaStream_t st) {
    auto kern = sieve_epilogue_kernel<MODE, CP>;
    static thread_local int blocks_per_sm[3][2] = {{0, 0}, {0, 0}, {0, 0}};
    static thread_local int cached_device = -1;
    if (cached_device != d.device) {
        for (auto &row : blocks_per_sm) row[0] = row[1] = 0;
        cached_device = d.device;
    }
    int &bps = blocks_per_sm[MODE][CP ? 1 : 0];
    if (bps == 0) {
        CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, kScanThreads, 0));
        if (bps < 1) return fail(ACB_ECUDA, "epilogue kernel does not fit on an SM");
        if (bps > 4) bps = 4;
    }
    void *args[] = {&E};
    const uint64_t n_work = E.n_tasks > (uint64_t)E.B.n_haystacks ? E.n_tasks : (uint64_t)E.B.n_haystacks;
    const int use_bps = epilogue_blocks_per_sm(bps, n_work);
    CUDA_OK(cudaLaunchCooperativeKernel(reinterpret_cast<void *>(kern), dim3(d.sms * use_bps), dim3(kScanThreads), args, 0, st));
    g_launches++;
    return ACB_OK;
}

int check_ws(const acb_workspace *ws) {
    if (!ws || !ws->dev_raw || !ws->dev_raw_seq || !ws->dev_raw_unit || !ws->dev_raw_aux || !ws->dev_unit_counts ||
        !ws->dev_unit_offsets || !ws->dev_seg_info || !ws->dev_scratch || !ws->dev_total || !ws->dev_out ||
        !ws->dev_match_offsets)
        return fail(ACB_EINVAL, "workspace has a null buffer");
    return ACB_OK;
}

}  // namespace

extern "C" {

int acb_profile(const acb_automaton *a, const void *dev_image, const uint8_t *dev_bytes, const int64_t *dev_offsets,
                int64_t n_haystacks, uint64_t total_bytes, int overlapping, uint32_t *dev_visits, void *stream) {
    if (!a || !dev_image || !dev_visits || !dev_offsets) return fail(ACB_EINVAL, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const ImageHeader &h = a->impl->hdr;
    CUDA_OK(cudaMemsetAsync(dev_visits, 0, uint64_t(h.n_states) * 4, st));
    if (n_haystacks < 1 || total_bytes == 0) return ACB_OK;
    Batch B{dev_bytes, dev_offsets, n_haystacks};
    int64_t n_samples = 256;
    if ((uint64_t)n_samples > total_bytes / 1024 + 1) n_samples = (int64_t)(total_bytes / 1024 + 1);
    const DevImage im = make_view(h, dev_image);
    const int restart = (!overlapping && h.match_kind == ACB_STANDARD) ? 1 : 0;
    profile_kernel<<<(unsigned)((n_samples + 127) / 128), 128, 0, st>>>(im, B, dev_visits, n_samples, 1024, restart);
    g_launches++;
    CUDA_OK(cudaGetLastError());
    return ACB_OK;
}

int acb_select_non_overlapping(const acb_automaton *a, const int64_t *dev_rows, uint64_t n_rows, int64_t *dev_out, uint64_t *dev_count,
                                void *stream) {
    if (!a || !dev_out || !dev_count || (n_rows && !dev_rows)) return fail(ACB_EINVAL, "null argument");
    const ImageHeader &h = a->impl->hdr;
    const int kind = (int)h.match_kind;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    select_rows_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const long long *>(dev_rows), n_rows, kind == ACB_STANDARD ? kModeStandard : kModeLeftmost,
                                         kind == ACB_LEFTMOST_LONGEST ? 1 : 0, (long long)h.max_pat_len, reinterpret_cast<long long *>(dev_out),
                                         reinterpret_cast<unsigned long long *>(dev_count));
    g_launches++;
    CUDA_OK(cudaGetLastError());
    return ACB_OK;
}

int acb_pack_gather_block(const uint64_t *dev_total, const acb_match *dev_out, uint32_t hay_base, uint64_t cap, void *dev_block, void *stream) {
    if (!dev_total || !dev_out || !dev_block) return fail(ACB_EINVAL, "null argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned blocks = (unsigned)((cap + 255) / 256);
    if (blocks > 296) blocks = 296;
    if (blocks < 1) blocks = 1;
    pack_gather_block_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const unsigned long long *>(dev_total), dev_out, hay_base, cap,
                                                     reinterpret_cast<uint4 *>(dev_block));
    g_launches++;
    CUDA_OK(cudaGetLastError());
    return ACB_OK;
}

int acb_scan_batch(const acb_automaton *a, const void *dev_image, const void *dev_hot, const acb_hot_desc *hot_desc,
                   const void *dev_sieve, const uint8_t *dev_bytes, const int64_t *dev_offsets, int64_t n_haystacks, uint64_t total_bytes,
                   int overlapping, int codepoints, const acb_plan *plan, const acb_workspace *ws, void *stream) {
    if (!a || !dev_image || !dev_offsets || n_haystacks < 0 || !plan) return fail(ACB_EINVAL, "bad argument");
    if (n_haystacks > 0xfffffffell) return fail(ACB_EINVAL, "too many haystacks in one batch");
    const ImageHeader &h = a->impl->hdr;
    const int kind = (int)h.match_kind;
    // overlapping == 2: the overlapping LIST, for any match kind -- the input of acb_select_non_overlapping; sieve only
    if (overlapping == 1 && kind != ACB_STANDARD)
        return fail(ACB_EUNSUPPORTED, std::string("match kind ") + (kind == ACB_LEFTMOST_FIRST ? "LeftmostFirst" : "LeftmostLongest") +
                                          " does not support overlapping searches");
    if (overlapping == 2 && !dev_sieve) return fail(ACB_EINVAL, "the overlapping list of a leftmost automaton needs the sieve image");
    int rc = check_ws(ws);
    if (rc) return rc;
    DeviceInfo d;
    if ((rc = device_info(d))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int mode = overlapping ? kModeOverlap : (kind == ACB_STANDARD ? kModeStandard : kModeLeftmost);
    const bool cp = codepoints != 0;
    const DevImage im = make_view(h, dev_image);
    Batch B{dev_bytes, dev_offsets, n_haystacks};

    // the plan must be the one acb_plan_scan gives for these arguments (it sizes the workspace)
    acb_plan want;
    acb_plan_scan(a, dev_bytes, total_bytes, (uint64_t)n_haystacks, &want);
    if (want.n_segments != plan->n_segments || want.segment_bytes != plan->segment_bytes || want.n_units != plan->n_units ||
        want.task_bytes != plan->task_bytes)
        return fail(ACB_EINVAL, "plan does not match the arguments (call acb_plan_scan again)");

    unsigned long long *totals = reinterpret_cast<unsigned long long *>(ws->dev_total);
    unsigned int *task_counter = reinterpret_cast<unsigned int *>(ws->dev_scratch);
    Sink out;
    out.raw = ws->dev_raw;
    out.raw_seq = ws->dev_raw_seq;
    out.raw_unit = ws->dev_raw_unit;
    out.raw_aux = ws->dev_raw_aux;
    out.cap = ws->raw_capacity;
    out.unit_counts = ws->dev_unit_counts;
    unsigned long long *acc = reinterpret_cast<unsigned long long *>(ws->dev_scratch);  // zero between scans (see kAcc*)
    out.raw_total = acc + kAccRaw;
    SegInfo *seg_info = reinterpret_cast<SegInfo *>(ws->dev_seg_info);

    unsigned long long *unit_offsets = reinterpret_cast<unsigned long long *>(ws->dev_unit_offsets);
    unsigned long long *match_offsets = reinterpret_cast<unsigned long long *>(ws->dev_match_offsets);
    if (n_haystacks == 0 || total_bytes == 0) {
        zero_outputs_kernel<<<(unsigned)((n_haystacks + 256) / 256), 256, 0, st>>>(unit_offsets, match_offsets, n_haystacks, totals);
        g_launches++;
        CUDA_OK(cudaGetLastError());
        return ACB_OK;
    }

    int kernel = g_tuning.kernel;
    if (kernel == 0) kernel = dev_sieve ? 5 : 2;  // the caller uploads a sieve image when it wants the position-parallel scan
    if (overlapping == 2) kernel = 5;
    // the caller's profile says the hot rows do not cover this data: scan from the image in global memory / L2
    if (kernel == 2 && g_tuning.kernel == 0 && hot_desc && (hot_desc->reserved & 1u)) kernel = 4;
    if (kernel == 5 && !dev_sieve) return fail(ACB_EINVAL, "the sieve kernel needs a sieve image (acb_sieve_build / acb_sieve_write)");
    if ((!dev_hot || !hot_desc) && kernel != 4 && kernel != 5) kernel = 1;  // no hot image: the plain kernel (one thread per haystack)
    if (kernel == 5) {
        // ---- position-parallel scan: filter + exact verification, then order (+ select) ----
        const Automaton &A = *a->impl;
        SieveHeader sh;
        {
            std::lock_guard<std::mutex> lock(a->impl->sieve_mutex);
            if (A.sieve.size() < sizeof(SieveHeader)) return fail(ACB_EINVAL, "acb_sieve_build has not been called");
            std::memcpy(&sh, A.sieve.data(), sizeof(sh));
        }
        const DevSieve sv = make_sieve_view(sh, dev_sieve);
        SievePlan SP;
        SP.origin = -(int64_t)(reinterpret_cast<uintptr_t>(dev_bytes) & 511u);
        SP.task_bytes = plan->task_bytes;
        SP.n_tasks = (int64_t)((total_bytes + (uint64_t)(-SP.origin) + plan->task_bytes - 1) / plan->task_bytes);
        SP.buf_bytes = total_bytes;
        SP.avg_len = total_bytes / (uint64_t)n_haystacks;
        if (SP.avg_len < 1) SP.avg_len = 1;
        const uint64_t cap = ws->raw_capacity < ws->out_capacity ? ws->raw_capacity : ws->out_capacity;
        // scratch: counters | unit tile sums | cont tile sums | cont_cum | cont tails (u32)
        const uint64_t tiles_max = (plan->n_units + kScanTile - 1) / kScanTile;
        unsigned long long *tile_sums = acc + kAccWords;
        unsigned long long *cont_tiles = tile_sums + tiles_max + 1;
        unsigned long long *cont_cum = cont_tiles + tiles_max + 1;
        const uint64_t per_piece = plan->n_segments > (uint64_t)SP.n_tasks ? plan->n_segments : (uint64_t)SP.n_tasks;
        uint32_t *cont_tail = reinterpret_cast<uint32_t *>(cont_cum + per_piece + 2);
        // a non-overlapping search orders the list into dev_raw's place and packs its selection into dev_out, so its
        // raw records go through dev_out first
        out.raw = mode == kModeOverlap ? ws->dev_raw : ws->dev_out;
        out.cap = cap;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (g_timing) {
            CUDA_OK(cudaEventCreate(&e0));
            CUDA_OK(cudaEventCreate(&e1));
            CUDA_OK(cudaEventRecord(e0, st));
        }
        // code points: the continuation bytes each task saw before a haystack that starts in it, per haystack; lives in
        // the match_offsets buffer until the epilogue's last phases write the offsets there
        uint32_t *hay_cont = reinterpret_cast<uint32_t *>(match_offsets);
        const bool fold = (sh.flags & kAsciiCaseInsensitive) != 0;
        rc = cp ? launch_sieve<true>(sv, fold, B, SP, out, cont_tail, hay_cont, task_counter, d, st)
                : launch_sieve<false>(sv, fold, B, SP, out, cont_tail, hay_cont, task_counter, d, st);
        if (rc) return rc;
        CUDA_OK(cudaGetLastError());
        if (e1) {
            CUDA_OK(cudaEventRecord(e1, st));
            g_timing_events.emplace_back(e0, e1);
        }
        SieveEpiArgs E;
        E.B = B;
        E.unit_counts = ws->dev_unit_counts;
        E.n_tasks = (uint64_t)SP.n_tasks;
        E.tile_sums = tile_sums;
        E.unit_offsets = unit_offsets;
        E.cont_tail = cont_tail;
        E.hay_cont = hay_cont;
        E.cont_tiles = cont_tiles;
        E.cont_cum = cont_cum;
        E.raw = out.raw;
        E.raw_seq = ws->dev_raw_seq;
        E.raw_unit = ws->dev_raw_unit;
        E.raw_aux = ws->dev_raw_aux;
        E.raw_cap = cap;
        E.ordered = mode == kModeOverlap ? ws->dev_out : ws->dev_raw;
        E.final_out = ws->dev_out;
        E.out_cap = cap;
        E.pat_cplen = im.pat_cplen;
        E.origin = SP.origin;
        E.task_bytes = SP.task_bytes;
        E.max_pat_len = h.max_pat_len;
        E.longest = kind == ACB_LEFTMOST_LONGEST ? 1 : 0;
        E.totals = totals;
        E.acc = acc;
        E.match_offsets = match_offsets;
        rc = mode == kModeStandard   ? (cp ? launch_sieve_epilogue<kModeStandard, true>(E, d, st) : launch_sieve_epilogue<kModeStandard, false>(E, d, st))
             : mode == kModeLeftmost ? (cp ? launch_sieve_epilogue<kModeLeftmost, true>(E, d, st) : launch_sieve_epilogue<kModeLeftmost, false>(E, d, st))
                                     : (cp ? launch_sieve_epilogue<kModeOverlap, true>(E, d, st) : launch_sieve_epilogue<kModeOverlap, false>(E, d, st));
        if (rc) return rc;
        CUDA_OK(cudaGetLastError());
        return ACB_OK;
    }
    const bool segments = kernel == 2 || kernel == 3 || kernel == 4;
    const int per_lane = kernel == 3 ? 2 : 1;  // segments per lane of the staged kernel (3: two interleaved chains)
    SegPlan P{};
    uint64_t n_units = (uint64_t)n_haystacks;

    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    if (g_timing) {
        CUDA_OK(cudaEventCreate(&ev0));
        CUDA_OK(cudaEventCreate(&ev1));
        CUDA_OK(cudaEventRecord(ev0, st));
    }
#define ACB_DISPATCH(FN, ...)                                                                                      \
    (mode == kModeStandard   ? (cp ? FN<kModeStandard, true>(__VA_ARGS__) : FN<kModeStandard, false>(__VA_ARGS__)) \
     : mode == kModeLeftmost ? (cp ? FN<kModeLeftmost, true>(__VA_ARGS__) : FN<kModeLeftmost, false>(__VA_ARGS__)) \
                             : (cp ? FN<kModeOverlap, true>(__VA_ARGS__) : FN<kModeOverlap, false>(__VA_ARGS__)))
    if (segments) {
        // the grid is anchored at the 64-byte aligned address at or before the buffer; the stream
        // bounds (offsets[0], offsets[n]) live on the device and are read by the kernels
        P.origin = -(int64_t)(reinterpret_cast<uintptr_t>(dev_bytes) & 63u);
        P.seg_bytes = plan->segment_bytes;
        P.warm = plan->warm_bytes;
        P.n_segments = (int64_t)plan->n_segments;
        P.lane_stride = plan->lane_stride;
        P.avg_len = n_haystacks > 0 ? total_bytes / (uint64_t)n_haystacks : 0;
        n_units = 2 * plan->n_segments;
    }
    if (kernel == 4) {
        rc = ACB_DISPATCH(launch_global, im, B, P, out, seg_info, d, st);
        if (rc) return rc;
        CUDA_OK(cudaGetLastError());
        if (ev1) {
            CUDA_OK(cudaEventRecord(ev1, st));
            g_timing_events.emplace_back(ev0, ev1);
        }
    } else if (segments) {
        DevHot hot;
        if ((rc = make_hot_view(a, dev_hot, *hot_desc, hot))) return rc;
        // the byte-indexed table is used when it exists and every row the profile saw fits on chip
        uint32_t fit128 = ascii_rows_that_fit(d);
        if (fit128 > hot.n_rows128) fit128 = hot.n_rows128;
        if (g_tuning.hot_rows > 0 && (uint32_t)g_tuning.hot_rows < fit128) fit128 = (uint32_t)g_tuning.hot_rows;
        // Byte-indexed (128-wide) rows make the transition two instructions per byte (IDP4A + LDS) instead of four,
        // but they are 256 bytes each (only ~230 fit below 64 KB) and on the config-2 text the kernel is bound by
        // the shared-memory pipe, not by instruction issue: measured equal to the compact table (162 vs 160 us).
        // Opt-in (tuning.table = 2), one segment per lane only (two per lane leave too little room for the rows).
        const bool ascii = g_tuning.table == 2 && fit128 > 0 && per_lane == 1;
        rc = ACB_DISPATCH(launch_staged_cols, h, im, hot, B, P, out, seg_info, d, task_counter, acc + kAccGroups, st, ascii, per_lane);
        if (rc) return rc;
        CUDA_OK(cudaGetLastError());
        if (ev1) {
            CUDA_OK(cudaEventRecord(ev1, st));
            g_timing_events.emplace_back(ev0, ev1);
        }
    } else {
        rc = ACB_DISPATCH(launch_plain, im, B, out, d, st);
        if (rc) return rc;
        CUDA_OK(cudaGetLastError());
        if (ev1) {
            CUDA_OK(cudaEventRecord(ev1, st));
            g_timing_events.emplace_back(ev0, ev1);
        }
    }
    // repair -> counts -> offsets -> ordered output -> per-haystack offsets: one cooperative kernel
    const uint64_t max_tiles = (plan->n_units + kScanTile - 1) / kScanTile;
    unsigned long long *tile_sums = reinterpret_cast<unsigned long long *>(ws->dev_scratch) + kAccWords;
    unsigned long long *cont_tiles = tile_sums + max_tiles + 1;
    unsigned long long *cont_cum = cont_tiles + max_tiles + 1;
    uint32_t *cont_dense = reinterpret_cast<uint32_t *>(cont_cum + plan->n_segments + 2);
    OrderArgs A;
    A.raw = ws->dev_raw;
    A.raw_seq = ws->dev_raw_seq;
    A.raw_unit = ws->dev_raw_unit;
    A.raw_aux = ws->dev_raw_aux;
    A.raw_cap = ws->raw_capacity;
    A.raw_total = acc + kAccRaw;
    A.unit_offsets = unit_offsets;
    A.unit_counts = ws->dev_unit_counts;
    A.seg_info = segments ? seg_info : nullptr;
    A.cont_cum = cont_cum;
    A.hay_offsets = dev_offsets;
    A.pat_cplen = im.pat_cplen;
    A.origin = P.origin;
    A.seg_bytes = P.seg_bytes;
    A.codepoints = cp ? 1 : 0;
    A.out = ws->dev_out;
    A.out_cap = ws->out_capacity;
    EpilogueArgs E;
    E.im = im;
    E.B = B;
    E.P = P;
    E.out = out;
    E.seg_info = seg_info;
    E.totals = totals;
    E.acc = acc;
    E.unit_counts = ws->dev_unit_counts;
    E.n_units = n_units;
    E.tile_sums = tile_sums;
    E.unit_offsets = unit_offsets;
    E.cont_tail = (segments && cp) ? reinterpret_cast<const uint32_t *>(seg_info) + 5 : nullptr;
    E.n_segments = plan->n_segments;
    E.cont_tiles = cont_tiles;
    E.cont_cum = cont_cum;
    E.cont_dense = cont_dense;
    E.order = A;
    E.match_offsets = match_offsets;
    E.need_repair = task_counter + 1;
    E.do_repair = (segments && mode != kModeOverlap) ? 1 : 0;
    rc = ACB_DISPATCH(launch_epilogue, E, d, st);
#undef ACB_DISPATCH
    if (rc) return rc;
    CUDA_OK(cudaGetLastError());
    return ACB_OK;
}

}  // extern "C"
