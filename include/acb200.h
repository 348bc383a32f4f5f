/*
 * acb200.h -- C ABI of the B200-native multi-pattern matcher (libacb200.so).
 *
 * This is the drop-in boundary for the reference's hot path.  The reference
 * (G-Research/ahocorasick_rs) has no C ABI of its own: its PyO3 shim
 * (src/lib.rs) calls straight into the Rust crate `aho-corasick` 1.1.4.  Each
 * entry point below names the reference call site it stands in for; a
 * maintainer of the reference would bind these from src/lib.rs through
 * `extern "C"` (see INTEGRATION.md) or, as this repo does, from Python with
 * ctypes (ahocorasick_rs_b200/_capi.py).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every function returns ACB_OK (0) or a negative ACB_E* code; text for the
 *     last error on the calling thread comes from acb_last_error();
 *   - "dev_" pointers are CUDA device pointers on the current device; the
 *     library never allocates device memory: the caller (PyTorch's caching
 *     allocator in this repo) owns every buffer and says how big it is;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it
 *     and nothing synchronises unless stated;
 *   - there is no CPU fallback: scan entry points fail with ACB_ECUDA when no
 *     device is usable.
 */
#ifndef ACB200_H
#define ACB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACB_OK 0
#define ACB_EINVAL (-1)      /* bad argument */
#define ACB_EBUILD (-2)      /* automaton construction failed (reference: BuildError -> ValueError, src/lib.rs:215,406) */
#define ACB_EUNSUPPORTED (-3) /* overlapping search on a non-Standard automaton (reference: MatchError -> ValueError, src/lib.rs:36-39,52-54) */
#define ACB_ECUDA (-4)       /* CUDA runtime error / no device */
#define ACB_ECAPACITY (-5)   /* a caller-provided buffer is too small */

/* MatchKind (reference: src/lib.rs:92-98) */
#define ACB_STANDARD 0
#define ACB_LEFTMOST_FIRST 1
#define ACB_LEFTMOST_LONGEST 2

/* Implementation (reference: src/lib.rs:111-118). -1 = None (heuristic).
 * Here it selects the device table layout only; results never depend on it. */
#define ACB_IMPL_AUTO (-1)
#define ACB_IMPL_NONCONTIGUOUS_NFA 0
#define ACB_IMPL_CONTIGUOUS_NFA 1
#define ACB_IMPL_DFA 2

typedef struct acb_automaton acb_automaton;

/* One match, as the reference's (pattern, start, end) tuple (src/lib.rs:240-246,
 * 431) plus the haystack it belongs to.  16 bytes, written with one store. */
typedef struct acb_match {
    uint32_t haystack; /* index into the batch (0 for single-haystack calls) */
    uint32_t pattern;  /* index into the pattern list given to acb_build */
    uint32_t start;    /* byte offset, or code point index when codepoints != 0 */
    uint32_t end;      /* exclusive */
} acb_match;

const char *acb_last_error(void);
const char *acb_version(void);

/*
 * Build an automaton on the host.
 * Stands in for AhoCorasickBuilder::new().kind(..).match_kind(..).build(..)
 * at src/lib.rs:186-215 (str) and 401-406 (bytes).
 * Pattern i is blob[offsets[i] .. offsets[i+1]); ids are input order.  Empty
 * patterns are an error here too (the reference rejects them before the crate
 * sees them, src/lib.rs:204-207,386-389).
 */
int acb_build(const uint8_t *blob, const uint64_t *offsets, uint64_t n_patterns, int match_kind,
              int implementation, acb_automaton **out);

/*
 * Build flags (acb_build_ex).
 * ACB_ASCII_CASE_INSENSITIVE stands in for AhoCorasickBuilder::ascii_case_insensitive(true): an ASCII letter in a
 * pattern matches either case of that letter in the haystack; no other byte changes (bytes >= 0x80 included, so
 * code point indexes are unaffected).  The matches are exactly those of the case-sensitive automaton of the folded
 * patterns (A-Z -> a-z) on the folded haystack, reported with the ORIGINAL pattern ids and lengths; patterns that
 * differ only in case keep their own ids.
 */
#define ACB_ASCII_CASE_INSENSITIVE 1u

/* acb_build with build flags; acb_build(...) == acb_build_ex(..., 0, ...).  Unknown flag bits: ACB_EINVAL. */
int acb_build_ex(const uint8_t *blob, const uint64_t *offsets, uint64_t n_patterns, int match_kind,
                 int implementation, uint32_t flags, acb_automaton **out);
/* The flags the automaton was built with. */
uint32_t acb_build_flags(const acb_automaton *a);
void acb_free(acb_automaton *a);

/* Facts about a built automaton. */
uint64_t acb_num_patterns(const acb_automaton *a);
uint64_t acb_num_states(const acb_automaton *a);
uint32_t acb_num_columns(const acb_automaton *a);
uint32_t acb_max_pattern_len(const acb_automaton *a);
uint32_t acb_min_pattern_len(const acb_automaton *a);
int acb_match_kind(const acb_automaton *a);

/*
 * The device image: the flat tables the kernels read (column map, dense
 * transition rows, per-state match lists, pattern lengths), serialised into
 * one buffer.  The caller allocates acb_image_bytes() on the device, fills it
 * from acb_image_write()'s host copy ("table uploaded once to HBM"), and
 * passes it to every scan.
 */
uint64_t acb_image_bytes(const acb_automaton *a);
int acb_image_write(const acb_automaton *a, void *host_dst, uint64_t dst_bytes);

/*
 * The hot image: the rows of the table the staged kernel keeps in shared memory,
 * hottest first.  "Hot" is decided from data: acb_profile() walks a sample of a
 * device-resident input through the automaton and counts state visits into
 * dev_visits (u32[acb_num_states], zeroed by the call); the caller copies the
 * counts to the host and hands them to acb_hot_build() (host_visits == NULL:
 * no profile, shallowest states first), then uploads the result and passes it,
 * with its row count, to the scans.  Which rows are hot changes speed only --
 * everything the fast path cannot prove uneventful is redone by the exact
 * scanner -- never results.  dev_hot == NULL selects the plain kernel.
 */
int acb_profile(const acb_automaton *a, const void *dev_image, const uint8_t *dev_bytes, const int64_t *dev_offsets,
                int64_t n_haystacks, uint64_t total_bytes, int overlapping, uint32_t *dev_visits, void *stream);
uint64_t acb_hot_bytes(const acb_automaton *a, uint32_t max_rows);
int acb_hot_build(const acb_automaton *a, const uint32_t *host_visits, uint32_t max_rows, void *host_dst,
                  uint64_t dst_bytes);
uint32_t acb_hot_rows(const void *host_hot);

/* What a hot image holds (read from its host copy; passed along with the device copy). */
typedef struct acb_hot_desc {
    uint32_t rows;     /* rows of the compact table (column-indexed) */
    uint32_t rows128;  /* rows of the byte-indexed 128-wide table (0: patterns use bytes >= 0x7f) */
    uint32_t visited;  /* rows the profile actually saw; the rest is filler */
    uint32_t reserved; /* flags set by the caller: bit 0 = the hot rows do not cover this data (dense automaton on
                          adversarial input): with tuning.kernel = 0 the scan then runs from the image in global
                          memory / L2 (kernel 4) instead of the shared-memory table */
} acb_hot_desc;
int acb_hot_describe(const void *host_hot, acb_hot_desc *desc);

/*
 * The sieve image: the position-parallel form of the matcher (csrc/sieve.h).  Instead of walking an automaton -- one
 * DEPENDENT table load per haystack byte -- every byte position is tested independently: the W bytes ending there are
 * hashed into a Bloom filter of the patterns' suffixes held in shared memory; survivors walk on through the filter's
 * deeper levels and are finally verified, exactly, against a reverse trie in global memory / L2, which names every
 * pattern ending at that position in the reference's order.  That is the overlapping match list
 * (try_find_overlapping_iter, src/lib.rs:52-54); the non-overlapping lists (try_find_iter, src/lib.rs:58-60) are
 * selected from it per haystack for all three match kinds.  This is the compact (non-DFA) table format: a few tens of
 * bytes per trie node instead of a dense row per state.
 * acb_sieve_build builds (or rebuilds, when the arguments change) the image on the host and returns its size (0 on
 * error): bloom_bytes_max = shared memory the filters may take when the scan keeps one 512-byte window of text per warp
 * on chip (the caller knows the device: shared memory per block minus 46 KB; the builder uses less for sparse pattern sets,
 * which leaves the scan a deeper ring of text), w_max = cap on the primary window in bytes (0 = automatic).  The caller uploads acb_sieve_write()'s copy and passes the device pointer to the
 * scans as dev_sieve (NULL = use the table kernels).
 */
uint64_t acb_sieve_build(acb_automaton *a, uint32_t bloom_bytes_max, uint32_t w_max);
int acb_sieve_write(acb_automaton *a, void *host_dst, uint64_t dst_bytes);
typedef struct acb_sieve_desc {
    uint32_t window;         /* W: bytes hashed per position by the fast path */
    uint32_t last_level;     /* longest suffix length held by the on-chip filter */
    uint32_t probes;         /* Bloom probes per key */
    uint32_t bloom_bytes;
    uint32_t nodes;          /* reverse-trie nodes (depth >= W) */
    uint32_t keys;           /* distinct W-byte suffixes = hash table entries */
    uint32_t filter_entries;
    uint32_t table_slots;
} acb_sieve_desc;
int acb_sieve_describe(const void *host_sieve, acb_sieve_desc *desc);

/*
 * How a scan is cut up.  The byte stream [offsets[0], offsets[n]) is divided into
 * fixed-size SEGMENTS on a grid anchored at the 64-byte aligned address at or
 * before dev_bytes; one GPU lane scans one segment, so the work per lane is the
 * same whatever the haystack lengths are (one huge haystack, a ragged batch, a
 * million short lines).  A segment that begins inside a haystack starts from a
 * speculated automaton state that is verified -- and, when wrong, repaired --
 * before results are delivered; see DESIGN.md.  The plan depends only on
 * host-known quantities: the automaton, the address of the byte buffer, its
 * length and the number of haystacks.
 */
typedef struct acb_plan {
    uint64_t n_segments;
    uint64_t n_units;       /* entries the unit arrays of the workspace need */
    uint64_t scratch_words; /* u64 words dev_scratch needs */
    uint32_t segment_bytes;
    uint32_t warm_bytes;    /* bytes scanned before a segment to guess its start state (>= longest pattern) */
    uint32_t lane_stride;   /* segments between neighbouring lanes of a warp */
    uint32_t task_bytes;    /* the sieve kernel's unit of work: bytes of the stream one warp walks (a multiple of 512) */
} acb_plan;

int acb_plan_scan(const acb_automaton *a, const void *dev_bytes, uint64_t total_bytes, uint64_t n_haystacks,
                  acb_plan *plan);

/* Caller-provided device workspace for one scan, sized from the plan. */
typedef struct acb_workspace {
    acb_match *dev_raw;      /* [raw_capacity] unordered matches as kernels emit them */
    uint32_t *dev_raw_seq;   /* [raw_capacity] rank of each raw match inside its unit */
    uint32_t *dev_raw_unit;  /* [raw_capacity] unit (segment slot / haystack) each raw match belongs to */
    uint32_t *dev_raw_aux;   /* [raw_capacity] code point bookkeeping per raw match */
    uint64_t raw_capacity;
    uint32_t *dev_unit_counts;   /* [plan.n_units] */
    uint64_t *dev_unit_offsets;  /* [plan.n_units + 1] */
    void *dev_seg_info;          /* [plan.n_segments * 32 bytes] per-segment summaries */
    uint64_t *dev_scratch;       /* [plan.scratch_words]; its first 8 words must be ZERO the first time a workspace is
                                    used: they hold the kernels' counters, and every completed scan leaves them zeroed
                                    again (so a scan needs no clearing launch in front of it) */
    uint64_t *dev_total;         /* [8]: [0] = matches found, [1] = 1 when dev_out holds all of them (0: buffers too
                                    small, retry), [2] = 16-byte groups in the stream, [3] = times a lane left the hot table
                                    for the exact scanner, [4] = raw matches emitted, [5] = segment boundaries repaired */
    acb_match *dev_out;          /* [out_capacity] final matches in the reference's order */
    uint64_t out_capacity;
    uint64_t *dev_match_offsets; /* [n_haystacks + 1] haystack h's matches are dev_out[off[h] .. off[h+1]) */
} acb_workspace;

/*
 * Scan a batch of haystacks resident in device memory:
 * haystack h = dev_bytes[dev_offsets[h] .. dev_offsets[h+1]); total_bytes =
 * length of the dev_bytes buffer (>= dev_offsets[n]).  One haystack of many
 * gigabytes is just n_haystacks = 1.
 *
 * Per haystack this is the drain of the reference's iterator: get_matches
 * (src/lib.rs:42-68) choosing try_find_iter (58-60) or
 * try_find_overlapping_iter (52-54), collected at 238-248 (str) / 433 (bytes).
 * codepoints != 0 reports start/end as code point indexes, i.e. it also does
 * the work of get_byte_to_code_point (src/lib.rs:73-88) for valid UTF-8.
 *
 * On return (after the stream has run): ws->dev_out holds
 * min(total, out_capacity) matches ordered by haystack and then in the
 * reference's iteration order; ws->dev_match_offsets brackets each haystack's
 * matches; ws->dev_total[0] is the true total.  If the matches did not fit
 * raw_capacity / out_capacity nothing is lost silently: dev_total[1] is 0 and
 * dev_total[0] / [4] say how much room a second call needs.
 * overlapping on a non-Standard automaton returns ACB_EUNSUPPORTED before any
 * byte is read, like the reference.  (overlapping = 2 asks for the overlapping LIST of any automaton -- the input of
 * acb_select_non_overlapping; it needs dev_sieve.)
 */
int acb_scan_batch(const acb_automaton *a, const void *dev_image, const void *dev_hot, const acb_hot_desc *hot_desc,
                   const void *dev_sieve, const uint8_t *dev_bytes, const int64_t *dev_offsets, int64_t n_haystacks, uint64_t total_bytes,
                   int overlapping, int codepoints, const acb_plan *plan, const acb_workspace *ws, void *stream);

/*
 * One haystack too large for one call (more than 2^31 bytes), non-overlapping search: the caller scans it as an
 * OVERLAPPING search in windows (exact: the matches ending at a position depend on max_pattern_len - 1 bytes before it),
 * concatenates the lists -- rows of four int64 (haystack, pattern, start, end), in the reference's order -- and this call
 * selects from them what the reference's non-overlapping iterator (try_find_iter, src/lib.rs:58-60) reports for the
 * automaton's match kind: dev_out gets the selected rows, *dev_count their number.  dev_out needs room for n_rows rows.
 */
int acb_select_non_overlapping(const acb_automaton *a, const int64_t *dev_rows, uint64_t n_rows, int64_t *dev_out, uint64_t *dev_count,
                                void *stream);

/*
 * Multi-GPU: the fixed-size block a rank contributes to the gather of the per-shard match lists (the only exchange
 * of the sharded path; NCCL all-gather over NVLink).  dev_block holds (cap + 1) records of 16 bytes: record 0 =
 * (match count, hay_base, complete flag, 0), then the first `cap` matches of a finished scan (dev_total / dev_out of
 * its workspace).  One launch on `stream`, no host round trip.
 */
int acb_pack_gather_block(const uint64_t *dev_total, const acb_match *dev_out, uint32_t hay_base, uint64_t cap, void *dev_block,
                          void *stream);

/* Kernel launch bookkeeping for bench.py's "gpu_launches". */
uint64_t acb_launch_count(void);

/*
 * Device-side timing of the scan kernel alone (CUDA events recorded on the
 * caller's stream around the scan kernel of every subsequent scan call), for
 * the roofline figure.  acb_timing_read synchronises on the recorded events,
 * returns their summed duration and count, and clears them.
 */
int acb_timing_enable(int on);
int acb_timing_read(double *total_ms, uint64_t *n_scans);

/* Tuning knobs (0 = library default), per calling thread. Affects speed only, never results. */
typedef struct acb_tuning {
    int kernel;        /* 0 auto (the sieve when dev_sieve is given), 1 = plain (one thread per haystack, table in global/L2),
                          2 = staged segments (hot rows in shared memory), 3 = staged, two segments per lane, 4 = segments
                          straight from global/L2, 5 = sieve (position-parallel filter + exact verification) */
    int hot_rows;      /* cap on rows kept in shared memory */
    int segment_bytes; /* segment size (rounded up to a multiple of 64 and to 8 x the warm-up); kernel 5: task size (multiple of 512) */
    int table;         /* 0 auto, 1 = column-indexed compact table only, 2 = byte-indexed 128-wide table when available */
} acb_tuning;
int acb_set_tuning(const acb_tuning *t);

#ifdef __cplusplus
}
#endif
#endif /* ACB200_H */
