/*
 * antiz_b200 - C ABI of the B200-native AntiZ precompression hot path.
 *
 * The reference (jagannatharjun/AntiZ) has no FFI; its seams are in-process C++
 * member functions (SURVEY.md 8b).  Each entry point below replaces one of those
 * seams and is what a binding (ctypes, or the `uncomp` host program in
 * antiz_b200/host/) calls.  Plain pointers and sizes only; no exceptions cross
 * this boundary; every function returns 0 on success or a negative ATZ_E_* code.
 * All work is done by hand-written sm_100a CUDA kernels; there is no CPU path:
 * without a usable CUDA device atz_ctx_create() fails with ATZ_E_NO_DEVICE.
 *
 * One context per GPU; a context is used from one host thread at a time.
 * Reference lines cite /root/reference/main.cpp unless noted.
 */
#ifndef ANTIZ_B200_H
#define ANTIZ_B200_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ATZ_OK 0
#define ATZ_E_NO_DEVICE  (-1)  /* no CUDA device / driver: the product never falls back to the CPU */
#define ATZ_E_CUDA       (-2)  /* a CUDA call or kernel failed; see atz_last_error() */
#define ATZ_E_ARG        (-3)  /* bad argument (NULL, level/window/memlevel out of range, chunksize < 2, ...) */
#define ATZ_E_STATE      (-10) /* calls out of order; same value as the reference's phase guard (main.cpp:263,278,289,302) */
#define ATZ_E_TOO_LARGE  (-4)  /* input >= 4 GiB (the reference's uInt limit, ZlibWrapper.h:29, main.cpp:628) */
#define ATZ_E_NOMEM      (-5)
#define ATZ_E_DATA       (-6)  /* atz_inflate_stream: not a complete valid zlib stream */
#define ATZ_E_SMALL      (-7)  /* output buffer too small */
#define ATZ_E_TRUNCATED  (-8)  /* atz_inflate_stream: the input ended before the end of the stream (zlib would wait for more) */

typedef struct atz_ctx atz_ctx;

/* ATZdata::programOptions, the fields the hot path reads (ATZData.h:7-35). */
typedef struct {
    uint64_t recompTresh;     /* default 128 */
    uint64_t sizediffTresh;   /* default 128 */
    uint64_t shortcutLength;  /* default 512 */
    uint64_t mismatchTol;     /* default 2   */
    int32_t  bruteforceWindow;/* --brute-window */
    int32_t  flags;           /* ATZ_F_* */
} atz_options;

/* Keep ATZdata::streamOffset::identBytes/zlibparams exact even for streams that end up NOT recompressed.
 * Without it, a trial is cut as soon as it has more than max(recompTresh, mismatchTol) mismatches: such a
 * trial can neither be a full match nor make the stream recompressible, so the ATZ bytes do not change
 * (DESIGN.md "early cut"); only the (never written) records of non-recompressed streams may differ. */
#define ATZ_F_EXACT_RECORDS 1
/* Extension (SURVEY.md 8 f4; not in the reference, which only ever passes Z_DEFAULT_STRATEGY, main.cpp:624): for a stream that the
 * reference's candidates (header class, then --brute-window if asked for) do not reproduce, also try zlib's other strategies -
 * Z_FILTERED (levels 4-9), Z_FIXED (levels 1-9), Z_RLE and Z_HUFFMAN_ONLY, each over memLevel 9..1 at the header's window
 * (Z/deflate.c:1861-1967, Z/trees.c:952).  A winner found this way is reported with the strategy in the high nibble of `clevel`
 * (ATZ_CLEVEL below); the ATZ file then differs from the reference's and only this library's reconstructor can read it. */
#define ATZ_F_STRATEGIES 2
/* `clevel` bytes (atz_stream.clevel, atz_deflate_stream / _batch / atz_trial arguments): level 0..9 in the low nibble, zlib strategy
 * 0..4 in bits 4-6 (0 = Z_DEFAULT_STRATEGY: plain levels are unchanged). */
#define ATZ_CLEVEL(level, strategy) ((uint8_t)((level) | ((strategy) << 4)))
/* Extension (SURVEY.md 8 f4; not in the reference): also recompress zlib streams inside the plaintext of recompressed streams, down to
 * `depth` levels (0..8; 0 = off; ATZ_E_ARG above 8).  After the level-d streams have been searched (d = 0: the file's), the plaintext P
 * of every recompressed level-d stream this context owns is walked ascending: at a position p where (P[p], P[p+1]) is a header of the
 * context's scan set (ATZ_SCAN_SMALL_WINDOWS counts; IDAT runs are not looked for), P[p:] is inflated with its input cut at the end of
 * P; a stream that ends there with a correct adler32 after more than 16 bytes (C) is accepted and the walk goes on at p + C, otherwise at
 * p + 1.  The level-(d+1) streams are searched like top-level ones (same candidate sequences, --brute-window, strategies, thresholds,
 * diff lists) and belong to their parent's owner; atz_get_nested returns them.  Stats n_streams / n_recomp stay top-level; ref_trials
 * and gpu_trials include the nested trials.  Carried in atz_options.flags, bits 8 and up, so that atz_options keeps its layout; any value
 * of those bits above 8 (a negative flags word too) is ATZ_E_ARG. */
#define ATZ_F_NESTED_DEPTH(d) ((d) << 8)

/* ATZdata::streamOffset (ATZData.h:42-77), flattened. */
typedef struct {
    uint64_t offset;          /* file offset of the 2-byte zlib header */
    uint64_t streamLength;    /* C: compressed bytes incl. header + adler */
    uint64_t inflatedLength;  /* U */
    uint64_t identBytes;
    int64_t  firstDiffByte;   /* -1 = none */
    uint64_t ndiff;           /* diffByteOffsets.size() (only filled for recomp streams) */
    uint64_t diff_index;      /* first entry of this stream in the arrays returned by atz_get_diffs() */
    int32_t  offsetType;      /* 0..23, parseOffsetType (main.cpp:168-203) = 4 * (CINFO - 2) + FLEVEL; with ATZ_SCAN_SMALL_WINDOWS
                                 also 24..31 = 24 + 4 * CINFO + FLEVEL (CINFO 0 and 1) */
    uint8_t  clevel, window, memlevel; /* zlibParamPack; ctor defaults 9/15/9 (ATZData.h:50-52) */
    uint8_t  recomp;
} atz_stream;

typedef struct {
    uint64_t n_candidates;      /* magic hits found by the scan kernel */
    uint64_t n_streams;
    uint64_t n_recomp;
    uint64_t ref_trials;        /* trials the reference would have executed (testDeflateParams calls) */
    uint64_t gpu_trials;        /* trials actually launched (>= ref_trials: waves are speculative) */
    uint64_t algo_bytes;        /* algorithmic bytes, SURVEY.md 8(d) */
    uint64_t kernel_launches;   /* kernels launched by this library since the last atz_load() */
    double ms_h2d, ms_scan, ms_inflate_probe, ms_inflate, ms_chains, ms_trials, ms_diff, ms_d2h; /* CUDA-event times on the ctx stream */
    double ms_trials_max_kernel; uint64_t n_trial_kernels;
    uint64_t trial_algo_bytes;  /* the part of algo_bytes the trial kernel is charged with */
    double ms_rows;             /* row tables (deflate.cu build_rows_kernel) */
} atz_stats;

const char *atz_version(void);
const char *atz_last_error(atz_ctx *ctx);

int  atz_ctx_create(int device, atz_ctx **out);
void atz_ctx_destroy(atz_ctx *ctx);
/* Upper bound of device memory the search may use for hash-chain structures (default: 60% of free memory). */
int  atz_ctx_set_budget(atz_ctx *ctx, uint64_t bytes);
/* Which zlib headers the scan accepts (ATZ_SCAN_* bits; default 0: the reference's 24).  Valid before the first atz_load /
 * atz_load_device / atz_attach; ATZ_E_STATE after that, ATZ_E_ARG for an unknown bit.  Every shard of a sharded run must use the
 * same set: atz_probe_import refuses the records of a shard that scanned with another one (ATZ_E_STATE). */
int  atz_ctx_set_scan_flags(atz_ctx *ctx, uint32_t flags);
/* Extension (SURVEY.md 8 f4; not in the reference, whose scan stops at CINFO 2): also accept the 8 headers with CINFO 0 and 1
 * (CMF 0x08 and 0x18; windows of 256 and 512 bytes).  zlib writes CINFO 1 for deflateInit2(windowBits 8 or 9); CINFO 0 comes from
 * encoders that rewrite the header of a small stream.  Both are searched at windowBits 9 (offsetType 24..31); a CINFO 0 stream that
 * zlib reproduces differs from its winner in the two header bytes, which go into its diff list.  The ATZ layout does not change, so
 * the reference's reconstructor still reads the file; it differs from the reference's own output because more streams are found. */
#define ATZ_SCAN_SMALL_WINDOWS 1
/* Extension (SURVEY.md 8 f4; not in the reference): PNG encoders split an image's zlib stream over consecutive IDAT chunks, with 12 bytes
 * of chunk framing (CRC, next length and type) between two pieces, so the scan's inflate fails at the end of the first piece.  With this
 * flag a K1 candidate that starts an IDAT run (header right behind an "IDAT" tag whose chunk is followed by another IDAT; see
 * atz_host_idat_run) is also inflated over the run's data, concatenated.  A stream that ends there (adler32 correct) beyond its first
 * chunk and is longer than 16 bytes is a split stream: its record has offset = the header, streamLength = C, the de-chunked compressed
 * length, and its span in the file is C + 12 * (pieces - 1) bytes (atz_get_pieces).  It replaces the accepted streams that lie inside
 * that span and is dropped if an accepted stream overlaps the span without lying inside it.  May be ORed with ATZ_SCAN_SMALL_WINDOWS.
 * The ATZ file of a run with split streams can only be read by this library's reconstructor. */
#define ATZ_SCAN_PNG_IDAT 4
/* Extension (SURVEY.md 8 f4; not in the reference): an animated PNG keeps every frame but its default image in a zlib stream of its own,
 * split over consecutive fdAT chunks whose data start with a 4-byte sequence number, so 16 bytes of framing (CRC, next length, type and
 * sequence number) lie between two pieces.  With this flag a K1 candidate that starts an fdAT run (header right behind an "fdAT" tag and
 * its sequence number, whose chunk is followed by another fdAT; see atz_host_fdat_run) is inflated over the run's pieces like an IDAT
 * run, with the same rule for what is a split stream; its span in the file is C + 16 * (pieces - 1) bytes (atz_get_framing).  Sequence
 * numbers and CRCs are not checked.  A header that starts both kinds of run (its sequence number spells "IDAT") is taken as an IDAT run
 * when ATZ_SCAN_PNG_IDAT is set.  Does not imply ATZ_SCAN_PNG_IDAT (an APNG's default image is in IDAT chunks); may be ORed with it and
 * with ATZ_SCAN_SMALL_WINDOWS.  Bits 2 and 8 stay unassigned.  The ATZ file of a run with split streams can only be read by this
 * library's reconstructor. */
#define ATZ_SCAN_APNG_FDAT 16

/* ---- precompress path ------------------------------------------------------------------------------ */

/* Copy the input file image to the device.  Replaces the per-chunk ifstream reads of searchInfile
 * (main.cpp:392-420) and the per-stream re-reads of findDeflateParams_ALL (main.cpp:431-436).
 * `file` may be pageable or pinned host memory.  n must be >= 1 and < 4 GiB. */
int atz_load(atz_ctx *ctx, const uint8_t *file, uint64_t n);

/* Same, but the image is already in device memory (benchmarks: "inputs resident in HBM"). */
int atz_load_device(atz_ctx *ctx, const void *dev_file, uint64_t n);

/* Phase 1: ZBuffSearcher over the whole file with the reference's per-chunk semantics
 * (main.cpp:205-246 and SURVEY.md A.1: 1-byte chunk overlap, total_in <= 16 rule, candidates inside an accepted
 * stream skipped, cross-chunk continuation with the duplicated byte).  Leaves every accepted stream's plaintext
 * resident on the device.  *n_streams receives streamOffsetList.size(). */
int atz_scan(atz_ctx *ctx, uint64_t chunksize, uint64_t *n_streams);

/* ---- one container over several GPUs (SURVEY.md 8e): one context per GPU, in one process (uncomp --gpus N) or one process each ----
 * The chunks of searchInfile (main.cpp:405-415) are split into nshards contiguous ranges.  Shard g probes the candidates that start in
 * its range (K1 + K2; main.cpp:205-246 up to the accept decision), and exports one fixed-size record per candidate the accept logic can
 * act on.  The host hands every shard's records to every context (memcpy in one process; any byte transport between processes - this is
 * the "host-side gather", there is no device collective); atz_scan_finish then replays ZBuffSearcher's sequential accept logic over all
 * of them (identical on every context), partitions the accepted streams over the shards (atz_host_partition: by plaintext length, a
 * stream staying on the shard that probed it where the balance allows) and
 * leaves the plaintext of the streams THIS shard owns resident.  atz_search_shard(ctx, opt, g, nshards) searches those; the per-stream
 * records are gathered by owner.  atz_scan(ctx, S, &n) is atz_scan_shard(ctx, S, 0, 1) + atz_scan_finish(ctx, &n).
 *
 * atz_attach: like atz_load, but the bytes stay in host memory (pageable or pinned; the caller keeps them alive and unchanged until the
 * search has returned) and only what this shard needs is copied to its GPU: its chunk range (plus the chunk a continuation may run
 * into) and the compressed bytes of the streams it owns. */
int atz_attach(atz_ctx *ctx, const uint8_t *file, uint64_t n);
int atz_scan_shard(atz_ctx *ctx, uint64_t chunksize, uint32_t shard, uint32_t nshards);
/* This shard's probe records as an opaque byte string (*nbytes receives its size; ATZ_E_SMALL if cap is too small, buf may be NULL). */
int atz_probe_export(atz_ctx *ctx, void *buf, uint64_t cap, uint64_t *nbytes);
/* The records another shard exported (each of the other nshards-1 shards exactly once before atz_scan_finish). */
int atz_probe_import(atz_ctx *ctx, uint32_t shard, const void *buf, uint64_t nbytes);
int atz_scan_finish(atz_ctx *ctx, uint64_t *n_streams);

/* Phase 3: findDeflateParams_ALL (main.cpp:421-460) = for every stream the sequential winner fold of
 * testDeflateParams (main.cpp:603-731) over the candidate order of main.cpp:487-602. */
int atz_search(atz_ctx *ctx, const atz_options *opt);
/* Multi-GPU: the same, restricted to the streams that atz_host_partition gives to `shard` (static partition of the stream x parameter
 * grid, SURVEY.md 8e).  After a sharded scan (shard, nshards) must be the scan's; after a plain atz_scan any partition may be asked for.
 * The host gathers stream i's record from the context that owns it. */
int atz_search_shard(atz_ctx *ctx, const atz_options *opt, uint32_t shard, uint32_t nshards);

/* A stream found inside the plaintext of another (ATZ_F_NESTED_DEPTH).  parent < n_streams: the top-level stream `parent`; otherwise
 * entry parent - n_streams of the same atz_get_nested list (always an earlier one).  depth: 1 under a top-level stream, 2 under a
 * depth-1 stream, ...  s.offset is relative to the start of the parent's plaintext; s.diff_index points into atz_get_diffs' arrays. */
typedef struct { uint64_t parent; uint32_t depth; uint32_t reserved; atz_stream s; } atz_nested;

/* Results.  `streams` must have room for n_streams entries. */
int atz_get_streams(atz_ctx *ctx, atz_stream *streams, uint64_t cap);
/* owner[i] = shard that owns stream i: set by atz_scan_finish (sharded scan) or by the last atz_search_shard (0 before that).  The
 * host gathers stream i's record, diff list and plaintext from that context; every context of a run reports the same list. */
int atz_get_owners(atz_ctx *ctx, uint32_t *owner, uint64_t cap);
/* The pieces of stream i in the file (ATZ_SCAN_PNG_IDAT, ATZ_SCAN_APNG_FDAT): *npieces = 0 for an ordinary stream, >= 2 for a split
 * one, whose piece lengths (summing to streamLength; piece k+1 starts atz_get_framing bytes after piece k ends) go to
 * len[0 .. min(npieces, cap)).  ATZ_E_SMALL if cap < npieces.  Every context of a sharded run reports the same pieces. */
int atz_get_pieces(atz_ctx *ctx, uint64_t stream_index, uint32_t *len, uint64_t cap, uint64_t *npieces);
/* The framing bytes between two pieces of stream i: 0 for an ordinary stream, 12 for one split over IDAT chunks (CRC, length, type),
 * 16 for one split over fdAT chunks (CRC, length, type, sequence number). */
int atz_get_framing(atz_ctx *ctx, uint64_t stream_index, uint32_t *bytes);
/* diffByteOffsets (delta-encoded, main.cpp:757-763) and diffByteVal of all recomp streams, concatenated: the top-level streams', then
 * those of the nested streams (atz_get_nested order). */
int atz_get_diffs(atz_ctx *ctx, uint64_t *offsets, uint8_t *values, uint64_t cap, uint64_t *n);
/* The nested streams the last search found under the streams this context owns, recompressed or not (ATZ_F_NESTED_DEPTH): level by
 * level, then by parent, then by offset.  *n receives their number; ATZ_E_SMALL if cap is smaller. */
int atz_get_nested(atz_ctx *ctx, atz_nested *out, uint64_t cap, uint64_t *n);
/* Inflated payload of stream i (what writeStreamdesc re-inflates, main.cpp:824-828); i = n_streams + j is nested entry j. */
int atz_get_inflated(atz_ctx *ctx, uint64_t stream_index, uint8_t *dst, uint64_t cap);
/* All payloads of recomp streams (of a sharded run: the ones this context owns), concatenated in stream order, into one host buffer (one D2H). */
int atz_get_inflated_recomp(atz_ctx *ctx, uint8_t *dst, uint64_t cap, uint64_t *n);
/* The payloads of the given streams (indices as atz_get_inflated takes them), concatenated in the given order (ATZ_E_STATE for a stream
 * another shard owns). */
int atz_get_inflated_list(atz_ctx *ctx, const uint64_t *indices, uint64_t count, uint8_t *dst, uint64_t cap, uint64_t *n);
int atz_get_stats(atz_ctx *ctx, atz_stats *st);
/* CUDA-event stopwatch on the context's stream (the stream every kernel of this library is launched on):
 * atz_timer_start records an event, atz_timer_stop records a second one, waits for it and returns the elapsed ms. */
int atz_timer_start(atz_ctx *ctx);
int atz_timer_stop(atz_ctx *ctx, double *ms);

/* ---- single-stream operators (ATZcreator::doInflate main.cpp:461-486, ATZreconstructor::doDeflate 976-1003) -- */

/* Whole zlib stream -> plaintext.  *consumed = total_in, *out_len = total_out (also on ATZ_E_DATA / _SMALL / _TRUNCATED,
 * where they are zlib's totals at the point inflate() stopped; up to `cap` bytes of output are returned).  ATZ_E_SMALL is zlib's
 * "output buffer full" state: *out_len = cap (the buffer is filled to the last byte, a match cut where the room ends) and
 * *consumed = the input used by then - what ZlibInflator::operator() / continuePrev report (ZlibWrapper.h:56-77). */
int atz_inflate_stream(atz_ctx *ctx, const uint8_t *in, uint64_t n, uint8_t *out, uint64_t cap,
                       uint64_t *out_len, uint64_t *consumed);
/* deflateInit2(clevel, Z_DEFLATED, window, memlevel, Z_DEFAULT_STRATEGY) + deflate(Z_FINISH): byte-identical
 * to zlib 1.2.8.  clevel 0..9 (a strategy may ride in its high nibble: ATZ_CLEVEL), window 9..15, memlevel 1..9. */
int atz_deflate_stream(atz_ctx *ctx, const uint8_t *in, uint64_t n, int clevel, int window, int memlevel,
                       uint8_t *out, uint64_t cap, uint64_t *out_len);

/* Reconstruct path: n independent doDeflate calls in one launch (reconstructATZ's loop, main.cpp:893-932).
 * in_off[i]/in_len[i] index `in`; out_off[i]/out_cap[i] index `out`; out_len[i] receives each length. */
int atz_deflate_batch(atz_ctx *ctx, const uint8_t *in, const uint64_t *in_off, const uint64_t *in_len,
                      const uint8_t *clevel, const uint8_t *window, const uint8_t *memlevel, uint64_t n,
                      uint8_t *out, const uint64_t *out_off, const uint64_t *out_cap, uint64_t *out_len);

/* One recompression trial, exposed for parity tests: the {bailed, C', ident} triple of testDeflateParams
 * (main.cpp:632-681) for plaintext `in` against the original stream `orig`.
 * status: 0 compared (valid size), 1 bailed at the shortcut, 2 size gate failed, 3 cut early (see flags). */
typedef struct { int32_t status; uint32_t in_consumed; uint64_t out_len; uint64_t ident; uint64_t kcycles, kcycles_flush; /* SM kilocycles: whole trial / block flushes */ } atz_trial_result;
int atz_trial(atz_ctx *ctx, const uint8_t *in, uint64_t n, const uint8_t *orig, uint64_t c,
              int clevel, int window, int memlevel, const atz_options *opt, atz_trial_result *res);

/* ---- host-logic hooks (pure host code, no device needed): the reference's candidate order (main.cpp:487-602), chunk list
 * (main.cpp:405-415) and ZBuffSearcher accept logic (main.cpp:205-246), exported so CPU tests can pin them. ---- */
/* brute: 0 = the header class's sequence (81 candidates), 1 = the --brute-window grid (405; 486 for offsetType 24..31, whose
 * header window 9 is not part of the grid), 2 = the ATZ_F_STRATEGIES extension (153; strategy in the high nibble of clevel).
 * offsetType 0..31 (24..31: ATZ_SCAN_SMALL_WINDOWS, searched at window 9).  Returns the length of the sequence. */
int atz_host_candidate_sequence(int offsetType, int brute, uint8_t *clevel, uint8_t *window, uint8_t *memlevel, uint32_t cap);
/* The header test of the scan (the same function K1 runs): offsetType of the zlib header (b0, b1) under the ATZ_SCAN_* set
 * scan_flags, or -1 if the set does not accept it. */
int atz_host_header_type(uint32_t scan_flags, uint32_t b0, uint32_t b1);
/* The IDAT run walker of ATZ_SCAN_PNG_IDAT (the same function the run-detection kernel runs) at file offset p: *npieces = number of
 * IDAT chunks of the run (0: p starts none; a run has >= 2), their data lengths into len[0 .. min(*npieces, cap)). */
int atz_host_idat_run(const uint8_t *file, uint64_t n, uint64_t p, uint32_t *len, uint64_t cap, uint64_t *npieces);
/* The same for the fdAT run walker of ATZ_SCAN_APNG_FDAT: p is where the stream's piece starts, behind the first chunk's sequence
 * number; the lengths are the pieces', L - 4 per chunk. */
int atz_host_fdat_run(const uint8_t *file, uint64_t n, uint64_t p, uint32_t *len, uint64_t cap, uint64_t *npieces);
/* owner[k] = shard that searches the k-th accepted stream of a scan, given the streams' inflated lengths.  probed_by == NULL: longest
 * first, each to the least loaded shard (what atz_search_shard uses after a plain atz_scan).  probed_by[k] = shard whose chunk range
 * stream k starts in (what atz_scan_finish uses): a stream stays where its plaintext already is unless that shard holds more than 2 %
 * above the mean load. */
int atz_host_partition(const uint64_t *inflated_len, const uint32_t *probed_by, uint32_t n, uint32_t nshards, uint32_t *owner);
int atz_host_chunks(uint64_t n, uint64_t chunksize, uint64_t *start, uint64_t *len, uint64_t cap);
/* How atz_search_shard splits the streams of a shard over its search lanes (host thread + CUDA stream each; DESIGN.md 5a): lane_of[k]
 * for the stream with inflated length inflated_len[k]; forced_lanes > 0 overrides the lane count.  Returns the number of lanes. */
int atz_host_lane_partition(const uint64_t *inflated_len, uint32_t n, int forced_lanes, uint32_t *lane_of);
int atz_host_scan_fold(uint64_t n, uint64_t chunksize, const uint32_t *cand, uint32_t ncand, const uint64_t *probe, const uint64_t *avail,
                       const int32_t *cont_of, const uint64_t *cont, uint32_t ncont, uint64_t *out, uint32_t cap);

#ifdef __cplusplus
}
#endif
#endif
