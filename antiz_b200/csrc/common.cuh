// antiz_b200 - shared device helpers and host<->device record layouts (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/antiz_b200.h"

#define FULL 0xffffffffu
#define ATZ_PAD 512u /* every device buffer that kernels read with unaligned word loads has >= this much zeroed slack */

namespace atz {

// ---------------------------------------------------------------------------------------------
// Records shared by host and kernels
// ---------------------------------------------------------------------------------------------
struct ChainRef {            // bucket lists of one (plaintext, hash_bits): see chains.cu
    const uint32_t *list;    // positions sorted by (hash, position)
    const uint32_t *idx;     // idx[p]  = slot of p in list
    const uint16_t *lsth;    // lsth[s] = hash of list[s]: the chain of p runs down from slot idx[p]-1 while this stays equal
    // optional row table (deflate.cu, build_rows_kernel): 32 bytes per position p < rlen
    const uint4 *rec; uint32_t rlen; uint32_t rbudget;   // rbudget: number of chain candidates the table has looked at
};
#define REC_VALID 0x08000000u
// token map of the ORIGINAL stream (one byte per plaintext position, written by the inflate kernel in produce mode):
// 0 = nothing known; 1 = a literal starts here; 3..250 = a match of that length starts here; TM_LONG = a match of
// 251..258 bytes starts here; TM_INNER + c = inside a match whose length is <= 4 (c = 3), 5 (c = 2), 6 (c = 1), longer (c = 0):
// deflate_fast at level L inserts the inner positions of a match iff its length <= max_insert_length = 3 + L (Z/deflate.c:1680).
#define RES_ABSENT 0x1ffu   /* resolved-table length field: no row here, walk the chain */
#define TM_LONG 251u
#define TM_INNER 252u

struct TrialDesc {
    const uint8_t *in;       // plaintext (any alignment; readable slack of ATZ_PAD bytes behind it and 3 before it)
    const uint8_t *orig;     // original compressed stream to compare with (any alignment) or nullptr
    uint8_t *out;            // store mode: output buffer (4 B aligned) or nullptr
    const uint8_t *tmap;     // token map of the original stream (8 B aligned) or nullptr: the hypothesis of deflate_fast rows, the speculation points of the burst parse
    const uint2 *res;        // levels 4-9: resolved table of this (level, window) for positions < ch.rlen (deflate.cu resolve_rows_kernel) or nullptr
    ChainRef ch;             // unused for level 0
    uint32_t n;              // plaintext length U
    uint32_t c;              // original stream length C
    uint32_t out_cap;        // store mode capacity in bytes (multiple of 4)
    uint32_t adler;          // adler32(plaintext)
    uint8_t level, wbits, memlevel, store;
    uint16_t phase1;         // 1 = stop with TR_PASSED once the --shortcut-len prefix has been compared and accepted
    uint16_t strategy;       // zlib's strategy: 0 Z_DEFAULT_STRATEGY (all the reference ever uses), 1 Z_FILTERED, 2 Z_HUFFMAN_ONLY, 3 Z_RLE, 4 Z_FIXED
};

struct TrialOpts {
    uint32_t shortcut;       // --shortcut-len S; the shortcut applies iff C > S (main.cpp:632)
    uint32_t bail_below;     // bail iff ident over the first min(S, C') bytes < this (main.cpp:649; 0xffffffff = always)
    uint32_t sizediff;       // --sizediff-tresh (main.cpp:671)
    uint32_t cut_mismatch;   // early cut when mismatches exceed this (0xffffffff = never; DESIGN.md "early cut")
    uint32_t compare;        // 1 = search trial (compare with orig), 0 = plain deflate
    uint32_t burst;          // 1 = burst parse where the original's token map allows it (0: test hook ATZ_BURST=0)
};

enum { TR_COMPARED = 0, TR_BAILED = 1, TR_SIZE = 2, TR_CUT = 3, TR_OVERFLOW = 4, TR_PASSED = 5 };
struct TrialResult {
    int32_t status;
    uint32_t in_consumed;    // plaintext bytes parsed when the trial stopped (algorithmic-bytes accounting)
    uint32_t out_len;        // C' (or bytes produced so far if stopped early)
    uint32_t ident;          // equal bytes over min(C', C)
    uint32_t kcycles, kcycles_flush;   // SM kilocycles spent in the trial / in its block flushes (profiling aid)
};

struct InflateJob {          // one candidate stream
    uint64_t off;            // file offset of the zlib header
    uint64_t avail;          // bytes available up to the end of the candidate's chunk
    uint64_t vtotal;         // virtual input length including the following chunks (== avail: no continuation)
    uint64_t out_off;        // offset of the output region in the arena
    uint64_t out_cap;        // size of the output region
    uint64_t tmap_off;       // offset of this stream's token map in the arena, or ~0 for none
    // The reference's chunk reader keeps the wrong byte for the overlap (searchInfile, main.cpp:411-414: `LastByte = rBuffer[f.gcount() - 1]`
    // is the last byte of chunk 0 but the SECOND TO LAST of every later chunk), so the first byte of chunk k >= 2 is file[start_k - 1]:
    //   bit 0      : this candidate starts at such a chunk start - its first input byte is file[off - 1], the rest file[off + 1 ...]
    //   bits 8..15 : how many of the chunk boundaries a continuation crosses still repeat the true last byte (1 for a candidate of chunk 0)
    uint64_t flags;
};
#define INFJ_FIRST_FROM_PREV 1ull
enum { INF_END = 0, INF_NEED_INPUT = 1, INF_DATA_ERROR = 2, INF_NEED_DICT = 3, INF_OUT_FULL = 4 };
struct InflateResult {
    int32_t status; uint32_t adler;
    uint64_t total_in, total_out, in_at_outcap;
};

// ---------------------------------------------------------------------------------------------
// The zlib headers the scan accepts (K1 in scan.cu, the chunk-start fix-up in api.cu).  `scan_flags` is the context's
// ATZ_SCAN_* set (include/antiz_b200.h).  The reference's 24 (ZBuffSearcher::parseOffsetType main.cpp:168-203): CM = 8,
// CINFO 2..7, FDICT = 0, (CMF*256 + FLG) % 31 == 0.  ATZ_SCAN_SMALL_WINDOWS adds CINFO 0 and 1 (CMF 0x08, 0x18): 8 more pairs.
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ bool zlib_header_ok(uint32_t b0, uint32_t b1, uint32_t scan_flags) {
    return (b0 & 0x8fu) == 0x08u && b0 >= ((scan_flags & ATZ_SCAN_SMALL_WINDOWS) ? 0x08u : 0x28u) && (b1 & 0x20u) == 0 && ((b0 << 8) | b1) % 31u == 0;
}
// offsetType of an accepted header: 4 * (CINFO - 2) + FLEVEL = 0..23 for the reference's set, 24 + 4 * CINFO + FLEVEL = 24..31 for
// CINFO 0 and 1
__host__ __device__ __forceinline__ int zlib_header_type_of(uint32_t b0, uint32_t b1) {
    return b0 >= 0x28u ? 4 * ((int)(b0 >> 4) - 2) + (int)(b1 >> 6) : 24 + 4 * (int)(b0 >> 4) + (int)(b1 >> 6);
}
// the same, -1 if the header is not in the set
__host__ __device__ __forceinline__ int zlib_header_type(uint32_t b0, uint32_t b1, uint32_t scan_flags) {
    return zlib_header_ok(b0, b1, scan_flags) ? zlib_header_type_of(b0, b1) : -1;
}

// ---------------------------------------------------------------------------------------------
// PNG chunk runs (ATZ_SCAN_PNG_IDAT, ATZ_SCAN_APNG_FDAT; png.cu, api.cu).  A chunk is a BE32 length L, a 4-byte tag, L data bytes and
// a CRC.  The data of an IDAT is a piece of the image's zlib stream; the data of an APNG fdAT is a 4-byte sequence number, then a piece
// of its frame's stream: `pre` = 0 or 4 bytes in front of each piece.  A header at p starts a run of `tag` chunks when p >= 8 + pre,
// the tag lies at file[p-pre-4 .. p-pre), the chunk's length L1 = BE32(file[p-pre-8 ..]) >= pre + 2 and the chunk behind its CRC is
// a `tag` chunk with L >= pre too.  The run goes on over consecutive `tag` chunks with L >= pre whose data and CRC lie inside the file
// [0, n) and ends at another chunk type, at a shorter one or at one that would run past the end.  Sequence numbers and CRCs are not
// looked at.  Returns the number of chunks (0: p starts no run; a run has >= 2) and their piece lengths L - pre in len[0 ..
// min(count, cap)); piece k+1 starts 12 + pre bytes after piece k ends.  Only [lo, lim) is read (the part of the file the caller can
// address); a walk that would need a byte outside returns IDAT_FAR, and the caller walks again over the whole file.  One dependent
// 8-byte read per chunk.
// ---------------------------------------------------------------------------------------------
#define IDAT_FAR 0xffffffffu
#define TAG_IDAT 0x49444154u    // "IDAT"
#define TAG_FDAT 0x66644154u    // "fdAT"
__host__ __device__ __forceinline__ uint32_t be32(const uint8_t *q) { return (uint32_t)q[0] << 24 | (uint32_t)q[1] << 16 | (uint32_t)q[2] << 8 | q[3]; }
__host__ __device__ inline uint32_t chunk_run(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, uint64_t p, uint32_t tag, uint32_t pre,
                                              uint32_t *len, uint32_t cap) {
    if (p < 8 + pre) return 0;
    if (p - 8 - pre < lo || p > lim) return IDAT_FAR;
    if (be32(file + p - pre - 4) != tag) return 0;
    uint64_t L = be32(file + p - pre - 8), d = p - pre;   // the current chunk: data at d, L bytes
    if (L < pre + 2) return 0;
    uint32_t cnt = 0;
    for (;;) {
        if (d + L + 4 > n) break;                 // data or CRC past the end of the file: not part of the run
        if (d + L + 4 > lim) return IDAT_FAR;
        if (cnt < cap) len[cnt] = (uint32_t)(L - pre);
        cnt++;
        const uint64_t q = d + L + 4;             // the next chunk's header
        if (q + 8 > n) break;
        if (q + 8 > lim) return IDAT_FAR;
        if (be32(file + q + 4) != tag) break;
        L = be32(file + q); d = q + 8;
        if (L < pre) break;
    }
    return cnt >= 2 ? cnt : 0;
}
__host__ __device__ __forceinline__ uint32_t idat_run(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, uint64_t p, uint32_t *len, uint32_t cap) {
    return chunk_run(file, n, lo, lim, p, TAG_IDAT, 0, len, cap);
}
__host__ __device__ __forceinline__ uint32_t fdat_run(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, uint64_t p, uint32_t *len, uint32_t cap) {
    return chunk_run(file, n, lo, lim, p, TAG_FDAT, 4, len, cap);
}
// The run the scan takes at p under the ATZ_SCAN_* set `flags`: an IDAT run if that flag is on and p starts one, otherwise an fdAT
// run if that flag is on (a header whose fdAT sequence number spells "IDAT" can start both).  The count of chunk_run, RUN_FDAT set
// for an fdAT run; IDAT_FAR as there.
#define RUN_FDAT 0x80000000u
__host__ __device__ __forceinline__ uint32_t split_run(const uint8_t *file, uint64_t n, uint64_t lo, uint64_t lim, uint64_t p, uint32_t flags, uint32_t *len, uint32_t cap) {
    if (flags & ATZ_SCAN_PNG_IDAT) {
        const uint32_t m = idat_run(file, n, lo, lim, p, len, cap);
        if (m) return m;
    }
    if (flags & ATZ_SCAN_APNG_FDAT) {
        const uint32_t m = fdat_run(file, n, lo, lim, p, len, cap);
        if (m) return m == IDAT_FAR ? m : m | RUN_FDAT;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// Unaligned 32-bit read through the read-only path. Touches up to 3 bytes before and 7 after p: callers
// guarantee the slack (ATZ_PAD, 16 B aligned arenas).
__device__ __forceinline__ uint32_t ldu32(const uint8_t *p) {
    uintptr_t a = (uintptr_t)p;
    const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
    uint32_t lo = __ldg(w), hi = __ldg(w + 1);
    return __funnelshift_r(lo, hi, (uint32_t)(a & 3) * 8u);
}
// Same for memory written earlier by this kernel (no .nc path).
__device__ __forceinline__ uint32_t ldu32_rw(const uint8_t *p) {
    uintptr_t a = (uintptr_t)p;
    const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
    uint32_t lo = w[0], hi = w[1];
    return __funnelshift_r(lo, hi, (uint32_t)(a & 3) * 8u);
}

__device__ __forceinline__ uint32_t warp_excl_scan(uint32_t v, uint32_t &total) {
    uint32_t lane = lane_id(), x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(FULL, x, d); if (lane >= (uint32_t)d) x += y; }
    total = __shfl_sync(FULL, x, 31);
    return x - v;
}

// zlib's 3-byte rolling hash after three updates (Z/deflate.c:167, hash_shift = (hash_bits+2)/3 Z/deflate.c:291)
__device__ __forceinline__ uint32_t hash3(uint32_t b0, uint32_t b1, uint32_t b2, uint32_t shift, uint32_t mask) {
    return ((((b0 << shift) ^ b1) << shift) ^ b2) & mask;
}

} // namespace atz
