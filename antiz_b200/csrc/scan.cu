// K1 - candidate scan: find every offset i with (file[i], file[i+1]) one of the zlib headers of the context's scan set: the 24 AntiZ
// accepts (ZBuffSearcher::parseOffsetType main.cpp:168-203: CM=8, CINFO 2..7, FDICT=0, (CMF*256+FLG) % 31 == 0), or those and the 8
// of CINFO 0 and 1 (ATZ_SCAN_SMALL_WINDOWS; common.cuh zlib_header_ok).
// HBM-bound by design: the file is read ONCE, with 16-byte vector loads; a word-at-a-time filter on the first header byte (low nibble 8,
// top bit clear: three integer instructions per four bytes) leaves the per-position test to the few bytes that can start a header.
// Pass 1 (scan_count_kernel) stores the 16-bit hit mask of every 16-byte group (N/8 bytes) and the hit count of every 64 KiB tile;
// a one-CTA scan turns the tile counts into output positions; pass 2 (scan_write_kernel) reads the masks, not the file, and writes the
// offsets in order - sorted output without a sort, exact buffer sizes, no spin-waits (a single-pass variant with tile tickets and
// decoupled look-back was built in round 2 and measured no faster inside the running program).
#include "common.cuh"

namespace atz {

#define SCAN_THREADS 256
#define SCAN_TILE (SCAN_THREADS * 16 * 16) /* 64 KiB per CTA */

// bytes of w whose low nibble is 8 and whose top bit is clear (0x08, 0x18, ... 0x78: every CMF of either set) -> 0x80 in that byte.  The zero-byte trick may
// also flag the byte above a true hit (borrow); never misses one - the exact test follows.
__device__ __forceinline__ uint32_t maybe_cmf(uint32_t w) {
    const uint32_t t = (w & 0x8f8f8f8fu) ^ 0x08080808u;
    return (t - 0x01010101u) & ~t & 0x80808080u;
}
// 16 consecutive positions starting at byte `pos` (a multiple of 16); bit k set <=> (pos+k, pos+k+1) is a header, pos+k is in
// [lo, hi) (the part of the file this launch scans: a shard's chunk range, api.cu atz_scan_shard) and pos+k+1 < n
__device__ __forceinline__ uint32_t magic_mask16(const uint8_t *file, uint64_t pos, uint64_t lo, uint64_t hi, uint64_t n, uint32_t flags) {
    if (pos >= hi || pos + 16 <= lo) return 0;
    const uint4 v = __ldg((const uint4 *)(file + pos));          // buffer is padded: always in bounds
    const uint32_t z0 = maybe_cmf(v.x), z1 = maybe_cmf(v.y), z2 = maybe_cmf(v.z), z3 = maybe_cmf(v.w);
    if (!(z0 | z1 | z2 | z3)) return 0;
    const uint64_t A = ((uint64_t)v.y << 32) | v.x, B = ((uint64_t)v.w << 32) | v.z;      // (dynamic byte picks without indexing registers)
    // one bit per flagged byte: bit 7 of byte j of a word -> bit j
    uint32_t q = (((z0 >> 7) * 0x00204081u) >> 21 & 0xfu) | ((((z1 >> 7) * 0x00204081u) >> 21 & 0xfu) << 4) |
                 ((((z2 >> 7) * 0x00204081u) >> 21 & 0xfu) << 8) | ((((z3 >> 7) * 0x00204081u) >> 21 & 0xfu) << 12);
    const uint32_t nxt = __ldg(file + pos + 16);
    const bool inside = pos >= lo && pos + 17 <= hi && pos + 17 <= n;       // no position of this group needs a bounds test
    uint32_t m = 0;
    while (q) {
        const uint32_t k = (uint32_t)__ffs((int)q) - 1; q &= q - 1;
        const uint32_t b0 = (uint32_t)((k < 8 ? A >> (8 * k) : B >> (8 * (k - 8))) & 0xff);
        const uint32_t b1 = k == 15 ? nxt : (uint32_t)((k < 7 ? A >> (8 * (k + 1)) : B >> (8 * (k - 7))) & 0xff);
        if (zlib_header_ok(b0, b1, flags) && (inside || (pos + k + 1 < n && pos + k >= lo && pos + k < hi))) m |= 1u << k;
    }
    return m;
}

// pass 1: masks[g] = hit mask of group g (g counts 16-byte groups from the tile base of this launch), tile_counts[t] = hits of tile t
__global__ void __launch_bounds__(SCAN_THREADS) scan_count_kernel(const uint8_t *file, uint64_t lo, uint64_t hi, uint64_t n, uint32_t flags, uint32_t *tile_counts, uint16_t *masks) {
    const uint64_t tile0 = (lo & ~(uint64_t)15) + (uint64_t)blockIdx.x * SCAN_TILE;
    uint16_t *tm = masks + (size_t)blockIdx.x * (SCAN_TILE / 16);
    uint32_t c = 0;
#pragma unroll 4
    for (int it = 0; it < 16; it++) {
        const uint32_t g = (uint32_t)it * SCAN_THREADS + threadIdx.x;
        const uint32_t m = magic_mask16(file, tile0 + (uint64_t)g * 16, lo, hi, n, flags);
        tm[g] = (uint16_t)m; c += __popc(m);
    }
    c = __reduce_add_sync(FULL, c);
    __shared__ uint32_t ws[SCAN_THREADS / 32];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int i = 0; i < SCAN_THREADS / 32; i++) t += ws[i]; tile_counts[blockIdx.x] = t; }
}

// exclusive scan of the tile counts in place; total -> *total (single CTA; tiles <= 65536 for a 4 GiB file)
__global__ void __launch_bounds__(1024) scan_tiles_kernel(uint32_t *tile_counts, uint32_t ntiles, uint32_t *total) {
    __shared__ uint32_t wsum[32]; __shared__ uint32_t carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (uint32_t b = 0; b < ntiles; b += 1024) {
        uint32_t i = b + threadIdx.x, v = i < ntiles ? tile_counts[i] : 0, tot, ex = warp_excl_scan(v, tot);
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = tot;
        __syncthreads();
        uint32_t woff = 0; for (uint32_t w = 0; w < (threadIdx.x >> 5); w++) woff += wsum[w];
        uint32_t carry = carry_s;
        if (i < ntiles) tile_counts[i] = carry + woff + ex;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = carry + woff + ex + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry_s;
}

// pass 2: the masks of a tile -> offsets and header types, in file order.  A thread owns 16 CONSECUTIVE groups (256 positions), so the
// order is thread-major and one block scan places everything; the file is touched only at the hits (for the type).
__global__ void __launch_bounds__(SCAN_THREADS) scan_write_kernel(const uint8_t *file, uint64_t lo, const uint16_t *masks, const uint32_t *tile_base, uint32_t *cand, uint8_t *ctype, uint32_t cap) {
    const uint64_t tile0 = (lo & ~(uint64_t)15) + (uint64_t)blockIdx.x * SCAN_TILE;
    const uint4 *tm = (const uint4 *)(masks + (size_t)blockIdx.x * (SCAN_TILE / 16)) + 2 * threadIdx.x;     // 16 masks = 32 bytes per thread
    const uint4 ma = __ldg(tm), mb = __ldg(tm + 1);
    const uint32_t mw[8] = {ma.x, ma.y, ma.z, ma.w, mb.x, mb.y, mb.z, mb.w};
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) c += __popc(mw[j]);
    uint32_t tot, ex = warp_excl_scan(c, tot);
    __shared__ uint32_t wsum[SCAN_THREADS / 32];
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = tot;
    __syncthreads();
    uint32_t woff = 0;
    for (uint32_t w = 0; w < (threadIdx.x >> 5); w++) woff += wsum[w];
    uint32_t o = tile_base[blockIdx.x] + woff + ex;
    if (!c) return;
    const uint64_t base = tile0 + (uint64_t)threadIdx.x * 256;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        uint32_t m = mw[j];      // two groups: bits 0-15 = group 2j, bits 16-31 = group 2j + 1 -> positions base + 32 j + bit
        while (m) {
            const uint32_t k = __ffs((int)m) - 1; m &= m - 1;
            const uint64_t p = base + 32u * j + k;
            if (o < cap) { cand[o] = (uint32_t)p; const uint32_t b0 = __ldg(file + p), b1 = __ldg(file + p + 1); ctype[o] = (uint8_t)zlib_header_type_of(b0, b1); }
            o++;
        }
    }
}

// `file` is the address of file offset 0 (16 B aligned; only [lo & ~15, hi + 16) has to be mapped), positions lo <= i < hi are scanned
uint32_t scan_tiles_for(uint64_t lo, uint64_t hi) { return hi > lo ? (uint32_t)((hi - (lo & ~(uint64_t)15) + SCAN_TILE - 1) / SCAN_TILE) : 0u; }
// masks: scan_tiles_for(lo, hi) * 8 KiB (2 bytes per 16-byte group)
cudaError_t launch_scan_count(const uint8_t *file, uint64_t lo, uint64_t hi, uint64_t n, uint32_t flags, uint32_t *tile_counts, uint16_t *masks, uint32_t *total, cudaStream_t s) {
    uint32_t nt = scan_tiles_for(lo, hi);
    if (nt) scan_count_kernel<<<nt, SCAN_THREADS, 0, s>>>(file, lo, hi, n, flags, tile_counts, masks);
    scan_tiles_kernel<<<1, 1024, 0, s>>>(tile_counts, nt, total);
    return cudaGetLastError();
}
cudaError_t launch_scan_write(const uint8_t *file, uint64_t lo, uint64_t hi, const uint16_t *masks, const uint32_t *tile_base, uint32_t *cand, uint8_t *ctype, uint32_t cap, cudaStream_t s) {
    if (scan_tiles_for(lo, hi)) scan_write_kernel<<<scan_tiles_for(lo, hi), SCAN_THREADS, 0, s>>>(file, lo, masks, tile_base, cand, ctype, cap);
    return cudaGetLastError();
}

// K4 - diff compaction for one winner: positions i < min(C', C) with out[i] != orig[i], then i in [C', C)
// (main.cpp:699-712).  One warp per job, ordered append by ballot.
struct DiffJob { const uint8_t *out; const uint8_t *orig; uint32_t cprime, c; uint32_t *pos; uint8_t *val; uint32_t cap; uint32_t *count; };
__global__ void __launch_bounds__(128) diff_kernel(const DiffJob *jobs, uint32_t njobs) {
    uint32_t wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = lane_id();
    if (wid >= njobs) return;
    const DiffJob j = jobs[wid];
    uint32_t smaller = j.cprime < j.c ? j.cprime : j.c, nd = 0;
    for (uint32_t i0 = 0; i0 < j.c; i0 += 32) {
        uint32_t i = i0 + lane; bool d = false; uint8_t ov = 0;
        if (i < j.c) { ov = j.orig[i]; d = i >= smaller || j.out[i] != ov; }
        uint32_t bm = __ballot_sync(FULL, d);
        if (d) { uint32_t o = nd + __popc(bm & ((1u << lane) - 1)); if (o < j.cap) { j.pos[o] = i; j.val[o] = ov; } }
        nd += __popc(bm);
    }
    if (lane == 0) *j.count = nd;
}
cudaError_t launch_diff(const DiffJob *jobs, uint32_t njobs, cudaStream_t s) {
    diff_kernel<<<(njobs + 3) / 4, 128, 0, s>>>(jobs, njobs);
    return cudaGetLastError();
}

// Gather: copy n bytes src -> dst for many (src, dst, n) jobs in one launch (the recompressed streams' plaintext, concatenated
// for a single D2H copy; what writeStreamdesc's per-stream re-inflate produced, main.cpp:824-828).  Sources are 16 B aligned
// with ATZ_PAD slack; destinations have any alignment: head/tail bytes singly, the middle as dst-aligned 32-bit words.
struct CopyJob { const uint8_t *src; uint8_t *dst; uint64_t n; };
__global__ void __launch_bounds__(256) gather_kernel(const CopyJob *jobs, uint32_t njobs) {
    for (uint32_t ji = blockIdx.x; ji < njobs; ji += gridDim.x) {
        const CopyJob j = jobs[ji];
        uint64_t head = (4 - ((uintptr_t)j.dst & 3)) & 3; if (head > j.n) head = j.n;
        const uint64_t words = (j.n - head) >> 2, tail0 = head + 4 * words;
        if (threadIdx.x < head) j.dst[threadIdx.x] = j.src[threadIdx.x];
        uint32_t *dw = (uint32_t *)(j.dst + head);
        for (uint64_t w = threadIdx.x; w < words; w += blockDim.x) dw[w] = ldu32(j.src + head + 4 * w);
        if (tail0 + threadIdx.x < j.n) j.dst[tail0 + threadIdx.x] = j.src[tail0 + threadIdx.x];
    }
}
cudaError_t launch_gather(const CopyJob *jobs, uint32_t njobs, cudaStream_t s) {
    if (!njobs) return cudaSuccess;
    uint32_t ctas = njobs < 148u * 8u ? njobs : 148u * 8u;
    gather_kernel<<<ctas, 256, 0, s>>>(jobs, njobs);
    return cudaGetLastError();
}

} // namespace atz
