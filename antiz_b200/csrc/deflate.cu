// K3 / K5 - bit-exact zlib 1.2.8 deflate, one warp per (stream x level x memLevel x windowBits) trial.
//
// What it replaces: testDeflateParams (main.cpp:603-731) and doDeflate (main.cpp:976-1003), i.e.
// deflateInit2 + deflate(Z_FINISH) of zlib 1.2.8 ("Z/" = includes, tools, stuff/zlib test/zlib128):
// deflate_stored/fast/slow Z/deflate.c:1564-1853, longest_match 1148-1289, fill_window 1390-1532,
// _tr_flush_block and helpers Z/trees.c:381-1226.  Not a port (DESIGN.md section 3):
//   * no window copy and no head[]/prev[] tables: the plaintext stays where K2 wrote it and the hash chain of
//     a position is a contiguous run of a per-(plaintext, hash_bits) bucket list built once by chains.cu and
//     shared by every level/window trial;
//   * longest_match is precomputed position-parallel: row tables (build_rows_kernel: the chain candidates that
//     improve on all earlier ones) and, per level and window, resolved tables (resolve_rows_kernel: the match
//     longest_match ends on); the serial loop of a trial is one small load and a few decisions per position,
//     with the bucket walk kept as the fallback wherever a table has nothing to say;
//   * deflate_fast (levels 1-3) runs under the hypothesis that it reproduces the original stream's tokens (token
//     map written by K2) for as long as that holds, then with zlib's own logic;
//   * the window slide survives only as `base` (absolute position of window index 0);
//   * symbols go to a per-warp buffer; the histogram, the Huffman bit packing and the compare with the original
//     stream are lane-parallel; only zlib's heap-based tree construction, whose tie-breaking must be reproduced
//     step by step, runs on one lane.
// Search trials never store their output: flushed words are compared with the original stream in flight
// (the --shortcut-len prefix test, the ident count, the size gate and the mismatch cut are warp reductions).
#include "common.cuh"
#include <cstdlib>

namespace atz {

#define MINM 3u
#define MAXM 258u
#define MIN_LOOK 262u
#define TOO_FAR_D 4096u
#define NLSYM 286
#define NDSYM 30
#define NBSYM 19
#define HEAPSZ 573
#define EOB 256

// per-warp shared memory layout (bytes)
#define OFF_LFC 0      /* u16[576] literal/length tree: freq -> code */
#define OFF_LDL 1152   /* u16[576]                      dad  -> len  */
#define OFF_HEAP 2304  /* u16[576]; with DEPTH also the u32 histogram scratch [320] */
#define OFF_DEPTH 3456 /* u8[576] */
#define OFF_DFC 4032   /* u16[64] distance tree */
#define OFF_DDL 4160
#define OFF_BFC 4288   /* u16[40] bit-length tree */
#define OFF_BDL 4368
#define OFF_BLC 4448   /* u16[16] bl_count */
#define OFF_STAGE 4480 /* u32[128] output bit staging */
#define OFF_ROWS 4992  /* uint4[64]: record rows of 32 consecutive positions */
#define OFF_RES 6016   /* uint2[32]: resolved entries of 32 consecutive positions */
#define WARP_SMEM 6272
#define STAGE_WORDS 128
#define STAGE_FLUSH_AT 64 /* flush once this many words are complete: the compare with the original stream is a dependent global load per
                             flush, so it is taken 64 words (2 per lane) at a time; a following 32-symbol parallel put (<= 1536 bits) still fits */

__constant__ uint8_t c_blord[NBSYM] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
// {good, lazy, nice, chain} per level, Z/deflate.c:131-143
__constant__ uint16_t c_cfg[10][4] = {{0, 0, 0, 0},     {4, 4, 8, 4},      {4, 5, 16, 8},      {4, 6, 32, 32},     {4, 4, 16, 16},
                                      {8, 16, 32, 32},  {8, 16, 128, 128}, {8, 32, 128, 256},  {32, 128, 258, 1024}, {32, 258, 258, 4096}};

// ---- code arithmetic (same values as Z/trees.h _length_code/_dist_code/base_*; derived, no tables) ----
__device__ __forceinline__ uint32_t len_code(uint32_t lc) {  // lc = length-3, 0..255 -> 0..28
    if (lc < 8) return lc;
    if (lc == 255) return 28;
    uint32_t k = 31 - __clz(lc);
    return 4 * k - 4 + ((lc >> (k - 2)) & 3);
}
__device__ __forceinline__ uint32_t len_extra_bits(uint32_t code) { return (code < 8 || code == 28) ? 0 : (code - 4) >> 2; }
__device__ __forceinline__ uint32_t dist_code(uint32_t d) {  // d = distance-1, 0..32767 -> 0..29
    if (d < 4) return d;
    uint32_t k = 31 - __clz(d);
    return 2 * k + ((d >> (k - 1)) & 1);
}
__device__ __forceinline__ uint32_t dist_extra_bits(uint32_t code) { return code < 4 ? 0 : (code - 2) >> 1; }
__device__ __forceinline__ uint32_t static_llen(uint32_t n) { return n <= 143 ? 8 : n <= 255 ? 9 : n <= 279 ? 7 : 8; }
__device__ __forceinline__ uint32_t static_lcode(uint32_t n) {  // bit-reversed fixed code (RFC1951 3.2.6)
    if (n <= 143) return __brev(0x30 + n) >> 24;
    if (n <= 255) return __brev(0x190 + (n - 144)) >> 23;
    if (n <= 279) return __brev(n - 256) >> 25;
    return __brev(0xC0 + (n - 280)) >> 24;
}

// ---------------------------------------------------------------------------------------------
struct Trial {
    // immutable
    const uint8_t *in, *orig; uint32_t n, C; uint32_t *outw; uint32_t out_cap;
    const uint32_t *list, *idx; const uint16_t *lsth; const uint4 *rec; const uint8_t *tmap; const uint2 *res; uint32_t rlen, rbudget, hbits;
    uint32_t wsize, maxd, litsz, level, good, lazy, nice, chain, strategy;
    uint32_t S, bail_below, sizediff, cut_mism; bool compare, store, phase1, burst;
    // warp scratch
    uint8_t *sm; uint32_t *symbuf; uint32_t *insmap;   // insmap: one bit per plaintext position (deflate_fast: inserted by this trial)
    // parse state (warp-uniform)
    uint32_t p, wend, base, nsym; int64_t block_start;
    // output state (warp-uniform)
    uint32_t bitpos, obase, ident_lo, ident_all; bool short_done, pass_pending; int stop; // stop: 0 run, else TR_* + 1
    // serial bit accumulator (uniform registers)
    uint64_t acc; uint32_t accbits, accw;
    long long cyc_flush;

    __device__ __forceinline__ uint16_t *lfc() { return (uint16_t *)(sm + OFF_LFC); }
    __device__ __forceinline__ uint16_t *ldl() { return (uint16_t *)(sm + OFF_LDL); }
    __device__ __forceinline__ uint16_t *dfc() { return (uint16_t *)(sm + OFF_DFC); }
    __device__ __forceinline__ uint16_t *ddl() { return (uint16_t *)(sm + OFF_DDL); }
    __device__ __forceinline__ uint16_t *bfc() { return (uint16_t *)(sm + OFF_BFC); }
    __device__ __forceinline__ uint16_t *bdl() { return (uint16_t *)(sm + OFF_BDL); }
    __device__ __forceinline__ uint16_t *heap() { return (uint16_t *)(sm + OFF_HEAP); }
    __device__ __forceinline__ uint8_t *depth() { return sm + OFF_DEPTH; }
    __device__ __forceinline__ uint16_t *blc() { return (uint16_t *)(sm + OFF_BLC); }
    __device__ __forceinline__ uint32_t *stage() { return (uint32_t *)(sm + OFF_STAGE); }
    __device__ __forceinline__ uint32_t *hist() { return (uint32_t *)(sm + OFF_HEAP); }

    // ================= output =================
    // Consume the complete 32-bit words of the staging area (all of it, byte-granular, when `final`).
    __device__ void flush_words(bool final) {
        __syncwarp();
        const uint32_t lane = lane_id();
        uint32_t *st = stage();
        uint32_t nw = final ? (bitpos + 31) >> 5 : bitpos >> 5;
        uint32_t nbytes = final ? (bitpos + 7) >> 3 : nw * 4;
        if (nw) {
            uint32_t e_lo = 0, e_all = 0;
            for (uint32_t j = lane; j < nw; j += 32) {
                uint32_t w = st[j], o = obase + 4 * j;
                uint32_t have = nbytes - 4 * j; if (have > 4) have = 4;
                if (compare) {
                    uint32_t ow = o < C ? ldu32(orig + o) : 0;
                    uint32_t eq = __vcmpeq4(w, ow) & 0x01010101u;
                    uint32_t lim_all = o >= C ? 0 : (C - o < have ? C - o : have);
                    uint32_t lim_lo = o >= S ? 0 : (S - o < lim_all ? S - o : lim_all);
                    e_all += __popc(eq & (lim_all >= 4 ? 0xffffffffu : ((1u << (8 * lim_all)) - 1)));
                    e_lo += __popc(eq & (lim_lo >= 4 ? 0xffffffffu : ((1u << (8 * lim_lo)) - 1)));
                }
                if (store) {
                    if (o + have <= out_cap) {
                        if (have == 4) outw[o >> 2] = w;
                        else { uint8_t *ob = (uint8_t *)outw + o; for (uint32_t b = 0; b < have; b++) ob[b] = (uint8_t)(w >> (8 * b)); }
                    }
                }
            }
            if (compare) {
                ident_all += __reduce_add_sync(FULL, e_all); ident_lo += __reduce_add_sync(FULL, e_lo);
                const uint32_t ahead = obase + nbytes + 256u + 128u * lane;     // the original stream's lines of the next flushes
                if (lane < 4 && ahead < C) asm volatile("prefetch.global.L2 [%0];" ::"l"(orig + ahead));
            }
            uint32_t carry = final ? 0 : st[nw];
            __syncwarp();
            for (uint32_t j = lane; j <= nw && j < STAGE_WORDS; j += 32) st[j] = 0;
            __syncwarp();
            if (lane == 0) st[0] = carry;
            obase += nbytes; bitpos = final ? 0 : (bitpos & 31);
            __syncwarp();
            if (store && obase > out_cap) { stop = TR_OVERFLOW + 1; return; }
        }
        if (!compare || stop) return;
        // --shortcut-len prefix test (main.cpp:632-653): evaluated on the first min(S, C') bytes
        if (!short_done && (obase >= S || final)) {
            short_done = true;
            if (C > S && ident_lo < bail_below) { stop = TR_BAILED + 1; return; }
            // the prefix is fine: the host will rerun this trial in full - unless the rest of this block, which is being emitted
            // anyway, already shows more mismatches than any useful result may have (the cut below)
            if (phase1 && C > S && !final) pass_pending = true;
        }
        if (obase > C && obase - C > sizediff) { stop = TR_SIZE + 1; return; }   // C' >= obase: size gate can no longer pass (main.cpp:671)
        uint32_t seen = obase < C ? obase : C;
        if (short_done && seen - ident_all > cut_mism) { stop = TR_CUT + 1; return; }
    }
    // --- serial puts: bits accumulate in registers, spilled to the staging words 32 at a time ---
    __device__ __forceinline__ void ser_begin() { __syncwarp(); accw = bitpos >> 5; accbits = bitpos & 31; acc = stage()[accw]; }
    __device__ __forceinline__ void ser_end() {
        if (lane_id() == 0) { stage()[accw] = (uint32_t)acc; }
        bitpos = accw * 32 + accbits; __syncwarp();
    }
    __device__ __forceinline__ void ser_put(uint32_t v, uint32_t nb) {
        acc |= (uint64_t)v << accbits; accbits += nb;
        if (accbits >= 32) {
            if (lane_id() == 0) stage()[accw] = (uint32_t)acc;
            acc >>= 32; accbits -= 32; accw++;
            if (accw >= STAGE_FLUSH_AT) { ser_end(); flush_words(false); ser_begin(); }
        }
    }
    // --- parallel put: every lane contributes nb (<= 48) bits ---
    __device__ __forceinline__ void par_put(uint64_t v, uint32_t nb) {
        uint32_t total, off = warp_excl_scan(nb, total);
        if (nb) {
            uint32_t o = bitpos + off, w = o >> 5, s = o & 31;
            uint32_t *st = stage();
            uint64_t lo = v << s;
            atomicOr(&st[w], (uint32_t)lo);
            if (s + nb > 32) atomicOr(&st[w + 1], (uint32_t)(lo >> 32));
            if (s + nb > 64) atomicOr(&st[w + 2], (uint32_t)(v >> (64 - s)));
        }
        bitpos += total;
        if (bitpos >= 32 * STAGE_FLUSH_AT) flush_words(false); else __syncwarp();
    }
    __device__ __forceinline__ void align_byte() { bitpos = (bitpos + 7) & ~7u; }

    // ================= Huffman construction, Z/trees.c:451-699 =================
    // The heap holds one 32-bit key per node: freq << 15 | depth << 10 | node.  zlib's smaller(n, m) - "freq[n] < freq[m], or equal
    // and depth[n] <= depth[m]" (Z/trees.c:443-445) - is then (key_n >> 10) <= (key_m >> 10): one load per heap entry instead of a
    // dependent chain of three.  Block frequencies sum to < 65536 (lit_bufsize <= 32768) and a tree over them is at most 23 deep.
    // The key heap lives where the parse loop stages its rows (dead during a flush; the parse re-stages afterwards).
    __device__ __forceinline__ uint32_t *keyheap() { return (uint32_t *)(sm + OFF_ROWS); }
    // Two levels per round of shared-memory loads: the two children and the four grandchildren are asked for together (the
    // chain of dependent loads is what a lone lane waits for), entries beyond the heap read as "never smaller".
    __device__ __forceinline__ void siftk(uint32_t *hk, int heap_len, int k) {  // pqdownheap
        const uint32_t v = hk[k], vk = v >> 10; int j = k << 1;
        while (j <= heap_len) {
            const uint32_t c0 = hk[j], c1 = j + 1 <= heap_len ? hk[j + 1] : 0xffffffffu;
            const int g = j << 1;
            const uint32_t g0 = g <= heap_len ? hk[g] : 0xffffffffu, g1 = g + 1 <= heap_len ? hk[g + 1] : 0xffffffffu;
            const uint32_t g2 = g + 2 <= heap_len ? hk[g + 2] : 0xffffffffu, g3 = g + 3 <= heap_len ? hk[g + 3] : 0xffffffffu;
            const bool r1 = (c1 >> 10) <= (c0 >> 10);                 // smaller(heap[j+1], heap[j]): the right child on ties
            const uint32_t cj = r1 ? c1 : c0; const int jj = j + (r1 ? 1 : 0);
            if (vk <= (cj >> 10)) break;
            hk[k] = cj; k = jj;
            const int j2 = jj << 1;
            if (j2 > heap_len) break;
            const uint32_t ga = r1 ? g2 : g0, gb = r1 ? g3 : g1;
            const bool r2 = (gb >> 10) <= (ga >> 10);
            const uint32_t gj = r2 ? gb : ga; const int jj2 = j2 + (r2 ? 1 : 0);
            if (vk <= (gj >> 10)) break;
            hk[k] = gj; k = jj2; j = jj2 << 1;
        }
        hk[k] = v;
    }
    // warp-wide: the initial heap (nonzero symbols in increasing order, Z/trees.c:633-641), Len = 0 for the others
    __device__ void tree_init(int kind, int &heap_len, int &max_code) {
        const uint32_t lane = lane_id();
        uint16_t *f = kind == 0 ? lfc() : kind == 1 ? dfc() : bfc();
        uint16_t *dl = kind == 0 ? ldl() : kind == 1 ? ddl() : bdl();
        const int elems = kind == 0 ? NLSYM : kind == 1 ? NDSYM : NBSYM;
        uint32_t *hk = keyheap();
        heap_len = 0; max_code = -1;
        __syncwarp();
        for (int n0 = 0; n0 < elems; n0 += 32) {
            const int n = n0 + (int)lane; const uint32_t fn = n < elems ? f[n] : 0u;
            const uint32_t m = __ballot_sync(FULL, fn != 0);
            if (fn) hk[heap_len + 1 + __popc(m & ((1u << lane) - 1))] = (fn << 15) | (uint32_t)n;
            else if (n < elems) dl[n] = 0;
            if (m) max_code = n0 + 31 - __clz((int)m);
            heap_len += __popc(m);
        }
        __syncwarp();
    }
    // lane 0: tree construction and code lengths.  kind 0 = literal/length, 1 = distance, 2 = bit-length tree.
    // Returns max_code; adds to opt/stat; leaves the lengths in dl[] and their counts in bl_count.
    __device__ int tree_build(int kind, int heap_len, int max_code, int &opt_len, int &static_len) {
        uint16_t *f = kind == 0 ? lfc() : kind == 1 ? dfc() : bfc();
        uint16_t *dl = kind == 0 ? ldl() : kind == 1 ? ddl() : bdl();
        const int elems = kind == 0 ? NLSYM : kind == 1 ? NDSYM : NBSYM;
        const int maxlen = kind == 2 ? 7 : 15;
        uint16_t *h = heap(); uint16_t *bc = blc(); uint32_t *hk = keyheap();
        int heap_max = HEAPSZ, node = elems;
        while (heap_len < 2) {   // Z/trees.c:648-654
            int nn = (max_code < 2 ? ++max_code : 0);
            hk[++heap_len] = (1u << 15) | (uint32_t)nn; f[nn] = 1; opt_len--;
            if (kind == 0) static_len -= (int)static_llen(nn); else if (kind == 1) static_len -= 5;
        }
        for (int n = heap_len / 2; n >= 1; n--) siftk(hk, heap_len, n);
        do {
            const uint32_t kn = hk[1]; hk[1] = hk[heap_len--]; siftk(hk, heap_len, 1);
            const uint32_t km = hk[1];
            const uint32_t n = kn & 1023u, m = km & 1023u;
            h[--heap_max] = (uint16_t)n; h[--heap_max] = (uint16_t)m;
            const uint32_t dn = (kn >> 10) & 31u, dm = (km >> 10) & 31u;
            dl[n] = dl[m] = (uint16_t)node;
            hk[1] = (((kn >> 15) + (km >> 15)) << 15) | (((dn >= dm ? dn : dm) + 1) << 10) | (uint32_t)node; node++;
            siftk(hk, heap_len, 1);
        } while (heap_len >= 2);
        h[--heap_max] = (uint16_t)(hk[1] & 1023u);
        // gen_bitlen Z/trees.c:488-565
        for (int b = 0; b < 16; b++) bc[b] = 0;
        int over = 0, hh;
        dl[h[heap_max]] = 0;
        int n_next = h[heap_max + 1 < HEAPSZ ? heap_max + 1 : heap_max], dad_next = dl[n_next];     // one node ahead: its index and its parent do not depend on this loop's stores
        for (hh = heap_max + 1; hh < HEAPSZ; hh++) {
            const int n = n_next, dad = dad_next;
            if (hh + 1 < HEAPSZ) { n_next = h[hh + 1]; dad_next = dl[n_next]; }
            int bits = dl[dad] + 1;
            if (bits > maxlen) { bits = maxlen; over++; }
            dl[n] = (uint16_t)bits;
            if (n > max_code) continue;
            bc[bits]++;
            int xb, sl = 0;
            if (kind == 0) { xb = n >= 257 ? (int)len_extra_bits(n - 257) : 0; sl = (int)static_llen(n); }
            else if (kind == 1) { xb = (int)dist_extra_bits(n); sl = 5; }
            else xb = n == 16 ? 2 : n == 17 ? 3 : n == 18 ? 7 : 0;
            opt_len += (int)f[n] * (bits + xb);
            if (kind != 2) static_len += (int)f[n] * (sl + xb);
        }
        if (over) {
            do {
                int bits = maxlen - 1;
                while (bc[bits] == 0) bits--;
                bc[bits]--; bc[bits + 1] += 2; bc[maxlen]--;
                over -= 2;
            } while (over > 0);
            for (int bits = maxlen; bits != 0; bits--) {
                int n = bc[bits];
                while (n != 0) {
                    int m = h[--hh];
                    if (m > max_code) continue;
                    if (dl[m] != (uint32_t)bits) { opt_len += (bits - (int)dl[m]) * (int)f[m]; dl[m] = (uint16_t)bits; }
                    n--;
                }
            }
        }
        return max_code;
    }
    // warp-wide gen_codes Z/trees.c:575-607: the code of symbol n is next_code[len] + (number of smaller symbols of that length),
    // bit-reversed; 32 symbols per step, ranked among equal lengths with __match_any_sync
    __device__ void tree_codes(int kind, int max_code) {
        const uint32_t lane = lane_id();
        uint16_t *f = kind == 0 ? lfc() : kind == 1 ? dfc() : bfc();
        uint16_t *dl = kind == 0 ? ldl() : kind == 1 ? ddl() : bdl();
        uint16_t *bc = blc(); uint32_t *next = keyheap();     // next_code[1..15]
        __syncwarp();
        if (lane == 0) { uint32_t code = 0; for (int b = 1; b <= 15; b++) { code = (code + bc[b - 1]) << 1; next[b] = code; } }
        __syncwarp();
        for (int n0 = 0; n0 <= max_code; n0 += 32) {
            const int n = n0 + (int)lane; const uint32_t l = n <= max_code ? dl[n] : 0u;
            const uint32_t peers = __match_any_sync(FULL, l), rank = __popc(peers & ((1u << lane) - 1));
            uint32_t base = 0;
            if (l) { base = next[l]; f[n] = (uint16_t)(__brev(base + rank) >> (32 - l)); }
            __syncwarp();
            if (l && rank == 0) next[l] = base + __popc(peers);
            __syncwarp();
        }
    }
    // scan_tree / send_tree Z/trees.c:705-795 (emit == false counts into the bit-length tree)
    __device__ void walk_lengths(int kind, int max_code, bool emit) {
        uint16_t *dl = kind == 0 ? ldl() : ddl(); uint16_t *bf = bfc(), *bl = bdl();
        int prevlen = -1, nextlen = dl[0], count = 0, maxc = 7, minc = 4;
        if (nextlen == 0) { maxc = 138; minc = 3; }
        if (!emit) { if (lane_id() == 0) dl[max_code + 1] = 0xffff; __syncwarp(); }
        for (int n = 0; n <= max_code; n++) {
            int cur = nextlen; nextlen = dl[n + 1];
            if (++count < maxc && cur == nextlen) continue;
            if (count < minc) {
                if (emit) { do ser_put(bf[cur], bl[cur]); while (--count != 0); } else if (lane_id() == 0) bf[cur] += (uint16_t)count;
            } else if (cur != 0) {
                if (cur != prevlen) { if (emit) { ser_put(bf[cur], bl[cur]); count--; } else if (lane_id() == 0) bf[cur]++; }
                if (emit) { ser_put(bf[16], bl[16]); ser_put((uint32_t)(count - 3), 2); } else if (lane_id() == 0) bf[16]++;
            } else if (count <= 10) {
                if (emit) { ser_put(bf[17], bl[17]); ser_put((uint32_t)(count - 3), 3); } else if (lane_id() == 0) bf[17]++;
            } else {
                if (emit) { ser_put(bf[18], bl[18]); ser_put((uint32_t)(count - 11), 7); } else if (lane_id() == 0) bf[18]++;
            }
            count = 0; prevlen = cur;
            if (nextlen == 0) { maxc = 138; minc = 3; } else if (cur == nextlen) { maxc = 6; minc = 3; } else { maxc = 7; minc = 4; }
            if (emit && stop) return;
        }
    }
    // compress_block Z/trees.c:1060-1105, 32 symbols per step
    __device__ void emit_symbols(bool dyn) {
        const uint32_t lane = lane_id();
        const uint16_t *lf = lfc(), *ll = ldl(), *df = dfc(), *dd = ddl();
        for (uint32_t i0 = 0; i0 < nsym + 1; i0 += 32) {      // the +1 slot is END_BLOCK
            uint32_t i = i0 + lane; uint64_t v = 0; uint32_t nb = 0;
            if (i < nsym) {
                uint32_t s = symbuf[i], dist = s >> 16, lc = s & 0xff;
                if (dist == 0) {
                    if (dyn) { v = lf[lc]; nb = ll[lc]; } else { v = static_lcode(lc); nb = static_llen(lc); }
                } else {
                    uint32_t c = len_code(lc), sym = c + 257, xb = len_extra_bits(c);
                    if (dyn) { v = lf[sym]; nb = ll[sym]; } else { v = static_lcode(sym); nb = static_llen(sym); }
                    if (xb) { v |= (uint64_t)(lc & ((1u << xb) - 1)) << nb; nb += xb; }   // lc - base_length[c]: bases are 2^xb aligned
                    uint32_t d = dist - 1, dc = dist_code(d), dxb = dist_extra_bits(dc);
                    if (dyn) { v |= (uint64_t)df[dc] << nb; nb += dd[dc]; } else { v |= (uint64_t)(__brev(dc) >> 27) << nb; nb += 5; }
                    if (dxb) { v |= (uint64_t)(d & ((1u << dxb) - 1)) << nb; nb += dxb; }
                }
            } else if (i == nsym) {
                if (dyn) { v = lf[EOB]; nb = ll[EOB]; } else { v = 0; nb = 7; }
            }
            par_put(v, nb);
            if (stop) return;
        }
    }
    // _tr_flush_block Z/trees.c:907-1004 + FLUSH_BLOCK_ONLY Z/deflate.c:1538-1546
    __device__ __noinline__ void flush_block(uint32_t last) {
        const long long t_in = clock64();
        flush_block_(last);
        cyc_flush += clock64() - t_in;
    }
    __device__ void flush_block_(uint32_t last) {
        const uint32_t lane = lane_id();
        const bool storable = block_start >= (int64_t)base;          // buf != NULL
        const uint32_t stored_len = (uint32_t)((int64_t)p - block_start);
        __syncwarp();   // the parse's symbol stores (lane 0) become visible to every lane
        int kindsel = 0;  // 0 stored, 1 static, 2 dynamic
        int l_max = 0, d_max = 0, max_bl = 0;
        if (level > 0) {
            uint32_t *hs = hist();
            for (uint32_t j = lane; j < 320; j += 32) hs[j] = 0;
            __syncwarp();
            for (uint32_t i = lane; i < nsym; i += 32) {
                uint32_t s = symbuf[i], dist = s >> 16, lc = s & 0xff;
                if (dist == 0) atomicAdd(&hs[lc], 1u);
                else { atomicAdd(&hs[257 + len_code(lc)], 1u); atomicAdd(&hs[288 + dist_code(dist - 1)], 1u); }
            }
            __syncwarp();
            uint16_t *lf = lfc(), *df = dfc(), *bf = bfc();
            for (uint32_t j = lane; j < NLSYM; j += 32) lf[j] = (uint16_t)(j == EOB ? 1 : hs[j]);
            if (lane < NDSYM) df[lane] = (uint16_t)hs[288 + lane];
            if (lane < NBSYM) bf[lane] = 0;
            __syncwarp();
            int opt_len = 0, static_len = 0, hl_l, hl_d, hl_b, mc;
            tree_init(0, hl_l, mc);
            if (lane == 0) l_max = tree_build(0, hl_l, mc, opt_len, static_len);
            l_max = __shfl_sync(FULL, l_max, 0);
            tree_codes(0, l_max);
            tree_init(1, hl_d, mc);
            if (lane == 0) d_max = tree_build(1, hl_d, mc, opt_len, static_len);
            d_max = __shfl_sync(FULL, d_max, 0);
            tree_codes(1, d_max);
            walk_lengths(0, l_max, false); walk_lengths(1, d_max, false);
            __syncwarp();
            tree_init(2, hl_b, mc);
            int b_max = 0;
            if (lane == 0) { int dummy = 0; b_max = tree_build(2, hl_b, mc, opt_len, dummy); }
            b_max = __shfl_sync(FULL, b_max, 0);
            tree_codes(2, b_max);
            if (lane == 0) {
                for (max_bl = NBSYM - 1; max_bl >= 3; max_bl--) if (bdl()[c_blord[max_bl]] != 0) break;
                opt_len += 3 * (max_bl + 1) + 5 + 5 + 4;
                uint32_t opt_lenb = (uint32_t)(opt_len + 3 + 7) >> 3, static_lenb = (uint32_t)(static_len + 3 + 7) >> 3;
                if (static_lenb <= opt_lenb) opt_lenb = static_lenb;
                if (stored_len + 4 <= opt_lenb && storable) kindsel = 0;
                else if (strategy == 4u || static_lenb == opt_lenb) kindsel = 1;      // Z_FIXED, Z/trees.c:952
                else kindsel = 2;
            }
            __syncwarp();
            kindsel = __shfl_sync(FULL, kindsel, 0); max_bl = __shfl_sync(FULL, max_bl, 0);
        }
        if (kindsel == 0) {   // _tr_stored_block + copy_block Z/trees.c:865-877,1205-1226
            ser_begin(); ser_put(last, 3); ser_end();
            align_byte();
            ser_begin(); ser_put(stored_len & 0xffff, 16); ser_put(~stored_len & 0xffff, 16); ser_end();
            const uint8_t *src = in + (uint32_t)block_start;
            for (uint32_t i0 = 0; i0 < stored_len && !stop; i0 += 128) {
                uint32_t i = i0 + 4 * lane, nb = 0; uint64_t v = 0;
                if (i < stored_len) { uint32_t k = stored_len - i; if (k > 4) k = 4; nb = 8 * k; v = ldu32(src + i); if (k < 4) v &= (1u << nb) - 1; }
                par_put(v, nb);
            }
        } else if (kindsel == 1) {
            ser_begin(); ser_put(2 + last, 3); ser_end();
            emit_symbols(false);
        } else {
            ser_begin();
            ser_put(4 + last, 3);
            ser_put((uint32_t)(l_max + 1 - 257), 5); ser_put((uint32_t)(d_max + 1 - 1), 5); ser_put((uint32_t)(max_bl + 1 - 4), 4);
            for (int r = 0; r <= max_bl; r++) ser_put(bdl()[c_blord[r]], 3);
            walk_lengths(0, l_max, true);
            if (!stop) walk_lengths(1, d_max, true);
            ser_end();
            if (!stop) emit_symbols(true);
        }
        nsym = 0;
        if (last && !stop) align_byte();
        block_start = (int64_t)p;
        if (!stop) flush_words(false);
        if (!stop && pass_pending) stop = TR_PASSED + 1;
    }
    __device__ void run_stored() {   // deflate_stored Z/deflate.c:1564-1619
        uint32_t pend = 4 * litsz, max_block = 0xffff; if (max_block > pend - 5) max_block = pend - 5;
        for (;;) {
            if (wend - p <= 1) {
                do {   // what is left of fill_window (Z/deflate.c:1390-1532): slide bookkeeping + how far the input has been read
                    uint32_t more = base + 2 * wsize - wend;
                    if (p - base >= wsize + maxd) { base += wsize; more += wsize; }
                    if (wend == n) break;
                    uint32_t k = n - wend; if (k > more) k = more;
                    wend += k;
                } while (wend - p < MIN_LOOK && wend != n);
                if (wend == p) break;
            }
            p = wend;
            uint64_t max_start = (uint64_t)block_start + max_block;
            if ((uint64_t)p >= max_start) { p = (uint32_t)max_start; flush_block(0); if (stop) return; }
            if (p - (uint32_t)block_start >= maxd) { flush_block(0); if (stop) return; }
        }
        flush_block(1);
    }
    // what is left of fill_window (Z/deflate.c:1390-1532) for the two strategy loops below
    __device__ __forceinline__ void refill() {
        do {
            uint32_t more = base + 2 * wsize - wend;
            if (p - base >= wsize + maxd) { base += wsize; more += wsize; }
            if (wend == n) break;
            uint32_t k = n - wend; if (k > more) k = more;
            wend += k;
        } while (wend - p < MIN_LOOK && wend != n);
    }
    // deflate_huff (Z_HUFFMAN_ONLY), Z/deflate.c:1929-1967: every byte a literal; the window is refilled when the lookahead is empty
    __device__ void run_huff() {
        const uint32_t lane = lane_id();
        for (;;) {
            if (wend == p) { refill(); if (wend == p) break; }
            // literals p .. wend-1, 32 at a time, up to the symbol that fills the block
            uint32_t room = litsz - 1 - nsym, cnt = wend - p; if (cnt > room) cnt = room; if (cnt > 32) cnt = 32;
            if (lane < cnt) symbuf[nsym + lane] = __ldg(in + p + lane);
            nsym += cnt; p += cnt;
            if (nsym == litsz - 1) { flush_block(0); if (stop) return; }
        }
        flush_block(1);
    }
    // deflate_rle (Z_RLE), Z/deflate.c:1861-1923: matches of distance one only; refill when the lookahead is <= MAX_MATCH
    __device__ void run_rle() {
        const uint32_t lane = lane_id();
        for (;;) {
            if (wend - p <= MAXM) { refill(); if (wend == p) break; }
            const uint32_t look = wend - p;
            uint32_t ml = 0;
            if (look >= MINM && p > 0) {
                // run length of in[p-1] from p on, at most MAX_MATCH: every lane checks eight bytes, first mismatch by ballot
                const uint32_t prev = __ldg(in + p - 1) * 0x01010101u;
                uint32_t run = 0;
                for (uint32_t o = 0; o < MAXM; o += 256) {
                    const uint32_t q = p + o + 8 * lane;
                    uint32_t mine = 0;                     // (bytes from 264 on are never needed: the run is capped at MAX_MATCH)
                    if (o + 8 * lane < 264) {
                        const uint32_t x0 = ldu32(in + q) ^ prev, x1 = ldu32(in + q + 4) ^ prev;
                        mine = x0 ? (uint32_t)(__ffs((int)x0) - 1) >> 3 : x1 ? 4 + ((uint32_t)(__ffs((int)x1) - 1) >> 3) : 8;
                    }
                    const uint32_t bad = __ballot_sync(FULL, mine < 8);
                    if (bad) { const uint32_t f = (uint32_t)__ffs((int)bad) - 1; run = o + 8 * f + __shfl_sync(FULL, mine, f); break; }
                    run = o + 256;
                }
                if (run > MAXM) run = MAXM;
                if (run >= MINM) { ml = run; if (ml > look) ml = look; }
            }
            bool fl;
            if (ml >= MINM) { if (lane == 0) symbuf[nsym] = (1u << 16) | (ml - MINM); nsym++; p += ml; }
            else { if (lane == 0) symbuf[nsym] = __ldg(in + p); nsym++; p++; }
            fl = nsym == litsz - 1;
            if (fl) { flush_block(0); if (stop) return; }
        }
        flush_block(1);
    }
};

// ---------------------------------------------------------------------------------------------
// The LZ77 parse.  Everything the serial loop touches lives in this struct, which only ever exists as a local of
// run_slow()/run_fast() with every helper force-inlined, so it is kept in registers (the Trial above is addressed through a
// pointer by the out-of-line block flush and therefore lives in local memory: touching it per position cost 5x).
//
// Rows (DESIGN.md "row tables"): 32 bytes per plaintext position, built position-parallel by build_rows_kernel:
//   7 records = the chain candidates of this position that strictly improve on all earlier ones, in chain order,
//               packed as (dist-1) | (len-3) << 15 | bits(chain index) << 23 | REC_VALID; 0 = end of row;
//               0xffffffff in slot 6 = more than 7 records, walk the chain instead;
//   1 meta    = plaintext byte | token code of the ORIGINAL stream at this position << 8 (fast rows only, see tmap).
// The serial loop of a trial reads one row per visited position (staged 32 rows at a time through shared memory,
// the next 32 prefetched into registers) and never touches the plaintext or the bucket lists.
struct Hot {
    const uint8_t *in; const uint32_t *list, *idx; const uint16_t *lsth; const uint4 *rows_g; uint32_t *symbuf; uint32_t *insmap; const uint8_t *tmap; uint4 *rows;
    uint32_t rc_base, pf_base; uint4 pf_a, pf_b;
    const uint2 *res_g; uint2 *res_st; uint32_t rs_base, rs_pf_base; uint2 rs_pf;   // resolved table + its 32-entry stage
    uint32_t n, rlen, wsize, maxd, litsz, good, lazy, nice, chain;
    uint32_t p, wend, base, match_len, prev_len, match_start, prev_match, nsym, cache_base, c_idx, hshift, hmask;
    uint32_t sw;   // fast levels: positions < sw were inserted as the original stream's tokens say (tmap); >= sw: insmap
    uint32_t im_idx, im_val;   // the inserted-map word marked last (h_mark_inserted)
};

__device__ __forceinline__ bool h_tally(Hot &h, uint32_t dist, uint32_t lc) {  // _tr_tally Z/trees.c:1010-1055 (counts are taken at flush time)
    if (lane_id() == 0) h.symbuf[h.nsym] = (dist << 16) | lc;
    h.nsym++;
    return h.nsym == h.litsz - 1;
}
// what is left of fill_window Z/deflate.c:1390-1532
__device__ __forceinline__ void h_refill(Hot &h) {
    do {
        uint32_t more = h.base + 2 * h.wsize - h.wend;
        if (h.p - h.base >= h.wsize + h.maxd) { h.base += h.wsize; more += h.wsize; }
        if (h.wend == h.n) break;
        uint32_t k = h.n - h.wend; if (k > more) k = more;
        h.wend += k;
    } while (h.wend - h.p < MIN_LOOK && h.wend != h.n);
}
__device__ __forceinline__ uint32_t common_len_free(const uint8_t *in, uint32_t p, uint32_t q, uint32_t maxlen, uint32_t best) {
    // quick reject exactly where zlib looks first (Z/deflate.c:1227-1230): positions best-1 and best
    if ((ldu32(in + p + best - 1) ^ ldu32(in + q + best - 1)) & 0xffffu) return 0;
    uint32_t l = 0;
    while (l < maxlen) {
        uint32_t x = ldu32(in + p + l) ^ ldu32(in + q + l);
        if (x) { l += (uint32_t)(__ffs((int)x) - 1) >> 3; break; }
        l += 4;
    }
    return l < maxlen ? l : maxlen;
}
// the same with the two bytes of p at best-1, best already fetched (they are the same for every candidate of a step)
__device__ __forceinline__ uint32_t common_len_tail(const uint8_t *in, uint32_t p, uint32_t q, uint32_t maxlen, uint32_t best, uint32_t p_tail) {
    if ((ldu32(in + q + best - 1) & 0xffffu) != p_tail) return 0;
    uint32_t l = 0;
    while (l < maxlen) {
        uint32_t x = ldu32(in + p + l) ^ ldu32(in + q + l);
        if (x) { l += (uint32_t)(__ffs((int)x) - 1) >> 3; break; }
        l += 4;
    }
    return l < maxlen ? l : maxlen;
}
// candidates of this step are in lane registers (q, valid); fold them the way the serial chain walk would
__device__ __forceinline__ bool h_fold_batch(Hot &h, uint32_t q, bool valid, uint32_t maxlen, uint32_t nice_c, uint32_t &best) {
    uint32_t len = valid ? common_len_free(h.in, h.p, q, maxlen, best) : 0;
    uint32_t nm = __ballot_sync(FULL, valid && len >= nice_c);
    uint32_t upto = nm ? (uint32_t)__ffs((int)nm) - 1 : 31;
    bool consider = valid && lane_id() <= upto;
    uint32_t mx = __reduce_max_sync(FULL, consider ? len : 0u);
    if (mx > best) {
        best = mx;
        uint32_t who = (uint32_t)__ffs((int)__ballot_sync(FULL, consider && len == mx)) - 1;
        h.match_start = __shfl_sync(FULL, q, who);
    }
    return nm != 0;
}
__device__ __forceinline__ void h_load_cache(Hot &h, uint32_t pos) {
    h.cache_base = pos & ~31u;
    uint32_t i = h.cache_base + lane_id();
    bool ok = i + 2 < h.n;
    h.c_idx = ok ? __ldg(h.idx + i) : 0;
    if (h.c_idx) {   // the head of this position's chain sits just below its slot: ask for those lines now
        const uint32_t s0 = h.c_idx > 32 ? h.c_idx - 32 : 0;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(h.list + s0)); asm volatile("prefetch.global.L2 [%0];" ::"l"(h.lsth + s0));
    }
}
// the row of position p (p < h.rlen), through the 32-row shared-memory stage
__device__ __forceinline__ void h_row(Hot &h, uint4 &r0, uint4 &r1) {
    const uint32_t pb = h.p & ~31u, lane = lane_id();
    if (pb != h.rc_base) {
        uint4 a, b;
        if (pb == h.pf_base) { a = h.pf_a; b = h.pf_b; }
        else {
            a = make_uint4(0, 0, 0, 0); b = a;
            const uint32_t i = pb + lane;
            if (i < h.rlen) { a = __ldg(h.rows_g + 2 * (size_t)i); b = __ldg(h.rows_g + 2 * (size_t)i + 1); }
        }
        __syncwarp();
        h.rows[2 * lane] = a; h.rows[2 * lane + 1] = b;
        h.rc_base = pb; h.pf_base = pb + 32;
        h.pf_a = make_uint4(0, 0, 0, 0); h.pf_b = h.pf_a;
        { const uint32_t i = pb + 32 + lane; if (i < h.rlen) { h.pf_a = __ldg(h.rows_g + 2 * (size_t)i); h.pf_b = __ldg(h.rows_g + 2 * (size_t)i + 1); } }
        __syncwarp();
    }
    r0 = h.rows[2 * (h.p & 31)]; r1 = h.rows[2 * (h.p & 31) + 1];
}
// longest_match (Z/deflate.c:1148-1289) through the row: the serial chain walk only ever acts on candidates that beat all
// earlier ones, and that list is a function of the data alone (shared by every level x window trial of this hash size).
//   emax  : log2 of the chain budget (records further down the chain than that are never reached)
//   dl_h  : largest distance the chain head may have, dl_f: the followers (Z/deflate.c:1158-1162,1284; SURVEY.md A.6)
__device__ __forceinline__ uint32_t h_eval_row(Hot &h, const uint4 &r0, const uint4 &r1, uint32_t best, uint32_t nice_c, uint32_t emax, uint32_t look) {
    const uint32_t pm1 = h.p - h.base - 1;
    const uint32_t dl_h = h.maxd < pm1 ? h.maxd : pm1, dl_f = (h.maxd - 1) < pm1 ? (h.maxd - 1) : pm1;
    const uint32_t rc[7] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z};
#pragma unroll
    for (int j = 0; j < 7; j++) {
        const uint32_t r = rc[j];
        if (!(r & REC_VALID)) break;
        const uint32_t d1 = r & 0x7fffu, e = (r >> 23) & 15u;
        uint32_t len = ((r >> 15) & 0xffu) + MINM;
        if (e > emax) break;
        if (d1 >= (e == 0 ? dl_h : dl_f)) break;
        if (len > look) len = look;
        if (len > best) { best = len; h.match_start = h.p - d1 - 1; if (len >= nice_c) break; }
    }
    return best <= look ? best : look;
}
// zlib's hash of position p (UPDATE_HASH x3, Z/deflate.c:167)
__device__ __forceinline__ uint32_t h_hash(const Hot &h, uint32_t p) {
    const uint32_t w = ldu32(h.in + p);
    return hash3(w & 0xff, (w >> 8) & 0xff, (w >> 16) & 0xff, h.hshift, h.hmask);
}
// longest_match for levels 4-9 by walking the bucket list: every earlier position of the bucket is on the chain
// (ip = number of list entries before p's own; the bucket ends where the stored hash changes)
__device__ __forceinline__ uint32_t h_longest_slow(Hot &h, uint32_t slot, uint32_t ip, uint32_t myh, uint32_t look) {
    uint32_t best = h.prev_len, nice_c = h.nice < look ? h.nice : look, maxlen = look < MAXM ? look : MAXM;
    if (best >= nice_c) return best <= look ? best : look;     // nothing can improve (see DESIGN.md)
    uint32_t ch = h.chain; if (h.prev_len >= h.good) ch >>= 2;
    const uint32_t navail = ip < ch ? ip : ch;
    uint32_t prel = h.p - h.base, limit = h.base + (prel > h.maxd ? prel - h.maxd : 0);
    const uint32_t lane = lane_id();
    for (uint32_t k0 = 0; k0 < navail; k0 += 32) {
        uint32_t k = k0 + lane; bool valid = k < navail;
        uint32_t q = valid ? __ldg(h.list + (slot - k)) : 0;
        valid = valid && (uint32_t)__ldg(h.lsth + (slot - k)) == myh && (k == 0 || q > limit);
        uint32_t vm = __ballot_sync(FULL, valid);
        uint32_t nv = vm == FULL ? 32 : (uint32_t)__ffs((int)~vm) - 1;    // validity is monotone along the chain
        valid = lane < nv;
        bool stopnow = h_fold_batch(h, q, valid, maxlen, nice_c, best);
        if (stopnow || nv < 32) break;
    }
    return best <= look ? best : look;
}
// the walk for one position of deflate_slow (row missing or overflowed)
__device__ __forceinline__ uint32_t h_walk_slow(Hot &h, uint32_t look) {
    if ((h.p & ~31u) != h.cache_base) h_load_cache(h, h.p);
    const uint32_t ip = __shfl_sync(FULL, h.c_idx, h.p & 31);
    if (!ip) return MINM - 1;
    const uint32_t slot = ip - 1, myh = h_hash(h, h.p);
    const uint32_t q0 = __ldg(h.list + slot);
    if ((uint32_t)__ldg(h.lsth + slot) != myh || !((h.p - q0 <= h.maxd) && (q0 > h.base))) return MINM - 1;
    return h_longest_slow(h, slot, ip, myh, look);
}
// was position q inserted into the hash table by this trial?  (levels 1-3, Z/deflate.c:1680-1704)
__device__ __forceinline__ bool h_inserted(const Hot &h, uint32_t q, uint32_t level) {
    if (q >= h.sw) return (h.insmap[q >> 5] >> (q & 31u)) & 1u;
    const uint32_t c = __ldg(h.tmap + q);
    return c != 0 && (c < TM_INNER || c - TM_INNER + level >= 4);
}
// fold a batch whose common lengths are already known (len == 0 where the lane does not count)
__device__ __forceinline__ bool h_fold_lens(Hot &h, uint32_t q, bool valid, uint32_t len, uint32_t nice_c, uint32_t &best) {
    uint32_t nm = __ballot_sync(FULL, valid && len >= nice_c);
    uint32_t upto = nm ? (uint32_t)__ffs((int)nm) - 1 : 31;
    bool consider = valid && lane_id() <= upto;
    uint32_t mx = __reduce_max_sync(FULL, consider ? len : 0u);
    if (mx > best) {
        best = mx;
        uint32_t who = (uint32_t)__ffs((int)__ballot_sync(FULL, consider && len == mx)) - 1;
        h.match_start = __shfl_sync(FULL, q, who);
    }
    return nm != 0;
}
// mark positions [a, a + n) (n <= 32) as inserted (warp-uniform call; lane 0 stores).  Marks only ever move forward, so the word
// a mark falls into is either the one marked last - kept in a register - or still all zero: a store, never a load the warp
// would have to wait for (the read-modify-write was 5 % of the stall samples of a dense launch)
__device__ __forceinline__ void h_mark_inserted(Hot &h, uint32_t a, uint32_t n) {
    const uint64_t m = ((n >= 32 ? 0xffffffffull : ((1ull << n) - 1ull))) << (a & 31u);
    const uint32_t w = a >> 5;
    h.im_val = (w == h.im_idx ? h.im_val : 0u) | (uint32_t)m; h.im_idx = w;
    if (lane_id() == 0) h.insmap[w] = h.im_val;
    if (m >> 32) { h.im_idx = w + 1; h.im_val = (uint32_t)(m >> 32); if (lane_id() == 0) h.insmap[w + 1] = h.im_val; }
}
// levels 1-3: the chain is the bucket list filtered by the inserted positions.  The inserted lookup and the compare of a
// bucket entry depend only on its position, so both are issued together for all 32 entries of a step (the compare of an
// entry that turns out not to be on the chain is wasted bandwidth, not latency) and the chain rank is applied afterwards.
// Measured on B200 (dense launch, the brute-window grid): asking for the flags first and then for the bytes of the chain members
// only (a third of the sectors for levels 1-2) is 20 % SLOWER - the extra dependent round trip costs more than the traffic it
// saves; evaluating the next 32 positions at once (several times the traffic) 2.4-4x slower.  The step is latency-bound at the
// 24 warps per SM its registers allow.
// (Also measured: asking for the bucket entries of p + 1 while the walk at p is in flight - no difference, 233.7 vs 234.2 M kilocycles.)
__device__ __forceinline__ uint32_t h_longest_fast(Hot &h, uint32_t look, uint32_t level, bool &have) {
    const uint32_t lane = lane_id();
    const uint32_t sl = __shfl_sync(FULL, h.c_idx, h.p & 31);     // entries before p's own in the list
    have = false;
    if (sl == 0) return h.match_len;
    const uint32_t hp = ldu32(h.in + h.p);      // p's first four bytes: its hash (UPDATE_HASH x3, Z/deflate.c:167) and the head of every compare
    const uint32_t myh = hash3(hp & 0xff, (hp >> 8) & 0xff, (hp >> 16) & 0xff, h.hshift, h.hmask);
    uint32_t best = h.prev_len; const uint32_t nice_c = h.nice < look ? h.nice : look, maxlen = look < MAXM ? look : MAXM;
    const uint32_t prel = h.p - h.base, limit = h.base + (prel > h.maxd ? prel - h.maxd : 0);
    uint32_t got = 0;
    for (uint32_t k0 = 1; k0 <= sl && got < h.chain; k0 += 32) {
        const uint32_t k = k0 + lane; bool inb = k <= sl;
        const uint32_t q = inb ? __ldg(h.list + (sl - k)) : 0;
        inb = inb && (uint32_t)__ldg(h.lsth + (sl - k)) == myh;
        const bool inwin = inb && (h.p - q <= h.maxd);
        // one round trip for everything that depends on q only: its inserted flag, its first four bytes and the two bytes zlib
        // looks at first (best-1, best: Z/deflate.c:1227-1230) - all loads issued before any of them is used
        const uint32_t p_tail = (best == MINM - 1 ? hp >> 8 : ldu32(h.in + h.p + best - 1)) & 0xffffu;
        uint32_t flag = 0, hq = 0, tq = 0;
        if (inwin) {
            flag = q >= h.sw ? ((h.insmap[q >> 5] >> (q & 31u)) & 1u) : (uint32_t)__ldg(h.tmap + q);
            hq = ldu32(h.in + q);
            tq = best == MINM - 1 ? 0u : ldu32(h.in + q + best - 1);
        }
        if (best == MINM - 1) tq = hq >> 8;
        const bool ins = inwin && flag != 0 && (q >= h.sw || flag < TM_INNER || flag - TM_INNER + level >= 4);
        uint32_t len = 0;
        if (inwin && ((tq ^ p_tail) & 0xffffu) == 0) {
            uint32_t x = hq ^ hp, l = 0;
            if (x) l = (uint32_t)(__ffs((int)x) - 1) >> 3;
            else for (l = 4; l < maxlen; l += 4) { x = ldu32(h.in + h.p + l) ^ ldu32(h.in + q + l); if (x) { l += (uint32_t)(__ffs((int)x) - 1) >> 3; break; } }
            len = l < maxlen ? l : maxlen;
        }
        const uint32_t im = __ballot_sync(FULL, ins), wm = __ballot_sync(FULL, inwin);
        if (im && !have) {   // the chain head
            const uint32_t q0 = __shfl_sync(FULL, q, (uint32_t)__ffs((int)im) - 1);
            if (!(q0 > h.base)) return h.match_len;            // window index 0 / slid out == NIL
            have = true;
            if (best >= nice_c) return best <= look ? best : look;
        }
        const uint32_t rank = got + __popc(im & ((1u << lane) - 1));
        // the walk ends at the first chain member beyond the budget or (past the head) beyond the distance limit
        const uint32_t bm = __ballot_sync(FULL, ins && !(rank < h.chain && (rank == 0 || q > limit)));
        const bool valid = ins && (bm == 0 || lane < (uint32_t)__ffs((int)bm) - 1);
        const bool stopnow = h_fold_lens(h, q, valid, valid ? len : 0u, nice_c, best);
        got += __popc(im);
        if (stopnow || bm || wm != FULL) break;    // left the window (or the bucket): older candidates are unreachable
    }
    if (!have) return h.match_len;
    return best <= look ? best : look;
}

#define HOT_FLUSH(last)                                                                                     \
    do {                                                                                                    \
        t.p = h.p; t.base = h.base; t.nsym = h.nsym;                                                        \
        t.flush_block(last);                                                                                \
        h.nsym = 0; h.rc_base = 0xffffffffu; h.rs_base = 0xffffffffu;   /* the flush built its trees where rows are staged */ \
    } while (0)

__device__ __forceinline__ void hot_init(Hot &h, Trial &t) {
    h.in = t.in; h.list = t.list; h.idx = t.idx; h.lsth = t.lsth; h.hshift = (t.hbits + 2) / 3; h.hmask = (1u << t.hbits) - 1; h.rows_g = t.rec; h.symbuf = t.symbuf; h.insmap = t.insmap; h.tmap = t.tmap;
    h.n = t.n; h.rlen = t.rec ? t.rlen : 0; h.wsize = t.wsize; h.maxd = t.maxd; h.litsz = t.litsz; h.good = t.good; h.lazy = t.lazy; h.nice = t.nice; h.chain = t.chain;
    h.p = 0; h.wend = 0; h.base = 0; h.match_len = h.prev_len = MINM - 1; h.match_start = h.prev_match = 0; h.nsym = 0;
    h.cache_base = 0xffffffffu; h.c_idx = 0; h.rc_base = 0xffffffffu; h.pf_base = 0xffffffffu; h.rows = (uint4 *)(t.sm + OFF_ROWS);
    h.pf_a = make_uint4(0, 0, 0, 0); h.pf_b = h.pf_a; h.sw = 0;
    h.res_g = t.res; h.res_st = (uint2 *)(t.sm + OFF_RES); h.rs_base = 0xffffffffu; h.rs_pf_base = 0xffffffffu; h.rs_pf = make_uint2(0, 0);
}

// the resolved entry of position p (p < h.rlen), through a 32-entry shared-memory stage
__device__ __forceinline__ uint2 h_res(Hot &h) {
    const uint32_t pb = h.p & ~31u, lane = lane_id();
    uint2 *st = h.res_st;
    if (pb != h.rs_base) {
        uint2 a;
        if (pb == h.rs_pf_base) a = h.rs_pf;
        else { a = make_uint2(0, 0); const uint32_t i = pb + lane; if (i < h.rlen) a = __ldg(h.res_g + i); }
        __syncwarp();
        st[lane] = a;
        h.rs_base = pb; h.rs_pf_base = pb + 32;
        h.rs_pf = make_uint2(0, 0);
        { const uint32_t i = pb + 32 + lane; if (i < h.rlen) h.rs_pf = __ldg(h.res_g + i); }
        __syncwarp();
    }
    return st[h.p & 31];
}

// ---------------------------------------------------------------------------------------------
// Burst parse (DESIGN.md "burst parse").  The serial loops above take one decision per step on one warp.  Where the ORIGINAL
// stream's token map is known, its token boundaries are used as speculation points: after a match has been emitted the state
// of deflate_slow is canonical (position only: match_available = 0, prev_length = 2), and deflate_fast's state is the position
// alone at every token start.  So 32 lanes parse 32 consecutive segments at once, each from the canonical state at a boundary
// of the original, and a segment's result is accepted iff the segment before it was accepted and ended exactly where this one
// began - then the concatenation is what the serial loop would have produced.  Nothing depends on the speculation being right:
// a segment that does not line up ends the accepted prefix and the next burst starts from the true state.
// Scratch: the tree-building area of the warp's shared memory (bytes 0..4480), which is dead between block flushes.
#define BURST_CAP 8u          /* symbols a lane may emit per burst */
#define BURST_SPAN 256u       /* positions scanned for boundaries per burst (8 per lane) */
#define BURST_STAGE 288u      /* resolved entries staged per burst: BURST_SPAN + BURST_CAP + slack, a multiple of 32 */
#define OFF_B_RES 0           /* uint2[BURST_STAGE] */
#define OFF_B_SEG 2304        /* u32[32] */
#define OFF_B_SYM 2432        /* u32[BURST_CAP][32] */

// token-map bytes of positions rb + 8*lane .. +7 as a bit mask of the positions whose code satisfies `start` and whose
// predecessor's code satisfies `inner` (slow: a token start right behind a match; fast: any token start), limited to (lo, hi)
template <bool NEED_INNER>
__device__ __forceinline__ uint32_t burst_marks(const uint8_t *tmap, uint32_t rb, uint32_t lo_excl_or_incl, uint32_t hi_excl) {
    const uint32_t lane = lane_id(), q0 = rb + 8u * lane;
    const uint2 w = __ldg((const uint2 *)(tmap + q0));
    uint32_t prev = __shfl_up_sync(FULL, w.y >> 24, 1);
    if (lane == 0) prev = rb ? (uint32_t)__ldg(tmap + rb - 1) : 0u;
    const uint32_t s_lo = __vcmpgeu4(w.x, 0x01010101u) & __vcmpleu4(w.x, 0x01010101u * TM_LONG);
    const uint32_t s_hi = __vcmpgeu4(w.y, 0x01010101u) & __vcmpleu4(w.y, 0x01010101u * TM_LONG);
    uint32_t m_lo = s_lo, m_hi = s_hi;
    if (NEED_INNER) {
        m_lo &= __vcmpgeu4((w.x << 8) | prev, 0x01010101u * TM_INNER);
        m_hi &= __vcmpgeu4((w.y << 8) | (w.x >> 24), 0x01010101u * TM_INNER);
    }
    uint32_t bits = ((m_lo & 1u) | ((m_lo >> 7) & 2u) | ((m_lo >> 14) & 4u) | ((m_lo >> 21) & 8u)) |
                    (((m_hi & 1u) | ((m_hi >> 7) & 2u) | ((m_hi >> 14) & 4u) | ((m_hi >> 21) & 8u)) << 4);
    // keep positions in [lo, hi)
    const uint32_t lo = lo_excl_or_incl > q0 ? lo_excl_or_incl - q0 : 0u, hi = hi_excl > q0 ? hi_excl - q0 : 0u;
    bits &= lo >= 8 ? 0u : (0xffu << lo) & 0xffu;
    bits &= hi >= 8 ? 0xffu : (1u << hi) - 1u;
    return bits;
}
// the first 31 (slow) / 32 (fast) marked positions go to segs[] in order; returns how many were stored
__device__ __forceinline__ uint32_t burst_collect(uint32_t bits, uint32_t rb, uint32_t *segs, uint32_t maxn) {
    uint32_t total, off = warp_excl_scan(__popc(bits), total);
    const uint32_t q0 = rb + 8u * lane_id();
    while (bits && off < maxn) { const uint32_t i = (uint32_t)__ffs((int)bits) - 1; bits &= bits - 1; segs[off++] = q0 + i; }
    __syncwarp();
    return total < maxn ? total : maxn;
}

// deflate_slow over resolved entries, 32 segments per call.  On entry the (uniform) state is h.p / h.match_len / h.match_start /
// match_avail / lit_prev as in the tight loop of run_slow; on return it is the state after the accepted segments.
// returns the number of accepted lanes (0: nothing could be accepted - the caller takes serial steps);
// reason_out: why the last accepted lane stopped (0 match emitted, 1 symbol cap, 2 reached pend, 3 entry absent); flush_out: a block is due
__device__ __forceinline__ uint32_t burst_slow(Hot &h, uint8_t *sm, bool &match_avail, uint32_t &lit_prev, uint32_t pend, uint32_t &reason_out, bool &flush_out) {
    const uint32_t lane = lane_id();
    uint2 *rs = (uint2 *)(sm + OFF_B_RES); uint32_t *segs = (uint32_t *)(sm + OFF_B_SEG), *syms = (uint32_t *)(sm + OFF_B_SYM);
    const uint32_t rb = h.p & ~7u;
    __syncwarp();
    // resolved entries of [rb, rb + BURST_STAGE), and a look ahead for the next bursts
#pragma unroll
    for (uint32_t k = 0; k < BURST_STAGE / 32; k++) {
        const uint32_t i = rb + 32u * k + lane;
        rs[32u * k + lane] = i < h.rlen ? __ldg(h.res_g + i) : make_uint2(RES_ABSENT, RES_ABSENT);
    }
    { const uint32_t i = rb + BURST_STAGE + 16u * lane; if (i < h.rlen) asm volatile("prefetch.global.L2 [%0];" ::"l"(h.res_g + i)); }
    const uint32_t nseg = burst_collect(burst_marks<true>(h.tmap, rb, h.p + 1, pend), rb, segs, 31u);   // also orders the stage stores
    // per-lane parse
    const bool live = lane <= nseg;
    uint32_t lp = h.p, pl = h.match_len, pm = h.match_start, lit = lit_prev; bool av = match_avail;
    if (lane) { lp = live ? segs[lane - 1] : 0u; pl = MINM - 1; pm = 0; lit = 0; av = false; }
    const uint32_t start = lp;
    uint32_t cnt = 0, reason = 1;
    if (live) {
        while (cnt < BURST_CAP) {
            if (lp >= pend) { reason = 2; break; }
            const uint2 e = rs[lp - rb];
            const uint32_t m = pl >= h.good ? e.y : e.x, len = m & 0x1ffu;
            if (len == RES_ABSENT) { reason = 3; break; }
            uint32_t ml = MINM - 1, ms = pm;
            if (pl < h.lazy && len > pl) { ml = len; ms = lp - ((m >> 9) & 0x7fffu) - 1; }
            if (pl >= MINM && ml <= pl) {
                syms[cnt * 32 + lane] = ((lp - 1 - pm) << 16) | (pl - MINM); cnt++;
                lp += pl - 1; av = false; pl = MINM - 1; reason = 0; break;
            }
            if (av) { syms[cnt * 32 + lane] = lit; cnt++; }
            av = true; lp++; pl = ml; pm = ms;
            lit = e.x >> 24;
        }
    }
    // accepted prefix: every lane starts where the lane before it ended, with a match
    const uint32_t prev_end = __shfl_up_sync(FULL, lp, 1), prev_fin = __shfl_up_sync(FULL, (uint32_t)(reason == 0), 1);
    const bool chained = lane == 0 || (live && prev_fin && prev_end == start);
    uint32_t tot, cexcl = warp_excl_scan(live ? cnt : 0u, tot);
    const uint32_t cincl = cexcl + cnt, rem = h.litsz - 1 - h.nsym;
    const bool fits = cincl < rem || (cincl == rem && reason == 0);     // a flush may only fall right behind a match (its p is canonical)
    const uint32_t okm = __ballot_sync(FULL, chained && fits);
    const uint32_t nacc = okm == FULL ? 32u : (uint32_t)__ffs((int)~okm) - 1;
    flush_out = false; reason_out = 0;
    if (nacc == 0) return 0;
    if (lane < nacc) for (uint32_t j = 0; j < cnt; j++) h.symbuf[h.nsym + cexcl + j] = syms[j * 32 + lane];
    const uint32_t last = nacc - 1;
    h.p = __shfl_sync(FULL, lp, last); h.match_len = __shfl_sync(FULL, pl, last); h.match_start = __shfl_sync(FULL, pm, last);
    match_avail = __shfl_sync(FULL, (uint32_t)av, last) != 0; lit_prev = __shfl_sync(FULL, lit, last);
    reason_out = __shfl_sync(FULL, reason, last);
    h.nsym += __shfl_sync(FULL, cincl, last);
    flush_out = h.nsym == h.litsz - 1;
    __syncwarp();
    return nacc;
}

// deflate_slow Z/deflate.c:1730-1853
__device__ __forceinline__ void run_slow(Trial &t) {
    Hot h; hot_init(h, t);
    bool match_avail = false;
    uint32_t lit_prev = 0;
    const bool filtered = t.strategy == 1u;      // Z_FILTERED: matches of up to 5 bytes are dropped (a resolved table has the rule folded in)
    const uint32_t jfull = 31 - __clz(h.chain), jgood = jfull >= 2 ? jfull - 2 : 0;
    const uint32_t res_len = h.res_g ? h.rlen : 0;
    uint32_t no_res_at = 0xffffffffu;   // a position whose resolved entry says "no usable row": handled the long way
    // burst parse where the original's token map is known; after a burst that got nowhere the serial loop runs for a while
    const bool burst_ok = t.burst && h.tmap != nullptr && h.res_g != nullptr && (((uintptr_t)h.tmap) & 7u) == 0;
    uint32_t serial_left = 0, backoff = 32;
    for (;;) {
        if (h.wend - h.p < MIN_LOOK) { h_refill(h); if (h.wend == h.p) break; }
        const uint32_t look = h.wend - h.p; bool fl; uint32_t lit_cur;
        h.prev_len = h.match_len; h.prev_match = h.match_start; h.match_len = MINM - 1;
        if (h.p < res_len && look >= MIN_LOOK && h.p != no_res_at) {
            // resolved table (resolve_rows_kernel): what longest_match returns here for this level and window, for the full and
            // for the quartered chain budget; lengths are not clipped because a whole MAX_MATCH fits in the lookahead.  Tight
            // loop over the positions up to which that holds; h.match_len / h.match_start carry the previous position's match.
            h.match_len = h.prev_len; h.match_start = h.prev_match;
            const uint32_t pend = res_len < h.wend - (MIN_LOOK - 1) ? res_len : h.wend - (MIN_LOOK - 1);
            while (h.p < pend) {
                if (burst_ok && serial_left == 0) {
                    uint32_t why; bool due;
                    const uint32_t nacc = burst_slow(h, t.sm, match_avail, lit_prev, pend, why, due);
                    h.rc_base = 0xffffffffu; h.rs_base = 0xffffffffu;     // (the serial stages are not touched by a burst; kept simple)
                    if (due) { HOT_FLUSH(0); if (t.stop) return; }
                    if (nacc <= 1) { serial_left = backoff; if (backoff < 2048) backoff *= 2; } else backoff = 32;
                    if (nacc && why == 3) { no_res_at = h.p; break; }
                    continue;
                }
                if (serial_left) serial_left--;
                const uint2 e = h_res(h);
                const uint32_t pl = h.match_len, m = pl >= h.good ? e.y : e.x, len = m & 0x1ffu;
                if (len == RES_ABSENT) { no_res_at = h.p; break; }
                const uint32_t pm = h.match_start;
                uint32_t ml = MINM - 1;
                if (pl < h.lazy && len > pl) { ml = len; h.match_start = h.p - ((m >> 9) & 0x7fffu) - 1; }
                fl = false;
                if (pl >= MINM && ml <= pl) {
                    fl = h_tally(h, h.p - 1 - pm, pl - MINM);
                    h.p += pl - 1; match_avail = false; h.match_len = MINM - 1;
                } else {
                    if (match_avail) { fl = h_tally(h, 0, lit_prev); if (fl) { HOT_FLUSH(0); if (t.stop) return; fl = false; } }   // flush before p++ (Z/deflate.c:1822-1826)
                    match_avail = true; h.p++; h.match_len = ml;
                }
                lit_prev = e.x >> 24;
                if (fl) { HOT_FLUSH(0); if (t.stop) return; }
            }
            continue;
        }
        {
            if (look >= MINM && h.p < h.rlen) {
                uint4 r0, r1; h_row(h, r0, r1);
                lit_cur = r1.w & 0xffu;
                if (h.prev_len < h.lazy) {
                    if (r1.z != 0xffffffffu) {
                        const uint32_t nice_c = h.nice < look ? h.nice : look;
                        if (h.prev_len >= nice_c) h.match_len = h.prev_len <= look ? h.prev_len : look;
                        else h.match_len = h_eval_row(h, r0, r1, h.prev_len, nice_c, h.prev_len >= h.good ? jgood : jfull, look);
                    } else h.match_len = h_walk_slow(h, look);
                    if (h.match_len <= 5 && (filtered || (h.match_len == MINM && h.p - h.match_start > TOO_FAR_D))) h.match_len = MINM - 1;   // Z/deflate.c:1774-1785
                }
            } else {
                lit_cur = __ldg(h.in + h.p);
                if (look >= MINM && h.prev_len < h.lazy) {
                    h.match_len = h_walk_slow(h, look);
                    if (h.match_len <= 5 && (filtered || (h.match_len == MINM && h.p - h.match_start > TOO_FAR_D))) h.match_len = MINM - 1;
                }
            }
        }
        if (h.prev_len >= MINM && h.match_len <= h.prev_len) {
            fl = h_tally(h, h.p - 1 - h.prev_match, h.prev_len - MINM);
            h.p += h.prev_len - 1; match_avail = false; h.match_len = MINM - 1;
            if (fl) { HOT_FLUSH(0); if (t.stop) return; }
        } else if (match_avail) {
            fl = h_tally(h, 0, lit_prev);
            if (fl) { HOT_FLUSH(0); if (t.stop) return; }   // before p++ (Z/deflate.c:1822-1826)
            h.p++;
        } else { match_avail = true; h.p++; }
        lit_prev = lit_cur;
    }
    if (match_avail) h_tally(h, 0, lit_prev);
    HOT_FLUSH(1);
}

// deflate_fast under the hypothesis (part 1 of run_fast), 32 tokens per call: every token start of the original is a state of
// its own (the position), so each lane evaluates the row of one token start; the accepted prefix is the run of lanes whose token
// equals the original's and which tile the plaintext without a gap.  Returns the number of tokens accepted (0: the serial step
// decides - normally the hypothesis has just failed); flush_out: a block is due.  Only called where a whole MAX_MATCH fits in the
// lookahead for every position it looks at (h.p < pend <= wend - 261: no clipping, no window slide inside the burst).
__device__ __forceinline__ uint32_t burst_fast(Hot &h, uint8_t *sm, uint32_t pend, uint32_t jfull, bool &flush_out) {
    const uint32_t lane = lane_id();
    uint32_t *segs = (uint32_t *)(sm + OFF_B_SEG);
    const uint32_t rb = h.p & ~7u;
    flush_out = false;
    __syncwarp();
    const uint32_t n = burst_collect(burst_marks<false>(h.tmap, rb, h.p, pend), rb, segs, 32u);
    { const uint32_t i = rb + BURST_SPAN + 4u * lane; if (i < h.rlen) asm volatile("prefetch.global.L2 [%0];" ::"l"(h.rows_g + 2 * (size_t)i)); }
    if (n == 0 || segs[0] != h.p) return 0;
    const bool live = lane < n;
    const uint32_t s0 = live ? segs[lane] : 0u;
    uint32_t ml = MINM - 1, mstart = 0, meta = 0;
    if (live) {
        const uint4 r0 = __ldg(h.rows_g + 2 * (size_t)s0), r1 = __ldg(h.rows_g + 2 * (size_t)s0 + 1);
        meta = r1.w;
        const uint32_t pm1 = s0 - h.base - 1;
        const uint32_t dl_h = h.maxd < pm1 ? h.maxd : pm1, dl_f = (h.maxd - 1) < pm1 ? (h.maxd - 1) : pm1;
        const uint32_t rc[7] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z};
#pragma unroll
        for (int j = 0; j < 7; j++) {      // h_eval_row for position s0, lookahead >= MIN_LOOKAHEAD
            const uint32_t r = rc[j];
            if (!(r & REC_VALID)) break;
            const uint32_t d1 = r & 0x7fffu, e = (r >> 23) & 15u, len = ((r >> 15) & 0xffu) + MINM;
            if (e > jfull) break;
            if (d1 >= (e == 0 ? dl_h : dl_f)) break;
            if (len > ml) { ml = len; mstart = s0 - d1 - 1; if (len >= h.nice) break; }
        }
    }
    const uint32_t mine = ml >= MINM ? (ml < TM_LONG ? ml : TM_LONG) : 1u;
    const uint32_t next = s0 + (ml >= MINM ? ml : 1u);
    const uint32_t prev_next = __shfl_up_sync(FULL, next, 1);
    const bool ok = live && mine == ((meta >> 8) & 0xffu) && (lane == 0 || prev_next == s0);
    const uint32_t okm = __ballot_sync(FULL, ok);
    uint32_t nacc = okm == FULL ? 32u : (uint32_t)__ffs((int)~okm) - 1;
    const uint32_t rem = h.litsz - 1 - h.nsym;
    if (nacc > rem) nacc = rem;
    if (nacc == 0) return 0;
    if (lane < nacc) h.symbuf[h.nsym + lane] = ml >= MINM ? (((s0 - mstart) << 16) | (ml - MINM)) : (meta & 0xffu);
    h.p = __shfl_sync(FULL, next, nacc - 1);
    h.match_len = 0;      // any value below MIN_MATCH is the same state
    h.nsym += nacc;
    flush_out = h.nsym == h.litsz - 1;
    __syncwarp();
    return nacc;
}

// deflate_fast Z/deflate.c:1628-1722
__device__ __forceinline__ void run_fast(Trial &t) {
    Hot h; hot_init(h, t);
    const uint32_t lane = lane_id(), level = t.level;
    h.prev_len = MINM - 1;
    // ---- part 1: while this trial reproduces the original stream's tokens, the inserted set is known in advance (tmap) and
    // the chains filtered by it have been folded into rows: no bucket walk, no inserted map ----
    if (h.rlen) {
        const uint32_t jfull = 31 - __clz(h.chain);
        const bool burst_ok = t.burst && h.tmap != nullptr && (((uintptr_t)h.tmap) & 7u) == 0;
        for (;;) {
            if (h.p >= h.rlen) break;
            if (h.wend - h.p < MIN_LOOK) { h_refill(h); if (h.wend == h.p) break; }
            if (burst_ok && h.wend - h.p >= MIN_LOOK) {
                const uint32_t pend = h.rlen < h.wend - (MIN_LOOK - 1) ? h.rlen : h.wend - (MIN_LOOK - 1);
                bool due; const uint32_t nacc = burst_fast(h, t.sm, pend, jfull, due);
                if (nacc) { h.rc_base = 0xffffffffu; if (due) { HOT_FLUSH(0); if (t.stop) return; } continue; }
            }
            const uint32_t look = h.wend - h.p;    // >= MINM here: rlen stays clear of the end of the stream
            uint4 r0, r1; h_row(h, r0, r1);
            uint32_t ml = h.match_len;
            if (r0.x & REC_VALID) {
                const uint32_t nice_c = h.nice < look ? h.nice : look;
                ml = h_eval_row(h, r0, r1, MINM - 1, nice_c, jfull, look);
            }
            const uint32_t mine = ml >= MINM ? (ml < TM_LONG ? ml : TM_LONG) : 1u;
            if (mine != ((r1.w >> 8) & 0xffu)) break;          // first token that differs from the original's: redo it the slow way
            bool fl;
            if (ml >= MINM) { fl = h_tally(h, h.p - h.match_start, ml - MINM); h.p += ml; h.match_len = 0; }
            else { h.match_len = ml; fl = h_tally(h, 0, r1.w & 0xffu); h.p++; }
            if (fl) { HOT_FLUSH(0); if (t.stop) return; }
        }
    }
    // ---- part 2: the trial's own inserted map from here on ----
    h.sw = h.p; h.im_idx = 0xffffffffu; h.im_val = 0;
    {   // clear the map for every position that can still be inserted
        const uint32_t w0 = h.sw >> 5, w1 = (h.n + 63) >> 5; uint32_t *im = h.insmap;
        for (uint32_t j = w0 + lane; j < w1; j += 32) im[j] = 0;
        __syncwarp();
    }
    for (;;) {
        if (h.wend - h.p < MIN_LOOK) { h_refill(h); if (h.wend == h.p) break; }
        uint32_t look = h.wend - h.p; bool fl;
        if (look >= MINM) {
            if ((h.p & ~31u) != h.cache_base) h_load_cache(h, h.p);
            bool have; uint32_t ml = h_longest_fast(h, look, level, have);
            if (have) h.match_len = ml;
            h_mark_inserted(h, h.p, 1);
        }
        if (h.match_len >= MINM) {
            fl = h_tally(h, h.p - h.match_start, h.match_len - MINM);
            look -= h.match_len;
            if (h.match_len <= h.lazy && look >= MINM) h_mark_inserted(h, h.p + 1, h.match_len - 1);
            h.p += h.match_len; h.match_len = 0;
        } else { fl = h_tally(h, 0, __ldg(h.in + h.p)); h.p++; }
        __syncwarp();
        if (fl) { HOT_FLUSH(0); if (t.stop) return; }
    }
    HOT_FLUSH(1);
}

// One warp = one trial at a time; trials are pulled from a queue (their lengths differ by orders of magnitude).
template <int MINB>
__global__ void __launch_bounds__(256, MINB) deflate_trials_kernel(const TrialDesc *descs, TrialResult *results, uint32_t ntrials,
                                                             uint32_t *queue, TrialOpts opts, uint32_t *symbuf_all,
                                                             uint8_t *insmap_all, uint64_t insmap_stride) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = lane_id(), slot = blockIdx.x;
    Trial t;
    t.sm = smem;
    t.symbuf = symbuf_all + (size_t)slot * 32768u;
    t.insmap = (uint32_t *)(insmap_all + (size_t)slot * insmap_stride);
    for (;;) {
        uint32_t ti = 0;
        if (lane == 0) ti = atomicAdd(queue, 1u);
        ti = __shfl_sync(FULL, ti, 0);
        if (ti >= ntrials) break;
        const TrialDesc d = descs[ti];
        t.in = d.in; t.orig = d.orig; t.n = d.n; t.C = d.c; t.outw = (uint32_t *)d.out; t.out_cap = d.out_cap;
        t.list = d.ch.list; t.idx = d.ch.idx; t.lsth = d.ch.lsth; t.hbits = (uint32_t)d.memlevel + 7; t.rec = d.ch.rec; t.rlen = d.ch.rlen; t.rbudget = d.ch.rbudget; t.tmap = d.tmap; t.res = d.res;
        t.level = d.level; t.strategy = d.strategy; t.wsize = 1u << d.wbits; t.maxd = t.wsize - MIN_LOOK; t.litsz = 1u << (d.memlevel + 6);
        t.good = c_cfg[d.level][0]; t.lazy = c_cfg[d.level][1]; t.nice = c_cfg[d.level][2]; t.chain = c_cfg[d.level][3];
        t.S = opts.shortcut; t.bail_below = opts.bail_below; t.sizediff = opts.sizediff; t.cut_mism = opts.cut_mismatch; t.phase1 = d.phase1 != 0; t.burst = opts.burst != 0;
        t.compare = opts.compare && d.orig != nullptr; t.store = d.store && d.out != nullptr;
        t.p = 0; t.wend = 0; t.base = 0; t.nsym = 0;
        t.block_start = 0;
        t.bitpos = 0; t.obase = 0; t.ident_lo = t.ident_all = 0; t.short_done = false; t.pass_pending = false; t.stop = 0;
        t.acc = 0; t.accbits = 0; t.accw = 0; t.cyc_flush = 0;
        const long long t_start = clock64();
        uint32_t *st = t.stage();
        for (uint32_t j = lane; j < STAGE_WORDS; j += 32) st[j] = 0;
        // Z/deflate.c:899-902: the strategy picks deflate_huff / deflate_rle before the level's function is looked at
        const int kind = d.strategy == 2 ? 3 : d.strategy == 3 ? 4 : d.level == 0 ? 0 : d.level <= 3 ? 1 : 2;
        __syncwarp();
        // zlib header, Z/deflate.c:738-754
        uint32_t hdr = (8u + ((uint32_t)(d.wbits - 8) << 4)) << 8, lf = (d.strategy >= 2 || d.level < 2) ? 0 : d.level < 6 ? 1 : d.level == 6 ? 2 : 3;
        hdr |= lf << 6; hdr += 31 - (hdr % 31);
        t.ser_begin(); t.ser_put(hdr >> 8, 8); t.ser_put(hdr & 0xff, 8); t.ser_end();
        if (kind == 0) t.run_stored(); else if (kind == 1) run_fast(t); else if (kind == 2) run_slow(t); else if (kind == 3) t.run_huff(); else t.run_rle();
        if (!t.stop) {   // trailer Z/deflate.c:967-968
            t.ser_begin();
            t.ser_put((d.adler >> 24) & 0xff, 8); t.ser_put((d.adler >> 16) & 0xff, 8); t.ser_put((d.adler >> 8) & 0xff, 8); t.ser_put(d.adler & 0xff, 8);
            t.ser_end();
            t.flush_words(true);
        }
        if (lane == 0) {
            TrialResult r;
            r.in_consumed = t.p; r.out_len = t.obase; r.ident = t.ident_all;
            r.kcycles = (uint32_t)((clock64() - t_start) >> 10); r.kcycles_flush = (uint32_t)(t.cyc_flush >> 10);
            if (t.stop) r.status = t.stop - 1;
            else if (t.compare) { uint32_t df = t.obase > d.c ? t.obase - d.c : d.c - t.obase; r.status = df <= opts.sizediff ? TR_COMPARED : TR_SIZE; }
            else r.status = TR_COMPARED;
            results[ti] = r;
        }
        __syncwarp();
    }
}


// ---------------------------------------------------------------------------------------------
// Row tables.  For every position p of a plaintext prefix, walk p's chain once, 32 candidates per step, and keep the
// candidates whose common length with p strictly exceeds that of every earlier candidate.  zlib's longest_match
// (Z/deflate.c:1148-1289) changes state only at such candidates, whatever the level (chain budget, nice/good length) or
// the window (distance limit): those parameters merely cut the list short, which the trial does on its own copy of the
// row.  Position-parallel (no serial dependence), so the expensive part of every trial of one hash size is done once,
// at full occupancy, instead of once per trial on a single warp.
//   level == 0 : rows for deflate_slow (levels 4-9): every earlier position of the bucket is on the chain;
//   level 1..3 : rows for deflate_fast at that level, under the hypothesis that the trial reproduces the ORIGINAL
//                stream's tokens (tmap, written by the inflate kernel): only positions where the original has a token
//                start get a row, and the chain is the bucket filtered by the positions that hypothesis inserts.
struct RowTask { const uint8_t *in; uint32_t n; const uint32_t *list, *idx; const uint16_t *lsth; const uint8_t *tmap; uint32_t *rows; uint32_t rlen, budget, chunk0, level, pbegin, visited_only; };

__global__ void __launch_bounds__(256, 8) build_rows_kernel(const RowTask *tasks, uint32_t ntasks, uint32_t nchunks, uint32_t *queue) {
    const uint32_t lane = lane_id();
    RowTask t = tasks[0]; uint32_t t_end = 0;      // chunks [t.chunk0, t_end) belong to the task held in t
    for (uint32_t ch = 0, ch_end = 0;; ch++) {
        if (ch == ch_end) {    // four chunks (128 positions) per pull
            if (lane == 0) ch = atomicAdd(queue, 4u);
            ch = __shfl_sync(FULL, ch, 0); ch_end = ch + 4;
        }
        if (ch >= nchunks) break;
        if (ch >= t_end || ch < t.chunk0) {
            uint32_t lo = 0, hi = ntasks - 1;   // task owning this chunk: last one with chunk0 <= ch
            while (lo < hi) { uint32_t mid = (lo + hi + 1) >> 1; if (tasks[mid].chunk0 <= ch) lo = mid; else hi = mid - 1; }
            t = tasks[lo]; t_end = lo + 1 < ntasks ? tasks[lo + 1].chunk0 : nchunks;
        }
        const uint32_t p0 = t.pbegin + (ch - t.chunk0) * 32;     // pbegin is a multiple of 32: rows below it were copied from an older table
        uint32_t my_idx = 0, my_h = 0, my_meta = 0; bool my_skip = false;
        if (p0 + lane < t.rlen) {
            my_idx = __ldg(t.idx + p0 + lane); my_h = __ldg(t.lsth + my_idx);
            my_meta = __ldg(t.in + p0 + lane) | (t.level ? (uint32_t)__ldg(t.tmap + p0 + lane) << 8 : 0u);
            if (t.visited_only) {
                // deflate_slow rows only where the ORIGINAL stream's parse called longest_match: at its token starts and at the
                // position after a match start (the lazy evaluation, Z/deflate.c:1766-1790).  A trial that reproduces the original
                // never looks anywhere else; one that does not finds the overflow mark there and walks the chain itself.
                const uint32_t p = p0 + lane, c0 = __ldg(t.tmap + p), c1 = p ? (uint32_t)__ldg(t.tmap + p - 1) : 0u;
                my_skip = !((c0 != 0 && c0 < TM_INNER) || (c1 >= MINM && c1 < TM_INNER));
            }
        }
        // every lane initialises the row of its own position (empty + meta; the overflow mark where no row is built), then the warp
        // walks the chains of the positions that get one - the others cost nothing more
        bool need = false;
        if (p0 + lane < t.rlen) {
            uint4 *row4 = (uint4 *)(t.rows + 8 * (size_t)(p0 + lane));
            row4[0] = make_uint4(0, 0, 0, 0); row4[1] = make_uint4(0, 0, my_skip ? 0xffffffffu : 0u, my_meta);
            const uint32_t tc = my_meta >> 8;
            need = !my_skip && (t.level == 0 || !(tc == 0 || tc >= TM_INNER));      // fast rows: token starts of the original only
        }
        uint32_t todo = __ballot_sync(FULL, need);
        __syncwarp();
        while (todo) {
            const uint32_t pi = (uint32_t)__ffs((int)todo) - 1; todo &= todo - 1;
            const uint32_t p = p0 + pi;
            const uint32_t ip = __shfl_sync(FULL, my_idx, pi), myh = __shfl_sync(FULL, my_h, pi), slot = ip - 1;
            uint32_t nav = ip;    // list entries before p's own; the bucket ends where the stored hash changes
            uint32_t *row = t.rows + 8 * (size_t)p;
            if (!t.level && nav > t.budget) nav = t.budget;
            const uint32_t maxlen = t.n - p < MAXM ? t.n - p : MAXM;
            uint32_t best = MINM - 1, nrec = 0, got = 0;
            uint32_t p_tail = ldu32(t.in + p + best - 1) & 0xffffu;
            for (uint32_t k0 = 0; k0 < nav; k0 += 32) {
                uint32_t kk = k0 + lane; bool valid = kk < nav;
                uint32_t q = valid ? __ldg(t.list + (slot - kk)) : 0, dist = p - q;
                valid = valid && (uint32_t)__ldg(t.lsth + (slot - kk)) == myh;
                const bool inwin = valid && dist <= 32506u;     // MAX_DIST of the largest window
                uint32_t k = kk;
                if (t.level) {   // chain index = rank among the inserted positions
                    bool ins = false;
                    if (inwin) { const uint32_t c = __ldg(t.tmap + q); ins = c != 0 && (c < TM_INNER || c - TM_INNER + t.level >= 4); }
                    const uint32_t im = __ballot_sync(FULL, ins);
                    k = got + __popc(im & ((1u << lane) - 1)); got += __popc(im);
                    valid = ins && k < t.budget && (k == 0 || dist <= 32505u);
                } else {
                    valid = inwin && (k == 0 || dist <= 32505u);   // head / followers
                    const uint32_t vm = __ballot_sync(FULL, valid);
                    const uint32_t nv = vm == FULL ? 32 : (uint32_t)__ffs((int)~vm) - 1;   // validity is monotone along the chain
                    valid = lane < nv;
                }
                const uint32_t wm = __ballot_sync(FULL, inwin);
                uint32_t len = valid ? common_len_tail(t.in, p, q, maxlen, best, p_tail) : 0;
                if (__ballot_sync(FULL, len > best)) {     // most steps far down a chain improve nothing: nothing to record
                    uint32_t pm = len;   // inclusive prefix maximum over lanes
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(FULL, pm, d); if (lane >= (uint32_t)d && y > pm) pm = y; }
                    uint32_t before = __shfl_up_sync(FULL, pm, 1); if (lane == 0) before = 0;
                    if (before < best) before = best;
                    const bool isrec = valid && len > before;
                    const uint32_t rm = __ballot_sync(FULL, isrec);
                    if (isrec) {
                        const uint32_t o = nrec + __popc(rm & ((1u << lane) - 1));
                        if (o < 7) row[o] = (dist - 1) | ((len - MINM) << 15) | ((k ? 32u - (uint32_t)__clz((int)k) : 0u) << 23) | REC_VALID;
                    }
                    nrec += __popc(rm);
                    const uint32_t top = __shfl_sync(FULL, pm, 31); if (top > best) { best = top; p_tail = ldu32(t.in + p + best - 1) & 0xffffu; }
                }
                if (best >= maxlen || wm != FULL || (t.level && got >= t.budget)) break;
            }
            __syncwarp();
            if (nrec > 7 && lane == 0) row[6] = 0xffffffffu;
        }
    }
}
cudaError_t launch_build_rows(const RowTask *tasks, uint32_t ntasks, uint32_t nchunks, uint32_t *queue, int ctas, cudaStream_t s) {
    build_rows_kernel<<<ctas, 256, 0, s>>>(tasks, ntasks, nchunks, queue);
    return cudaGetLastError();
}

// Resolved tables.  For one (level, window) the answer of longest_match at a position depends on the parse only through
// prev_length, and only in two ways: the chain budget is quartered when prev_length >= good_match, and a result that is not
// longer than prev_length changes nothing.  Along a row the record lengths grow strictly, so the walk ends on the same record
// whatever prev_length is: the first one in reach that attains nice_match, else the last one in reach.  This kernel finds
// that record for both budgets, position-parallel, and the trial's serial loop is left with one 8-byte load per position:
//   x = len | (dist-1) << 9 | literal << 24 (full budget), y = len | (dist-1) << 9 (quartered); len 2 = no match,
//   RES_ABSENT = no usable row.  The TOO_FAR rule for length-3 matches (Z/deflate.c:1774-1785) is folded in.
// Valid where a whole MAX_MATCH fits in the lookahead (no clipping) - the trial checks that; the distance limits are those
// of SURVEY.md A.6 (head: min(MAX_DIST, p-1), followers one less), positional once the lookahead is full.
struct ResTask { const uint4 *rows; uint2 *out; uint32_t rlen, nice, jfull, jgood, maxd, chunk0, filtered; };

__device__ __forceinline__ uint32_t resolve_one(const uint32_t (&rc)[7], uint32_t emax, uint32_t nice, uint32_t dl_h, uint32_t dl_f, uint32_t filtered) {
    uint32_t best = MINM - 1, bd1 = 0;
#pragma unroll
    for (int j = 0; j < 7; j++) {
        const uint32_t r = rc[j];
        if (!(r & REC_VALID)) break;
        const uint32_t d1 = r & 0x7fffu, e = (r >> 23) & 15u, len = ((r >> 15) & 0xffu) + MINM;
        if (e > emax) break;
        if (d1 >= (e == 0 ? dl_h : dl_f)) break;
        if (len > best) { best = len; bd1 = d1; if (len >= nice) break; }
    }
    if (best <= 5 && (filtered || (best == MINM && bd1 + 1 > TOO_FAR_D))) best = MINM - 1;
    return best | (bd1 << 9);
}
__global__ void __launch_bounds__(256) resolve_rows_kernel(const ResTask *tasks, uint32_t ntasks, uint32_t nchunks) {
    for (uint32_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
        uint32_t lo = 0, hi = ntasks - 1;
        while (lo < hi) { uint32_t mid = (lo + hi + 1) >> 1; if (tasks[mid].chunk0 <= ch) lo = mid; else hi = mid - 1; }
        const ResTask t = tasks[lo];
        const uint32_t p = (ch - t.chunk0) * 256 + threadIdx.x;
        if (p >= t.rlen) continue;
        const uint4 r0 = __ldg(t.rows + 2 * (size_t)p), r1 = __ldg(t.rows + 2 * (size_t)p + 1);
        const uint32_t rc[7] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z};
        uint2 o;
        if (r1.z == 0xffffffffu) { o.x = RES_ABSENT | (r1.w << 24); o.y = RES_ABSENT; }
        else {
            const uint32_t pm1 = p - 1;   // p == 0 has no candidates
            const uint32_t dl_h = t.maxd < pm1 ? t.maxd : pm1, dl_f = (t.maxd - 1) < pm1 ? (t.maxd - 1) : pm1;
            o.x = resolve_one(rc, t.jfull, t.nice, dl_h, dl_f, t.filtered) | (r1.w << 24);
            o.y = resolve_one(rc, t.jgood, t.nice, dl_h, dl_f, t.filtered);
        }
        t.out[p] = o;
    }
}
cudaError_t launch_resolve_rows(const ResTask *tasks, uint32_t ntasks, uint32_t nchunks, cudaStream_t s) {
    uint32_t ctas = nchunks < 148u * 16u ? nchunks : 148u * 16u;
    resolve_rows_kernel<<<ctas, 256, 0, s>>>(tasks, ntasks, nchunks);
    return cudaGetLastError();
}

// one warp per CTA: a warp that finds the queue empty gives its registers and shared memory back at once, so the tail of a launch
// (a few long trials) leaves room for the kernels launched next to it
cudaError_t launch_deflate_trials(const TrialDesc *descs, TrialResult *results, uint32_t ntrials, uint32_t *queue, const TrialOpts &opts,
                                  uint32_t *symbuf_all, uint8_t *insmap_all, uint64_t insmap_stride, int ctas, bool dense, cudaStream_t stream) {
    // dense launches (more trials than 16 warps/SM can hold) use the 80-register build: more resident warps hide the
    // latency of the serial parse better than the extra registers do
    if (dense) deflate_trials_kernel<3><<<ctas, 32, WARP_SMEM, stream>>>(descs, results, ntrials, queue, opts, symbuf_all, insmap_all, insmap_stride);
    else deflate_trials_kernel<2><<<ctas, 32, WARP_SMEM, stream>>>(descs, results, ntrials, queue, opts, symbuf_all, insmap_all, insmap_stride);
    return cudaGetLastError();
}

} // namespace atz
