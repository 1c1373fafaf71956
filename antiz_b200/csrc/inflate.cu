// K2 - batched trial inflate, one warp per candidate stream.
//
// Replaces ZlibInflator/zlib inflate as ZBuffSearcher and doInflate drive it (main.cpp:205-246, 461-486;
// Z/inflate.c:605-1252, Z/inffast.c, Z/inftrees.c).  It reproduces zlib's accept/reject set and its byte
// accounting: total_in at Z_STREAM_END, at an error (ceil(bits consumed / 8): zlib pulls whole bytes only as
// needed and inflate_fast hands unused ones back), when the input runs out (everything), and at the moment the
// scanner's first output buffer is full - the four numbers ZBuffSearcher's accept logic reads (SURVEY.md A.1).
// Every job writes its output (plaintext + token map, common.cuh TM_*) into a region of its own; a job whose region is
// too small stops with INF_OUT_FULL and is rerun by the host with a larger one (api.cu: small first-stage slots for all
// candidates, exact-ish regions for the few that outgrow them).
// Continuation: when the input of a candidate ends at the end of its chunk, the scanner keeps the z_stream and feeds it
// "chunk k+1 starting with its duplicated overlap byte, ..." (refillInput, main.cpp:207-217).  The kernel does the same
// in place: it records the state at the chunk end as the probe result, then goes on over the virtual input
// (file position = off + v - (#chunk boundaries crossed)) and reports the final state as the continuation result.
// Huffman decode tables live in shared memory (10-bit primary for literal/length, 8-bit for distance, canonical
// bit-serial fallback for longer codes and for exact behaviour at the end of input).  Tokens are decoded 32 at a time and
// their bytes produced together (Inflater::batch); table builds and the final adler32 are lane-parallel.
#include "common.cuh"

namespace atz {

#define LPB 10
#define DPB 8
#define CPB 7
#define STAGE_BYTES 2048u
// per-warp shared memory (bytes)
#define I_LTAB 0      /* u16[1024] primary literal/length table: (sym << 4) | len, 0 = not here */
#define I_DTAB 2048   /* u16[256]  primary distance table */
#define I_LSYM 2560   /* u16[288]  symbols sorted by (len, sym) */
#define I_DSYM 3136   /* u16[32] */
#define I_LCNT 3200   /* u16[16] count per length */
#define I_DCNT 3232
#define I_CCNT 3264   /* code-length code */
#define I_CSYM 3296   /* u16[19] -> 40 B */
#define I_LENS 3336   /* u8[320] */
#define I_TMP 3656    /* u16[16] first code, u16[16] start index, u16[16] fill cursor, u32[16] counters = 160 B */
#define I_CTAB 3816   /* u16[128] primary table of the code-length code */
#define I_STAGE 4080  /* u8[STAGE_BYTES] output bytes of one token batch, then u8[STAGE_BYTES] their token-map codes (16 B aligned) */
#define I_WARP (4080 + 2 * 2048)
// CTA-wide fixed tables
#define F_LTAB 0
#define F_DTAB 2048
#define F_LSYM 2560
#define F_DSYM 3136
#define F_LCNT 3200
#define F_DCNT 3232
#define F_SIZE 3264

__constant__ uint16_t c_lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_clord[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct Code { const uint16_t *tab; const uint16_t *sym; const uint16_t *cnt; uint32_t pb; uint32_t maxlen; };

__device__ __noinline__ void write_probe(InflateResult *r, uint32_t adler, uint64_t avail, uint64_t nout, uint64_t in_at_cap) {
    if (lane_id() == 0) { r->status = INF_NEED_INPUT; r->adler = adler; r->total_in = avail; r->total_out = nout; r->in_at_outcap = in_at_cap; }
}

struct Writer {
    uint8_t *out, *tmap, *sm;
    __device__ __forceinline__ void put_literal(uint64_t nout, uint32_t v) {
        if (lane_id() == 0) { out[nout] = (uint8_t)v; if (tmap) tmap[nout] = 1; }
    }
    __device__ __forceinline__ void put_match(uint64_t nout, uint32_t len, uint32_t dist) {
        const uint32_t lane = lane_id();
        const uint32_t tin = TM_INNER + (len <= 4 ? 3u : len == 5 ? 2u : len == 6 ? 1u : 0u), tst = len < TM_LONG ? len : TM_LONG;
        __syncwarp();
        for (uint32_t i = lane; i < len; i += 32) {
            const uint32_t r = i < dist ? i : i % dist;
            out[nout + i] = out[nout - dist + r];
            if (tmap) tmap[nout + i] = (uint8_t)(i ? tin : tst);
        }
        __syncwarp();
    }
    // The bytes of one batch (lane k holds token k, ntok of them), written at out[nout..]: literals and matches are assembled in a
    // shared-memory stage - sources that lie before the batch are fetched from global memory four tokens at a time so that their
    // latencies overlap, sources inside the batch are copied stage to stage in token order - and written out with coalesced stores.
    __device__ __forceinline__ void produce(uint32_t my_len, uint32_t my_dist, uint32_t my_lit, uint32_t ntok, uint64_t nout) {
        const uint32_t lane = lane_id();
        const bool is_tok = lane < ntok, is_match = is_tok && my_dist != 0;
        uint32_t tot; const uint32_t off = warp_excl_scan(is_tok ? my_len : 0u, tot);
        const uint32_t tin = TM_INNER + (my_len <= 4 ? 3u : my_len == 5 ? 2u : my_len == 6 ? 1u : 0u), tst = my_len < TM_LONG ? my_len : TM_LONG;
        if (tot <= STAGE_BYTES) {
            uint8_t *st = sm + I_STAGE, *tt = st + STAGE_BYTES;
            __syncwarp();
            const uint32_t span = my_len < my_dist ? my_len : my_dist;
            const bool indep = is_match && my_dist >= off + span;        // every source byte lies before this batch
            // Byte-parallel: every lane owns output bytes q, q+32, ... of the batch, finds the token a byte belongs to by a binary search
            // over the token offsets (shuffles), and fetches it - a literal, or a source byte that lies before the batch - with the
            // loads of 8 x 32 bytes in flight together: one memory round trip per 256 output bytes instead of one per four tokens
            // (under load the sources, written a moment ago by this warp, come back from L2 or DRAM).  Tokens with a source inside
            // the batch are left to the ordered pass below.
            const uint32_t pack = my_len | ((uint32_t)indep << 9) | ((uint32_t)(is_tok && !is_match) << 10) | (off << 11);   // off <= 2048
            const uint32_t val = is_match ? my_dist : my_lit;
            for (uint32_t q0 = 0; q0 < tot; q0 += 256) {
                uint32_t xb[8], cb[8]; bool wr[8];
#pragma unroll
                for (int g = 0; g < 8; g++) {
                    const uint32_t q = q0 + 32u * g + lane;
                    wr[g] = false; xb[g] = 0; cb[g] = 0;
                    if (q0 + 32u * g >= tot) continue;
                    uint32_t t = 0;
#pragma unroll
                    for (uint32_t sft = 16; sft >= 1; sft >>= 1) {   // largest t < ntok with off[t] <= q
                        const uint32_t c = t + sft, o = __shfl_sync(FULL, off, c & 31);
                        if (c < ntok && o <= q) t = c;
                    }
                    const uint32_t pk = __shfl_sync(FULL, pack, t), v = __shfl_sync(FULL, val, t);
                    const uint32_t len = pk & 0x1ffu, o = pk >> 11, i = q - o;
                    const bool in = q < tot, lit = (pk >> 10) & 1u, ind = (pk >> 9) & 1u;
                    wr[g] = in && (lit || ind); xb[g] = v; cb[g] = 1;
                    if (in && ind) {
                        uint32_t r = i; if (i >= v) r = i % v;       // (overlapping copy: only the first token of a batch can be both)
                        xb[g] = out[nout + o + r - v];
                        cb[g] = i ? TM_INNER + (len <= 4 ? 3u : len == 5 ? 2u : len == 6 ? 1u : 0u) : (len < TM_LONG ? len : TM_LONG);
                    }
                }
#pragma unroll
                for (int g = 0; g < 8; g++) if (wr[g]) { const uint32_t q = q0 + 32u * g + lane; st[q] = (uint8_t)xb[g]; tt[q] = (uint8_t)cb[g]; }
            }
            __syncwarp();
            uint32_t dm = __ballot_sync(FULL, is_match && !indep);
            while (dm) {   // sources inside the batch: token order, stage to stage
                const uint32_t t = (uint32_t)__ffs((int)dm) - 1; dm &= dm - 1;
                const uint32_t len = __shfl_sync(FULL, my_len, t), dist = __shfl_sync(FULL, my_dist, t), o = __shfl_sync(FULL, off, t);
                const uint32_t ci = __shfl_sync(FULL, tin, t), cs = __shfl_sync(FULL, tst, t);
                for (uint32_t i = lane; i < len; i += 32) {
                    const uint32_t r = i < dist ? i : i % dist;
                    const int32_t srel = (int32_t)(o + r) - (int32_t)dist;
                    st[o + i] = srel < 0 ? out[nout + o + r - dist] : st[srel];
                    tt[o + i] = (uint8_t)(i ? ci : cs);
                }
                __syncwarp();
            }
            for (uint32_t q = lane; q < tot; q += 32) { out[nout + q] = st[q]; if (tmap) tmap[nout + q] = tt[q]; }
            __syncwarp();
        } else {   // a batch of long matches: token by token, straight to global memory
            for (uint32_t t = 0; t < ntok; t++) {
                const uint32_t len = __shfl_sync(FULL, my_len, t), dist = __shfl_sync(FULL, my_dist, t), lit = __shfl_sync(FULL, my_lit, t);
                if (dist == 0) { put_literal(nout, lit); nout += 1; } else { put_match(nout, len, dist); nout += len; }
            }
            __syncwarp();
        }
    }
};

struct Inflater {
    const uint8_t *file; uint64_t off, avail, first_len, vtotal, chunk; // input: avail = current end (first_len, then vtotal)
    bool first_prev; uint32_t good_dups;   // InflateJob::flags: the reference's overlap-byte quirk (common.cuh)
    bool switched; InflateResult *probe_res;
    uint64_t seg_end, seg_delta;   // the input is physically contiguous for virtual indices < seg_end: file position = off + v - seg_delta
    uint64_t buf; uint32_t bcnt; uint64_t next; // bit buffer: bcnt valid bits, next = index of next unread byte
    uint8_t *out; uint64_t out_cap, nout;
    uint8_t *tmap;      // produce mode: token map of this stream (common.cuh TM_*), or nullptr
    uint64_t first_cap, in_at_cap; bool cap_seen;
    uint32_t a, b;
    uint8_t *sm;

    __device__ __forceinline__ uint32_t in_byte(uint64_t v) {
        uint64_t fp = off + v;
        if (v >= first_len) {
            const uint64_t c = (v - first_len) / chunk;
            fp -= 1 + c;
            if ((v - first_len) % chunk == 0 && c >= good_dups) fp -= 1;     // the repeated byte of this boundary is the one before the true last byte
        } else if (v == 0 && first_prev) fp = off - 1;
        return __ldg(file + fp);
    }
    __device__ __forceinline__ void fill() {
        if (bcnt > 32) return;
        if (next == 0 && first_prev) { buf |= (uint64_t)__ldg(file + off - 1) << bcnt; bcnt += 8; next = 1; }
        if (next + 4 <= seg_end) { buf |= (uint64_t)ldu32(file + off + next - seg_delta) << bcnt; bcnt += 32; next += 4; return; }
        while (bcnt <= 56 && next < avail) {
            uint64_t quirk = 0;
            if (next >= seg_end) {   // entering the next chunk of a continuation: it starts with the duplicated overlap byte
                const uint64_t c = (next - first_len) / chunk;
                seg_delta = 1 + c; seg_end = first_len + (c + 1) * chunk; if (seg_end > avail) seg_end = avail;
                if (c >= good_dups) quirk = 1;      // (... which for all but the boundary between chunks 0 and 1 is the byte before it)
            }
            buf |= (uint64_t)__ldg(file + off + next - seg_delta - quirk) << bcnt; bcnt += 8; next++;
        }
    }
    // The input of the first chunk is used up: what inflate() would report now is the probe result; then carry on over
    // the following chunks, if any.  false = there is nothing more.
    __device__ __forceinline__ bool more_input() {
        if (switched || vtotal <= avail) return false;
        write_probe(probe_res, (b << 16) | a, avail, nout, cap_seen ? in_at_cap : avail);
        switched = true; avail = vtotal;
        return true;
    }
    // n <= 16.  false = input exhausted (everything counts as consumed, like NEEDBITS draining `have`)
    __device__ __forceinline__ bool need(uint32_t nb, uint32_t &v) {
        fill();
        if (bcnt < nb) {
            if (more_input()) fill();
            if (bcnt < nb) { next = avail; bcnt = 0; buf = 0; return false; }   // everything counts as consumed
        }
        v = (uint32_t)buf & ((1u << nb) - 1); buf >>= nb; bcnt -= nb;
        return true;
    }
    // bits consumed so far = 8 * next - bcnt (the buffer always holds whole unread bytes above the current one)
    __device__ __forceinline__ uint64_t bitpos() const { return next * 8 - bcnt; }
    __device__ __forceinline__ void byte_align() { const uint32_t r = bcnt & 7; buf >>= r; bcnt -= r; }
    __device__ __forceinline__ uint64_t bytes_used() const { return (bitpos() + 7) >> 3; }
    __device__ __forceinline__ void note_cap() { if (!cap_seen && nout >= first_cap) { cap_seen = true; in_at_cap = bytes_used(); } }

    // canonical bit-serial decode (exact at the end of input and for the filler entries of incomplete codes,
    // Z/inftrees.c:118-125,290-296).  1 ok, 0 out of input, -1 invalid code (1 bit consumed)
    __device__ int decode_slow(const uint16_t *cnt, const uint16_t *symtab, uint32_t maxlen, uint32_t &sym) {
        uint32_t bit;
        if (maxlen == 0) { if (!need(1, bit)) return 0; return -1; }
        int code = 0, first = 0, index = 0;
        for (uint32_t len = 1; len <= maxlen; len++) {
            if (!need(1, bit)) return 0;
            code |= (int)bit;
            int c = cnt[len];
            if (code - c < first) { sym = symtab[index + (code - first)]; return 1; }
            index += c; first += c; first <<= 1; code <<= 1;
        }
        return -1;
    }
    __device__ __forceinline__ int decode(const Code &c, uint32_t &sym) {
        fill();
        uint32_t e = c.tab[(uint32_t)buf & ((1u << c.pb) - 1)], l = e & 15;
        if (l && l <= bcnt) { buf >>= l; bcnt -= l; sym = e >> 4; return 1; }
        return decode_slow(c.cnt, c.sym, c.maxlen, sym);
    }

    // Canonical code from lens[0..n): counts, validity (Z/inftrees.c:100-139), sorted symbols, primary table.
    // returns 0 ok / -1 rejected; maxlen_out = longest code length (0 = no codes).  Lane-parallel except the 15-step
    // validity / first-code recurrences.
    __device__ int build(const uint8_t *lens, uint32_t n, uint16_t *cnt, uint16_t *symtab, uint16_t *tab, uint32_t pb, bool is_cl, uint32_t &maxlen_out) {
        const uint32_t lane = lane_id();
        uint16_t *first = (uint16_t *)(sm + I_TMP), *start = first + 16, *offs = first + 32; uint32_t *cw = (uint32_t *)(first + 48);
        int rc = 0; uint32_t maxl = 0;
        __syncwarp();
        if (lane < 16) cw[lane] = 0;
        __syncwarp();
        for (uint32_t i = lane; i < n; i += 32) atomicAdd(&cw[lens[i]], 1u);
        __syncwarp();
        if (lane == 0) {
            maxl = 15; while (maxl >= 1 && cw[maxl] == 0) maxl--;
            if (maxl > 0) {
                int left = 1;
                for (int l = 1; l <= 15; l++) { left <<= 1; left -= (int)cw[l]; if (left < 0) { rc = -1; break; } }
                if (rc == 0 && left > 0 && (is_cl || maxl != 1)) rc = -1;
            }
            uint32_t code = 0, idx = 0;
            cnt[0] = 0;
            for (int l = 1; l <= 15; l++) { cnt[l] = (uint16_t)cw[l]; first[l] = (uint16_t)code; start[l] = (uint16_t)idx; offs[l] = (uint16_t)idx; code = (code + cw[l]) << 1; idx += cw[l]; }
        }
        rc = __shfl_sync(FULL, rc, 0); maxl = __shfl_sync(FULL, maxl, 0);
        maxlen_out = maxl;
        __syncwarp();
        if (rc) return rc;
        for (uint32_t i0 = 0; i0 < n; i0 += 32) {   // symbols sorted by (length, symbol): 32 symbols per step, ranked among equal lengths
            const uint32_t i = i0 + lane, l = i < n ? lens[i] : 0;
            const uint32_t peers = __match_any_sync(FULL, l), rank = __popc(peers & ((1u << lane) - 1));
            uint32_t base = 0;
            if (l) { base = offs[l]; symtab[base + rank] = (uint16_t)i; }
            __syncwarp();
            if (l && rank == 0) offs[l] = (uint16_t)(base + __popc(peers));
            __syncwarp();
        }
        if (tab == nullptr) return 0;
        const uint32_t tsize = 1u << pb;
        for (uint32_t j = lane; j < tsize; j += 32) tab[j] = 0;
        __syncwarp();
        uint32_t total = 0; for (int l = 1; l <= 15; l++) total += cnt[l];
        for (uint32_t j0 = 0; j0 < total; j0 += 32) {
            const uint32_t j = j0 + lane; uint32_t s = 0, l = 0, rev = 0;
            if (j < total) { s = symtab[j]; l = lens[s]; if (l <= pb) rev = __brev((uint32_t)first[l] + (j - start[l])) >> (32 - l); else l = 0; }
            const bool wide = l && (tsize >> l) >= 32;      // many replicas: the whole warp fills them
            if (l && !wide) for (uint32_t k = rev; k < tsize; k += 1u << l) tab[k] = (uint16_t)((s << 4) | l);
            uint32_t wm = __ballot_sync(FULL, wide);
            while (wm) {
                const uint32_t w = (uint32_t)__ffs((int)wm) - 1; wm &= wm - 1;
                const uint32_t ws = __shfl_sync(FULL, s, w), wl = __shfl_sync(FULL, l, w), wr = __shfl_sync(FULL, rev, w);
                for (uint32_t k = wr + (lane << wl); k < tsize; k += 32u << wl) tab[k] = (uint16_t)((ws << 4) | wl);
            }
        }
        __syncwarp();
        return 0;
    }

    __device__ __forceinline__ uint8_t *optr(uint64_t pos) { return out + pos; }
    __device__ __forceinline__ void put_literal(uint32_t v) {
        if (lane_id() == 0) { *optr(nout) = (uint8_t)v; if (tmap) tmap[nout] = 1; }
        nout++;
    }
    // copy `len` bytes from distance `dist` (lane-parallel; handles overlap)
    __device__ __forceinline__ void put_match(uint32_t len, uint32_t dist) {
        const uint32_t lane = lane_id();
        const uint32_t tin = TM_INNER + (len <= 4 ? 3u : len == 5 ? 2u : len == 6 ? 1u : 0u), tst = len < TM_LONG ? len : TM_LONG;
        __syncwarp();
        for (uint32_t i = lane; i < len; i += 32) {
            const uint32_t r = i < dist ? i : i % dist;
            *optr(nout + i) = *optr(nout - dist + r);
            if (tmap) tmap[nout + i] = (uint8_t)(i ? tin : tst);
        }
        nout += len;
        __syncwarp();
    }
    // adler32 (Z/adler32.c:65-133) of the whole output, once, when the stream has ended: every lane sums a contiguous
    // slice, the slices are combined in order (b_total += b_k + len_k * a_running).
    __device__ void adler_of_output() {
        const uint32_t lane = lane_id();
        const uint64_t per = (nout + 31) / 32;
        uint64_t beg = (uint64_t)lane * per, end = beg + per; if (beg > nout) beg = nout; if (end > nout) end = nout;
        uint32_t sa = 0, sb = 0; const uint32_t slen = (uint32_t)((end - beg) % 65521u);
        __syncwarp();
        for (uint64_t i = beg; i < end;) {
            uint32_t k = (uint32_t)(end - i < 3800 ? end - i : 3800);
            for (uint32_t e = 0; e < k; e++) { sa += out[i + e]; sb += sa; }
            sa %= 65521u; sb %= 65521u; i += k;
        }
        uint64_t A = 1, B = 0;
        for (uint32_t k = 0; k < 32; k++) {
            const uint32_t ka = __shfl_sync(FULL, sa, k), kb = __shfl_sync(FULL, sb, k), kl = __shfl_sync(FULL, slen, k);
            B = (B + kb + (uint64_t)kl * A) % 65521u; A = (A + ka) % 65521u;
        }
        a = (uint32_t)A; b = (uint32_t)B;
    }

    // One batch: decode up to 32 tokens (uniform code; lane k keeps token k), then produce their bytes together: literals and
    // matches are assembled in a shared-memory stage - sources that lie before the batch are fetched from global memory four
    // tokens at a time so that their latencies overlap, sources inside the batch are copied stage to stage in token order -
    // and written out with coalesced stores.  Only entered where a whole batch is sure to have input and output room.
    // returns 0 = 32 tokens done, 1 = end of block, 2 = data error (bits / nout are exact at the point of the error).
    __device__ __forceinline__ int batch(const Code &L, const Code &D) {
        const uint32_t lane = lane_id();
        uint32_t my_len = 0, my_dist = 0, my_lit = 0, k = 0; uint64_t vout = nout; int ev = 0;
        const uint16_t *ltab = L.tab, *dtab = D.tab;
        // input is guaranteed here (the caller checked that 288 bytes are left in this segment): the next input word is always
        // requested one refill ahead, so its load is not on the decode's dependency chain
        const uint8_t *ip = file + off + next - seg_delta;     // address of the next unread input byte
        uint32_t ahead = ldu32(ip);
#define BATCH_REFILL() do { if (bcnt <= 32) { buf |= (uint64_t)ahead << bcnt; bcnt += 32; next += 4; ip += 4; ahead = ldu32(ip); } } while (0)
        while (k < 32) {
            // refill 32 bits whenever at most 32 are left, so a literal/length code with its extra bits (<= 20) and then a
            // distance code with its extra bits (<= 28) always find their bits
            BATCH_REFILL();
            uint32_t e = ltab[(uint32_t)buf & ((1u << LPB) - 1)], l = e & 15, sym = e >> 4;
            if (l) { buf >>= l; bcnt -= l; }
            else { const int rc = decode_slow(L.cnt, L.sym, L.maxlen, sym); if (rc <= 0) { ev = 2; break; } ip = file + off + next - seg_delta; ahead = ldu32(ip); }   // (long code: bit-serial, refills on its own)
            if (sym < 256) { if (lane == k) { my_len = 1; my_lit = sym; my_dist = 0; } k++; vout++; continue; }
            if (sym == 256) { ev = 1; break; }
            if (sym > 285) { ev = 2; break; }
            const uint32_t lc = sym - 257, xb = (lc < 8 || lc == 28) ? 0 : (lc - 4) >> 2;
            uint32_t len = lc < 8 ? lc + 3 : lc == 28 ? 258u : 3 + ((4 + (lc & 3)) << xb);      // base_length, Z/trees.h
            len += (uint32_t)buf & ((1u << xb) - 1); buf >>= xb; bcnt -= xb;
            BATCH_REFILL();
            e = dtab[(uint32_t)buf & ((1u << DPB) - 1)]; l = e & 15; sym = e >> 4;
            if (l) { buf >>= l; bcnt -= l; }
            else { const int rc = decode_slow(D.cnt, D.sym, D.maxlen, sym); if (rc <= 0) { ev = 2; break; } ip = file + off + next - seg_delta; ahead = ldu32(ip); }
            if (sym > 29) { ev = 2; break; }
            const uint32_t dxb = sym < 4 ? 0 : (sym - 2) >> 1; uint32_t dist = sym < 4 ? sym + 1 : ((2 + (sym & 1)) << dxb) + 1;
            dist += (uint32_t)buf & ((1u << dxb) - 1); buf >>= dxb; bcnt -= dxb;
            if ((uint64_t)dist > vout) { ev = 2; break; }
            if (lane == k) { my_len = len; my_dist = dist; }
            k++; vout += len;
        }
#undef BATCH_REFILL
        const uint32_t ntok = k;
        if (ntok == 0) return ev;
        Writer{out, tmap, sm}.produce(my_len, my_dist, my_lit, ntok, nout);
        nout = vout;
        return ev;
    }

    __device__ int run(InflateResult *res, InflateResult *cont) {
        const uint32_t lane = lane_id();
        uint16_t *ltab = (uint16_t *)(sm + I_LTAB), *dtab = (uint16_t *)(sm + I_DTAB), *lsym = (uint16_t *)(sm + I_LSYM), *dsym = (uint16_t *)(sm + I_DSYM);
        uint16_t *lcnt = (uint16_t *)(sm + I_LCNT), *dcnt = (uint16_t *)(sm + I_DCNT), *ccnt = (uint16_t *)(sm + I_CCNT), *csym = (uint16_t *)(sm + I_CSYM), *ctab = (uint16_t *)(sm + I_CTAB);
        uint8_t *lens = sm + I_LENS;
        extern __shared__ __align__(16) uint8_t smem_all[];
        const uint8_t *fx = smem_all;
        int status = INF_DATA_ERROR; uint32_t v, last = 0;
#define NEED(nb, v) do { if (!need((nb), (v))) { status = INF_NEED_INPUT; goto done; } } while (0)
#define FAILD() do { status = INF_DATA_ERROR; goto done; } while (0)
        NEED(16, v);   // zlib header, Z/inflate.c:636-679
        { uint32_t cmf = v & 0xff, flg = v >> 8;
          if (((cmf << 8) + flg) % 31) FAILD();
          if ((cmf & 15) != 8) FAILD();
          if ((cmf >> 4) + 8 > 15) FAILD();
          if (flg & 0x20) { NEED(16, v); NEED(16, v); status = INF_NEED_DICT; goto done; } }
        while (!last) {
            uint32_t type;
            NEED(3, v); last = v & 1; type = v >> 1;
            if (type == 3) FAILD();
            if (type == 0) {   // stored, Z/inflate.c:866-901
                byte_align();
                uint32_t len, nlen; NEED(16, len); NEED(16, nlen);
                if (len != (nlen ^ 0xffff)) FAILD();
                // the bit buffer holds whole bytes now; hand them back and copy from the byte position
                uint64_t bp = bitpos() >> 3; buf = 0; bcnt = 0; next = bp;
                uint32_t left = len;
                for (;;) {
                    uint64_t can = avail - bp; uint32_t take = left < can ? left : (uint32_t)can;
                    if (!cap_seen && nout + take > first_cap) { cap_seen = true; in_at_cap = bp + (first_cap - nout); }
                    if (nout + take > out_cap) { status = INF_OUT_FULL; goto done; }
                    __syncwarp();
                    for (uint32_t i = lane; i < take; i += 32) { *optr(nout + i) = (uint8_t)in_byte(bp + i); if (tmap) tmap[nout + i] = 0; }   // stored: no tokens known
                    __syncwarp();
                    nout += take; bp += take; left -= take; next = bp;
                    if (!left) break;
                    if (!more_input()) { status = INF_NEED_INPUT; goto done; }
                }
                continue;
            }
            Code L, D;
            if (type == 1) {
                L.tab = (const uint16_t *)(fx + F_LTAB); L.sym = (const uint16_t *)(fx + F_LSYM); L.cnt = (const uint16_t *)(fx + F_LCNT); L.pb = LPB; L.maxlen = 9;
                D.tab = (const uint16_t *)(fx + F_DTAB); D.sym = (const uint16_t *)(fx + F_DSYM); D.cnt = (const uint16_t *)(fx + F_DCNT); D.pb = DPB; D.maxlen = 5;
            } else {   // dynamic, Z/inflate.c:903-1016
                uint32_t nlen, ndist, ncode;
                NEED(14, v); nlen = (v & 31) + 257; ndist = ((v >> 5) & 31) + 1; ncode = (v >> 10) + 4;
                if (nlen > 286 || ndist > 30) FAILD();
                __syncwarp();
                if (lane < 19) lens[lane] = 0;
                __syncwarp();
                for (uint32_t i = 0; i < ncode; i++) { NEED(3, v); if (lane == 0) lens[c_clord[i]] = (uint8_t)v; }
                uint32_t cmax;
                if (build(lens, 19, ccnt, csym, ctab, CPB, true, cmax)) FAILD();
                Code Cc; Cc.tab = ctab; Cc.sym = csym; Cc.cnt = ccnt; Cc.pb = CPB; Cc.maxlen = cmax;
                uint32_t have = 0, prevlen = 0;
                while (have < nlen + ndist) {
                    uint32_t sym; int rc;
                    if (cmax == 0) { NEED(1, v); sym = 0; rc = 1; }   // filler entries decode as length 0 (Z/inflate.c:944-953)
                    else rc = decode(Cc, sym);
                    if (rc == 0) { status = INF_NEED_INPUT; goto done; }
                    if (rc < 0) sym = 0;
                    if (sym < 16) { if (lane == 0) lens[have] = (uint8_t)sym; prevlen = sym; have++; continue; }
                    uint32_t rep, val = 0;
                    if (sym == 16) { NEED(2, v); if (have == 0) FAILD(); val = prevlen; rep = 3 + v; }
                    else if (sym == 17) { NEED(3, v); rep = 3 + v; }
                    else { NEED(7, v); rep = 11 + v; }
                    if (have + rep > nlen + ndist) FAILD();
                    for (uint32_t i = lane; i < rep; i += 32) lens[have + i] = (uint8_t)val;
                    have += rep; prevlen = val;
                }
                __syncwarp();
                if (lens[256] == 0) FAILD();
                uint32_t lmax, dmax;
                if (build(lens, nlen, lcnt, lsym, ltab, LPB, false, lmax)) FAILD();
                if (build(lens + nlen, ndist, dcnt, dsym, dtab, DPB, false, dmax)) FAILD();
                L.tab = ltab; L.sym = lsym; L.cnt = lcnt; L.pb = LPB; L.maxlen = lmax;
                D.tab = dtab; D.sym = dsym; D.cnt = dcnt; D.pb = DPB; D.maxlen = dmax;
            }
            for (;;) {   // Z/inflate.c:1018-1172, Z/inffast.c:120-307
                // batches where 32 tokens (<= 6 B of input, <= 258 B of output each) are sure to fit before the input ends, the
                // scanner's first output buffer fills (in_at_cap must be exact) or the output region does
                if (next + 288 <= seg_end && (cap_seen || nout + 8300 < first_cap) && nout + 8300 <= out_cap) {
                    const int ev = batch(L, D);
                    if (ev == 1) break;
                    if (ev == 2) FAILD();
                    continue;
                }
                uint32_t sym; int rc = decode(L, sym);
                if (rc == 0) { status = INF_NEED_INPUT; goto done; }
                if (rc < 0 || sym > 285) FAILD();
                if (sym < 256) {
                    note_cap();
                    if (nout >= out_cap) { status = INF_OUT_FULL; goto done; }
                    put_literal(sym); continue;
                }
                if (sym == 256) break;
                uint32_t lc = sym - 257, len = c_lbase[lc], xb = (lc < 8 || lc == 28) ? 0 : (lc - 4) >> 2, dist;
                if (xb) { NEED(xb, v); len += v; }
                rc = decode(D, sym);
                if (rc == 0) { status = INF_NEED_INPUT; goto done; }
                if (rc < 0 || sym > 29) FAILD();
                { uint32_t dxb = sym < 4 ? 0 : (sym - 2) >> 1;
                  dist = sym < 4 ? sym + 1 : ((2 + (sym & 1)) << dxb) + 1;
                  if (dxb) { NEED(dxb, v); dist += v; } }
                note_cap();   // MATCH leaves on left == 0 before it checks the distance (Z/inflate.c:1137-1147)
                if (!cap_seen && nout + len > first_cap) { cap_seen = true; in_at_cap = bytes_used(); }
                if ((uint64_t)dist > nout) FAILD();
                if (nout + len > out_cap) { status = INF_OUT_FULL; goto done; }
                put_match(len, dist);
            }
        }
        byte_align();   // CHECK, Z/inflate.c:1174-1195
        { uint32_t hi, lo; NEED(16, hi); NEED(16, lo);
          uint32_t want = ((hi & 0xff) << 24) | ((hi >> 8) << 16) | ((lo & 0xff) << 8) | (lo >> 8);
          adler_of_output();
          if (want != ((b << 16) | a)) FAILD();
          status = INF_END; }
    done:
#undef NEED
#undef FAILD
        if (lane == 0) {
            InflateResult *r = switched ? cont : res;
            r->status = status; r->adler = (b << 16) | a; r->total_in = bytes_used(); r->total_out = nout;
            r->in_at_outcap = cap_seen ? in_at_cap : bytes_used();
            if (!switched) cont->status = -1;
        }
        return status;
    }
};

__global__ void __launch_bounds__(128) inflate_kernel(const uint8_t *file, const InflateJob *jobs, InflateResult *results, InflateResult *cont, uint32_t njobs,
                                                      uint32_t *queue, uint8_t *arena, uint64_t first_cap, uint64_t chunk) {
    extern __shared__ __align__(16) uint8_t smem_all[];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    Inflater inf;
    inf.sm = smem_all + F_SIZE + warp * I_WARP;
    // fixed Huffman tables once per CTA (Z/inffixed.h is what zlib uses; here they are rebuilt from the RFC lengths)
    {
        uint8_t *lens = inf.sm + I_LENS; uint32_t mx;
        if (warp == 0) {
            for (uint32_t i = lane; i < 288; i += 32) lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
            __syncwarp();
            inf.build(lens, 288, (uint16_t *)(smem_all + F_LCNT), (uint16_t *)(smem_all + F_LSYM), (uint16_t *)(smem_all + F_LTAB), LPB, false, mx);
            lens[lane] = 5;
            __syncwarp();
            inf.build(lens, 32, (uint16_t *)(smem_all + F_DCNT), (uint16_t *)(smem_all + F_DSYM), (uint16_t *)(smem_all + F_DTAB), DPB, false, mx);
        }
        __syncthreads();
    }
    for (;;) {
        uint32_t ji = 0;
        if (lane == 0) ji = atomicAdd(queue, 1u);
        ji = __shfl_sync(FULL, ji, 0);
        if (ji >= njobs) break;
        const InflateJob j = jobs[ji];
        inf.file = file; inf.off = j.off; inf.avail = j.avail; inf.first_len = j.avail; inf.vtotal = j.vtotal; inf.chunk = chunk;
        inf.first_prev = (j.flags & INFJ_FIRST_FROM_PREV) != 0; inf.good_dups = (uint32_t)((j.flags >> 8) & 0xff);
        inf.switched = false; inf.probe_res = &results[ji]; inf.seg_end = j.avail; inf.seg_delta = 0;
        inf.buf = 0; inf.bcnt = 0; inf.next = 0;
        inf.out = arena + j.out_off;
        inf.out_cap = j.out_cap; inf.nout = 0;
        inf.tmap = j.tmap_off != ~0ull ? arena + j.tmap_off : nullptr;
        inf.first_cap = first_cap ? first_cap : ~0ull; inf.in_at_cap = 0; inf.cap_seen = false;
        inf.a = 1; inf.b = 0;
        inf.run(&results[ji], &cont[ji]);
        __syncwarp();
    }
}

cudaError_t launch_inflate(const uint8_t *file, const InflateJob *jobs, InflateResult *results, InflateResult *cont, uint32_t njobs, uint32_t *queue,
                           uint8_t *arena, uint64_t first_cap, uint64_t chunk, int ctas, int warps_per_cta, cudaStream_t s) {
    const size_t smem = F_SIZE + (size_t)warps_per_cta * I_WARP;
    inflate_kernel<<<ctas, warps_per_cta * 32, smem, s>>>(file, jobs, results, cont, njobs, queue, arena, first_cap, chunk);
    return cudaGetLastError();
}

} // namespace atz
