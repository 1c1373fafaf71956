/*
 * ORACLE - TEST INFRASTRUCTURE ONLY.  Never linked into, called by, or shipped
 * with the product library (libantiz_b200.so).  Only tests/, bench.py's
 * cpu_baseline/--impl reference leg and __graft_entry__.smoke() may use it.
 *
 * CPU restatement of zlib 1.2.8's deflate as AntiZ drives it
 *   deflateInit2(level, Z_DEFLATED, windowBits, memLevel, Z_DEFAULT_STRATEGY)
 *   + deflate(Z_FINISH) with the whole plaintext available
 * (reference call sites: main.cpp:621-661 testDeflateParams, main.cpp:976-1003
 * doDeflate).  It is a *faithful* restatement: 16-bit window-relative head/prev
 * tables, the window slide, the symbol buffer and zlib's heap-based Huffman
 * construction are all kept, so that it can pin every tie-break.  Cited lines
 * are in "/root/reference/includes, tools, stuff/zlib test/zlib128/" (Z/).
 *
 * Parity pin: tests/test_oracle_deflate.py checks this file byte-for-byte
 * against oracle/_ref/libz128.so (the reference's own zlib, compiled from
 * /root/reference) over level 0-9 x wbits 10-15 x memLevel 1-9 and against the
 * reference's five golden vectors (tests/golden/zlibtest_out_*.bin).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define MINM 3
#define MAXM 258
#define MIN_LOOK (MAXM + MINM + 1) /* Z/deflate.h:278 */
#define TOO_FAR_D 4096             /* Z/deflate.c:1727 */
#define NLIT 256
#define NLEN 29
#define NLSYM 286 /* L_CODES */
#define NDSYM 30  /* D_CODES */
#define NBSYM 19  /* BL_CODES */
#define HEAPSZ (2 * NLSYM + 1)
#define EOB 256

/* ---- constant tables (Z/trees.c:62-73, Z/trees.h; regenerated, not copied) ---- */
static const uint8_t XL[NLEN] = {0,0,0,0,0,0,0,0,1,1,1,1,2,2,2,2,3,3,3,3,4,4,4,4,5,5,5,5,0};
static const uint8_t XD[NDSYM] = {0,0,0,0,1,1,2,2,3,3,4,4,5,5,6,6,7,7,8,8,9,9,10,10,11,11,12,12,13,13};
static const uint8_t XB[NBSYM] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,2,3,7};
static const uint8_t BLORD[NBSYM] = {16,17,18,0,8,7,9,6,10,5,11,4,12,3,13,2,14,1,15};

static uint8_t  g_lcode[256];   /* (len-3) -> length code 0..28 */
static uint16_t g_lbase[NLEN];
static uint8_t  g_dcode[512];   /* Z/trees.c:317-331 two-level distance code map */
static uint16_t g_dbase[NDSYM];
static uint16_t g_sl_code[NLSYM + 2]; static uint8_t g_sl_len[NLSYM + 2];
static uint16_t g_sd_code[NDSYM];     static uint8_t g_sd_len[NDSYM];
static int g_init = 0;

static unsigned rev_bits(unsigned c, int n) { unsigned r = 0; while (n--) { r = (r << 1) | (c & 1); c >>= 1; } return r; }

static void init_tables(void) { /* what tr_static_init computes, Z/trees.c:235-323 */
    if (g_init) return;
    int len = 0;
    for (int c = 0; c < NLEN - 1; c++) { g_lbase[c] = (uint16_t)len; for (int n = 0; n < (1 << XL[c]); n++) g_lcode[len++] = (uint8_t)c; }
    g_lcode[255] = NLEN - 1; g_lbase[NLEN - 1] = 255; /* length 258 has its own code, Z/trees.c:269-272 */
    int d = 0, c = 0;
    for (; c < 16; c++) { g_dbase[c] = (uint16_t)d; for (int n = 0; n < (1 << XD[c]); n++) g_dcode[d++] = (uint8_t)c; }
    d >>= 7;
    for (; c < NDSYM; c++) { g_dbase[c] = (uint16_t)(d << 7); for (int n = 0; n < (1 << (XD[c] - 7)); n++) g_dcode[256 + d++] = (uint8_t)c; }
    /* fixed literal/length code: 8,9,7,8 bits (RFC1951 3.2.6) */
    unsigned cnt[16] = {0}, next[16];
    for (int n = 0; n < NLSYM + 2; n++) { g_sl_len[n] = n <= 143 ? 8 : n <= 255 ? 9 : n <= 279 ? 7 : 8; cnt[g_sl_len[n]]++; }
    unsigned code = 0; for (int b = 1; b <= 15; b++) { code = (code + cnt[b - 1]) << 1; next[b] = code; }
    for (int n = 0; n < NLSYM + 2; n++) g_sl_code[n] = (uint16_t)rev_bits(next[g_sl_len[n]]++, g_sl_len[n]);
    for (int n = 0; n < NDSYM; n++) { g_sd_len[n] = 5; g_sd_code[n] = (uint16_t)rev_bits((unsigned)n, 5); }
    g_init = 1;
}
static inline int dist_code(unsigned d) { return d < 256 ? g_dcode[d] : g_dcode[256 + (d >> 7)]; }

/* level table, Z/deflate.c:131-143 */
static const struct { uint16_t good, lazy, nice, chain; uint8_t kind; } CFG[10] = {
    {0,0,0,0,0},{4,4,8,4,1},{4,5,16,8,1},{4,6,32,32,1},{4,4,16,16,2},
    {8,16,32,32,2},{8,16,128,128,2},{8,32,128,256,2},{32,128,258,1024,2},{32,258,258,4096,2}};

typedef struct { uint16_t fc; uint16_t dl; } node_t; /* freq|code, dad|len as in ct_data */

/* Branch counters of the block flush (tests only: they write nothing into the output).  oracle_flush_counts() reads and resets them. */
enum { FC_OVER_L, FC_OVER_D, FC_OVER_B,                                  /* gen_bitlen depth-limit repair, per tree kind */
       FC_FORCE_L_LOW, FC_FORCE_L_HIGH, FC_FORCE_D_LOW, FC_FORCE_D_HIGH,  /* heap_len < 2 forcing, max_code < 2 / >= 2 */
       FC_FORCE_B_LOW, FC_FORCE_B_HIGH,
       FC_STORED, FC_STATIC, FC_DYNAMIC, FC_UNSTORABLE,                   /* block kinds; flushes with buf == NULL after a slide */
       FC_TIE_STORED, FC_TIE_STATIC,                                      /* stored_len + 4 == opt_lenb; static_lenb == opt_lenb == opt_len */
       FC_REP16_6, FC_REP17_3, FC_REP17_10, FC_REP18_11, FC_REP18_138,   /* scan_tree runs at the limits of their codes */
       FC_ZRUN_SPLIT,                                                     /* a run of more than 138 zero lengths, split */
       FC_N };
static uint64_t g_fc[FC_N];
int oracle_flush_counts(uint64_t *out, int n) {
    if (out) for (int i = 0; i < n && i < FC_N; i++) out[i] = g_fc[i];
    memset(g_fc, 0, sizeof g_fc);
    return FC_N;
}

typedef struct {
    const uint8_t *in; uint32_t in_len, in_pos;
    uint8_t *out; uint64_t out_cap, out_len; int overflow;
    uint64_t bitbuf; int bitcnt;
    int level, wbits, memlevel;
    uint32_t wsize, wmask, hbits, hsize, hmask, hshift, litsz, pend_sz;
    uint8_t *win; uint16_t *prev, *head;
    uint32_t strstart, lookahead, match_start, match_len, prev_len, prev_match, ins_h;
    int match_avail; long block_start;
    uint16_t *dbuf; uint8_t *lbuf; uint32_t nsym;
    node_t lt[HEAPSZ], dt[2 * NDSYM + 1], bt[2 * NBSYM + 1];
    int heap[HEAPSZ], heap_len, heap_max; uint8_t depth[HEAPSZ];
    uint16_t blcount[16];
    long opt_len, static_len;
    int l_max, d_max;
    uint32_t adler_a, adler_b;
    /* instrumentation for tests / bench accounting */
    uint64_t out_at_first_flush; uint32_t in_at_limit; uint64_t limit_out; int limit_hit; uint32_t base;
    int abs_mode; uint32_t wend; /* design model only (oracle_deflate_listmode) */
} zd_t;

/* ---- output ---- */
static void put8(zd_t *s, unsigned b) { if (s->out_len < s->out_cap) s->out[s->out_len] = (uint8_t)b; else s->overflow = 1; s->out_len++; }
static void putbits(zd_t *s, unsigned v, int n) { /* LSB-first packing == Z/trees.c:213-225 send_bits + put_short */
    s->bitbuf |= (uint64_t)v << s->bitcnt; s->bitcnt += n;
    while (s->bitcnt >= 8) { put8(s, (unsigned)(s->bitbuf & 0xff)); s->bitbuf >>= 8; s->bitcnt -= 8; }
}
static void align_byte(zd_t *s) { if (s->bitcnt > 0) { put8(s, (unsigned)(s->bitbuf & 0xff)); } s->bitbuf = 0; s->bitcnt = 0; } /* bi_windup Z/trees.c:1186 */

/* ---- Huffman construction: Z/trees.c:451-699 ---- */
static int tree_kind(zd_t *s, node_t *t) { return t == s->lt ? 0 : t == s->dt ? 1 : 2; }
#define LESS(t, n, m) ((t)[n].fc < (t)[m].fc || ((t)[n].fc == (t)[m].fc && s->depth[n] <= s->depth[m]))
static void sift(zd_t *s, node_t *t, int k) { /* pqdownheap Z/trees.c:451-478 */
    int v = s->heap[k], j = k << 1;
    while (j <= s->heap_len) {
        if (j < s->heap_len && LESS(t, s->heap[j + 1], s->heap[j])) j++;
        if (LESS(t, v, s->heap[j])) break;
        s->heap[k] = s->heap[j]; k = j; j <<= 1;
    }
    s->heap[k] = v;
}
static void bit_lengths(zd_t *s, node_t *t, int max_code, const uint8_t *st_len, const uint8_t *extra, int xbase, int maxlen) { /* gen_bitlen Z/trees.c:488-565 */
    int over = 0, h;
    memset(s->blcount, 0, sizeof s->blcount);
    t[s->heap[s->heap_max]].dl = 0;
    for (h = s->heap_max + 1; h < HEAPSZ; h++) {
        int n = s->heap[h], bits = t[t[n].dl].dl + 1;
        if (bits > maxlen) { bits = maxlen; over++; }
        t[n].dl = (uint16_t)bits;
        if (n > max_code) continue;
        s->blcount[bits]++;
        int xb = n >= xbase ? extra[n - xbase] : 0;
        s->opt_len += (long)t[n].fc * (bits + xb);
        if (st_len) s->static_len += (long)t[n].fc * (st_len[n] + xb);
    }
    if (!over) return;
    g_fc[FC_OVER_L + tree_kind(s, t)]++;
    do {
        int bits = maxlen - 1;
        while (s->blcount[bits] == 0) bits--;
        s->blcount[bits]--; s->blcount[bits + 1] += 2; s->blcount[maxlen]--;
        over -= 2;
    } while (over > 0);
    for (int bits = maxlen; bits != 0; bits--) {
        int n = s->blcount[bits];
        while (n != 0) {
            int m = s->heap[--h];
            if (m > max_code) continue;
            if (t[m].dl != (unsigned)bits) { s->opt_len += ((long)bits - (long)t[m].dl) * (long)t[m].fc; t[m].dl = (uint16_t)bits; }
            n--;
        }
    }
}
static void assign_codes(zd_t *s, node_t *t, int max_code) { /* gen_codes Z/trees.c:575-607 */
    unsigned next[16], code = 0;
    for (int b = 1; b <= 15; b++) { code = (code + s->blcount[b - 1]) << 1; next[b] = code; }
    for (int n = 0; n <= max_code; n++) { int l = t[n].dl; if (l) t[n].fc = (uint16_t)rev_bits(next[l]++, l); }
}
static int make_tree(zd_t *s, node_t *t, int elems, const uint8_t *st_len, const uint8_t *extra, int xbase, int maxlen) { /* build_tree Z/trees.c:617-699 */
    int max_code = -1, node = elems, n, m;
    s->heap_len = 0; s->heap_max = HEAPSZ;
    for (n = 0; n < elems; n++) {
        if (t[n].fc != 0) { s->heap[++s->heap_len] = max_code = n; s->depth[n] = 0; } else t[n].dl = 0;
    }
    if (s->heap_len < 2) g_fc[FC_FORCE_L_LOW + 2 * tree_kind(s, t) + (max_code >= 2)]++;
    while (s->heap_len < 2) { /* force two codes, Z/trees.c:648-654 */
        int nn = s->heap[++s->heap_len] = (max_code < 2 ? ++max_code : 0);
        t[nn].fc = 1; s->depth[nn] = 0; s->opt_len--; if (st_len) s->static_len -= st_len[nn];
    }
    for (n = s->heap_len / 2; n >= 1; n--) sift(s, t, n);
    do {
        n = s->heap[1]; s->heap[1] = s->heap[s->heap_len--]; sift(s, t, 1);
        m = s->heap[1];
        s->heap[--s->heap_max] = n; s->heap[--s->heap_max] = m;
        t[node].fc = (uint16_t)(t[n].fc + t[m].fc);
        s->depth[node] = (uint8_t)((s->depth[n] >= s->depth[m] ? s->depth[n] : s->depth[m]) + 1);
        t[n].dl = t[m].dl = (uint16_t)node;
        s->heap[1] = node++; sift(s, t, 1);
    } while (s->heap_len >= 2);
    s->heap[--s->heap_max] = s->heap[1];
    bit_lengths(s, t, max_code, st_len, extra, xbase, maxlen);
    assign_codes(s, t, max_code);
    return max_code;
}
/* run-length walk over a code-length array; emit==0 counts into bt (scan_tree Z/trees.c:705-744), emit==1 sends (send_tree 750-795) */
static void walk_lengths(zd_t *s, node_t *t, int max_code, int emit) {
    int prevlen = -1, nextlen = t[0].dl, count = 0, maxc = 7, minc = 4;
    if (nextlen == 0) { maxc = 138; minc = 3; }
    if (!emit) t[max_code + 1].dl = 0xffff;
    for (int n = 0; n <= max_code; n++) {
        int cur = nextlen; nextlen = t[n + 1].dl;
        if (++count < maxc && cur == nextlen) continue;
        if (!emit && count >= minc) {
            if (cur != 0) g_fc[FC_REP16_6] += count - (cur != prevlen) == 6;
            else if (count <= 10) { g_fc[FC_REP17_3] += count == 3; g_fc[FC_REP17_10] += count == 10; }
            else { g_fc[FC_REP18_11] += count == 11; g_fc[FC_REP18_138] += count == 138; g_fc[FC_ZRUN_SPLIT] += count == 138 && nextlen == 0; }
        }
        if (count < minc) {
            if (emit) { do putbits(s, s->bt[cur].fc, s->bt[cur].dl); while (--count != 0); } else s->bt[cur].fc += (uint16_t)count;
        } else if (cur != 0) {
            if (cur != prevlen) { if (emit) { putbits(s, s->bt[cur].fc, s->bt[cur].dl); count--; } else s->bt[cur].fc++; }
            if (emit) { putbits(s, s->bt[16].fc, s->bt[16].dl); putbits(s, (unsigned)(count - 3), 2); } else s->bt[16].fc++;
        } else if (count <= 10) {
            if (emit) { putbits(s, s->bt[17].fc, s->bt[17].dl); putbits(s, (unsigned)(count - 3), 3); } else s->bt[17].fc++;
        } else {
            if (emit) { putbits(s, s->bt[18].fc, s->bt[18].dl); putbits(s, (unsigned)(count - 11), 7); } else s->bt[18].fc++;
        }
        count = 0; prevlen = cur;
        if (nextlen == 0) { maxc = 138; minc = 3; } else if (cur == nextlen) { maxc = 6; minc = 3; } else { maxc = 7; minc = 4; }
    }
}
static void reset_block(zd_t *s) { /* init_block Z/trees.c:409-422 */
    for (int n = 0; n < NLSYM; n++) s->lt[n].fc = 0;
    for (int n = 0; n < NDSYM; n++) s->dt[n].fc = 0;
    for (int n = 0; n < NBSYM; n++) s->bt[n].fc = 0;
    s->lt[EOB].fc = 1; s->opt_len = s->static_len = 0; s->nsym = 0;
}
static void emit_symbols(zd_t *s, int dyn) { /* compress_block Z/trees.c:1060-1105 */
    for (uint32_t i = 0; i < s->nsym; i++) {
        unsigned dist = s->dbuf[i], lc = s->lbuf[i];
        if (dist == 0) { if (dyn) putbits(s, s->lt[lc].fc, s->lt[lc].dl); else putbits(s, g_sl_code[lc], g_sl_len[lc]); continue; }
        unsigned c = g_lcode[lc], sym = c + NLIT + 1;
        if (dyn) putbits(s, s->lt[sym].fc, s->lt[sym].dl); else putbits(s, g_sl_code[sym], g_sl_len[sym]);
        if (XL[c]) putbits(s, lc - g_lbase[c], XL[c]);
        dist--; c = (unsigned)dist_code(dist);
        if (dyn) putbits(s, s->dt[c].fc, s->dt[c].dl); else putbits(s, g_sd_code[c], g_sd_len[c]);
        if (XD[c]) putbits(s, dist - g_dbase[c], XD[c]);
    }
    if (dyn) putbits(s, s->lt[EOB].fc, s->lt[EOB].dl); else putbits(s, g_sl_code[EOB], g_sl_len[EOB]);
}
/* _tr_flush_block Z/trees.c:907-1004 (+ FLUSH_BLOCK_ONLY Z/deflate.c:1538-1546) */
static void flush_block(zd_t *s, int last) {
    const uint8_t *buf = (s->abs_mode ? s->block_start >= (long)s->base : s->block_start >= 0) ? s->win + s->block_start : NULL;
    unsigned long stored_len = (unsigned long)((long)s->strstart - s->block_start);
    unsigned long opt_lenb, static_lenb; int max_bl = 0;
    if (s->level > 0) {
        s->l_max = make_tree(s, s->lt, NLSYM, g_sl_len, XL, NLIT + 1, 15);
        s->d_max = make_tree(s, s->dt, NDSYM, g_sd_len, XD, 0, 15);
        walk_lengths(s, s->lt, s->l_max, 0); walk_lengths(s, s->dt, s->d_max, 0);
        make_tree(s, s->bt, NBSYM, NULL, XB, 0, 7);
        for (max_bl = NBSYM - 1; max_bl >= 3; max_bl--) if (s->bt[BLORD[max_bl]].dl != 0) break;
        s->opt_len += 3 * (max_bl + 1) + 5 + 5 + 4;
        opt_lenb = (unsigned long)(s->opt_len + 3 + 7) >> 3; static_lenb = (unsigned long)(s->static_len + 3 + 7) >> 3;
        if (static_lenb <= opt_lenb) opt_lenb = static_lenb;
        if (stored_len + 4 == opt_lenb && buf != NULL) g_fc[FC_TIE_STORED]++;
        else if (!(stored_len + 4 <= opt_lenb && buf != NULL) && static_lenb == opt_lenb && static_lenb == (unsigned long)(s->opt_len + 3 + 7) >> 3) g_fc[FC_TIE_STATIC]++;
    } else opt_lenb = static_lenb = stored_len + 5;
    if (buf == NULL) g_fc[FC_UNSTORABLE]++;
    if (stored_len + 4 <= opt_lenb && buf != NULL) { /* _tr_stored_block + copy_block Z/trees.c:865-877,1205-1226 */
        g_fc[FC_STORED]++;
        putbits(s, (unsigned)last, 3); align_byte(s);
        put8(s, stored_len & 0xff); put8(s, (stored_len >> 8) & 0xff); put8(s, ~stored_len & 0xff); put8(s, (~stored_len >> 8) & 0xff);
        for (unsigned long i = 0; i < stored_len; i++) put8(s, buf[i]);
    } else if (static_lenb == opt_lenb) {
        g_fc[FC_STATIC]++;
        putbits(s, 2 + (unsigned)last, 3); emit_symbols(s, 0);
    } else {
        g_fc[FC_DYNAMIC]++;
        putbits(s, 4 + (unsigned)last, 3);
        putbits(s, (unsigned)(s->l_max + 1 - 257), 5); putbits(s, (unsigned)(s->d_max + 1 - 1), 5); putbits(s, (unsigned)(max_bl + 1 - 4), 4);
        for (int r = 0; r <= max_bl; r++) putbits(s, s->bt[BLORD[r]].dl, 3);
        walk_lengths(s, s->lt, s->l_max, 1); walk_lengths(s, s->dt, s->d_max, 1);
        emit_symbols(s, 1);
    }
    reset_block(s);
    if (last) align_byte(s);
    s->block_start = (long)s->strstart;
    if (s->out_at_first_flush == 0) s->out_at_first_flush = s->out_len;
    if (!s->limit_hit && s->limit_out && s->out_len >= s->limit_out) { s->limit_hit = 1; s->in_at_limit = s->abs_mode ? s->strstart : s->base + s->strstart; }
}
static int tally(zd_t *s, unsigned dist, unsigned lc) { /* _tr_tally Z/trees.c:1010-1055 */
    s->dbuf[s->nsym] = (uint16_t)dist; s->lbuf[s->nsym++] = (uint8_t)lc;
    if (dist == 0) s->lt[lc].fc++; else { s->lt[g_lcode[lc] + NLIT + 1].fc++; s->dt[dist_code(dist - 1)].fc++; }
    return s->nsym == s->litsz - 1;
}

/* ---- window management: fill_window Z/deflate.c:1390-1532, read_buf 1076-1101 ---- */
static void adler_feed(zd_t *s, const uint8_t *p, uint32_t n) { /* Z/adler32.c:65-133, BASE 65521 */
    uint32_t a = s->adler_a, b = s->adler_b;
    while (n) { uint32_t k = n < 5552 ? n : 5552; n -= k; while (k--) { a += *p++; b += a; } a %= 65521u; b %= 65521u; }
    s->adler_a = a; s->adler_b = b;
}
static void refill(zd_t *s) {
    uint32_t maxd = s->wsize - MIN_LOOK;
    do {
        uint32_t more = 2 * s->wsize - s->lookahead - s->strstart;
        if (s->strstart >= s->wsize + maxd) { /* slide, Z/deflate.c:1419-1451 */
            memcpy(s->win, s->win + s->wsize, s->wsize);
            s->match_start -= s->wsize; s->strstart -= s->wsize; s->block_start -= (long)s->wsize; s->base += s->wsize;
            for (uint32_t i = 0; i < s->hsize; i++) s->head[i] = (uint16_t)(s->head[i] >= s->wsize ? s->head[i] - s->wsize : 0);
            for (uint32_t i = 0; i < s->wsize; i++) s->prev[i] = (uint16_t)(s->prev[i] >= s->wsize ? s->prev[i] - s->wsize : 0);
            more += s->wsize;
        }
        if (s->in_pos == s->in_len) break;
        uint32_t n = s->in_len - s->in_pos; if (n > more) n = more;
        memcpy(s->win + s->strstart + s->lookahead, s->in + s->in_pos, n);
        adler_feed(s, s->in + s->in_pos, n);
        s->in_pos += n; s->lookahead += n;
        if (s->lookahead >= MINM) { s->ins_h = s->win[s->strstart]; s->ins_h = ((s->ins_h << s->hshift) ^ s->win[s->strstart + 1]) & s->hmask; }
    } while (s->lookahead < MIN_LOOK && s->in_pos != s->in_len);
    /* bytes past the data are never allowed to influence output (Z/deflate.c:1496-1528); keep them zero */
    { uint32_t curr = s->strstart + s->lookahead, z = 2 * s->wsize - curr; if (z > MAXM) z = MAXM; memset(s->win + curr, 0, z); }
}
static uint32_t insert_str(zd_t *s, uint32_t pos) { /* INSERT_STRING Z/deflate.c:186-189 */
    s->ins_h = ((s->ins_h << s->hshift) ^ s->win[pos + 2]) & s->hmask;
    uint32_t h = s->prev[pos & s->wmask] = s->head[s->ins_h];
    s->head[s->ins_h] = (uint16_t)pos;
    return h;
}
static uint32_t find_longest(zd_t *s, uint32_t cur) { /* longest_match Z/deflate.c:1148-1289 */
    uint32_t chain = CFG[s->level].chain, maxd = s->wsize - MIN_LOOK;
    const uint8_t *scan = s->win + s->strstart;
    int best = (int)s->prev_len, nice = CFG[s->level].nice;
    uint32_t limit = s->strstart > maxd ? s->strstart - maxd : 0;
    if (s->prev_len >= CFG[s->level].good) chain >>= 2;
    if ((uint32_t)nice > s->lookahead) nice = (int)s->lookahead;
    do {
        const uint8_t *m = s->win + cur;
        if (m[best] != scan[best] || m[best - 1] != scan[best - 1] || m[0] != scan[0] || m[1] != scan[1]) continue;
        int len = 2; /* byte 2 equal by hash construction; compare up to MAXM as Z/deflate.c:1249-1258 */
        while (len < MAXM && scan[len] == m[len]) len++;
        if (len > best) { s->match_start = cur; best = len; if (len >= nice) break; }
    } while ((cur = s->prev[cur & s->wmask]) > limit && --chain != 0);
    return (uint32_t)best <= s->lookahead ? (uint32_t)best : s->lookahead;
}

static void run_stored(zd_t *s) { /* deflate_stored Z/deflate.c:1564-1619 (flush == Z_FINISH) */
    unsigned long max_block = 0xffff; if (max_block > s->pend_sz - 5) max_block = s->pend_sz - 5;
    uint32_t maxd = s->wsize - MIN_LOOK;
    for (;;) {
        if (s->lookahead <= 1) { refill(s); if (s->lookahead == 0) break; }
        s->strstart += s->lookahead; s->lookahead = 0;
        unsigned long max_start = (unsigned long)s->block_start + max_block;
        if (s->strstart == 0 || (unsigned long)s->strstart >= max_start) {
            s->lookahead = (uint32_t)(s->strstart - max_start); s->strstart = (uint32_t)max_start; flush_block(s, 0);
        }
        if (s->strstart - (uint32_t)s->block_start >= maxd) flush_block(s, 0);
    }
    flush_block(s, 1);
}
static void run_fast(zd_t *s) { /* deflate_fast Z/deflate.c:1628-1722 */
    uint32_t maxd = s->wsize - MIN_LOOK;
    for (;;) {
        if (s->lookahead < MIN_LOOK) { refill(s); if (s->lookahead == 0) break; }
        uint32_t hh = 0; int fl;
        if (s->lookahead >= MINM) hh = insert_str(s, s->strstart);
        if (hh != 0 && s->strstart - hh <= maxd) s->match_len = find_longest(s, hh);
        if (s->match_len >= MINM) {
            fl = tally(s, s->strstart - s->match_start, s->match_len - MINM);
            s->lookahead -= s->match_len;
            if (s->match_len <= CFG[s->level].lazy && s->lookahead >= MINM) {
                s->match_len--;
                do { s->strstart++; insert_str(s, s->strstart); } while (--s->match_len != 0);
                s->strstart++;
            } else {
                s->strstart += s->match_len; s->match_len = 0;
                s->ins_h = s->win[s->strstart]; s->ins_h = ((s->ins_h << s->hshift) ^ s->win[s->strstart + 1]) & s->hmask;
            }
        } else { fl = tally(s, 0, s->win[s->strstart]); s->lookahead--; s->strstart++; }
        if (fl) flush_block(s, 0);
    }
    flush_block(s, 1);
}
static void run_slow(zd_t *s) { /* deflate_slow Z/deflate.c:1730-1853 */
    uint32_t maxd = s->wsize - MIN_LOOK;
    for (;;) {
        if (s->lookahead < MIN_LOOK) { refill(s); if (s->lookahead == 0) break; }
        uint32_t hh = 0; int fl;
        if (s->lookahead >= MINM) hh = insert_str(s, s->strstart);
        s->prev_len = s->match_len; s->prev_match = s->match_start; s->match_len = MINM - 1;
        if (hh != 0 && s->prev_len < CFG[s->level].lazy && s->strstart - hh <= maxd) {
            s->match_len = find_longest(s, hh);
            if (s->match_len <= 5 && s->match_len == MINM && s->strstart - s->match_start > TOO_FAR_D) s->match_len = MINM - 1;
        }
        if (s->prev_len >= MINM && s->match_len <= s->prev_len) {
            uint32_t max_ins = s->strstart + s->lookahead - MINM;
            fl = tally(s, s->strstart - 1 - s->prev_match, s->prev_len - MINM);
            s->lookahead -= s->prev_len - 1; s->prev_len -= 2;
            do { if (++s->strstart <= max_ins) insert_str(s, s->strstart); } while (--s->prev_len != 0);
            s->match_avail = 0; s->match_len = MINM - 1; s->strstart++;
            if (fl) flush_block(s, 0);
        } else if (s->match_avail) {
            fl = tally(s, 0, s->win[s->strstart - 1]);
            if (fl) flush_block(s, 0); /* before strstart++, Z/deflate.c:1822-1826 */
            s->strstart++; s->lookahead--;
        } else { s->match_avail = 1; s->strstart++; s->lookahead--; }
    }
    if (s->match_avail) { tally(s, 0, s->win[s->strstart - 1]); s->match_avail = 0; }
    flush_block(s, 1);
}

/*
 * Whole-stream deflate.  Returns the zlib-stream length (even if > out_cap; then
 * only out_cap bytes were stored), or -1 on bad parameters.
 *   limit_out / in_at_limit: if limit_out != 0, *in_at_limit receives the number
 *   of plaintext bytes zlib had read when the first block flush left >= limit_out
 *   output bytes (the "--shortcut-len" stopping point, main.cpp:635-636).
 */
long long oracle_deflate(const uint8_t *in, uint32_t in_len, int level, int wbits, int memlevel,
                         uint8_t *out, uint64_t out_cap, uint64_t limit_out, uint32_t *in_at_limit) {
    if (level < 0 || level > 9 || wbits < 9 || wbits > 15 || memlevel < 1 || memlevel > 9) return -1;
    init_tables();
    zd_t *s = (zd_t *)calloc(1, sizeof(zd_t));
    s->in = in; s->in_len = in_len; s->out = out; s->out_cap = out_cap; s->limit_out = limit_out;
    s->level = level; s->wbits = wbits; s->memlevel = memlevel;
    s->wsize = 1u << wbits; s->wmask = s->wsize - 1;                     /* Z/deflate.c:284-291 */
    s->hbits = (uint32_t)memlevel + 7; s->hsize = 1u << s->hbits; s->hmask = s->hsize - 1; s->hshift = (s->hbits + MINM - 1) / MINM;
    s->litsz = 1u << (memlevel + 6); s->pend_sz = 4 * s->litsz;           /* Z/deflate.c:298-303 */
    s->win = (uint8_t *)calloc(2 * s->wsize + MAXM + 8, 1); s->prev = (uint16_t *)calloc(s->wsize, 2); s->head = (uint16_t *)calloc(s->hsize, 2);
    s->dbuf = (uint16_t *)malloc(2 * s->litsz); s->lbuf = (uint8_t *)malloc(s->litsz);
    s->match_len = s->prev_len = MINM - 1; s->adler_a = 1; s->adler_b = 0;   /* lm_init Z/deflate.c:1106-1132 */
    reset_block(s);
    /* zlib header, Z/deflate.c:738-754 */
    unsigned hdr = (8u + ((unsigned)(wbits - 8) << 4)) << 8;
    unsigned lf = level < 2 ? 0 : level < 6 ? 1 : level == 6 ? 2 : 3;
    hdr |= lf << 6; hdr += 31 - (hdr % 31);
    put8(s, hdr >> 8); put8(s, hdr & 0xff);
    if (CFG[level].kind == 0) run_stored(s); else if (CFG[level].kind == 1) run_fast(s); else run_slow(s);
    uint32_t ad = (s->adler_b << 16) | s->adler_a;                        /* trailer Z/deflate.c:967-968 */
    put8(s, ad >> 24); put8(s, (ad >> 16) & 0xff); put8(s, (ad >> 8) & 0xff); put8(s, ad & 0xff);
    if (in_at_limit) *in_at_limit = s->limit_hit ? s->in_at_limit : in_len;
    long long n = (long long)s->out_len;
    free(s->win); free(s->prev); free(s->head); free(s->dbuf); free(s->lbuf); free(s);
    return n;
}

uint32_t oracle_adler32(const uint8_t *p, uint64_t n) {
    zd_t t; t.adler_a = 1; t.adler_b = 0;
    while (n) { uint32_t k = n > (1u << 30) ? (1u << 30) : (uint32_t)n; adler_feed(&t, p, k); p += k; n -= k; }
    return (t.adler_b << 16) | t.adler_a;
}

/* =====================================================================================
 * DESIGN MODEL of the GPU algorithm (still test infrastructure; scalar, one candidate at
 * a time).  Same output as oracle_deflate(), but computed the way antiz_b200/csrc/deflate.cu
 * does it, so the equivalence argument of DESIGN.md ("list mode") is machine-checked on the
 * CPU against zlib 1.2.8 before any GPU time is spent:
 *   - no window copy, no head[]/prev[]: positions are absolute offsets into the plaintext;
 *   - per (plaintext, hash_bits) one bucket list = all positions sorted by (hash, position),
 *     idx[p] = slot of p in it, cnt[p] = number of earlier positions in p's bucket.  The hash
 *     chain zlib would walk from p is list[idx[p]-1], list[idx[p]-2], ... (levels 4-9 insert
 *     every position, Z/deflate.c:1757-1759,1806-1810); for levels 1-3 the same list filtered
 *     by a per-trial "inserted" map (Z/deflate.c:1680-1704 skips positions inside long matches);
 *   - the slide (Z/deflate.c:1419-1451) survives only as `base`, the absolute position of
 *     window index 0: it decides NIL (index 0 is never a match source), the `limit` of
 *     longest_match, and whether a block is still storable (block_start >= 0).
 * ===================================================================================== */
typedef struct { uint32_t *list, *idx; uint16_t *cnt; } chains_t;
static void build_chains(const uint8_t *in, uint32_t n, uint32_t hbits, chains_t *c) {
    uint32_t np = n >= 3 ? n - 2 : 0, hsize = 1u << hbits, hmask = hsize - 1, hshift = (hbits + 2) / 3;
    uint32_t *start = (uint32_t *)calloc(hsize + 1, 4), *fill = (uint32_t *)calloc(hsize, 4);
    c->list = (uint32_t *)malloc(4 * (np + 1)); c->idx = (uint32_t *)malloc(4 * (np + 1)); c->cnt = (uint16_t *)malloc(2 * (np + 1));
#define H3(p) ((((((uint32_t)in[p] << hshift) ^ in[(p) + 1]) << hshift) ^ in[(p) + 2]) & hmask)
    for (uint32_t p = 0; p < np; p++) start[H3(p) + 1]++;
    for (uint32_t h = 0; h < hsize; h++) start[h + 1] += start[h];
    for (uint32_t p = 0; p < np; p++) { uint32_t h = H3(p), r = fill[h]++; c->idx[p] = start[h] + r; c->cnt[p] = (uint16_t)(r > 65535 ? 65535 : r); c->list[start[h] + r] = p; }
#undef H3
    free(start); free(fill);
}
static void refill_abs(zd_t *s) {
    uint32_t maxd = s->wsize - MIN_LOOK;
    do {
        uint32_t more = s->base + 2 * s->wsize - s->wend;
        if (s->strstart - s->base >= s->wsize + maxd) { s->base += s->wsize; more += s->wsize; }
        if (s->wend == s->in_len) break;
        uint32_t n = s->in_len - s->wend; if (n > more) n = more;
        s->wend += n;
    } while (s->wend - s->strstart < MIN_LOOK && s->wend != s->in_len);
}
static uint32_t common_len(const uint8_t *in, uint32_t p, uint32_t q, uint32_t maxlen) { uint32_t l = 0; while (l < maxlen && in[p + l] == in[q + l]) l++; return l; }
/* chain walk; k0 = list slot of the head candidate, navail = candidates available at and below k0 */
static uint32_t find_longest_abs(zd_t *s, const chains_t *c, const uint8_t *insmap, uint32_t slot, uint32_t navail) {
    uint32_t p = s->strstart, look = s->wend - p, maxd = s->wsize - MIN_LOOK, prel = p - s->base;
    uint32_t chain = CFG[s->level].chain, nice = CFG[s->level].nice, best = s->prev_len;
    uint32_t limit = s->base + (prel > maxd ? prel - maxd : 0);
    uint32_t maxlen = look < MAXM ? look : MAXM;
    if (s->prev_len >= CFG[s->level].good) chain >>= 2;
    if (nice > look) nice = look;
    int first = 1;
    for (uint32_t k = 0; k < navail; k++) {
        uint32_t q = c->list[slot - k];
        if (insmap && !insmap[q]) { if (q <= limit) break; continue; }
        if (!first) { if (!(q > limit)) break; if (--chain == 0) break; }
        first = 0;
        uint32_t len = common_len(s->in, p, q, maxlen);
        if (len > best) { s->match_start = q; best = len; if (len >= nice) break; }
    }
    return best <= look ? best : look;
}
/* head of chain: most recent inserted earlier position with the same hash, or NIL (returns 0 = none) */
static int chain_head(zd_t *s, const chains_t *c, const uint8_t *insmap, uint32_t p, uint32_t *slot, uint32_t *navail, uint32_t *head) {
    uint32_t n = c->cnt[p], sl = c->idx[p], maxd = s->wsize - MIN_LOOK;
    for (uint32_t k = 1; k <= n; k++) {
        uint32_t q = c->list[sl - k];
        if (p - q > maxd) return 0;                 /* farther candidates only get older */
        if (insmap && !insmap[q]) continue;
        if (q <= s->base) return 0;                 /* window index 0 (or slid out) == NIL */
        *slot = sl - k; *navail = n - k + 1; *head = q; return 1;
    }
    return 0;
}
long long oracle_deflate_listmode(const uint8_t *in, uint32_t in_len, int level, int wbits, int memlevel, uint8_t *out, uint64_t out_cap) {
    if (level < 0 || level > 9 || wbits < 9 || wbits > 15 || memlevel < 1 || memlevel > 9) return -1;
    init_tables();
    zd_t *s = (zd_t *)calloc(1, sizeof(zd_t));
    s->abs_mode = 1; s->in = in; s->in_len = in_len; s->out = out; s->out_cap = out_cap; s->level = level;
    s->wsize = 1u << wbits; s->hbits = (uint32_t)memlevel + 7; s->litsz = 1u << (memlevel + 6); s->pend_sz = 4 * s->litsz;
    s->win = (uint8_t *)in; s->dbuf = (uint16_t *)malloc(2 * s->litsz); s->lbuf = (uint8_t *)malloc(s->litsz);
    s->match_len = s->prev_len = MINM - 1;
    reset_block(s);
    unsigned hdr = (8u + ((unsigned)(wbits - 8) << 4)) << 8, lf = level < 2 ? 0 : level < 6 ? 1 : level == 6 ? 2 : 3;
    hdr |= lf << 6; hdr += 31 - (hdr % 31); put8(s, hdr >> 8); put8(s, hdr & 0xff);
    uint32_t maxd = s->wsize - MIN_LOOK, n = in_len;
    if (CFG[level].kind == 0) {
        unsigned long max_block = 0xffff; if (max_block > s->pend_sz - 5) max_block = s->pend_sz - 5;
        for (;;) {
            if (s->wend - s->strstart <= 1) { refill_abs(s); if (s->wend == s->strstart) break; }
            s->strstart = s->wend;
            unsigned long max_start = (unsigned long)s->block_start + max_block;
            if ((unsigned long)s->strstart >= max_start) { s->strstart = (uint32_t)max_start; flush_block(s, 0); }
            if (s->strstart - (uint32_t)s->block_start >= maxd) flush_block(s, 0);
        }
        flush_block(s, 1);
    } else {
        chains_t c; build_chains(in, n, s->hbits, &c);
        uint8_t *insmap = CFG[level].kind == 1 ? (uint8_t *)calloc(n + 1, 1) : NULL;
        for (;;) {
            if (s->wend - s->strstart < MIN_LOOK) { refill_abs(s); if (s->wend == s->strstart) break; }
            uint32_t p = s->strstart, look = s->wend - p, slot = 0, navail = 0, head = 0; int have = 0, fl;
            if (look >= MINM) { have = chain_head(s, &c, insmap, p, &slot, &navail, &head); if (insmap) insmap[p] = 1; }
            if (CFG[level].kind == 1) {
                if (have) s->match_len = find_longest_abs(s, &c, insmap, slot, navail);
                if (s->match_len >= MINM) {
                    fl = tally(s, p - s->match_start, s->match_len - MINM);
                    look -= s->match_len;
                    if (s->match_len <= CFG[level].lazy && look >= MINM) {
                        s->match_len--;
                        do { s->strstart++; insmap[s->strstart] = 1; } while (--s->match_len != 0);
                        s->strstart++;
                    } else { s->strstart += s->match_len; s->match_len = 0; }
                } else { fl = tally(s, 0, in[p]); s->strstart++; }
                if (fl) flush_block(s, 0);
            } else {
                s->prev_len = s->match_len; s->prev_match = s->match_start; s->match_len = MINM - 1;
                if (have && s->prev_len < CFG[level].lazy) {
                    s->match_len = find_longest_abs(s, &c, NULL, slot, navail);
                    if (s->match_len == MINM && p - s->match_start > TOO_FAR_D) s->match_len = MINM - 1;
                }
                if (s->prev_len >= MINM && s->match_len <= s->prev_len) {
                    fl = tally(s, p - 1 - s->prev_match, s->prev_len - MINM);
                    s->strstart += s->prev_len - 1; s->match_avail = 0; s->match_len = MINM - 1;
                    if (fl) flush_block(s, 0);
                } else if (s->match_avail) {
                    fl = tally(s, 0, in[p - 1]);
                    if (fl) flush_block(s, 0);
                    s->strstart++;
                } else { s->match_avail = 1; s->strstart++; }
            }
        }
        if (s->match_avail) tally(s, 0, in[s->strstart - 1]);
        flush_block(s, 1);
        free(c.list); free(c.idx); free(c.cnt); free(insmap);
    }
    uint32_t ad = oracle_adler32(in, in_len);
    put8(s, ad >> 24); put8(s, (ad >> 16) & 0xff); put8(s, (ad >> 8) & 0xff); put8(s, ad & 0xff);
    long long r = (long long)s->out_len;
    free(s->dbuf); free(s->lbuf); free(s);
    return r;
}
