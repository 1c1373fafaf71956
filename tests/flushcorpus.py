"""Seeded inputs that drive zlib 1.2.8's block flush (_tr_flush_block, build_tree, gen_bitlen, scan_tree) into the branches that
ordinary text and binary inputs do not reach, and a small deflate token decoder that shows what a stream's blocks hold.
Which branch an input reaches is measured with the CPU oracle's branch counters (zref.oracle_flush_counts), in
test_flush_coverage.py.  TEST INFRASTRUCTURE ONLY."""
import random

import numpy as np

LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LXB = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DXB = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
BLORD = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


# ---------------------------------------------------------------------------------------------------------------------------------
# token decoder
class _Bits:
    def __init__(self, b, pos):
        self.b, self.p = b, pos

    def get(self, n):
        v = 0
        for i in range(n):
            v |= ((self.b[self.p >> 3] >> (self.p & 7)) & 1) << i
            self.p += 1
        return v


def _canon(lens):
    count = [0] * 16
    for n in lens:
        if n:
            count[n] += 1
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1
        nxt[b] = code
    t = {}
    for s, n in enumerate(lens):
        if n:
            t[(n, nxt[n])] = s
            nxt[n] += 1
    return t


def _sym(br, t):
    c = 0
    for n in range(1, 16):
        c = (c << 1) | br.get(1)
        if (n, c) in t:
            return t[(n, c)]
    raise ValueError("invalid code")


_FIXED_L = _canon([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8)
_FIXED_D = _canon([5] * 30)


def blocks(z):
    """Blocks of a zlib stream, in order: dicts with `type` (0 stored, 1 static, 2 dynamic), `start`/`end` (bit offsets in z of the block
    header and of the bit after END_BLOCK), and for dynamic blocks `header_end` (bit offset of the first symbol) and `lengths` (the
    code lengths sent); `lit` (286 counts: literals, END_BLOCK, length codes) and `dist` (30 counts) for compressed blocks."""
    br = _Bits(z, 16)
    out = []
    while True:
        blk = dict(start=br.p)
        last = br.get(1)
        blk["type"] = bt = br.get(2)
        if bt == 0:
            br.p = (br.p + 7) & ~7
            n = br.get(16)
            br.get(16)
            br.p += 8 * n
        else:
            if bt == 2:
                hl, hd, hc = br.get(5) + 257, br.get(5) + 1, br.get(4) + 4
                cl = [0] * 19
                for i in range(hc):
                    cl[BLORD[i]] = br.get(3)
                ct = _canon(cl)
                lens = []
                while len(lens) < hl + hd:
                    s = _sym(br, ct)
                    if s < 16:
                        lens.append(s)
                    elif s == 16:
                        lens += [lens[-1]] * (3 + br.get(2))
                    elif s == 17:
                        lens += [0] * (3 + br.get(3))
                    else:
                        lens += [0] * (11 + br.get(7))
                lt, dt = _canon(lens[:hl]), _canon(lens[hl:])
                blk.update(header_end=br.p, lengths=lens, hlit=hl)
            else:
                lt, dt = _FIXED_L, _FIXED_D
            lh, dh = np.zeros(286, np.int64), np.zeros(30, np.int64)
            while True:
                s = _sym(br, lt)
                lh[s] += 1
                if s == 256:
                    break
                if s > 256:
                    br.get(LXB[s - 257])
                    c = _sym(br, dt)
                    dh[c] += 1
                    br.get(DXB[c])
            blk.update(lit=lh, dist=dh)
        blk["end"] = br.p
        out.append(blk)
        if last:
            return out


def max_code_length(blk, kind):
    """longest code of a dynamic block's literal/length (kind 0) or distance (kind 1) tree"""
    lens = blk["lengths"]
    return max(lens[:blk["hlit"]] if kind == 0 else lens[blk["hlit"]:])


# ---------------------------------------------------------------------------------------------------------------------------------
# generators
def _unique_trigram_bytes(n, r):
    """n random bytes in which no 3-byte string occurs twice: deflate finds no match in them"""
    seen = set()
    d = bytearray(r.randbytes(2))
    while len(d) < n:
        b = r.randrange(256)
        t = (d[-2], d[-1], b)
        if t not in seen:
            seen.add(t)
            d.append(b)
    return d


def lit_overflow(memlevel, seed, ncodes=17):
    """A literal/length tree deeper than 15 bits in the last block.

    Blocks of lit_bufsize - 1 = 2^(memLevel+6) - 1 literals with no repeated 3-byte string (so no matches) fill the first ~32 KB; the
    last block then holds only copies of 4+ bytes out of them, one per token, with the counts 1, 2, 3, 5, 8, ... 1597 on the length
    codes 258.. (END_BLOCK is the chain's first 1).  Those Fibonacci weights make a Huffman chain one level deeper per code: 17 leaves,
    depth 16.  A byte is skipped between copied sources, chosen so that no match runs on into the next copy.

    memLevel 6 and below cannot overflow this tree: a block holds at most 4,095 symbols plus END_BLOCK, and a Huffman tree with a
    16-bit code needs a total weight of at least 1+1+2+...+987+1597 = 4,180.  Level 1 does not reach it either: its 4-entry chain walk
    misses some of the sources, and the literals that replace those copies break the chain."""
    r = random.Random(seed)
    per = (1 << (memlevel + 6)) - 1
    P = per * (32767 // per)
    d = _unique_trigram_bytes(P, r)
    counts = [1, 2]
    while len(counts) < ncodes - 1:
        counts.append(counts[-1] + counts[-2])
    toks = [c + 1 for c, k in enumerate(counts[::-1]) for _ in range(k)]    # heaviest count on the shortest length (4)
    r.shuffle(toks)
    a = P - sum(LBASE[c] + 1 for c in toks) - 64
    assert a >= 0 and P - a <= 32506, (P, a)
    for c in toks:
        L = LBASE[c]
        d += d[a:a + L]
        a += L + 1
        while d[a] == d[a - 1]:     # the byte after this source differs from the next copy's first byte
            a += 1
    return bytes(d)


DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193,
         12289, 16385, 24577]


def dist_overflow(seed, tail=b""):
    """A distance tree deeper than 15 bits in the last block (memLevel 9).

    One block of 32,767 literals with no repeated 3-byte string comes first.  The last block then holds 4,180 tokens, each five fresh
    literals and a copy of 4 bytes, with the Fibonacci counts 1, 1, 2, 3, ... 987, 1597 on the distance codes 13-29 (heaviest on code
    29): a 17-leaf chain, depth 16.  A copy's source is 4 fresh bytes not copied from before, taken first-fit inside its code's distance
    range (code 29 capped at 31,000, below MAX_DIST = 32,506), so that zlib finds it at exactly that distance.  Every 3-byte string
    that starts at a fresh byte or spans a copy's edge is new, and the literal after a copy differs from the byte after its source, so
    no match starts early or runs on.  The codes come in an order that meets each one's last usable position.

    memLevel 9 only: the last block holds 25,080 symbols.  memLevel 6 and below cannot overflow a distance tree at all (a block holds at
    most 4,095 matches, and a 16-bit code needs a total weight of 1+1+2+...+1597 = 4,180); memLevels 7 and 8 are not reached here.

    With a `tail`, fresh literals fill the repaired block to its 32,767 symbols and `tail` follows in a block of its own."""
    r = random.Random(seed)
    P = 32767
    d = _unique_trigram_bytes(P, r)
    seen = {bytes(d[i:i + 3]) for i in range(P - 2)}
    free = bytearray(b"\1" * P)                # fresh bytes not yet copied from
    counts = [1, 1]
    while len(counts) < 17:
        counts.append(counts[-1] + counts[-2])
    cnt = {13 + i: k for i, k in enumerate(counts)}
    L, K = 4, 5
    after = -1
    for c in [c for c in list(range(13, 27)) + [29, 27, 28] for _ in range(cnt[c])]:
        for k in range(K):                      # fresh literals
            while True:
                g = r.randrange(256)
                t = bytes([d[-2], d[-1], g])
                if t not in seen and not (k == 0 and g == after):
                    break
            seen.add(t)
            d.append(g)
            free.append(1)
        pos = len(d)
        lo, hi = DBASE[c], min(DBASE[c] + (1 << DXB[c]) - 1, 31000)
        s = next(s for s in range(pos - hi, pos - lo + 1)
                 if all(free[s:s + L]) and bytes([d[-2], d[-1], d[s]]) not in seen and bytes([d[-1], d[s], d[s + 1]]) not in seen)
        free[s:s + L] = bytes(L)
        seen.update((bytes([d[-2], d[-1], d[s]]), bytes([d[-1], d[s], d[s + 1]])))
        after = d[s + L]
        d += d[s:s + L]
        free += bytes(L)
    if tail:
        for _ in range(P - 6 * sum(counts)):
            while True:
                g = r.randrange(256)
                t = bytes([d[-2], d[-1], g])
                if t not in seen and g != after:
                    break
            seen.add(t)
            d.append(g)
            after = -1
        d += tail
    return bytes(d)


def forced_lit():
    """literal trees with no symbol besides END_BLOCK (empty blocks: build_tree forces two codes) and with one"""
    return [b"", b"x", b"\0" * 3, bytes(1000), b"ab" * 2000]


def single_distance_code(seed):
    """blocks whose distance tree has one code, 0 (distance 1: a run), 1 (distance 2) or >= 2 (3, 7, 200): build_tree forces a second
    code, code 1 when max_code < 2 and code 0 otherwise"""
    r = random.Random(seed)
    out = []
    for period in (1, 2, 3, 7, 200):
        unit = r.randbytes(period)
        out.append(r.randbytes(5) + unit * (3000 // period))
    return out


def stored_ties(seed, n=40):
    """short random inputs, short texts and repeated random units: stored, static and dynamic sizes within a few bytes of each other,
    so that some blocks tie at stored_len + 4 == opt_lenb (a stored block is written)"""
    r = random.Random(seed)
    out = []
    for i in range(n):
        k = r.randrange(3)
        if k == 0:
            out.append(r.randbytes(r.randint(5, 400)))
        elif k == 1:
            out.append(bytes(r.choice(b"abcdefgh ") for _ in range(r.randint(10, 300))))
        else:
            out.append(r.randbytes(r.randint(2, 60)) * r.randint(1, 4))
    return out


def static_ties(n=16):
    """4,000-byte word texts: at memLevel 1 and 2 (blocks of 127 and 255 symbols) the static and dynamic block sizes are close, and
    some blocks tie at static_lenb == opt_lenb (a static block is written)"""
    import corpus
    return [corpus.text(4000, i, 300) for i in range(n)]


def slid_blocks(seed, wbits):
    """blocks that start more than a window before they end, after a slide: not storable (buf == NULL).  Incompressible bytes with a
    few repeats make blocks of lit_bufsize - 1 symbols longer than the window of 512 or 1,024 bytes."""
    r = random.Random(seed)
    ws = 1 << wbits
    d = bytearray(r.randbytes(6 * ws))
    for p in range(0, len(d) - 64, 97):
        src = r.randrange(max(0, p - ws // 2), p) if p else 0
        d[p:p + 8] = d[src:src + 8]
    return bytes(d)


def length_runs(seed):
    """code-length sequences at scan_tree's limits: a repeat of 6 (code 16), zero runs of exactly 3, 10, 11 and 138 (codes 17, 18)
    and of 139 (split), made from which literals are present"""
    r = random.Random(seed)
    out = []
    for gap in (3, 10, 11, 138, 139, 150):
        lits = [0x20 + i for i in range(7)] + [0x20 + 7 + gap + i for i in range(6)]
        lits = [x for x in lits if x < 256]
        out.append(bytes(r.choice(lits) for _ in range(3000)))
    return out
