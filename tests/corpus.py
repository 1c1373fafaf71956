"""Seeded synthetic deflate-bearing containers (SURVEY.md 8d), built with zref.zlib_lib(): the reference's own zlib 1.2.8 where it
has been built, else the host's zlib and, at level 0, the oracle: the same bytes (Z_FIXED aside, where zlib 1.2.12 changed).
TEST / BENCH INFRASTRUCTURE ONLY."""
import random
import numpy as np
import zref

_JUNK_ALPHABET = np.frombuffer(b"abcdefgijklmnopqrstuvwyzABCDEFGIJKLMNOPQRSTUVWYZ01234567 9/<>[]{}%\n.-_", dtype=np.uint8)  # no ( 8 H X h x


def text(n, seed, nwords=3000):
    """word-list pseudo text: `nwords` random 2-9 letter words, space separated, 8 % newlines"""
    rng = np.random.default_rng(seed)
    r = random.Random(seed)
    words = [''.join(r.choice('abcdefghijklmnopqrstuvwxyz') for _ in range(r.randint(2, 9))) for _ in range(nwords)]
    need = n // 4 + 16
    idx = rng.integers(0, nwords, size=need)
    nl = rng.random(need) < 0.08
    parts = [words[i] + ('\n' if b else ' ') for i, b in zip(idx, nl)]
    s = ''.join(parts).encode()
    while len(s) < n:
        s += s
    return s[:n]


def binaryish(n, seed):
    """PNG-filter-like bytes: small signed deltas with runs"""
    rng = np.random.default_rng(seed)
    d = rng.integers(-3, 4, size=n, dtype=np.int64)
    d[rng.random(n) < 0.6] = 0
    return (np.cumsum(d) & 0xff).astype(np.uint8).tobytes()


def junk(n, seed):
    rng = np.random.default_rng(seed)
    return _JUNK_ALPHABET[rng.integers(0, len(_JUNK_ALPHABET), size=n)].tobytes()


def container(streams, seed, gap=(20, 200)):
    """streams: list of zlib streams -> (file bytes, [offsets])"""
    r = random.Random(seed)
    out = [junk(r.randint(100, 300), seed)]
    offs = []
    pos = len(out[0])
    for i, s in enumerate(streams):
        offs.append(pos)
        out.append(s); pos += len(s)
        g = junk(r.randint(*gap), seed * 7919 + i); out.append(g); pos += len(g)
    return b''.join(out), offs


def c1(seed=1234, n=1 << 20):
    """config 1: one 1 MiB text stream, level 6 / memLevel 8 / 32K window"""
    d = text(n, seed)
    return container([zref.ref_deflate(d, 6, 15, 8)], seed)[0]


def c2(nstreams=2000, seed=2, umin=1 << 10, umax=256 << 10):
    """config 2: PDF-like, levels 1-9, wbits 15, memLevel 8"""
    r = random.Random(seed)
    ss = []
    for i in range(nstreams):
        u = r.randint(umin, umax)
        ss.append(zref.ref_deflate(text(u, seed * 100003 + i), r.randint(1, 9), 15, 8))
    return container(ss, seed)[0]


def c3(nstreams=500, seed=3, umin=20_000, umax=200_000, filtered_frac=0.5):
    """config 3: PNG-style IDAT corpus, varied memLevel/windowBits, a fraction Z_FILTERED (no parameter set matches)"""
    r = random.Random(seed)
    ss = []
    for i in range(nstreams):
        u = r.randint(umin, umax)
        d = binaryish(u, seed * 100003 + i) if i % 2 else text(u, seed * 100003 + i)
        lvl, w, m = r.randint(1, 9), r.randint(10, 15), r.randint(1, 9)
        strat = 1 if (r.random() < filtered_frac and lvl >= 4) else 0
        ss.append(zref.ref_deflate(d, lvl, w, m, strat))
    return container(ss, seed)[0]


def c4(nstreams=50000, seed=4, umin=512, umax=8192):
    """config 4: JAR-like many small streams, levels {1,6,6,6,9}, defaults"""
    r = random.Random(seed)
    big = text(4 << 20, seed)
    ss = []
    for i in range(nstreams):
        u = r.randint(umin, umax); o = r.randint(0, len(big) - u)
        ss.append(zref.ref_deflate(big[o:o + u], r.choice([1, 6, 6, 6, 9]), 15, 8))
    return container(ss, seed, gap=(30, 120))[0]


def mixed(total_bytes, seed=5):
    """config 5 style: mix of c2/c3/c4-like streams up to ~total_bytes of container"""
    r = random.Random(seed)
    ss = []; size = 0; i = 0
    big = text(4 << 20, seed)
    while size < total_bytes:
        k = r.random(); i += 1
        if k < 0.4:
            u = r.randint(1 << 10, 256 << 10); s = zref.ref_deflate(text(u, seed * 100003 + i), r.randint(1, 9), 15, 8)
        elif k < 0.7:
            u = r.randint(20_000, 200_000); d = binaryish(u, seed * 100003 + i) if i % 2 else text(u, seed * 100003 + i)
            lvl = r.randint(1, 9); s = zref.ref_deflate(d, lvl, r.randint(10, 15), r.randint(1, 9), 1 if (r.random() < 0.5 and lvl >= 4) else 0)
        else:
            u = r.randint(512, 8192); o = r.randint(0, len(big) - u); s = zref.ref_deflate(big[o:o + u], r.choice([1, 6, 6, 6, 9]), 15, 8)
        ss.append(s); size += len(s) + 100
    return container(ss, seed)[0]


def fast_mix(nstreams=36, seed=61):
    """levels 1-3 at several sizes and memLevels, some made with another strategy (Z_FILTERED / Z_HUFFMAN_ONLY / Z_RLE /
    Z_FIXED): the original's tokens are then valid deflate but not what any deflate_fast trial produces"""
    r = random.Random(seed)
    ss = []
    for i in range(nstreams):
        u = r.choice([900, 2100, 5000, 30000, 70000, 150000])
        d = binaryish(u, seed * 100003 + i) if i % 3 == 2 else text(u, seed * 100003 + i, 300 if i % 2 else 3000)
        ss.append(zref.ref_deflate(d, r.randint(1, 3), 15, r.choice([8, 8, 9, 5]), r.choice([0, 0, 0, 1, 2, 3, 4])))
    return container(ss, seed)[0]


def extremes(seed=71):
    """streams at the ends of the expansion range: 8 MiB of zeros (ratio ~1000:1, outgrows every first-guess output region),
    incompressible bytes (stored blocks: no tokens to learn from), a level-0 stream, and ordinary text in between"""
    r = random.Random(seed)
    ss = [zref.ref_deflate(bytes(8 << 20), 6, 15, 8), zref.ref_deflate(r.randbytes(90000), 6, 15, 8), zref.ref_deflate(text(50000, seed), 0, 15, 8),
          zref.ref_deflate(text(120000, seed + 1), 9, 15, 8), zref.ref_deflate(r.randbytes(3000) + bytes(40000) + text(30000, seed + 2), 1, 15, 8)]
    return container(ss, seed)[0]


def imperfect(seed=101, small=False):
    """streams no plain parameter set reproduces exactly (SURVEY.md 8 a16: the diff list, incl. the tail bytes when the best trial's
    output is shorter than the original, main.cpp:699-715, and the reconstructor's patching, main.cpp:916-926):
      * a flush (Z_SYNC_FLUSH / Z_PARTIAL_FLUSH / Z_BLOCK) right before the end: the last block loses its BFINAL bit and an empty block
        follows - one differing byte plus a tail the trial does not have (C' < C);
      * the same flush a little before the end: the last bytes are parsed in a block of their own;
      * deflateTune'd encoders and flushes in the middle (small streams: with --recomp-tresh / --sizediff-tresh raised they are
        recompressed with long diff lists, either sign of C' - C)."""
    r = random.Random(seed)
    ss = []
    for i in range(28 if not small else 40):
        u = r.randint(600, 3000) if small else r.choice([900, 2500, 7000, 30000, 90000, 200000])
        d = binaryish(u, seed * 100003 + i) if i % 4 == 3 else text(u, seed * 100003 + i, 300 if i % 2 else 3000)
        lvl, w, m = r.randint(1, 9), (15 if i % 3 else r.randint(10, 15)), (8 if i % 3 else r.randint(1, 9))
        kind = i % 7
        if small:
            if kind < 3:
                s = zref.ref_deflate_ex(d, lvl, w, m, tune=r.choice([(4, 4, 8, 2), (8, 16, 64, 64), (32, 258, 258, 300), (4, 6, 16, 16)]))
            elif kind < 5:
                s = zref.ref_deflate_ex(d, lvl, w, m, flushes=[(r.randint(u // 3, 2 * u // 3), r.choice([1, 2, 5]))])
            else:
                s = zref.ref_deflate_ex(d, lvl, w, m, flushes=[(u, r.choice([1, 2]))])
        else:
            if kind < 3:
                s = zref.ref_deflate_ex(d, lvl, w, m, flushes=[(u, r.choice([1, 2, 5]))])
            elif kind < 5:
                s = zref.ref_deflate_ex(d, lvl, w, m, flushes=[(u - r.randint(1, 40), r.choice([1, 2, 5]))])
            elif kind == 5:
                s = zref.ref_deflate_ex(d, lvl, w, m, flushes=[(u - r.randint(2, 30), 2), (u, 1)])
            else:
                s = zref.ref_deflate(d, lvl, w, m)
        ss.append(s)
    return container(ss, seed)[0]


def at_chunk_starts(S=5000, seed=91, nchunks=9):
    """streams (and bare header pairs) placed exactly on the chunk starts k(S-1), and one byte either side of them: the reference's
    reader keeps the wrong overlap byte from chunk 1 on (searchInfile, main.cpp:408-413: `rBuffer[f.gcount() - 1]`), so the first
    position of chunk k >= 2 is compared and inflated with file[start - 1] in place of file[start]; a stream that starts exactly
    there is missed (unless the byte before it happens to be its own first byte), one that starts a byte later is found, and a header
    pair split around the boundary can appear where the file has none"""
    r = random.Random(seed)
    out = bytearray()
    for k in range(1, nchunks):
        start = k * (S - 1) + r.choice([0, 0, 0, 1, -1])
        if len(out) > start:
            continue
        out += junk(start - len(out), seed * 31 + k)
        mode = k % 4
        if mode == 3:      # the byte before the boundary repeats the stream's first byte: found even with the wrong overlap byte
            out[-1:] = b"\x78"
        z = zref.ref_deflate(text(r.randint(200, 2 * S), seed * 77 + k, 300), r.choice([1, 6, 9]), 15, 8)
        if mode == 2:      # a header pair split around the boundary position: (file[start - 1], file[start + 1])
            out[-1:] = b"\x78"; out += b"Q\x9c" + junk(40, seed + k)
        out += z
    out += junk(300, seed)
    return bytes(out)
