"""-m gpu: ATZ_SCAN_PNG_IDAT (uncomp --png).  PNG encoders split an image's zlib stream over consecutive IDAT chunks; with the flag the
scan finds such a stream over its IDAT run, the search recompresses it like any other, and the ATZ file keeps the 12 framing bytes
between its pieces.  PNGs are written here (signature, IHDR, ancillary chunks, IDAT run, IEND) around zlib's own streams."""
import hashlib
import os
import random
import struct
import subprocess
import tempfile
import zlib

import pytest

import antiz_b200 as az
import corpus
import zref
from test_png_idat import chunk, py_run

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")
PNG = az.ATZ_SCAN_PNG_IDAT
SW = az.ATZ_SCAN_SMALL_WINDOWS
TMP = "/dev/shm" if os.path.isdir("/dev/shm") else None


def idat_sizes(c, kind, r):
    """chunk sizes for a c-byte zlib stream: a fixed size, "random", or "zero" (1000-byte chunks with a zero-length one after the first)"""
    if kind == "random":
        out = []
        while sum(out) < c:
            out.append(r.randint(1, 20000))
        out[-1] -= sum(out) - c
        return out
    if kind == "zero":
        out = idat_sizes(c, 1000, r)
        return out[:1] + [0] + out[1:]
    return [kind] * (c // kind) + ([c % kind] if c % kind else [])


def png_image(z, sizes, seed, idat_extra=b"", after=b"", bad_crc=False):
    """a PNG around zlib stream z (+ idat_extra, bytes behind it in the IDAT data) in IDATs of `sizes` (their sum: len(z + idat_extra));
    `after`: chunks between the IDATs and IEND.  Returns (bytes, offset of the first IDAT's data)"""
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", 97 + seed % 50, 64, 8, 0, 0, 0, 0))
    out += chunk(b"gAMA", struct.pack(">I", 45455)) + chunk(b"tEXt", b"Software\0pytest %d" % seed)
    first = len(out) + 8
    body, at = z + idat_extra, 0
    assert sum(sizes) == len(body)
    for k, s in enumerate(sizes):
        c = chunk(b"IDAT", body[at:at + s]); at += s
        if bad_crc and k == 0:
            c = c[:-4] + bytes(b ^ 0x5a for b in c[-4:])
        out += c
    return out + after + chunk(b"IEND", b""), first


def cut(lens, c):
    """the pieces of a c-byte stream over chunks of lengths `lens`"""
    out, got = [], 0
    for n in lens:
        if got >= c:
            break
        out.append(min(n, c - got)); got += out[-1]
    return out


def plain(u, seed):
    return corpus.binaryish(u, seed) if seed % 2 else corpus.text(u, seed)


class Corpus:
    """PNGs among junk and ordinary zlib streams; pngs[i] = (offset of the header, C, zlib stream, pieces or None for a single IDAT, strategy,
    header bytes)"""

    def __init__(self, seed, n=20, strategies=(0,), small=False, sizes=(8192, 65536, 1000, "random", "zero"), umax=60000):
        r = random.Random(seed)
        items, meta = [], []
        for k in range(n):
            d = plain(r.randint(3000, umax), seed * 1000 + k)
            lvl, w, m = r.randint(1, 9), r.choice([15, 15, 12, 10]), r.randint(1, 9)
            st = strategies[k % len(strategies)]
            if st == 1:
                lvl = max(lvl, 4)
            if small and k % 3 == 1:
                w = 9
            z = zref.ref_deflate(d, lvl, w, m, st)
            if small and k % 6 == 4:
                flg = z[1] & 0xc0
                z = bytes([0x08, flg | (31 - ((0x0800 | flg) % 31)) % 31]) + z[2:]      # CINFO 0 rewrite of a window-9 stream
            sz = idat_sizes(len(z), sizes[k % len(sizes)], r)
            img, first = png_image(z, sz, seed * 100 + k)
            items.append(img); meta.append((first, z, sz, st))
            if k % 3 == 0:     # an ordinary zlib stream in between
                items.append(zref.ref_deflate(plain(r.randint(500, 30000), seed * 7 + k), r.randint(1, 9), 15, 8)); meta.append(None)
        self.data, offs = corpus.container(items, seed)
        self.pngs = []
        for off, mt in zip(offs, meta):
            if mt:
                first, z, sz, st = mt
                p = off + first
                multi = len([x for x in sz if x]) > 1
                self.pngs.append((p, len(z), z, cut(py_run(self.data, p), len(z)) if multi else None, st))

    def spans(self):
        return [(p, p + c + 12 * (len(pc) - 1)) for p, c, z, pc, st in self.pngs if pc]


def rec(s):
    return (s.offset, s.streamLength, s.inflatedLength, s.offsetType, s.clevel, s.window, s.memlevel, s.identBytes, s.recomp, s.ndiff, s.firstDiffByte)


def run(data, flags, opt=None, chunksize=524288, env=None):
    """(records, diffs, pieces) of one context"""
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update({k: str(v) for k, v in (env or {}).items()})
    try:
        c = az.Context(0)
        if flags:
            c.set_scan_flags(flags)
        c.load(data); n = c.scan(chunksize); c.search(opt or az.Options())
        ss = c.streams()
        out = ([rec(s) for s in ss], c.diffs(), [c.pieces(i) for i in range(n)])
        c.close()
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
    return out


def outside(recs, spans):
    return [x for x in recs if not any(a <= x[0] < b for a, b in spans)]


@pytest.fixture(scope="module")
def base():
    return Corpus(11)


# ---------------------------------------------------------------------------------------------------------------------------------
def test_flag_off_unchanged(base):
    """without the flag no stream starts at a multi-IDAT run and the .atz is the reference's where its binary exists"""
    recs, _, pieces = run(base.data, 0)
    starts = {p for p, c, z, pc, st in base.pngs if pc}
    assert len(starts) >= 10 and not starts & {x[0] for x in recs}
    assert all(pc == [] for pc in pieces)
    if os.path.exists(zref.REF_BIN):
        with tempfile.TemporaryDirectory(dir=TMP) as tmp:
            f = os.path.join(tmp, "in.bin"); open(f, "wb").write(base.data)
            a = subprocess.run([UNCOMP, "-i", f, "-o", f + ".a", "--notest"], capture_output=True)
            b = subprocess.run([zref.REF_BIN, "-i", f, "-o", f + ".b", "--notest"], capture_output=True)
            assert a.returncode == 0 and b.returncode == 0 and open(f + ".a", "rb").read() == open(f + ".b", "rb").read()


def check_pngs(cp, recs, pieces, want):
    by = {x[0]: (x, pc) for x, pc in zip(recs, pieces)}
    n = 0
    for p, c, z, pc, st in cp.pngs:
        if pc and want(st, z):
            x, got = by[p]
            # exact for zlib's default strategy (a CINFO 0 header: its two bytes are diffs); another strategy's winner may be a full match
            # within --mismatch-tol 2
            exact = c - (2 if z[0] == 0x08 else 0)
            assert x[1] == c and (x[7] == exact if st == 0 else x[7] + 2 >= c) and x[8] == 1, (p, x)
            assert got == pc, (p, got[:4], pc[:4])
            n += 1
        elif not pc:
            assert by[p][1] == [] if p in by else True
    return n


def test_png_records(base):
    """--png: every multi-IDAT default-strategy PNG is recompressed exactly with the parser's pieces; ordinary streams keep their records"""
    off = run(base.data, 0)[0]
    recs, _, pieces = run(base.data, PNG)
    assert check_pngs(base, recs, pieces, lambda st, z: True) >= 10
    assert outside(recs, base.spans()) == outside(off, base.spans())
    # single-IDAT PNGs are ordinary streams, found with and without the flag
    singles = {p for p, c, z, pc, st in base.pngs if not pc}
    assert singles and singles <= {x[0] for x in off} and all(pc == [] for x, pc in zip(recs, pieces) if x[0] in singles)


@pytest.mark.parametrize("gpus", [1, 2, 4])
def test_uncomp_png_round_trip(base, gpus):
    """uncomp --png: the self-test passes, uncomp -r restores the input, and --gpus N (contexts sharing a device where there are fewer)
    writes the same file as --gpus 1"""
    import torch
    env = dict(os.environ)
    if torch.cuda.device_count() < gpus:
        env["ATZ_TEST_ONE_DEVICE"] = "1"
    with tempfile.TemporaryDirectory(dir=TMP) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(base.data)
        p = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--png", "--chunksize", "65536", "--gpus", str(gpus)], capture_output=True, text=True, env=env)
        assert p.returncode == 0 and "OK! Restoration is bit by bit identical" in p.stdout, p.stdout + p.stderr
        rec = subprocess.run([UNCOMP, "-r", "-i", f + ".atz", "-o", f + ".rec"], capture_output=True, text=True)
        assert rec.returncode == 0 and open(f + ".rec", "rb").read() == base.data
        if gpus > 1:
            one = subprocess.run([UNCOMP, "-i", f, "-o", f + ".g1", "--png", "--chunksize", "65536", "--notest"], capture_output=True, text=True)
            assert one.returncode == 0
            h = lambda q: hashlib.sha256(open(q, "rb").read()).hexdigest()
            assert h(f + ".g1") == h(f + ".atz")


@pytest.mark.parametrize("combo", ["strategies", "small-windows", "brute-window"])
def test_png_combinations(combo):
    """--png with --strategies recompresses the Z_FILTERED PNGs too; with --small-windows the window-9 and CINFO 0 bodies; --brute-window"""
    if combo == "strategies":
        cp = Corpus(21, n=12, strategies=(0, 1), sizes=(8192, 1000, "random"))
        recs, _, pieces = run(cp.data, PNG, az.Options(flags=az.ATZ_F_STRATEGIES))
        assert check_pngs(cp, recs, pieces, lambda st, z: True) >= 8
        assert any(st == 1 and pc for p, c, z, pc, st in cp.pngs)
        args = ["--strategies"]
    elif combo == "small-windows":
        cp = Corpus(22, n=12, small=True, sizes=(1000, 4096, "random"))
        recs, _, pieces = run(cp.data, PNG | SW)
        assert check_pngs(cp, recs, pieces, lambda st, z: True) >= 8
        assert sum(1 for p, c, z, pc, st in cp.pngs if pc and z[0] in (0x08, 0x18)) >= 4
        args = ["--small-windows"]
    else:
        cp = Corpus(23, n=8, sizes=(8192, "zero"))
        recs, _, pieces = run(cp.data, PNG, az.Options(bruteforceWindow=True))
        assert check_pngs(cp, recs, pieces, lambda st, z: True) >= 5
        args = ["--brute-window"]
    with tempfile.TemporaryDirectory(dir=TMP) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(cp.data)
        p = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--png"] + args, capture_output=True, text=True)
        assert p.returncode == 0 and "OK! Restoration is bit by bit identical" in p.stdout, p.stdout + p.stderr


# ---------------------------------------------------------------------------------------------------------------------------------
def edge_corpus():
    r = random.Random(31)
    items, cases = [], {}

    def add(name, img, first, **kw):
        cases[name] = (len(items), first, kw); items.append(img)

    z = zref.ref_deflate(plain(20000, 1), 6, 15, 8)
    add("ends_in_first", *png_image(z, [len(z) + 7, 300], 1, idat_extra=bytes(range(7)) + bytes(300)))
    z = zref.ref_deflate(plain(30000, 3), 6, 15, 8)
    img, first = png_image(z, idat_sizes(len(z), 2000, r), 2)
    g = bytearray(img); g[first + 2000 + 12 + 700] ^= 0x10
    add("bitflip", bytes(g), first)
    z = zref.ref_deflate(plain(25000, 4), 9, 15, 9)
    add("bad_crc", *png_image(z, idat_sizes(len(z), 3000, r), 3, bad_crc=True), want=len(z))
    z = zref.ref_deflate(plain(25000, 5), 5, 13, 7)
    sz = idat_sizes(len(z) + 10, 4096, r)
    add("trailing", *png_image(z, sz, 4, idat_extra=b"TRAILING!!", after=chunk(b"IDAT", b"extra idat") + chunk(b"IDAT", bytes(50))), want=len(z))
    inner, _ = png_image(z, idat_sizes(len(z), 2048, r), 5)
    add("in_level0", zref.ref_deflate(b"prefix" + inner + b"suffix", 0, 15, 8), 0, outer=True)
    d = plain(40000, 7)
    zs = zref.ref_deflate_ex(d, 6, 15, 8, flushes=[(len(d) - 25, 2)])
    add("sync_flush", *png_image(zs, idat_sizes(len(zs), 8192, r), 6), want=len(zs), sync=True)
    big = random.Random(8).randbytes(2 << 20) + plain(1 << 20, 9)
    zb = zref.ref_deflate(big, 6, 15, 8)
    assert len(zb) >= 2 << 20
    add("big", *png_image(zb, idat_sizes(len(zb), 8192, r), 7), want=len(zb))
    data, offs = corpus.container(items, 32)
    out = {name: (offs[i] + first, kw) for name, (i, first, kw) in cases.items()}
    out["_item_ranges"] = {name: (offs[i], offs[i] + len(items[i])) for name, (i, first, kw) in cases.items()}
    return data, out


def test_png_edge_cases():
    data, cs = edge_corpus()
    rng = cs["_item_ranges"]
    opt = az.Options(recompTresh=400)      # (below --shortcut-len 512: above it every trial of a longer stream bails, main.cpp:649)
    off = run(data, 0, opt)
    on = run(data, PNG, opt)
    by_on = {x[0]: (x, pc) for x, pc in zip(on[0], on[2])}
    within = lambda recs, name: [x for x in recs if rng[name][0] <= x[0] < rng[name][1]]
    # a stream that ends inside the first of two IDATs keeps its record; a bit flip in piece 2 leaves the PNG as it is without the flag
    p = cs["ends_in_first"][0]
    assert p in {x[0] for x in off[0]} and within(on[0], "ends_in_first") == within(off[0], "ends_in_first") and by_on[p][1] == []
    assert within(on[0], "bitflip") == within(off[0], "bitflip")
    # wrong CRC, trailing bytes + extra IDATs, mid-stream Z_SYNC_FLUSH, a 2 MB run: split streams of the stream's own length
    for name in ("bad_crc", "trailing", "sync_flush", "big"):
        p, kw = cs[name]
        x, pc = by_on[p]
        assert x[1] == kw["want"] and x[8] == 1 and len(pc) >= 2 and sum(pc) == kw["want"], (name, x)
    assert cs["trailing"][0] + cs["trailing"][1]["want"] + 12 * (len(by_on[cs["trailing"][0]][1]) - 1) < rng["trailing"][1] - 12 - 30
    x = by_on[cs["sync_flush"][0]][0]
    assert x[9] > 0, x        # diffs, in de-chunked coordinates (the round trip below checks them)
    assert len(by_on[cs["big"][0]][1]) >= 256
    # a PNG inside a level-0 stream: the outer stream is kept, nothing is split inside it
    o = rng["in_level0"][0]
    assert o in by_on and by_on[o][0] == next(y for y in off[0] if y[0] == o) and within(on[0], "in_level0") == [by_on[o][0]]
    with tempfile.TemporaryDirectory(dir=TMP) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        pr = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--png", "--recomp-tresh", "400"], capture_output=True, text=True)
        assert pr.returncode == 0 and "OK! Restoration is bit by bit identical" in pr.stdout, pr.stdout + pr.stderr
        rec = subprocess.run([UNCOMP, "-r", "-i", f + ".atz", "-o", f + ".rec"], capture_output=True, text=True)
        assert rec.returncode == 0 and open(f + ".rec", "rb").read() == data


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nsh,chunksize", [(2, 524288), (3, 65536), (4, 20000), (5, 5000)])
def test_sharded_png_equal_single(base, nsh, chunksize):
    """2..5 emulated shards (runs across shard boundaries): the same stream list, records, diffs and pieces as one context"""
    opt = az.Options(flags=az.ATZ_F_EXACT_RECORDS)
    one = az.Context(0); one.set_scan_flags(PNG); one.load(base.data); n1 = one.scan(chunksize); one.search(opt)
    want = [rec(s) for s in one.streams()]; wd = one.diffs(); wp = [one.pieces(i) for i in range(n1)]
    one.close()
    assert sum(1 for pc in wp if pc) >= 10
    ctxs = [az.Context(0) for _ in range(nsh)]
    for g, c in enumerate(ctxs):
        c.set_scan_flags(PNG); c.attach(base.data); c.scan_shard(chunksize, g, nsh)
    blobs = [c.probe_export() for c in ctxs]
    for g, c in enumerate(ctxs):
        for h in range(nsh):
            if h != g:
                c.probe_import(h, blobs[h])
        assert c.scan_finish() == n1
    for g, c in enumerate(ctxs):
        c.search(opt, g, nsh)
        assert [c.pieces(i) for i in range(n1)] == wp
    own = ctxs[0].owners(); got = []; offs = []; vals = b""
    for i in range(n1):
        c = ctxs[own[i]]; s = c.streams()[i]
        got.append(rec(s))
        o, v = c.diffs()
        offs += list(o[s.diff_index:s.diff_index + s.ndiff]); vals += bytes(v[s.diff_index:s.diff_index + s.ndiff])
    assert got == want and (offs, vals) == (list(wd[0]), bytes(wd[1]))
    for c in ctxs:
        c.close()


def test_png_flag_state_and_shard_mismatch():
    """the PNG flag is known and ORs with the small windows (bits 2 and 8 stay unknown); the flags are fixed by the first load; shards
    that scanned with other flags refuse each other's records"""
    c = az.Context(0)
    for bad in (2, 8, PNG | 8):
        with pytest.raises(az.AtzError) as e:
            c.set_scan_flags(bad)
        assert e.value.code == az.ATZ_E_ARG
    c.set_scan_flags(SW); c.set_scan_flags(PNG | SW); c.set_scan_flags(PNG)
    c.load(b"x" * 1000)
    with pytest.raises(az.AtzError) as e:
        c.set_scan_flags(0)
    assert e.value.code == az.ATZ_E_STATE
    c.close()
    data = Corpus(41, n=6).data
    for fa, fb in ((PNG, 0), (SW, 0), (PNG, PNG | SW)):
        a, b = az.Context(0), az.Context(0)
        a.set_scan_flags(fa)
        if fb:
            b.set_scan_flags(fb)
        for g, x in enumerate((a, b)):
            x.attach(data); x.scan_shard(20000, g, 2)
        for g, x in enumerate((a, b)):
            with pytest.raises(az.AtzError) as e:
                x.probe_import(1 - g, (b, a)[g].probe_export())
            assert e.value.code == az.ATZ_E_STATE
        a.close(); b.close()


def test_probe_export_without_flag_is_unchanged(base):
    """the blob of a context without the flag is the flags word and the probe records only; with it, the split part and its size follow"""
    a, b = az.Context(0), az.Context(0)
    b.set_scan_flags(PNG)
    for x in (a, b):
        x.attach(base.data); x.scan_shard(20000, 0, 2)
    ea, eb = a.probe_export(), b.probe_export()
    assert struct.unpack_from("<Q", ea)[0] == 0 and struct.unpack_from("<Q", eb)[0] == PNG
    split = struct.unpack_from("<Q", eb, len(eb) - 8)[0]
    assert split > 0 and ea[8:] == eb[8:len(eb) - 8 - split]
    a.close(); b.close()


def test_search_schedule_does_not_change_png_records(base):
    want = run(base.data, PNG, az.Options(flags=az.ATZ_F_EXACT_RECORDS), env=dict(ATZ_BURST=1, ATZ_LANES=1))
    for env in (dict(ATZ_BURST=0), dict(ATZ_LANES=2)):
        assert run(base.data, PNG, az.Options(flags=az.ATZ_F_EXACT_RECORDS), env=env) == want, env
