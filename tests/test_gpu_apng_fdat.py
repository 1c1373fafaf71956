"""-m gpu: ATZ_SCAN_APNG_FDAT (uncomp --apng).  An animated PNG keeps each frame but its default image in a zlib stream of its own, split
over consecutive fdAT chunks whose data start with a sequence number; with the flag the scan finds such a stream over its fdAT run, the
search recompresses it like any other, and the ATZ file keeps the 16 framing bytes between its pieces.  APNGs are written here
(signature, IHDR, acTL, fcTL + IDAT run, fcTL + fdAT run per frame, IEND, correct CRCs and sequence numbers) around zlib's own streams."""
import hashlib
import os
import random
import struct
import subprocess
import tempfile

import pytest

import antiz_b200 as az
import corpus
import zref
from test_apng_fdat import fdat, py_fdat_run
from test_gpu_png_idat import Corpus as PngCorpus
from test_gpu_png_idat import cut, idat_sizes, plain, rec
from test_png_idat import chunk, py_run

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")
PNG = az.ATZ_SCAN_PNG_IDAT
APNG = az.ATZ_SCAN_APNG_FDAT
SW = az.ATZ_SCAN_SMALL_WINDOWS
TMP = "/dev/shm" if os.path.isdir("/dev/shm") else None


def fctl(seq, w=64, h=64):
    return chunk(b"fcTL", struct.pack(">IIIIIHHBB", seq, w, h, 0, 0, 1, 10, 0, 0))


def apng_file(default, frames, seed, bad_crc=False, bad_seq=False, tail=b""):
    """an APNG: the default image's zlib stream `default` = (z, IDAT sizes), then frames [(z + extra, fdAT piece sizes)], IEND.  bad_crc /
    bad_seq: every second fdAT gets a wrong CRC / sequence number.  tail: bytes appended to the last fdAT's data.  Returns (bytes,
    offset of the default image's first IDAT data, [offset of each frame's first piece])"""
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", 80 + seed % 40, 64, 8, 0, 0, 0, 0))
    out += chunk(b"acTL", struct.pack(">II", 1 + len(frames), 0)) + chunk(b"tEXt", b"Software\0pytest %d" % seed)
    seq = 0
    out += fctl(seq); seq += 1
    first_idat = len(out) + 8
    z, sizes = default
    at = 0
    for s in sizes:
        out += chunk(b"IDAT", z[at:at + s]); at += s
    starts = []
    for fi, (body, sizes) in enumerate(frames):
        out += fctl(seq); seq += 1
        starts.append(len(out) + 12)
        at = 0
        for k, s in enumerate(sizes):
            data = body[at:at + s]; at += s
            if fi == len(frames) - 1 and k == len(sizes) - 1:
                data += tail
            c = fdat(seq ^ (0x5a5a if bad_seq and k % 2 else 0), data); seq += 1
            if bad_crc and k % 2 == 0:
                c = c[:-4] + bytes(b ^ 0xa5 for b in c[-4:])
            out += c
        assert at == len(body)
    return out + chunk(b"IEND", b""), first_idat, starts


def frame_sizes(c, kind, r):
    """fdAT piece sizes for a c-byte stream: 4096, 8192, "random", or "zero" (3000-byte pieces with empty fdATs in between)"""
    if kind == "zero":
        out = idat_sizes(c, 3000, r)
        return out[:1] + [0] + out[1:2] + [0, 0] + out[2:]
    return idat_sizes(c, kind, r)


class Corpus:
    """APNGs among junk and ordinary zlib streams.  frames[i] = (offset of the header, C, zlib stream, pieces or None for a frame in one
    fdAT, strategy, kind: 12 for a default image in IDATs, 16 for a frame in fdATs)"""

    def __init__(self, seed, n=8, nframes=3, strategies=(0,), small=False, sizes=(4096, 8192, "random", "zero"), umax=50000):
        r = random.Random(seed)
        items, meta = [], []
        for k in range(n):
            streams = []
            for f in range(1 + nframes):
                d = plain(r.randint(2000, umax), seed * 1000 + 10 * k + f)
                lvl, w, m = r.randint(1, 9), r.choice([15, 15, 13, 11, 10]), r.randint(1, 9)
                st = strategies[(k + f) % len(strategies)]
                if st == 1:
                    lvl = max(lvl, 4)
                if small and f % 2 == 1:
                    w = 9
                streams.append((zref.ref_deflate(d, lvl, w, m, st), st))
            (z0, st0), fr = streams[0], streams[1:]
            if k % 4 == 3:           # a frame small enough for one fdAT
                d = plain(r.randint(200, 1500), seed * 7 + k)
                fr[0] = (zref.ref_deflate(d, 6, 15, 8), 0)
            dflt = (z0, idat_sizes(len(z0), 8192, r))
            frs = [(z, [len(z)] if len(z) < 3000 else frame_sizes(len(z), sizes[(k + i) % len(sizes)], r)) for i, (z, st) in enumerate(fr)]
            img, first, starts = apng_file(dflt, frs, seed * 100 + k)
            items.append(img); meta.append((first, starts, [(z0, st0, dflt[1])] + [(z, st, sz) for (z, st), (_, sz) in zip(fr, frs)]))
            if k % 2 == 0:
                items.append(zref.ref_deflate(plain(r.randint(500, 20000), seed * 7 + k), r.randint(1, 9), 15, 8)); meta.append(None)
        self.data, offs = corpus.container(items, seed)
        self.frames = []
        for off, mt in zip(offs, meta):
            if not mt:
                continue
            first, starts, zs = mt
            for j, (z, st, sz) in enumerate(zs):
                p = off + (first if j == 0 else starts[j - 1])
                multi = len([x for x in sz if x]) > 1
                walk = (py_run if j == 0 else py_fdat_run)(self.data, p)
                self.frames.append((p, len(z), z, cut(walk, len(z)) if multi else None, st, 12 if j == 0 else 16))

    def spans(self, kinds=(12, 16)):
        return [(p, p + c + fr * (len(pc) - 1)) for p, c, z, pc, st, fr in self.frames if pc and fr in kinds]


def run(data, flags, opt=None, chunksize=524288, env=None):
    """(records, diffs, pieces, framing) of one context"""
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update({k: str(v) for k, v in (env or {}).items()})
    try:
        c = az.Context(0)
        if flags:
            c.set_scan_flags(flags)
        c.load(data); n = c.scan(chunksize); c.search(opt or az.Options())
        out = ([rec(s) for s in c.streams()], c.diffs(), [c.pieces(i) for i in range(n)], [c.framing(i) for i in range(n)])
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


def check_frames(cp, res, kinds):
    """every multi-chunk stream of the given kinds is recompressed exactly with the restated pieces and framing; the others have none"""
    recs, _, pieces, framing = res
    by = {x[0]: (x, pc, fr) for x, pc, fr in zip(recs, pieces, framing)}
    n = 0
    for p, c, z, pc, st, kind in cp.frames:
        if pc and kind in kinds:
            x, got, fr = by[p]
            exact = c - (2 if z[0] == 0x08 else 0)
            assert x[1] == c and (x[7] == exact if st == 0 else x[7] + 2 >= c) and x[8] == 1, (p, kind, x)
            assert got == pc and fr == kind, (p, got[:4], pc[:4], fr)
            n += 1
        elif p in by:
            assert by[p][1] == [] and by[p][2] == 0, (p, kind)
    assert all((fr == 0) == (pc == []) for pc, fr in zip(pieces, framing))
    return n


@pytest.fixture(scope="module")
def base():
    return Corpus(11)


# ---------------------------------------------------------------------------------------------------------------------------------
def test_flag_off_unchanged(base):
    """without the flag no stream starts at a multi-fdAT frame, with or without --png; single-fdAT frames are ordinary streams"""
    for flags in (0, PNG):
        res = run(base.data, flags)
        starts = {p for p, c, z, pc, st, fr in base.frames if pc and fr == 16}
        assert len(starts) >= 12 and not starts & {x[0] for x in res[0]}
        assert check_frames(base, res, (12,) if flags else ()) >= (6 if flags else 0)
    singles = {p for p, c, z, pc, st, fr in base.frames if not pc and fr == 16}
    off, on = run(base.data, 0), run(base.data, PNG | APNG)
    assert singles and singles <= {x[0] for x in off[0]} and singles <= {x[0] for x, pc in zip(on[0], on[2]) if pc == []}


@pytest.mark.parametrize("flags", [APNG, PNG | APNG])
def test_apng_records(base, flags):
    """--apng: every multi-fdAT default-strategy frame is recompressed exactly with the restated pieces and 16 framing bytes; streams
    outside the split spans keep their records; with --png the default images are IDAT-split streams next to them"""
    off = run(base.data, 0)
    res = run(base.data, flags)
    kinds = (12, 16) if flags & PNG else (16,)
    assert check_frames(base, res, kinds) >= 12
    assert outside(res[0], base.spans(kinds)) == outside(off[0], base.spans(kinds))


@pytest.mark.parametrize("combo", ["strategies", "small-windows", "brute-window"])
@pytest.mark.parametrize("png", [False, True])
def test_apng_combinations(combo, png):
    flags = APNG | (PNG if png else 0)
    kinds = (12, 16) if png else (16,)
    if combo == "strategies":
        cp = Corpus(21, n=5, strategies=(0, 1), sizes=(8192, 4096, "random"))
        res = run(cp.data, flags, az.Options(flags=az.ATZ_F_STRATEGIES))
        assert any(st == 1 and pc and fr == 16 for p, c, z, pc, st, fr in cp.frames)
        args = ["--strategies"]
    elif combo == "small-windows":
        cp = Corpus(22, n=5, small=True, sizes=(4096, "random"))
        res = run(cp.data, flags | SW)
        assert sum(1 for p, c, z, pc, st, fr in cp.frames if pc and fr == 16 and z[0] == 0x18) >= 3
        args = ["--small-windows"]
    else:
        cp = Corpus(23, n=4, sizes=(8192, "zero"))
        res = run(cp.data, flags, az.Options(bruteforceWindow=True))
        args = ["--brute-window"]
    assert check_frames(cp, res, kinds) >= 8
    with tempfile.TemporaryDirectory(dir=TMP) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(cp.data)
        p = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--apng"] + (["--png"] if png else []) + args, capture_output=True, text=True)
        assert p.returncode == 0 and "OK! Restoration is bit by bit identical" in p.stdout, p.stdout + p.stderr


@pytest.mark.parametrize("gpus", [1, 2, 4])
def test_uncomp_apng_round_trip(base, gpus):
    """uncomp --png --apng: the self-test passes, uncomp -r restores the input, and --gpus N (contexts sharing a device where there are
    fewer) writes the same file as --gpus 1"""
    import torch
    env = dict(os.environ)
    if torch.cuda.device_count() < gpus:
        env["ATZ_TEST_ONE_DEVICE"] = "1"
    with tempfile.TemporaryDirectory(dir=TMP) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(base.data)
        p = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--png", "--apng", "--chunksize", "65536", "--gpus", str(gpus)], capture_output=True, text=True, env=env)
        assert p.returncode == 0 and "OK! Restoration is bit by bit identical" in p.stdout, p.stdout + p.stderr
        r = subprocess.run([UNCOMP, "-r", "-i", f + ".atz", "-o", f + ".rec"], capture_output=True, text=True)
        assert r.returncode == 0 and open(f + ".rec", "rb").read() == base.data
        if gpus > 1:
            one = subprocess.run([UNCOMP, "-i", f, "-o", f + ".g1", "--png", "--apng", "--chunksize", "65536", "--notest"], capture_output=True, text=True)
            assert one.returncode == 0
            h = lambda q: hashlib.sha256(open(q, "rb").read()).hexdigest()
            assert h(f + ".g1") == h(f + ".atz")
        else:     # the records of fdAT-split streams carry bits 7 and 5 of the window byte, those of IDAT-split ones bit 7
            w = atz_windows(open(f + ".atz", "rb").read())
            for p, c, z, pc, st, fr in base.frames:
                if pc:
                    assert w[p] & 0xe0 == (0xa0 if fr == 16 else 0x80), (p, fr, w[p])


def atz_windows(atz):
    """offset -> window byte of every top-level record of an ATZ1 file (uncomp.cpp writeATZfile; no nested records)"""
    q, out = 28, {}
    for _ in range(struct.unpack_from("<Q", atz, 20)[0]):
        off, c, u = struct.unpack_from("<QQQ", atz, q)
        w, nd = atz[q + 25], struct.unpack_from("<Q", atz, q + 27)[0]
        assert not w & 0x40
        q += 35 + (8 + 9 * nd if nd else 0)
        if w & 0x80:
            np_ = struct.unpack_from("<Q", atz, q)[0]
            q += 8 + 4 * np_ + (16 if w & 0x20 else 12) * (np_ - 1)
        q += u
        out[off] = w
    return out


# ---------------------------------------------------------------------------------------------------------------------------------
def edge_corpus():
    r = random.Random(31)
    items, cases = [], {}

    def add(name, img, starts, **kw):
        cases[name] = (len(items), starts[0], kw); items.append(img)

    dflt = lambda s: (lambda z: (z, idat_sizes(len(z), 8192, r)))(zref.ref_deflate(plain(12000, s), 6, 15, 8))
    z = zref.ref_deflate(plain(20000, 1), 6, 15, 8)
    add("ends_in_first", *apng_file(dflt(1), [(z + bytes(range(7)) + bytes(300), [len(z) + 7, 300])], 1)[::2])
    z = zref.ref_deflate(plain(30000, 3), 6, 15, 8)
    img, _, st = apng_file(dflt(2), [(z, frame_sizes(len(z), 2000, r))], 2)
    g = bytearray(img); g[st[0] + 2000 + 16 + 700] ^= 0x10
    add("bitflip", bytes(g), st)
    z = zref.ref_deflate(plain(25000, 4), 9, 15, 9)
    add("bad_crc_seq", *apng_file(dflt(3), [(z, frame_sizes(len(z), 3000, r))], 3, bad_crc=True, bad_seq=True)[::2], want=len(z))
    z = zref.ref_deflate(plain(25000, 5), 5, 13, 7)
    add("trailing", *apng_file(dflt(4), [(z, frame_sizes(len(z), 4096, r))], 4, tail=b"TRAILING!!")[::2], want=len(z))
    inner, _, _ = apng_file(dflt(5), [(z, frame_sizes(len(z), 2048, r))], 5)
    add("in_level0", zref.ref_deflate(b"prefix" + inner + b"suffix", 0, 15, 8), [0], outer=True)
    d = plain(40000, 7)
    zs = zref.ref_deflate_ex(d, 6, 15, 8, flushes=[(len(d) - 25, 2)])
    add("sync_flush", *apng_file(dflt(6), [(zs, frame_sizes(len(zs), 8192, r))], 6)[::2], want=len(zs), sync=True)
    data, offs = corpus.container(items, 32)
    out = {name: (offs[i] + first, kw) for name, (i, first, kw) in cases.items()}
    out["_item_ranges"] = {name: (offs[i], offs[i] + len(items[i])) for name, (i, first, kw) in cases.items()}
    return data, out


def test_apng_edge_cases():
    data, cs = edge_corpus()
    rng = cs["_item_ranges"]
    opt = az.Options(recompTresh=400)
    off = run(data, PNG, opt)
    on = run(data, PNG | APNG, opt)
    by_on = {x[0]: (x, pc, fr) for x, pc, fr in zip(on[0], on[2], on[3])}
    within = lambda recs, name: [x for x in recs if rng[name][0] <= x[0] < rng[name][1]]
    # a frame that ends inside the first of two fdATs keeps its record; a bit flip in piece 2 leaves the APNG as it is without the flag
    p = cs["ends_in_first"][0]
    assert p in {x[0] for x in off[0]} and within(on[0], "ends_in_first") == within(off[0], "ends_in_first") and by_on[p][1] == []
    assert within(on[0], "bitflip") == within(off[0], "bitflip")
    # wrong CRCs and sequence numbers, trailing bytes in the last fdAT, a mid-stream Z_SYNC_FLUSH: split streams of their own length
    for name in ("bad_crc_seq", "trailing", "sync_flush"):
        p, kw = cs[name]
        x, pc, fr = by_on[p]
        assert x[1] == kw["want"] and x[8] == 1 and len(pc) >= 2 and sum(pc) == kw["want"] and fr == 16, (name, x)
    assert by_on[cs["sync_flush"][0]][0][9] > 0      # diffs, in de-chunked coordinates (the round trip below checks them)
    # an APNG inside a level-0 stream: the outer stream is kept, nothing is split inside it
    o = rng["in_level0"][0]
    assert o in by_on and by_on[o][0] == next(y for y in off[0] if y[0] == o) and within(on[0], "in_level0") == [by_on[o][0]]
    # a small chunksize: the runs cross many scan chunks and give the same split streams (where the reference's chunking no longer finds
    # the level-0 stream, the frame inside it is split instead)
    split = lambda res: [(x, pc, fr) for x, pc, fr in zip(res[0], res[2], res[3]) if fr and not rng["in_level0"][0] <= x[0] < rng["in_level0"][1]]
    small = run(data, PNG | APNG, opt, chunksize=3000)
    assert len(split(on)) >= 3 and split(small) == split(on)
    with tempfile.TemporaryDirectory(dir=TMP) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        pr = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--png", "--apng", "--recomp-tresh", "400"], capture_output=True, text=True)
        assert pr.returncode == 0 and "OK! Restoration is bit by bit identical" in pr.stdout, pr.stdout + pr.stderr
        r = subprocess.run([UNCOMP, "-r", "-i", f + ".atz", "-o", f + ".rec"], capture_output=True, text=True)
        assert r.returncode == 0 and open(f + ".rec", "rb").read() == data


@pytest.mark.parametrize("which", ["png", "c2"])
def test_atz_unchanged_without_fdat_runs(which):
    """on corpora without fdAT runs --apng writes the same .atz bytes and stdout"""
    data, args = (PngCorpus(11).data, ["--png"]) if which == "png" else (corpus.c2(nstreams=300), [])
    with tempfile.TemporaryDirectory(dir=TMP) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        outs = []
        for extra in ([], ["--apng"]):
            p = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--notest"] + args + extra, capture_output=True, text=True)
            assert p.returncode == 0, p.stdout
            outs.append(open(f + ".atz", "rb").read())
        assert outs[0] == outs[1] and struct.unpack_from("<Q", outs[0], 20)[0] > 0      # (some streams are recompressed)


# ---------------------------------------------------------------------------------------------------------------------------------
def split_offsets(blob):
    """the header offsets and kinds (16: fdAT) of the split streams in a probe export"""
    flags = struct.unpack_from("<Q", blob)[0]
    assert flags & (PNG | APNG)
    sb = struct.unpack_from("<Q", blob, len(blob) - 8)[0]
    q, e, out = len(blob) - 8 - sb, len(blob) - 8, []
    while q < e:
        off, t, np_ = struct.unpack_from("<Q", blob, q)[0], struct.unpack_from("<I", blob, q + 28)[0], struct.unpack_from("<I", blob, q + 32)[0]
        out.append((off, 16 if t & 0x10000 else 12))
        q += 36 + 4 * np_
    return out


@pytest.mark.parametrize("nsh,chunksize", [(2, 524288), (3, 65536), (4, 20000), (5, 5000)])
def test_sharded_apng_equal_single(base, nsh, chunksize):
    """2..5 emulated shards (runs across shard boundaries): the same stream list, records, diffs, pieces and framing as one context.  The
    APNGs are in the first third of the file, so the partition moves some of the streams away from the shard that probed them."""
    opt = az.Options(flags=az.ATZ_F_EXACT_RECORDS)
    flags = PNG | APNG
    data = base.data + corpus.junk(2 * len(base.data), 5)
    one = az.Context(0); one.set_scan_flags(flags); one.load(data); n1 = one.scan(chunksize); one.search(opt)
    want = [rec(s) for s in one.streams()]; wd = one.diffs(); wp = [one.pieces(i) for i in range(n1)]; wf = [one.framing(i) for i in range(n1)]
    one.close()
    assert sum(1 for f in wf if f == 16) >= 12
    ctxs = [az.Context(0) for _ in range(nsh)]
    for g, c in enumerate(ctxs):
        c.set_scan_flags(flags); c.attach(data); c.scan_shard(chunksize, g, nsh)
    blobs = [c.probe_export() for c in ctxs]
    probed = {off: (g, kind) for g, b in enumerate(blobs) for off, kind in split_offsets(b)}
    for g, c in enumerate(ctxs):
        for h in range(nsh):
            if h != g:
                c.probe_import(h, blobs[h])
        assert c.scan_finish() == n1
    for g, c in enumerate(ctxs):
        c.search(opt, g, nsh)
        assert [c.pieces(i) for i in range(n1)] == wp and [c.framing(i) for i in range(n1)] == wf
    own = ctxs[0].owners(); got = []; offs = []; vals = b""
    for i in range(n1):
        c = ctxs[own[i]]; s = c.streams()[i]
        got.append(rec(s))
        o, v = c.diffs()
        offs += list(o[s.diff_index:s.diff_index + s.ndiff]); vals += bytes(v[s.diff_index:s.diff_index + s.ndiff])
    assert got == want and (offs, vals) == (list(wd[0]), bytes(wd[1]))
    fdat_streams = [i for i in range(n1) if wf[i] == 16]
    assert all(probed[want[i][0]][1] == 16 for i in fdat_streams)
    assert any(probed[want[i][0]][0] != own[i] for i in fdat_streams), "no fdAT stream owned away from the shard that probed it"
    for c in ctxs:
        c.close()


def test_apng_flag_state_and_shard_mismatch(base):
    """the fdAT flag is known and ORs with the others; shards that scanned with other flags refuse each other's records; an export
    without the flag carries no fdAT records and IDAT records keep their type word"""
    c = az.Context(0)
    for ok in (APNG, APNG | PNG, APNG | PNG | SW, APNG | SW):
        c.set_scan_flags(ok)
    for bad in (2, 8, APNG | 8):
        with pytest.raises(az.AtzError) as e:
            c.set_scan_flags(bad)
        assert e.value.code == az.ATZ_E_ARG
    c.close()
    for fa, fb in ((APNG, PNG), (APNG, 0), (APNG | PNG, PNG)):
        a, b = az.Context(0), az.Context(0)
        a.set_scan_flags(fa)
        if fb:
            b.set_scan_flags(fb)
        for g, x in enumerate((a, b)):
            x.attach(base.data); x.scan_shard(65536, g, 2)
        for g, x in enumerate((a, b)):
            with pytest.raises(az.AtzError) as e:
                x.probe_import(1 - g, (b, a)[g].probe_export())
            assert e.value.code == az.ATZ_E_STATE
        a.close(); b.close()
    a, b = az.Context(0), az.Context(0)
    a.set_scan_flags(PNG); b.set_scan_flags(PNG | APNG)
    for x in (a, b):
        x.attach(base.data); x.scan_shard(65536, 0, 2)
    sa, sb = split_offsets(a.probe_export()), split_offsets(b.probe_export())
    assert sa and all(k == 12 for o, k in sa) and any(k == 16 for o, k in sb) and [x for x in sb if x[1] == 12] == sa
    a.close(); b.close()


def test_search_schedule_does_not_change_apng_records(base):
    want = run(base.data, PNG | APNG, az.Options(flags=az.ATZ_F_EXACT_RECORDS), env=dict(ATZ_BURST=1, ATZ_LANES=1))
    for env in (dict(ATZ_BURST=0), dict(ATZ_LANES=2)):
        assert run(base.data, PNG | APNG, az.Options(flags=az.ATZ_F_EXACT_RECORDS), env=env) == want, env
