"""-m gpu parity tests proper: the CUDA kernels, called through the C ABI, against the reference's zlib 1.2.8
(oracle/_ref; the host's zlib where it writes the same bytes, see zref.host_zlib) and the CPU oracle on the same seeded inputs.  Bit-exact (byte/integer work): no tolerance."""
import json
import os
import random
import zlib

import pytest

import antiz_b200 as az
import corpus
import zref
from test_oracle_inflate import INFCOVER_RAW, wrap

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ctx():
    c = az.Context(0)
    yield c
    c.close()


def expect_deflate(d, lvl, w, m):
    return zref.ref_deflate(d, lvl, w, m) if zref.have_ref() else zref.oracle_deflate(d, lvl, w, m)


def test_deflate_full_parameter_grid(ctx):
    R = random.Random(1)
    ins = {"text70k": corpus.text(70000, 2), "bin": corpus.binaryish(60000, 9), "mixed": corpus.text(20000, 5) + R.randbytes(3000) + bytes(5000) + corpus.text(40000, 6)}
    for name, d in ins.items():
        items = [(d, lvl, w, m) for lvl in range(10) for w in range(10, 16) for m in range(1, 10)]
        outs = ctx.deflate_batch(items)
        for (dd, lvl, w, m), o in zip(items, outs):
            assert o == expect_deflate(dd, lvl, w, m), (name, lvl, w, m)


def test_deflate_edge_inputs(ctx):
    R = random.Random(2)
    ins = [b"", b"x", b"ab", b"abc", b"aaaa", bytes(100000), R.randbytes(70000), b"asd" * 4608, corpus.text(3000, 3), bytes(range(256)) * 300,
           corpus.text(1 << 20, 1234)]
    items = [(d, lvl, w, m) for d in ins for lvl in range(10) for (w, m) in ((15, 8), (10, 1), (12, 9), (9, 5))]
    outs = ctx.deflate_batch(items)
    for (d, lvl, w, m), o in zip(items, outs):
        assert o == expect_deflate(d, lvl, w, m), (len(d), lvl, w, m)


def test_deflate_reference_golden_vectors(ctx):
    asd = b"asd" * 4608
    for name, lvl, w in (("c1", 1, 15), ("c5", 5, 15), ("c6", 6, 15), ("c9", 9, 15), ("2k", 9, 11)):
        want = open(os.path.join(GOLD, f"zlibtest_out_{name}.bin"), "rb").read()
        for m in (1, 8, 9):
            assert ctx.deflate_stream(asd, lvl, w, m) == want


def test_deflate_window_edges(ctx):
    """slide timing, MAX_DIST, window index 0 == NIL (incl. the post-slide corner), stored-block eligibility"""
    R = random.Random(5)
    items = []
    for w in (10, 11):
        ws = 1 << w; md = ws - 262
        for k in (1, 2):
            pslide = k * ws + ws + md
            for extra in (3, 20, 261):
                for delta in (-1, 0, 1):
                    n = pslide + extra; d = bytearray(R.randbytes(n)); src = (k + 1) * ws + delta; L = min(20, n - pslide)
                    d[pslide:pslide + L] = d[src:src + L]
                    items += [(bytes(d), lvl, w, 8) for lvl in (1, 3, 4, 6, 9)]
    for it in range(300):
        w = R.choice([10, 10, 11, 12]); ws = 1 << w; md = ws - 262
        L = max(1, R.choice([1, 2, 3]) * ws + R.randrange(-400, 400) + R.choice([0, md, ws])); kind = R.randrange(4)
        if kind == 0:
            per = md + R.choice([-2, -1, 0, 1, 2, 262, 261, 260]); base = R.randbytes(per); d = (base * (L // per + 2))[:L]
        elif kind == 1:
            d = bytes(R.choice(b"ab") for _ in range(L))
        elif kind == 2:
            blk = R.randbytes(40); d = bytearray(R.randbytes(L))
            for pos in range(0, L - 40, R.choice([md - 1, md, md + 1, ws, 700])):
                d[pos:pos + 40] = blk
            d = bytes(d[:L])
        else:
            unit = bytes(R.choice(b"xyz") for _ in range(R.randrange(1, 50))); d = (unit * (L // len(unit) + 1))[:L]
        items.append((d, R.randrange(0, 10), w, R.randrange(1, 10)))
    outs = ctx.deflate_batch(items)
    for (d, lvl, w, m), o in zip(items, outs):
        assert o == expect_deflate(d, lvl, w, m), (len(d), lvl, w, m)


def _inflate_expect(buf, cap):
    """(rc class, total_in, total_out) of zlib's inflate over buf with a cap-byte output buffer"""
    if zref.have_ref():
        fi, ret, ti, to, ai = zref.ref_inflate_scan(buf, 0, 1 << 22)
        st = {1: 0, -3: 2, 2: 3}.get(ret, 1)
    else:
        r, _ = zref.oracle_inflate(buf, None, 0); st, ti, to = r.status, r.total_in, r.total_out
    return st, ti, to


def test_inflate_status_and_byte_accounting(ctx):
    R = random.Random(7)
    streams = []
    for seed in range(3):
        d = corpus.text(R.choice([10, 700, 5000]), seed, 300)
        for lvl in (0, 1, 6, 9):
            streams.append(zref.oracle_deflate(d, lvl, R.choice([10, 15]), R.choice([1, 8, 9])))
    streams.append(zref.oracle_deflate(bytes(3000), 6, 15, 8)); streams.append(zref.oracle_deflate(b"", 6, 15, 8))
    rcmap = {0: az.ATZ_OK, 1: az.ATZ_E_TRUNCATED, 2: az.ATZ_E_DATA, 3: az.ATZ_E_DATA}
    n = 0
    for s in streams:
        cases = [s, s + b"xyz"] + [s[:c] for c in range(0, len(s), max(1, len(s) // 25))]
        for _ in range(25):
            b = bytearray(s); b[R.randrange(len(b))] ^= 1 << R.randrange(8); cases.append(bytes(b))
        for buf in cases:
            if not buf:
                continue
            st, ti, to = _inflate_expect(buf, 1 << 22)
            rc, out, used = ctx.inflate_stream(buf, 1 << 16)
            assert rc == rcmap[st] and used == ti, (buf[:10].hex(), len(buf), rc, st, used, ti)
            n += 1
    assert n > 400


def test_inflate_output_full_state_equals_zlib(ctx):
    """ATZ_E_SMALL is zlib's "output buffer full": the buffer is filled to the last byte and *consumed is the input zlib has used by
    then - what ZlibInflator::operator() reports to the scanner (ZlibWrapper.h:56-69, main.cpp:228-232)"""
    R = random.Random(11)
    n = 0
    for seed in range(6):
        d = corpus.text(R.choice([3000, 20000, 70000]), seed, 300) if seed % 3 else corpus.binaryish(30000, seed)
        for lvl in (0, 1, 6, 9):
            z = zref.ref_deflate(d, lvl, 15, R.choice([1, 8, 9]))
            for cap in (1, 2, 100, 257, 258, 259, 1000, len(d) // 3, len(d) - 1):
                first_in, ret, ti, to, _ = zref.ref_inflate_scan(z + b"junk", 0, cap)
                import ctypes as C
                out = (C.c_uint8 * cap)(); olen, used = C.c_uint64(), C.c_uint64()
                addr, ln, keep = az._buf(z + b"junk")
                rc = az.lib().atz_inflate_stream(ctx._h, addr, ln, out, cap, C.byref(olen), C.byref(used))
                assert rc == az.ATZ_E_SMALL and olen.value == cap and used.value == first_in, (lvl, cap, rc, olen.value, used.value, first_in)
                assert bytes(out) == d[:cap]
                n += 1
    assert n > 150


def test_inflate_infcover_vectors(ctx):
    gold = json.load(open(os.path.join(GOLD, "inflate_vectors.json")))
    for hexs, what in INFCOVER_RAW:
        g = gold[hexs]
        rc, out, used = ctx.inflate_stream(wrap(hexs), 1 << 16)
        want = {1: az.ATZ_OK, -3: az.ATZ_E_DATA}.get(g["ret"], az.ATZ_E_TRUNCATED)
        assert rc == want and used == g["total_in"], (what, rc, used, g)


def test_inflate_round_trip_and_adler(ctx):
    for d in (corpus.text(1 << 20, 1234), corpus.binaryish(300000, 5), bytes(500000), random.Random(3).randbytes(200000)):
        for lvl, w, m in ((6, 15, 8), (1, 10, 1), (0, 15, 8), (9, 13, 9)):
            z = ctx.deflate_stream(d, lvl, w, m)
            assert zlib.decompress(z) == d                       # any inflater accepts it, adler included
            rc, out, used = ctx.inflate_stream(z, len(d))
            assert rc == az.ATZ_OK and out == d and used == len(z)


def test_deflate_strategies_bit_exact(ctx):
    """ATZ_F_STRATEGIES extension: deflate with Z_FILTERED / Z_HUFFMAN_ONLY / Z_RLE / Z_FIXED equals zlib 1.2.8's
    deflateInit2(level, 8, wbits, memLevel, strategy) + deflate(Z_FINISH) (Z/deflate.c:1861-1967, 1774-1785, Z/trees.c:952)"""
    R = random.Random(21)
    inputs = [corpus.text(40000, 3, 300), corpus.binaryish(60000, 4), bytes(5000) + corpus.text(3000, 5) + bytes([7]) * 70000 + b"ab" * 500,
              R.randbytes(20000), b"", b"a", b"aaaa", corpus.text(300000, 6)]
    items, want = [], []
    for d in inputs:
        for strat in (1, 2, 3, 4):
            for lvl, w, m in ((1, 15, 8), (3, 12, 9), (4, 15, 8), (6, 10, 1), (6, 15, 8), (9, 14, 3), (9, 15, 9), (5, 9, 5)):
                items.append((d, az.clevel(lvl, strat), w, m)); want.append(zref.ref_deflate(d, lvl, w, m, strat))
    got = ctx.deflate_batch(items)
    bad = [(len(it[0]), it[1] & 15, it[1] >> 4, it[2], it[3]) for it, g, x in zip(items, got, want) if g != x]
    assert not bad, bad[:10]


def _trial_expect(plain, orig, lvl, w, m, opt):
    """testDeflateParams' {bailed, valid, ident} (main.cpp:632-681) from the reference zlib's output"""
    cp = expect_deflate(plain, lvl, w, m); C, Cp = len(orig), len(cp)
    S, R_, SD = opt.shortcutLength, opt.recompTresh, opt.sizediffTresh
    if C > S:
        p = min(S, Cp); ident = sum(1 for i in range(p) if cp[i] == orig[i])
        if ident < ((S - R_) & 0xFFFFFFFFFFFFFFFF):
            return az.TR_BAILED, None, None
    if abs(Cp - C) > SD:
        return az.TR_SIZE, Cp, None
    sm = min(Cp, C)
    return az.TR_COMPARED, Cp, sum(1 for i in range(sm) if cp[i] == orig[i])


def test_trial_compare_shortcut_sizegate(ctx):
    R = random.Random(9)
    plain = corpus.text(60000, 77)
    exact = az.Options(flags=az.ATZ_F_EXACT_RECORDS)
    for (ol, ow, om) in ((6, 15, 8), (9, 15, 8), (1, 15, 9), (4, 12, 3), (0, 15, 8)):
        orig = zref.oracle_deflate(plain, ol, ow, om)
        mut = bytearray(orig)
        for _ in range(5):
            mut[R.randrange(600, len(mut))] ^= 0x55
        for o in (orig, bytes(mut), orig[:-40], orig + b"\0" * 300):
            for (lvl, w, m) in ((ol, ow, om), (6, 15, 8), (5, 15, 8), (1, 15, 8), (9, 14, 9), (0, 15, 8), (ol, ow, (om % 9) + 1)):
                for opt in (exact, az.Options(shortcutLength=100, recompTresh=10, sizediffTresh=10, flags=az.ATZ_F_EXACT_RECORDS), az.Options(recompTresh=1000, flags=1)):
                    st, cp, ident = _trial_expect(plain, o, lvl, w, m, opt)
                    r = ctx.trial(plain, o, lvl, w, m, opt)
                    assert r.status == st, (ol, ow, om, lvl, w, m, len(o), r.status, st)
                    if st == az.TR_COMPARED:
                        assert (r.out_len, r.ident) == (cp, ident)
    # default mode (early cut): a cut trial is one the exact mode would also never accept as recompressible
    orig = zref.oracle_deflate(plain, 6, 15, 8)
    r = ctx.trial(plain, orig, 6, 15, 7, az.Options())
    e = ctx.trial(plain, orig, 6, 15, 7, exact)
    assert r.status in (az.TR_CUT, az.TR_BAILED, az.TR_SIZE) or (r.status == e.status and r.ident == e.ident)
    if r.status == az.TR_CUT:
        assert e.status != az.TR_COMPARED or len(orig) - e.ident > 128


def test_deflate_chain_walk_fallback(ctx):
    """the same kernel with row tables switched off (ATZ_FORCE_REC=0): every longest_match walks the bucket lists"""
    d = corpus.text(50000, 12) + corpus.binaryish(30000, 13)
    items = [(d, lvl, w, m) for lvl in (1, 3, 4, 6, 9) for (w, m) in ((15, 8), (11, 2), (13, 9))]
    for var in ("ATZ_FORCE_REC", "ATZ_FORCE_RES"):   # no rows at all / rows but no resolved tables
        os.environ[var] = "0"
        try:
            outs = ctx.deflate_batch(items)
        finally:
            del os.environ[var]
        for (dd, lvl, w, m), o in zip(items, outs):
            assert o == expect_deflate(dd, lvl, w, m), (var, lvl, w, m)
