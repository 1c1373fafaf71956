"""The CPU oracle (oracle/zdeflate.c) against the reference's golden vectors and its own zlib 1.2.8 build (the host's zlib at
levels 1-9 where that build is absent: see zref.host_zlib)."""
import hashlib
import json
import os
import random

import pytest

import corpus
import zref

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ASD = b"asd" * 4608   # the input of the reference's zlib harness (ZT/main.cpp), SURVEY.md section 4


@pytest.mark.parametrize("name,level,wbits", [("c1", 1, 15), ("c5", 5, 15), ("c6", 6, 15), ("c9", 9, 15), ("2k", 9, 11)])
def test_reference_golden_vectors(name, level, wbits):
    want = open(os.path.join(GOLD, f"zlibtest_out_{name}.bin"), "rb").read()
    for m in range(1, 10):   # the fixtures do not depend on memLevel (SURVEY.md section 4)
        assert zref.oracle_deflate(ASD, level, wbits, m) == want
        assert zref.oracle_deflate_listmode(ASD, level, wbits, m) == want
    r, out = zref.oracle_inflate(want, len(ASD))
    assert r.status == zref.OI_END and out == ASD and r.total_in == len(want)


def test_header_flevel_table():
    """docs/stream type tables.txt: FLEVEL 0 <-> clevel 0-1, 1 <-> 2-5, 2 <-> 6, 3 <-> 7-9 (Z/deflate.c:741-748)"""
    want = {0: 0x7801, 1: 0x7801, 2: 0x785e, 5: 0x785e, 6: 0x789c, 7: 0x78da, 9: 0x78da}
    for lvl, hdr in want.items():
        z = zref.oracle_deflate(b"hello hello hello", lvl, 15, 8)
        assert (z[0] << 8 | z[1]) == hdr
    assert zref.oracle_deflate(b"x", 9, 14, 8)[:2] == bytes([0x68, 0xde])
    assert zref.oracle_deflate(b"x", 1, 14, 8)[:2] == bytes([0x68, 0x05])


def _inputs():
    R = random.Random(1)
    return {
        "text40k": corpus.text(40000, 2), "text3k": corpus.text(3000, 3), "zeros": bytes(70000), "rand": R.randbytes(30000),
        "short": b"ab", "empty": b"", "one": b"x", "bin": corpus.binaryish(50000, 9),
        "mixed": corpus.text(20000, 5) + R.randbytes(3000) + bytes(5000) + corpus.text(30000, 6),
    }


# levels at which zref's zlib is zlib 1.2.8's equal (level 0 only with the reference's own build)
LEVELS = range(10) if zref.have_ref() else range(1, 10)


def test_golden_digests():
    """committed digests of the reference zlib's output (tests/golden/make_golden.py) - works without oracle/_ref"""
    gold = json.load(open(os.path.join(GOLD, "deflate_digests.json")))
    ins = _inputs()
    for key, want in gold.items():
        name, lvl, w, m = key.split(":")
        got = zref.oracle_deflate(ins[name], int(lvl), int(w), int(m))
        assert hashlib.sha256(got).hexdigest() == want, key


def test_host_zlib_equals_the_golden_digests_above_level_0():
    """the seeded corpora and, where the reference's zlib has not been built, the comparisons below use the host's zlib: its output
    at levels 1-9 must be the one zlib 1.2.8 wrote into the committed digests"""
    gold = json.load(open(os.path.join(GOLD, "deflate_digests.json")))
    ins = _inputs()
    z = zref.host_zlib()
    n = 0
    for key, want in gold.items():
        name, lvl, w, m = key.split(":")
        if int(lvl) == 0:
            continue
        got = zref.ref_deflate(ins[name], int(lvl), int(w), int(m), z=z)
        assert hashlib.sha256(got).hexdigest() == want, (key, z.zlibVersion())
        n += 1
    assert n >= 200


def test_against_reference_zlib_grid():
    ins = _inputs()
    R = random.Random(7)
    for name, d in ins.items():
        for lvl in LEVELS:
            for w in range(10, 16):
                for m in (R.sample(range(1, 10), 3)):
                    want = zref.ref_deflate(d, lvl, w, m)
                    assert zref.oracle_deflate(d, lvl, w, m) == want, (name, lvl, w, m)
                    assert zref.oracle_deflate_listmode(d, lvl, w, m) == want, ("listmode", name, lvl, w, m)


def test_nil_after_slide_corner():
    """A match source at window index 0 after the last slide of a stream is NIL for zlib (Z/deflate.c:1158-1162,1766)
    although its distance (exactly MAX_DIST) would be legal: the one place where the slide is not a no-op."""
    R = random.Random(5)
    for w in (10, 11):
        ws = 1 << w; md = ws - 262
        for k in (1, 2):
            pslide = k * ws + ws + md
            for extra in (3, 20, 261):
                for delta in (-1, 0, 1):
                    n = pslide + extra
                    d = bytearray(R.randbytes(n))
                    src = (k + 1) * ws + delta
                    L = min(20, n - pslide)
                    d[pslide:pslide + L] = d[src:src + L]
                    d = bytes(d)
                    for lvl in (1, 3, 4, 6, 9):
                        want = zref.ref_deflate(d, lvl, w, 8)
                        assert zref.oracle_deflate(d, lvl, w, 8) == want
                        assert zref.oracle_deflate_listmode(d, lvl, w, 8) == want


def test_window_edge_stress():
    R = random.Random(11)
    for it in range(250):
        w = R.choice([10, 10, 11, 12]); ws = 1 << w; md = ws - 262
        L = max(1, R.choice([1, 2, 3]) * ws + R.randrange(-400, 400) + R.choice([0, md, ws]))
        kind = R.randrange(4)
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
        lvl = R.randrange(0, 10); m = R.randrange(1, 10)
        if lvl not in LEVELS:
            continue
        want = zref.ref_deflate(d, lvl, w, m)
        assert zref.oracle_deflate(d, lvl, w, m) == want, (it, lvl, w, m)
        assert zref.oracle_deflate_listmode(d, lvl, w, m) == want, ("listmode", it, lvl, w, m)


def test_adler():
    import zlib
    R = random.Random(3)
    for n in (0, 1, 5551, 5552, 5553, 100000):
        d = R.randbytes(n)
        assert zref.oracle().oracle_adler32(d, n) == zlib.adler32(d)
