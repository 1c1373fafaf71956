"""The CPU oracle (oracle/zinflate.c) against zlib 1.2.8 (or the host's zlib, whose inflate accounting is the same: zref.host_zlib):
accept/reject set and the byte accounting ZBuffSearcher reads."""
import json
import os
import random

import corpus
import zref

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# Raw-deflate known-answer vectors restated from the reference's vendored Z/test/infcover.c:583-659 (hex bytes, what they
# exercise).  AntiZ only ever sees zlib-wrapped streams, so each is wrapped in a 78 9c header (no trailer).
INFCOVER_RAW = [
    ("0 0 0 0 0", "invalid stored block lengths"), ("3 0", "fixed"), ("6", "invalid block type"), ("1 1 0 fe ff 0", "stored"),
    ("fc 0 0", "too many length or distance symbols"), ("4 0 fe ff", "invalid code lengths set"),
    ("4 0 24 49 0", "invalid bit length repeat"), ("4 0 24 e9 ff ff", "invalid bit length repeat"),
    ("4 0 24 e9 ff 6d", "invalid code -- missing end-of-block"),
    ("4 80 49 92 24 49 92 24 71 ff ff 93 11 0", "invalid literal/lengths set"),
    ("4 80 49 92 24 49 92 24 f b4 ff ff c3 84", "invalid distances set"),
    ("4 c0 81 8 0 0 0 0 20 7f eb b 0 0", "invalid literal/length code"), ("2 7e ff ff", "invalid distance code"),
    ("c c0 81 0 0 0 0 0 90 ff 6b 4 0", "invalid distance too far back"),
    ("5 c0 21 d 0 0 0 80 b0 fe 6d 2f 91 6c", "pull 17"),
    ("5 e0 81 91 24 cb b2 2c 49 e2 f 2e 8b 9a 47 56 9f fb fe ec d2 ff 1f", "long code"),
    ("ed c0 1 1 0 0 0 40 20 ff 57 1b 42 2c 4f", "length extra"),
    ("ed cf c1 b1 2c 47 10 c4 30 fa 6f 35 1d 1 82 59 3d fb be 2e 2a fc f c", "long distance and extra"),
    ("2 8 20 80 0 3 0", "inflate_fast TYPE return"), ("63 18 5 40 c 0", "window wrap"),
    ("e5 e0 81 ad 6d cb b2 2c c9 01 1e 59 63 ae 7d ee fb 4d fd b5 35 41 68 ff 7f 0f 0 0 0", "fast length extra bits"),
    ("25 fd 81 b5 6d 59 b6 6a 49 ea af 35 6 34 eb 8c b9 f6 b9 1e ef 67 49 50 fe ff ff 3f 0 0", "fast distance extra bits"),
    ("3 7e 0 0 0 0 0", "fast invalid distance code"), ("1b 7 0 0 0 0 0", "fast invalid literal/length code"),
    ("d c7 1 ae eb 38 c 4 41 a0 87 72 de df fb 1f b8 36 b1 38 5d ff ff 0", "fast 2nd level codes and too far back"),
    ("63 18 5 8c 10 8 0 0 0 0", "very common case"), ("63 60 60 18 c9 0 8 18 18 18 26 c0 28 0 29 0 0 0", "contiguous and wrap around window"),
    ("63 0 3 0 0 0 0 0", "copy direct from output"),
]
# zlib-wrapper cases, Z/test/infcover.c:399-411 (already wrapped)
INFCOVER_ZLIB = [("77 85", 2), ("78 90", 2), ("78 9c 63 0 0 0 1 0 1", 0), ("78 9c 63 0", 1), ("8 b8 0 0 0 1", 3)]


def wrap(hexs):
    return bytes([0x78, 0x9c]) + bytes(int(x, 16) for x in hexs.split())


def cls(ret):
    return {1: zref.OI_END, -3: zref.OI_DATA_ERROR, 2: zref.OI_NEED_DICT}.get(ret, zref.OI_NEED_INPUT)


def test_infcover_known_answers():
    gold = json.load(open(os.path.join(GOLD, "inflate_vectors.json")))
    for hexs, what in INFCOVER_RAW:
        r, _ = zref.oracle_inflate(wrap(hexs), None, 1 << 16)
        g = gold[hexs]
        assert (r.status, r.total_in, r.total_out) == (cls(g["ret"]), g["total_in"], g["total_out"]), what
        if what.startswith(("invalid", "too many", "fast invalid", "fast 2nd", "fast length", "fast distance")):
            assert r.status == zref.OI_DATA_ERROR, what
    for hexs, want in INFCOVER_ZLIB:
        z = bytes(int(x, 16) for x in hexs.split())
        r, _ = zref.oracle_inflate(z, None, 1 << 16)
        assert r.status == want, hexs


def _check(buf, outcap):
    fi, ret, ti, to, ai = zref.ref_inflate_scan(buf, 0, outcap)
    r, _ = zref.oracle_inflate(buf, None, outcap)
    assert (r.in_at_outcap, r.status, r.total_in, r.total_out, len(buf) - r.total_in) == (fi, cls(ret), ti, to, ai), (buf[:12].hex(), len(buf), outcap)


def test_against_reference_zlib_truncations_and_bitflips():
    R = random.Random(7)
    streams = []
    for seed in range(4):
        d = corpus.text(R.choice([10, 100, 700, 5000]), seed, 300)
        for lvl in (0, 1, 6, 9):
            streams.append(zref.ref_deflate(d, lvl, R.choice([10, 12, 15]), R.choice([1, 5, 8, 9])))
    streams += [zref.ref_deflate(bytes(3000), 6, 15, 8), zref.ref_deflate(R.randbytes(2000), 6, 15, 8), zref.ref_deflate(b"", 6, 15, 8), zref.ref_deflate(b"a", 1, 15, 8)]
    for s in streams:
        for outcap in (64, 300, 1 << 16):
            step = 1 if len(s) < 400 else 13
            for cut in range(0, len(s) + 1, step):
                _check(s[:cut], outcap)
            _check(s + b"xyz", outcap)
            for _ in range(120):
                b = bytearray(s); pos = R.randrange(len(b)); b[pos] ^= 1 << R.randrange(8)
                if R.random() < 0.3:
                    b = b[:R.randrange(1, len(b) + 1)]
                _check(bytes(b), outcap)


def test_against_reference_zlib_garbage_after_magic():
    R = random.Random(8)
    magics = [0x7801, 0x785e, 0x789c, 0x78da, 0x2815, 0x68de, 0x5885]
    for _ in range(6000):
        m = R.choice(magics)
        _check(bytes([m >> 8, m & 0xff]) + R.randbytes(R.choice([3, 5, 9, 17, 40, 200])), R.choice([64, 1 << 16]))


def test_round_trip_large():
    d = corpus.text(300000, 4)
    for lvl, w, m in ((6, 15, 8), (1, 10, 1), (9, 12, 9), (0, 15, 8)):
        z = zref.oracle_deflate(d, lvl, w, m)
        r, out = zref.oracle_inflate(z, len(d))
        assert r.status == zref.OI_END and out == d and r.total_in == len(z)
