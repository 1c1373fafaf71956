"""ATZ_SCAN_SMALL_WINDOWS (uncomp --small-windows): zlib headers with CINFO 0 and 1 (256- and 512-byte windows), offsetType 24..31,
searched at windowBits 9.  Host logic only: no GPU needed."""
import ctypes as C
import os
import subprocess

import antiz_b200 as az
import zref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")

REFERENCE_24 = [0x2815, 0x2853, 0x2891, 0x28cf, 0x3811, 0x384f, 0x388d, 0x38cb, 0x480d, 0x484b, 0x4889, 0x48c7,
                0x5809, 0x5847, 0x5885, 0x58c3, 0x6805, 0x6843, 0x6881, 0x68de, 0x7801, 0x785e, 0x789c, 0x78da]
SMALL_8 = [0x081d, 0x085b, 0x0899, 0x08d7, 0x1819, 0x1857, 0x1895, 0x18d3]    # CINFO 0 (types 24..27), CINFO 1 (types 28..31)


def header_type(flags, b0, b1):
    return az.lib().atz_host_header_type(flags, b0, b1)


def seq(ot, brute):
    c = (C.c_uint8 * 600)(); w = (C.c_uint8 * 600)(); m = (C.c_uint8 * 600)()
    n = az.lib().atz_host_candidate_sequence(ot, brute, c, w, m, 600)
    return [(c[i], w[i], m[i]) for i in range(n)]


def test_header_set_over_all_pairs():
    """the scan's header test (common.cuh zlib_header_type, what K1 and the chunk-start fix-up run) over all 65,536 byte pairs: the
    reference's 24 with types 0..23 without the flag; those and the 8 small-window pairs with types 24..31 with it"""
    want_off = {h: i for i, h in enumerate(REFERENCE_24)}
    want_on = {**want_off, **{h: 24 + i for i, h in enumerate(SMALL_8)}}
    got_off, got_on = {}, {}
    for b0 in range(256):
        for b1 in range(256):
            h = b0 << 8 | b1
            t0, t1 = header_type(0, b0, b1), header_type(az.ATZ_SCAN_SMALL_WINDOWS, b0, b1)
            if t0 >= 0:
                got_off[h] = t0
            if t1 >= 0:
                got_on[h] = t1
            # K1's word-at-a-time prefilter (low nibble 8, top bit clear) must never drop a header of either set
            assert t1 < 0 or ((b0 & 0x8f) == 0x08)
    assert got_off == want_off and got_on == want_on
    # the types of the new pairs follow 24 + 4 * CINFO + FLEVEL; FLEVEL is the header's, as for 0..23
    for h in SMALL_8:
        assert want_on[h] == 24 + 4 * (h >> 12) + ((h & 0xff) >> 6)
    # FDICT headers stay out (zlib cannot inflate them without the dictionary)
    assert all(header_type(az.ATZ_SCAN_SMALL_WINDOWS, b0, b1) < 0 for b0 in (0x08, 0x18) for b1 in range(256) if b1 & 0x20)


def test_zlib_writes_cinfo_1_for_windows_8_and_9():
    """what the new types are for: zlib's own header for windowBits 8 and 9 is one of the CINFO 1 pairs, with the level's FLEVEL"""
    flevel = {0: 0, 1: 0, 2: 1, 3: 1, 4: 1, 5: 1, 6: 2, 7: 3, 8: 3, 9: 3}
    for wb in (8, 9):
        for lvl in range(10):
            z = zref.ref_deflate(b"small window " * 40, lvl, wb, 8, z=zref.zlib_lib())   # (only the header is looked at)
            assert header_type(az.ATZ_SCAN_SMALL_WINDOWS, z[0], z[1]) == 28 + flevel[lvl], (wb, lvl, z[:2].hex())
            assert header_type(0, z[0], z[1]) == -1


def test_candidate_sequences_of_small_window_types():
    """types 24..31 follow the reference's rules at window 9: the FLEVEL class's sequence, the --brute-window grid over windows 15..10,
    the strategy sequence"""
    for ot in range(24, 32):
        cls = ot % 4
        s = seq(ot, 0)
        ref = seq(20 + cls, 0)                                    # the same class at window 15
        assert s == [(c, 9, m) for c, _, m in ref]
        b = seq(ot, 1)
        assert len(b) == 486 and len(set(b)) == 486
        assert [x[1] for x in b[::81]] == [15, 14, 13, 12, 11, 10]
        assert b[:81] == [(c, 15, m) for m in range(9, 0, -1) for c in range(9, 0, -1)]      # memLevel 9..1 x level 9..1 per window
        st = seq(ot, 2)
        assert st == [(c, 9, m) for c, _, m in seq(20 + cls, 2)]
    # the sequences of the reference's types are untouched
    assert seq(0, 1)[0] == (9, 15, 9) and len(seq(0, 1)) == 405
    for bad in (-1, 32):
        assert az.lib().atz_host_candidate_sequence(bad, 0, (C.c_uint8 * 600)(), (C.c_uint8 * 600)(), (C.c_uint8 * 600)(), 600) == az.ATZ_E_ARG


def test_help_lists_small_windows_after_the_extensions():
    h = subprocess.run(["uncomp", "--help"], executable=UNCOMP, capture_output=True, text=True)
    assert h.returncode == 0
    ext = h.stdout.index("antiz_b200 extensions:")
    at = h.stdout.index("--small-windows")
    assert at > ext
    tail = " ".join(h.stdout[at:].split())
    assert "256- and 512-byte windows" in tail and "differs from the reference's" in tail and "reference can still reconstruct" in tail
    # the brief usage of a parse error stays the reference's: no extension in it
    p = subprocess.run(["uncomp", "--bogus"], executable=UNCOMP, capture_output=True, text=True)
    assert p.returncode == 1 and "--small-windows" not in p.stderr and "--brute-window" in p.stderr
