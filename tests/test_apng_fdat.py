"""ATZ_SCAN_APNG_FDAT (uncomp --apng): zlib streams of APNG frames split over consecutive fdAT chunks.  Host logic only: the fdAT run
walker (the function the run-detection kernel runs) against a restatement, the reconstructor's checks of fdAT-split descriptors, which
come before any GPU work, the help text and the constants against C."""
import ctypes as C
import mmap
import os
import struct
import subprocess
import tempfile
import zlib

import antiz_b200 as az
from test_nested import atz_file, outer, record
from test_png_idat import chunk, py_run

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")


def py_fdat_run(f, p):
    """the fdAT run whose first piece starts at p (include/antiz_b200.h ATZ_SCAN_APNG_FDAT): its piece lengths, [] if there is none"""
    n = len(f)
    if p < 12 or p >= n or f[p - 8:p - 4] != b"fdAT":
        return []
    L = struct.unpack(">I", f[p - 12:p - 8])[0]
    if L < 6:
        return []
    out, d = [], p - 4
    while d + L + 4 <= n:
        out.append(L - 4)
        q = d + L + 4
        if q + 8 > n or f[q + 4:q + 8] != b"fdAT":
            break
        L = struct.unpack(">I", f[q:q + 4])[0]
        d = q + 8
        if L < 4:
            break
    return out if len(out) >= 2 else []


def host_run(f, p, cap=4096, fn="atz_host_fdat_run"):
    buf = (C.c_uint8 * max(len(f), 1)).from_buffer_copy(f or b"\0")
    lens = (C.c_uint32 * cap)()
    n = C.c_uint64()
    assert getattr(az.lib(), fn)(buf, len(f), p, lens, cap, C.byref(n)) == az.ATZ_OK
    return list(lens[:min(n.value, cap)]) if n.value else []


def fdat(seq, data):
    return chunk(b"fdAT", struct.pack(">I", seq) + data)


def apng(sizes, tail=b"", body=None, lens=None):
    """signature, IHDR, acTL, fcTL + IDAT, fcTL, then fdAT chunks holding pieces of the given sizes behind their sequence numbers (a
    zlib header then filler), `tail`; offset of the first piece.  lens: chunk lengths to write instead of 4 + size."""
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", 64, 64, 8, 2, 0, 0, 0)) + chunk(b"acTL", struct.pack(">II", 2, 0))
    out += chunk(b"fcTL", struct.pack(">IIIIIHHBB", 0, 64, 64, 0, 0, 1, 10, 0, 0)) + chunk(b"IDAT", zlib.compress(bytes(64 * 193)))
    out += chunk(b"fcTL", struct.pack(">IIIIIHHBB", 2, 64, 64, 0, 0, 1, 10, 0, 0))
    first = len(out) + 12
    body = body if body is not None else b"\x78\x9c" + bytes((i * 7) & 255 for i in range(sum(sizes)))
    at = 0
    for k, s in enumerate(sizes):
        c = fdat(3 + k, body[at:at + s]); at += s
        if lens is not None:
            c = struct.pack(">I", lens[k]) + c[4:]
        out += c
    return out + tail, first


def check(f, p, want_len):
    got = host_run(f, p)
    assert got == py_fdat_run(f, p)
    assert len(got) == want_len, (got, want_len)
    return got


IEND = chunk(b"IEND", b"")


def test_walker_runs():
    check(*apng([8192], IEND), 0)                                 # 1 chunk: no run
    f, p = apng([8192, 100], IEND)
    assert check(f, p, 2) == [8192, 100]
    for k in (3, 17, 300):
        f, p = apng([37] * k, IEND)
        assert check(f, p, k) == [37] * k
    f, p = apng([500, 0, 0, 300, 9], IEND)                        # fdATs with a sequence number and no data (L == 4) in the middle
    assert check(f, p, 5) == [500, 0, 0, 300, 9]
    # the run ends at another chunk type (fcTL of the next frame), and the walk does not go on behind it
    f, p = apng([400, 400], chunk(b"fcTL", bytes(26)) + fdat(9, b"later") + fdat(10, b"later"))
    assert check(f, p, 2) == [400, 400]
    f, p = apng([400], chunk(b"tIME", b"1234567") + fdat(9, b"later"))
    check(f, p, 0)
    # the IDAT walker does not see an fdAT run, nor the fdAT walker the default image's IDAT
    f, p = apng([400, 400], IEND)
    assert host_run(f, p, fn="atz_host_idat_run") == py_run(f, p) == []
    assert host_run(f, f.index(b"IDAT") + 4) == []


def test_walker_short_chunks():
    """an fdAT with L < 4 ends the run (it holds no whole sequence number); a first chunk with L1 < 6 starts none"""
    f, p = apng([400, 400, 0, 300], IEND, lens=[404, 404, 3, 304])
    assert check(f, p, 2) == [400, 400]
    f, p = apng([400, 0, 300], IEND, lens=[404, 2, 304])
    check(f, p, 0)
    f, p = apng([400, 400], IEND)
    for l1 in (0, 3, 4, 5):
        h = bytearray(f); h[p - 12:p - 8] = struct.pack(">I", l1)
        assert host_run(bytes(h), p) == py_fdat_run(bytes(h), p) == [], l1
    f, p = apng([2, 400], IEND)                                   # L1 == 6: the smallest first chunk
    assert check(f, p, 2) == [2, 400]


def test_walker_end_of_file():
    f, p = apng([300, 200, 100], b"")                             # no IEND: the last chunk ends exactly at the end of the file
    assert check(f, p, 3) == [300, 200, 100]
    check(f[:-1], p, 2)                                           # the last chunk's CRC cut off: it is not part of the run
    check(f[:-4], p, 2)
    check(f[:-4 - 50], p, 2)                                      # cut in the last chunk's data
    check(f[:-(4 + 104 + 8) - 1], p, 0)                           # second chunk cut: only one left
    for k in range(1, 8):                                         # the next header itself cut off
        check(f[:p + 300 + 4 + k], p, 0)
    # lengths that run past the end of the file
    f, p = apng([300, 200], b"")
    g = bytearray(f); q = p + 300 + 4
    g[q:q + 4] = struct.pack(">I", 10 ** 6)
    check(bytes(g), p, 0)
    f, p = apng([300, 200, 50], b"")
    g = bytearray(f); q = p + 300 + 4 + 12 + 200 + 4
    g[q:q + 4] = struct.pack(">I", 0xffffffff)
    assert check(bytes(g), p, 2) == [300, 200]
    g = bytearray(f); g[p - 12:p - 8] = struct.pack(">I", 0xffffffff)
    check(bytes(g), p, 0)


def test_walker_rejects_and_cap():
    f, p = apng([400, 400], IEND)
    for q in (p - 1, p + 1, p - 4, p + 400 + 4, p + 400 + 16, 0, len(f) - 1, len(f), len(f) + 5):   # not at a piece start (or outside the file)
        assert host_run(f, q) == py_fdat_run(f, q) == [], q
    for q in range(12):                                           # p < 12, even right behind an fdAT tag and its sequence number
        g = (struct.pack(">I", 300) + b"fdAT" + struct.pack(">I", 1))[max(0, 12 - q):]
        g = (g + bytes(800))[:800]
        assert host_run(g, q) == [], q
    h = bytearray(f); h[p - 7] = ord("D")                         # "fDAT" is another chunk type
    assert host_run(bytes(h), p) == []
    # sequence numbers and CRCs are not looked at
    h = bytearray(f); h[p - 4:p] = b"\xff\xff\xff\xff"; h[p + 400:p + 404] = bytes(4)
    assert host_run(bytes(h), p) == [400, 400]
    # cap: the count is reported, only cap lengths are written
    f, p = apng([20] * 10, IEND)
    lens = (C.c_uint32 * 4)(); n = C.c_uint64()
    buf = (C.c_uint8 * len(f)).from_buffer_copy(f)
    assert az.lib().atz_host_fdat_run(buf, len(f), p, lens, 4, C.byref(n)) == 0 and n.value == 10 and list(lens) == [20] * 4
    assert az.lib().atz_host_fdat_run(buf, len(f), p, None, 0, C.byref(n)) == 0 and n.value == 10
    assert az.lib().atz_host_fdat_run(buf, len(f), p, None, 4, C.byref(n)) == az.ATZ_E_ARG


def test_both_walkers_accept_a_sequence_number_that_spells_idat():
    """the one header both kinds can start: an fdAT sequence number "IDAT" makes the 4 bytes before it ("fdAT") an IDAT length of
    0x66644154, so the IDAT run needs a 1.7 GB file; the scan takes it as an IDAT run (common.cuh split_run).  The file is an anonymous
    mapping, so only the pages written here are touched."""
    L = 0x66644154
    p = 4096
    n = p + L + 4 + 12 + 64
    mm = mmap.mmap(-1, n)
    try:
        mm[p - 12:p] = struct.pack(">I", 104) + b"fdAT" + b"IDAT"
        mm[p - 4 + 104 + 4:p - 4 + 104 + 4 + 12] = struct.pack(">I", 54) + b"fdAT" + struct.pack(">I", 7)
        q = p + L + 4                                             # the IDAT walker's second chunk: empty
        mm[q:q + 8] = struct.pack(">I", 0) + b"IDAT"
        buf = (C.c_uint8 * n).from_buffer(mm)
        lens = (C.c_uint32 * 4)(); cnt = C.c_uint64()
        assert az.lib().atz_host_fdat_run(buf, n, p, lens, 4, C.byref(cnt)) == 0 and cnt.value == 2 and list(lens[:2]) == [100, 50]
        assert az.lib().atz_host_idat_run(buf, n, p, lens, 4, C.byref(cnt)) == 0 and cnt.value == 2 and list(lens[:2]) == [L, 0]
        del buf
    finally:
        mm.close()


# ---------------------------------------------------------------------------------------------------------------------------------
def split_atz(pieces, window=0xa0 | 15, frame=16, cut=0, origlen=None):
    """an ATZ1 file with one recompressed stream split over fdAT chunks (16 framing bytes per gap); `cut` bytes are taken off its end"""
    plain = b"hello hello hello"
    z = zlib.compress(plain, 9)
    span = len(z) + frame * (len(pieces) - 1)
    desc = struct.pack("<QQQ", 5, len(z), len(plain)) + bytes([9, window, 9]) + struct.pack("<Q", 0)
    desc += struct.pack("<Q", len(pieces)) + b"".join(struct.pack("<I", x) for x in pieces) + bytes(frame * (len(pieces) - 1))
    return atz_file([desc + plain], origlen if origlen is not None else 5 + span + 5, bytes(10), cut)


def reconstruct(atz):
    with tempfile.TemporaryDirectory() as tmp:
        f = os.path.join(tmp, "x.atz")
        open(f, "wb").write(atz)
        return subprocess.run([UNCOMP, "-r", "-i", f, "-o", f + ".rec"], capture_output=True, text=True)


def test_broken_fdat_descriptors_are_rejected():
    """every broken descriptor ends in `Invalid file` and a non-zero exit before a CUDA context is created (no GPU here)"""
    c = len(zlib.compress(b"hello hello hello", 9))
    plain = b"hello hello hello"
    p1, z1 = outer()
    zin = zlib.compress(b"inner text, inner text, inner text " * 20, 9)
    kid = lambda window: (10, len(zin), record(10, len(zin), b"inner text, inner text, inner text " * 20, window))
    nested = lambda window: atz_file([record(5, len(z1), p1, 15, [kid(window)])], 5 + len(z1) + 5, bytes(10))
    cases = {
        "bit 5 without bit 7": split_atz((6, c - 6), window=0x20 | 15),
        "bit 5 without bit 7, not split": atz_file([struct.pack("<QQQ", 5, c, len(plain)) + bytes([9, 0x20 | 15, 9]) + struct.pack("<Q", 0) + plain],
                                                   5 + c + 5, bytes(10)),
        "bit 5 on a nested record": nested(0x20 | 15),
        "bits 7 and 5 on a nested record": nested(0xa0 | 15),
        "framing cut": split_atz((6, c - 6), cut=len(plain) + 10 + 5),
        "framing cut by 12-byte reading": split_atz((6, c - 6), cut=len(plain) + 10 + 2),
        "table cut": split_atz((6, c - 6), cut=len(plain) + 10 + 16 + 2),
        "span outside (16-byte gaps)": split_atz((6, c - 6), origlen=5 + c + 16 - 1),
        "span outside, three pieces": split_atz((6, 5, c - 11), origlen=5 + c + 32 - 1),
        "piece sum": split_atz((6, c - 5)),
        "npieces 1": split_atz((c,)),
        "window 0xa8": split_atz((6, c - 6), window=0xa8),
    }
    for name, atz in cases.items():
        p = reconstruct(atz)
        assert p.returncode != 0 and "Invalid file" in p.stdout, (name, p.returncode, p.stdout, p.stderr)
    # well formed (with the span that 12-byte gaps would give, it is still inside): past the checks, stopping at the device here
    from conftest import has_gpu
    for atz in (split_atz((6, c - 6)), split_atz((6, 5, c - 11)), split_atz((6, c - 6), origlen=5 + c + 16)):
        p = reconstruct(atz)
        assert "Invalid file" not in p.stdout, p.stdout
        if not has_gpu():
            assert p.returncode != 0 and "no usable CUDA device" in p.stdout


def test_help_lists_apng_after_nested():
    h = subprocess.run(["uncomp", "--help"], executable=UNCOMP, capture_output=True, text=True)
    assert h.returncode == 0
    ext = h.stdout.index("antiz_b200 extensions:")
    at = h.stdout.index("--apng")
    assert at > h.stdout.index("--nested <integer>") > ext
    tail = " ".join(h.stdout[at:].split())
    assert "fdAT" in tail and "--png" in tail and "only this program can reconstruct" in tail
    p = subprocess.run(["uncomp", "--bogus"], executable=UNCOMP, capture_output=True, text=True)
    assert p.returncode == 1 and "--apng" not in p.stderr and "--brute-window" in p.stderr


def test_constants_match_c():
    src = r'''
    #include "antiz_b200.h"
    #include <stdio.h>
    int main(){ printf("%d %d %d\n", ATZ_SCAN_SMALL_WINDOWS, ATZ_SCAN_PNG_IDAT, ATZ_SCAN_APNG_FDAT); return 0; }'''
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "consts")
        subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    assert got == [az.ATZ_SCAN_SMALL_WINDOWS, az.ATZ_SCAN_PNG_IDAT, az.ATZ_SCAN_APNG_FDAT]
    assert az.ATZ_SCAN_APNG_FDAT & (2 | 8) == 0 and bin(az.ATZ_SCAN_APNG_FDAT).count("1") == 1
    assert "atz_get_framing" in az.EXPORTS and "atz_host_fdat_run" in az.EXPORTS
