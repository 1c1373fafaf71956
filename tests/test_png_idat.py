"""ATZ_SCAN_PNG_IDAT (uncomp --png): zlib streams split over consecutive PNG IDAT chunks.  Host logic only: the IDAT run walker (the
function the run-detection kernel runs) against a restatement, and the reconstructor's checks of split-stream descriptors, which
come before any GPU work."""
import ctypes as C
import os
import struct
import subprocess
import tempfile
import zlib

import antiz_b200 as az

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")


def chunk(kind, data):
    return struct.pack(">I", len(data)) + kind + data + struct.pack(">I", zlib.crc32(kind + data))


def py_run(f, p):
    """the IDAT run that starts at p (include/antiz_b200.h ATZ_SCAN_PNG_IDAT): the data lengths of its chunks, [] if there is none"""
    n = len(f)
    if p < 8 or p >= n or f[p - 4:p] != b"IDAT":
        return []
    L = struct.unpack(">I", f[p - 8:p - 4])[0]
    if L < 2:
        return []
    out, d = [], p
    while d + L + 4 <= n:
        out.append(L)
        q = d + L + 4
        if q + 8 > n or f[q + 4:q + 8] != b"IDAT":
            break
        L = struct.unpack(">I", f[q:q + 4])[0]
        d = q + 8
    return out if len(out) >= 2 else []


def host_run(f, p, cap=4096):
    buf = (C.c_uint8 * max(len(f), 1)).from_buffer_copy(f or b"\0")
    lens = (C.c_uint32 * cap)()
    n = C.c_uint64()
    assert az.lib().atz_host_idat_run(buf, len(f), p, lens, cap, C.byref(n)) == az.ATZ_OK
    return list(lens[:min(n.value, cap)]) if n.value else []


def png(sizes, tail=b"", body=None):
    """signature, IHDR, the IDATs of the given sizes (their data a zlib header then filler), `tail`; offset of the first IDAT's data"""
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", 64, 64, 8, 2, 0, 0, 0)) + chunk(b"tEXt", b"Comment\0walker")
    first = len(out) + 8
    body = body if body is not None else b"\x78\x9c" + bytes((i * 7) & 255 for i in range(sum(sizes)))
    at = 0
    for s in sizes:
        out += chunk(b"IDAT", body[at:at + s]); at += s
    return out + tail, first


def check(f, p, want_len):
    got = host_run(f, p)
    assert got == py_run(f, p)
    assert len(got) == want_len, (got, want_len)
    return got


def test_walker_runs():
    iend = chunk(b"IEND", b"")
    check(*png([8192], iend), 0)                                  # 1 chunk: no run
    f, p = png([8192, 100], iend)
    assert check(f, p, 2) == [8192, 100]
    f, p = png([37] * 300, iend)
    assert check(f, p, 300) == [37] * 300
    f, p = png([500, 0, 0, 300, 9], iend)                         # zero-length IDATs in the middle
    assert check(f, p, 5) == [500, 0, 0, 300, 9]
    # the run ends at another chunk type, and the walk does not go on behind it
    f, p = png([400, 400], chunk(b"tIME", b"1234567") + chunk(b"IDAT", b"later"))
    assert check(f, p, 2) == [400, 400]
    f, p = png([400], chunk(b"tIME", b"1234567") + chunk(b"IDAT", b"later"))
    check(f, p, 0)


def test_walker_end_of_file():
    f, p = png([300, 200, 100], b"")                              # no IEND: the last chunk ends exactly at the end of the file
    assert check(f, p, 3) == [300, 200, 100]
    check(f[:-1], p, 2)                                           # the last chunk's CRC cut off: it is not part of the run
    check(f[:-4], p, 2)
    check(f[:-(4 + 100 + 8) - 1], p, 0)                           # second chunk cut: only one left
    # a length that runs past the end of the file
    f, p = png([300, 200], b"")
    g = bytearray(f); q = p + 300 + 4
    g[q:q + 4] = struct.pack(">I", 10 ** 6)
    check(bytes(g), p, 0)
    f, p = png([300, 200, 50], b"")
    g = bytearray(f); q = p + 300 + 4 + 8 + 200 + 4
    g[q:q + 4] = struct.pack(">I", 0xffffffff)
    assert check(bytes(g), p, 2) == [300, 200]
    check(f[:p + 300 + 4 + 7], p, 0)                              # the next header itself cut off


def test_walker_rejects():
    iend = chunk(b"IEND", b"")
    f, p = png([400, 400], iend)
    for q in (p - 1, p + 1, p + 400 + 4, 0, len(f) - 1, len(f), len(f) + 5):   # not at an IDAT data start (or outside the file)
        assert host_run(f, q) == py_run(f, q) == [], q
    for q in range(8):                                            # p < 8, even right behind an IDAT tag
        g = struct.pack(">I", 300)[:max(0, q - 4)] + b"IDAT"[-q:] if q else b""
        g = (g + bytes(400))[:400]
        assert host_run(g, q) == [], q
    h = bytearray(f); h[p - 8:p - 4] = struct.pack(">I", 1)       # L1 < 2
    assert host_run(bytes(h), p) == py_run(bytes(h), p) == []
    h = bytearray(f); h[p - 3] = ord("d")                         # "IdAT" is another chunk type
    assert host_run(bytes(h), p) == []
    # cap: the count is reported, only cap lengths are written
    f, p = png([20] * 10, iend)
    lens = (C.c_uint32 * 4)(); n = C.c_uint64()
    buf = (C.c_uint8 * len(f)).from_buffer_copy(f)
    assert az.lib().atz_host_idat_run(buf, len(f), p, lens, 4, C.byref(n)) == 0 and n.value == 10 and list(lens) == [20] * 4


# ---------------------------------------------------------------------------------------------------------------------------------
def split_atz(npieces=2, pieces=(6, 5), window=0x80 | 15, cut=0):
    """an ATZ1 file with one recompressed split stream; `cut` bytes are taken off its end"""
    plain = b"hello hello hello"
    z = zlib.compress(plain, 9)
    origlen = 5 + len(z) + 12 * max(0, len(pieces) - 1) + 5     # 5 bytes of residue before the stream, 5 after
    desc = struct.pack("<QQQ", 5, len(z), len(plain)) + bytes([9, window, 9]) + struct.pack("<Q", 0)
    desc += struct.pack("<Q", npieces) + b"".join(struct.pack("<I", x) for x in pieces)
    desc += bytes(12 * max(0, len(pieces) - 1))
    body = desc + plain + bytes(10)
    total = 28 + len(body) - cut
    return (b"ATZ\x01" + struct.pack("<QQQ", total, origlen, 1) + body)[:total]


def reconstruct(atz):
    with tempfile.TemporaryDirectory() as tmp:
        f = os.path.join(tmp, "x.atz")
        open(f, "wb").write(atz)
        return subprocess.run([UNCOMP, "-r", "-i", f, "-o", f + ".rec"], capture_output=True, text=True)


def test_broken_split_descriptors_are_rejected():
    """every broken split descriptor ends in `Invalid file` and a non-zero exit before a CUDA context is created (no GPU here)"""
    c = len(zlib.compress(b"hello hello hello", 9))
    cases = {
        "npieces 0": split_atz(npieces=0, pieces=()),
        "npieces 1": split_atz(npieces=1, pieces=(c,)),
        "npieces 2^61": split_atz(npieces=1 << 61, pieces=(6, c - 6)),
        "piece sum": split_atz(pieces=(6, c - 5)),
        "table cut": split_atz(pieces=(6, c - 6), cut=len(b"hello hello hello") + 10 + 12 + 2),
        "gaps cut": split_atz(pieces=(6, c - 6), cut=len(b"hello hello hello") + 10 + 5),
        "window 0x88": split_atz(pieces=(6, c - 6), window=0x88),
    }
    good = split_atz(pieces=(6, c - 6))
    cases["span outside"] = good[:12] + struct.pack("<Q", 5 + c + 12 - 1) + good[20:]      # original length one byte short of the span
    for name, atz in cases.items():
        p = reconstruct(atz)
        assert p.returncode != 0 and "Invalid file" in p.stdout, (name, p.returncode, p.stdout, p.stderr)


def test_help_lists_png_after_the_extensions():
    h = subprocess.run(["uncomp", "--help"], executable=UNCOMP, capture_output=True, text=True)
    assert h.returncode == 0
    ext = h.stdout.index("antiz_b200 extensions:")
    at = h.stdout.index("--png")
    assert at > ext
    tail = " ".join(h.stdout[at:].split())
    assert "IDAT" in tail and "only this program can reconstruct" in tail
    p = subprocess.run(["uncomp", "--bogus"], executable=UNCOMP, capture_output=True, text=True)
    assert p.returncode == 1 and "--png" not in p.stderr and "--brute-window" in p.stderr
