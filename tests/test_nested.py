"""ATZ_F_NESTED_DEPTH (uncomp --nested N): zlib streams inside the plaintext of recompressed streams.  Host logic only: the header
property that lets the scan buffer put parents side by side with zero gaps, the reconstructor's checks of nested records, which come
before any GPU work, and the help text."""
import ctypes as C
import os
import struct
import subprocess
import tempfile
import zlib

import antiz_b200 as az

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")


def test_no_header_starts_in_or_runs_into_a_zero_gap():
    """K1 runs over parents separated by zero bytes without segment logic: no accepted header has a 0x00 byte on either side"""
    for flags in (0, az.ATZ_SCAN_SMALL_WINDOWS):
        assert az.lib().atz_host_header_type(flags, 0, 0) == -1
        for b in range(256):
            assert az.lib().atz_host_header_type(flags, b, 0) == -1, (flags, b)
            assert az.lib().atz_host_header_type(flags, 0, b) == -1, (flags, b)


# ---------------------------------------------------------------------------------------------------------------------------------
# A writer of the nested layout (uncomp.cpp writeATZfile): descriptor, diffs, then the payload - or, with bit 6 of the window byte,
# u64 nchild, the child records in offset order and the parent's plaintext without the children's bytes.
def record(off, c, plain, window=15, kids=None, nchild=None):
    """kids: list of (offset in plain, compressed length, record bytes); nchild overrides the count written"""
    d = struct.pack("<QQQ", off, c, len(plain))
    if not kids:
        return d + bytes([9, window, 9]) + struct.pack("<Q", 0) + plain
    body = struct.pack("<Q", len(kids) if nchild is None else nchild) + b"".join(k[2] for k in kids)
    res, at = b"", 0
    for o, cl, _ in sorted(kids, key=lambda k: k[0]):
        res += plain[at:o]; at = max(at, o + cl)
    return d + bytes([9, window | 0x40, 9]) + struct.pack("<Q", 0) + body + res + plain[at:]


def atz_file(recs, origlen, residue, cut=0):
    body = b"".join(recs) + residue
    total = 28 + len(body) - cut
    return (b"ATZ\x01" + struct.pack("<QQQ", total, origlen, len(recs)) + body)[:total]


INNER = b"inner text, inner text, inner text " * 20
ZIN = zlib.compress(INNER, 9)


def outer(kids_at=(10,), n=None):
    """(plaintext of the outer stream with ZIN at each offset of kids_at, its zlib stream)"""
    p = bytearray(b"-" * (n or 400 + max(kids_at) + len(ZIN)))
    for o in kids_at:
        p[o:o + len(ZIN)] = ZIN
    p = bytes(p)
    return p, zlib.compress(p, 6)


def one(kids, plain, z, window=15, nchild=None):
    return atz_file([record(5, len(z), plain, window, kids, nchild)], 5 + len(z) + 5, bytes(10))


def child(o, window=15, kids=None):
    return (o, len(ZIN), record(o, len(ZIN), INNER, window, kids))


def reconstruct(atz):
    with tempfile.TemporaryDirectory() as tmp:
        f = os.path.join(tmp, "x.atz")
        open(f, "wb").write(atz)
        return subprocess.run([UNCOMP, "-r", "-i", f, "-o", f + ".rec"], capture_output=True, text=True)


def chain(levels):
    """a record nested `levels` deep: every level holds one child at offset 0 (the sizes only have to fit the file)"""
    rec = record(0, 20, bytes(100))
    for _ in range(levels):
        rec = struct.pack("<QQQ", 0, 20, 100) + bytes([9, 15 | 0x40, 9]) + struct.pack("<Q", 0) + struct.pack("<Q", 1) + rec + bytes(80)
    return rec


def test_broken_nested_descriptors_are_rejected():
    """every broken nested record ends in `Invalid file` and a non-zero exit before a CUDA context is created"""
    p2, z2 = outer((10, 200))
    p1, z1 = outer()
    cases = {
        "not ascending": one([child(200), child(10)], p2, z2),
        "overlapping": one([child(10), child(10 + len(ZIN) - 1)], p2, z2),
        "offset at U": one([(len(p1), len(ZIN), record(len(p1), len(ZIN), INNER))], p1, z1),
        "past U": one([(len(p1) - 5, len(ZIN), record(len(p1) - 5, len(ZIN), INNER))], p1, z1),
        "nchild 0": one([child(10)], p1, z1, nchild=0),
        "nchild 2^61": one([child(10)], p1, z1, nchild=1 << 61),
        "bit 7 on a child": one([(10, len(ZIN), record(10, len(ZIN), INNER, window=0x80 | 15))], p1, z1),
        "bad child window": one([(10, len(ZIN), record(10, len(ZIN), INNER, window=8))], p1, z1),
        "truncated": one([child(10)], p1, z1)[:-11],
        "child payload cut": one([child(10)], p1, z1)[:28 + 35 + 8 + 35 + 40],
        "depth 9": atz_file([struct.pack("<QQQ", 0, 20, 100) + bytes([9, 15 | 0x40, 9]) + struct.pack("<Q", 0) + struct.pack("<Q", 1) + chain(8) + bytes(80)],
                            20, b""),
    }
    for name, atz in cases.items():
        p = reconstruct(atz)
        assert p.returncode != 0 and "Invalid file" in p.stdout, (name, p.returncode, p.stdout, p.stderr)
    # the same layouts, well formed, get past the checks (here they stop at the device, or reconstruct on a GPU)
    for name, atz in {"one": one([child(10)], p1, z1), "two": one([child(10), child(200)], p2, z2),
                      "depth 8": atz_file([struct.pack("<QQQ", 0, 20, 100) + bytes([9, 15 | 0x40, 9]) + struct.pack("<Q", 0) + struct.pack("<Q", 1) + chain(7) + bytes(80)], 20, b"")}.items():
        p = reconstruct(atz)
        assert "Invalid file" not in p.stdout, (name, p.stdout)


def test_good_nested_file_reconstructs_where_there_is_a_gpu():
    from conftest import has_gpu
    p1, z1 = outer((0, 10 + len(ZIN)))
    kids = [child(0), child(10 + len(ZIN), kids=[])]
    atz = one(kids, p1, z1)
    p = reconstruct(atz)
    if not has_gpu():
        assert p.returncode != 0 and "no usable CUDA device" in p.stdout and "Invalid file" not in p.stdout
        return
    assert p.returncode == 0, p.stdout


def test_help_lists_nested_after_the_extensions():
    h = subprocess.run(["uncomp", "--help"], executable=UNCOMP, capture_output=True, text=True)
    assert h.returncode == 0
    ext = h.stdout.index("antiz_b200 extensions:")
    at = h.stdout.index("--nested <integer>")
    assert at > ext
    tail = " ".join(h.stdout[at:].split())
    assert "only this program can reconstruct" in tail
    p = subprocess.run(["uncomp", "--bogus"], executable=UNCOMP, capture_output=True, text=True)
    assert p.returncode == 1 and "--nested" not in p.stderr
    p = subprocess.run(["uncomp", "--nested", "9", "-i", "x"], executable=UNCOMP, capture_output=True, text=True)
    assert p.returncode == 1 and "at most 8" in p.stderr


def test_nested_struct_matches_c():
    src = r'''
    #include "antiz_b200.h"
    #include <stdio.h>
    #include <stddef.h>
    int main(){ printf("%zu %zu %d\n", sizeof(atz_nested), offsetof(atz_nested, s), ATZ_F_NESTED_DEPTH(3)); return 0; }'''
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "sizes")
        subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    assert got == [C.sizeof(az.Nested), az.Nested.s.offset, az.nested_depth(3)]
    assert "atz_get_nested" in az.EXPORTS
