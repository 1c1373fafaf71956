"""ctypes access to zlib - the *reference's own* zlib 1.2.8 (oracle/_ref/libz128.so, built by oracle/build_ref.sh where the
reference sources are present), else the host's zlib - and to the CPU oracle (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY - nothing under antiz_b200/ imports this module.
"""
import ctypes as C
import ctypes.util
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libz128.so")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "uncomp_ref")
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")

Z_OK, Z_STREAM_END, Z_NEED_DICT, Z_DATA_ERROR, Z_BUF_ERROR = 0, 1, 2, -3, -5
Z_SYNC_FLUSH, Z_FINISH = 2, 4


class ZStream(C.Structure):
    _fields_ = [
        ("next_in", C.c_void_p), ("avail_in", C.c_uint), ("total_in", C.c_ulong),
        ("next_out", C.c_void_p), ("avail_out", C.c_uint), ("total_out", C.c_ulong),
        ("msg", C.c_char_p), ("state", C.c_void_p),
        ("zalloc", C.c_void_p), ("zfree", C.c_void_p), ("opaque", C.c_void_p),
        ("data_type", C.c_int), ("adler", C.c_ulong), ("reserved", C.c_ulong),
    ]


_ref = None
_host = None
_oracle = None


def have_ref():
    return os.path.exists(REF_SO)


def ref():
    global _ref
    if _ref is None:
        _ref = C.CDLL(REF_SO)
        _ref.zlibVersion.restype = C.c_char_p
        assert _ref.zlibVersion() == b"1.2.8", _ref.zlibVersion()
    return _ref


def host_zlib():
    """the host's zlib (the library Python's zlib module uses).  Its deflate output equals zlib 1.2.8's at levels 1-9 with the
    default and Z_FILTERED strategies (test_oracle_deflate checks that against the committed 1.2.8 digests), and on the inputs of
    test_deflate_strategies_bit_exact with every strategy; level 0 differs (stored blocks, rewritten in zlib 1.2.11), and Z_FIXED
    can (block choice changed in 1.2.12).  Its inflate accounting agrees with the oracle's (test_oracle_inflate)."""
    global _host
    if _host is None:
        _host = C.CDLL(ctypes.util.find_library("z") or "libz.so.1")
        _host.zlibVersion.restype = C.c_char_p
    return _host


def zlib_lib():
    """what the ref_* helpers call: zlib 1.2.8 where the reference has been built, the host's zlib everywhere else (ref_deflate
    then takes level 0 from the oracle, which lays out stored blocks as 1.2.8 does)"""
    return ref() if have_ref() else host_zlib()


def build_oracle():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"])


def oracle():
    global _oracle
    if _oracle is None:
        if not os.path.exists(ORACLE_SO):
            build_oracle()
        o = C.CDLL(ORACLE_SO)
        o.oracle_deflate.restype = C.c_longlong
        o.oracle_deflate.argtypes = [C.c_char_p, C.c_uint32, C.c_int, C.c_int, C.c_int,
                                     C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint32)]
        o.oracle_adler32.restype = C.c_uint32
        o.oracle_adler32.argtypes = [C.c_char_p, C.c_uint64]
        _oracle = o
    return _oracle


def ref_deflate(data: bytes, level: int, wbits: int, memlevel: int, strategy: int = 0, z=None) -> bytes:
    """deflateInit2(level, 8, wbits, memlevel, strategy) + deflate(Z_FINISH) with `z` or zlib_lib() (strategy 1 = Z_FILTERED)."""
    if z is None and not have_ref() and level == 0 and strategy == 0:
        return oracle_deflate(data, level, wbits, memlevel)
    z = z or zlib_lib()
    s = ZStream()
    rc = z.deflateInit2_(C.byref(s), level, 8, wbits, memlevel, strategy, b"1.2.8", C.sizeof(ZStream))
    assert rc == Z_OK, rc
    z.deflateBound.restype = C.c_ulong
    cap = z.deflateBound(C.byref(s), C.c_ulong(len(data))) + 64
    src = C.create_string_buffer(data, len(data) + 1)
    dst = C.create_string_buffer(cap)
    s.next_in = C.addressof(src); s.avail_in = len(data)
    s.next_out = C.addressof(dst); s.avail_out = cap
    rc = z.deflate(C.byref(s), Z_FINISH)
    assert rc == Z_STREAM_END, rc
    n = s.total_out
    z.deflateEnd(C.byref(s))
    return dst.raw[:n]


def ref_deflate_ex(data: bytes, level: int, wbits: int, memlevel: int, strategy: int = 0, flushes=(), tune=None) -> bytes:
    """zlib_lib() driven the way other encoders drive it: `flushes` = [(input offset, flush mode)] (1 Z_PARTIAL_FLUSH, 2 Z_SYNC_FLUSH,
    3 Z_FULL_FLUSH, 5 Z_BLOCK) applied once the input up to that offset has been fed, then Z_FINISH; `tune` = deflateTune's
    (good_length, max_lazy, nice_length, max_chain).  Streams made like this inflate to `data` but are not what any plain
    deflateInit2 + deflate(Z_FINISH) produces: the search finds an imperfect winner or none."""
    z = zlib_lib()
    s = ZStream()
    rc = z.deflateInit2_(C.byref(s), level, 8, wbits, memlevel, strategy, b"1.2.8", C.sizeof(ZStream))
    assert rc == Z_OK, rc
    if tune:
        assert z.deflateTune(C.byref(s), *tune) == Z_OK
    cap = len(data) + len(data) // 4 + 1024 + 64 * (len(flushes) + 1)
    src = C.create_string_buffer(data, len(data) + 1)
    dst = C.create_string_buffer(cap)
    s.next_out = C.addressof(dst); s.avail_out = cap
    fed = 0
    for off, mode in list(flushes) + [(len(data), Z_FINISH)]:
        s.next_in = C.addressof(src) + fed; s.avail_in = off - fed; fed = off
        rc = z.deflate(C.byref(s), mode)
        assert rc in (Z_OK, Z_STREAM_END) and s.avail_in == 0, rc
    assert rc == Z_STREAM_END
    n = s.total_out
    z.deflateEnd(C.byref(s))
    return dst.raw[:n]


def oracle_deflate(data: bytes, level: int, wbits: int, memlevel: int, limit_out: int = 0):
    o = oracle()
    cap = len(data) + len(data) // 8 + 1024
    dst = C.create_string_buffer(cap)
    at = C.c_uint32(0)
    n = o.oracle_deflate(data, len(data), level, wbits, memlevel, dst, cap, limit_out, C.byref(at))
    assert 0 <= n <= cap, n
    if limit_out:
        return dst.raw[:n], at.value
    return dst.raw[:n]


FLUSH_COUNTERS = ("over_lit", "over_dist", "over_bl",
                  "force_lit_low", "force_lit_high", "force_dist_low", "force_dist_high", "force_bl_low", "force_bl_high",
                  "stored", "static", "dynamic", "unstorable", "tie_stored", "tie_static",
                  "rep16_6", "rep17_3", "rep17_10", "rep18_11", "rep18_138", "zrun_split")


def oracle_flush_counts():
    """Branch counters of the oracle's block flush since the last call (which resets them), by name:
    over_*: gen_bitlen's depth-limit repair of the literal/length, distance and bit-length tree (Z/trees.c:530-564);
    force_*_low / _high: build_tree's heap_len < 2 forcing with max_code < 2 / >= 2 (Z/trees.c:648-654);
    stored / static / dynamic: block kinds written; unstorable: flushes whose block start has slid out of the window (buf == NULL);
    tie_stored: stored_len + 4 == opt_lenb with a stored block written; tie_static: static_lenb == opt_lenb == the dynamic size;
    rep16_6, rep17_3, rep17_10, rep18_11, rep18_138: scan_tree runs at the limits of their codes; zrun_split: a zero run over 138."""
    o = oracle()
    n = len(FLUSH_COUNTERS)
    buf = (C.c_uint64 * n)()
    assert o.oracle_flush_counts(buf, n) == n
    return dict(zip(FLUSH_COUNTERS, buf))


def ref_inflate_scan(buf: bytes, start: int, outcap: int, segments=None):
    """Re-enact ZBuffSearcher's calls on one candidate (main.cpp:228-239): inflateInit,
    inflate(Z_SYNC_FLUSH) with avail_in = len(buf)-start, avail_out = outcap, then drain
    while avail_out == 0.  Returns (first_total_in, ret, total_in, total_out, avail_in).
    """
    z = zlib_lib()
    s = ZStream()
    rc = z.inflateInit_(C.byref(s), b"1.2.8", C.sizeof(ZStream))
    assert rc == Z_OK
    src = C.create_string_buffer(buf, len(buf) + 1)
    dst = C.create_string_buffer(outcap)
    s.next_in = C.addressof(src) + start; s.avail_in = len(buf) - start
    s.next_out = C.addressof(dst); s.avail_out = outcap
    ret = z.inflate(C.byref(s), Z_SYNC_FLUSH)
    first_in = s.total_in
    while s.avail_out == 0:
        s.next_out = C.addressof(dst); s.avail_out = outcap
        ret = z.inflate(C.byref(s), Z_SYNC_FLUSH)
    res = (first_in, ret, s.total_in, s.total_out, s.avail_in)
    z.inflateEnd(C.byref(s))
    return res


def ref_inflate(data: bytes, outlen: int):
    """doInflate (main.cpp:461-486): one-shot inflate(Z_FINISH)."""
    z = zlib_lib()
    s = ZStream()
    assert z.inflateInit_(C.byref(s), b"1.2.8", C.sizeof(ZStream)) == Z_OK
    src = C.create_string_buffer(data, len(data) + 1)
    dst = C.create_string_buffer(max(outlen, 1))
    s.next_in = C.addressof(src); s.avail_in = len(data)
    s.next_out = C.addressof(dst); s.avail_out = outlen
    ret = z.inflate(C.byref(s), Z_FINISH)
    n, ti = s.total_out, s.total_in
    z.inflateEnd(C.byref(s))
    return ret, dst.raw[:n], ti


class OIResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("err", C.c_int32), ("total_in", C.c_uint64),
                ("total_out", C.c_uint64), ("in_at_outcap", C.c_uint64), ("adler", C.c_uint32)]


class OISeg(C.Structure):
    _fields_ = [("p", C.c_void_p), ("n", C.c_uint64)]


OI_END, OI_NEED_INPUT, OI_DATA_ERROR, OI_NEED_DICT, OI_OUT_FULL = 0, 1, 2, 3, 4


def oracle_inflate(data: bytes, out_cap=None, first_out_cap=0):
    """Returns (OIResult, output bytes or None).  out_cap=None -> discard mode (32K ring)."""
    o = oracle()
    r = OIResult()
    src = C.create_string_buffer(data, len(data) + 1)
    if out_cap is None:
        o.oracle_inflate(src, C.c_uint64(len(data)), None, C.c_uint64(0), C.c_uint64(first_out_cap), C.byref(r))
        return r, None
    dst = C.create_string_buffer(max(out_cap, 1))
    o.oracle_inflate(src, C.c_uint64(len(data)), dst, C.c_uint64(out_cap), C.c_uint64(first_out_cap), C.byref(r))
    return r, dst.raw[:min(r.total_out, out_cap)]


def oracle_deflate_listmode(data: bytes, level: int, wbits: int, memlevel: int) -> bytes:
    """CPU design model of the GPU 'list mode' deflate (oracle/zdeflate.c, bottom)."""
    o = oracle()
    o.oracle_deflate_listmode.restype = C.c_longlong
    cap = len(data) + len(data) // 8 + 1024
    dst = C.create_string_buffer(cap)
    n = o.oracle_deflate_listmode(data, C.c_uint32(len(data)), level, wbits, memlevel, dst, C.c_uint64(cap))
    assert 0 <= n <= cap, n
    return dst.raw[:n]
