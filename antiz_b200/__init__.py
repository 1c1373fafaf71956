"""antiz_b200 - B200-native AntiZ precompression hot path.

Thin ctypes binding over the C ABI in include/antiz_b200.h (libantiz_b200.so: hand-written sm_100a CUDA
kernels + host scheduler).  This module adds no compute of its own and has no CPU path: if the shared library
or a CUDA device is missing it raises.  The reference-facing host program is antiz_b200/host/uncomp.cpp.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libantiz_b200.so")

ATZ_OK, ATZ_E_NO_DEVICE, ATZ_E_CUDA, ATZ_E_ARG, ATZ_E_TOO_LARGE = 0, -1, -2, -3, -4
ATZ_E_NOMEM, ATZ_E_DATA, ATZ_E_SMALL, ATZ_E_TRUNCATED, ATZ_E_STATE = -5, -6, -7, -8, -10
ATZ_F_EXACT_RECORDS = 1
ATZ_F_STRATEGIES = 2     # extension: also try Z_FILTERED / Z_FIXED / Z_RLE / Z_HUFFMAN_ONLY (include/antiz_b200.h)
ATZ_SCAN_SMALL_WINDOWS = 1   # extension: the scan also accepts CINFO 0 and 1 headers (offsetType 24..31, searched at window 9)
ATZ_SCAN_PNG_IDAT = 4        # extension: the scan also finds zlib streams split over consecutive PNG IDAT chunks (Context.pieces)
ATZ_SCAN_APNG_FDAT = 16      # extension: the same for APNG frames split over consecutive fdAT chunks (Context.framing)


def clevel(level, strategy=0):
    """`clevel` byte with a zlib strategy in its high nibble (ATZ_CLEVEL)"""
    return level | (strategy << 4)


def nested_depth(d):
    """Options.flags bits asking the search to recompress zlib streams nested inside recompressed ones, d levels deep (ATZ_F_NESTED_DEPTH)"""
    return d << 8
TR_COMPARED, TR_BAILED, TR_SIZE, TR_CUT = 0, 1, 2, 3


class AtzError(RuntimeError):
    def __init__(self, code, msg=""):
        super().__init__(f"antiz_b200 error {code}: {msg}")
        self.code = code


class Options(C.Structure):
    """ATZdata::programOptions (ATZData.h:7-35), defaults of parseCLI (main.cpp:1085-1093)."""
    _fields_ = [("recompTresh", C.c_uint64), ("sizediffTresh", C.c_uint64), ("shortcutLength", C.c_uint64),
                ("mismatchTol", C.c_uint64), ("bruteforceWindow", C.c_int32), ("flags", C.c_int32)]

    def __init__(self, recompTresh=128, sizediffTresh=128, shortcutLength=512, mismatchTol=2, bruteforceWindow=False, flags=0):
        super().__init__(recompTresh, sizediffTresh, shortcutLength, mismatchTol, int(bool(bruteforceWindow)), flags)


class Stream(C.Structure):
    """ATZdata::streamOffset (ATZData.h:42-77)."""
    _fields_ = [("offset", C.c_uint64), ("streamLength", C.c_uint64), ("inflatedLength", C.c_uint64), ("identBytes", C.c_uint64),
                ("firstDiffByte", C.c_int64), ("ndiff", C.c_uint64), ("diff_index", C.c_uint64), ("offsetType", C.c_int32),
                ("clevel", C.c_uint8), ("window", C.c_uint8), ("memlevel", C.c_uint8), ("recomp", C.c_uint8)]


class Nested(C.Structure):
    """atz_nested: a stream inside the plaintext of `parent` (< n_streams: a top-level stream; else entry parent - n_streams of the same list)"""
    _fields_ = [("parent", C.c_uint64), ("depth", C.c_uint32), ("reserved", C.c_uint32), ("s", Stream)]


class Stats(C.Structure):
    _fields_ = [("n_candidates", C.c_uint64), ("n_streams", C.c_uint64), ("n_recomp", C.c_uint64), ("ref_trials", C.c_uint64),
                ("gpu_trials", C.c_uint64), ("algo_bytes", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("ms_h2d", C.c_double), ("ms_scan", C.c_double), ("ms_inflate_probe", C.c_double), ("ms_inflate", C.c_double),
                ("ms_chains", C.c_double), ("ms_trials", C.c_double), ("ms_diff", C.c_double), ("ms_d2h", C.c_double),
                ("ms_trials_max_kernel", C.c_double), ("n_trial_kernels", C.c_uint64), ("trial_algo_bytes", C.c_uint64), ("ms_rows", C.c_double)]


class TrialResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("in_consumed", C.c_uint32), ("out_len", C.c_uint64), ("ident", C.c_uint64),
                ("kcycles", C.c_uint64), ("kcycles_flush", C.c_uint64)]


_lib = None


def lib():
    """Load libantiz_b200.so; fail loudly if it has not been built (python antiz_b200/build.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AtzError(ATZ_E_NO_DEVICE, f"{LIB_PATH} is missing: build it with `python antiz_b200/build.py` (there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.atz_version.restype = C.c_char_p
        L.atz_last_error.restype = C.c_char_p
        L.atz_last_error.argtypes = [C.c_void_p]
        L.atz_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.atz_ctx_destroy.argtypes = [C.c_void_p]
        L.atz_ctx_set_budget.argtypes = [C.c_void_p, C.c_uint64]
        L.atz_ctx_set_scan_flags.argtypes = [C.c_void_p, C.c_uint32]
        L.atz_load.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.atz_load_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.atz_scan.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_attach.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.atz_scan_shard.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32]
        L.atz_probe_export.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_probe_import.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64]
        L.atz_scan_finish.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.atz_host_partition.argtypes = [C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]
        L.atz_get_owners.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.c_uint64]
        L.atz_get_pieces.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32), C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_get_framing.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32)]
        L.atz_host_idat_run.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint32), C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_host_fdat_run.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint32), C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_search.argtypes = [C.c_void_p, C.POINTER(Options)]
        L.atz_search_shard.argtypes = [C.c_void_p, C.POINTER(Options), C.c_uint32, C.c_uint32]
        L.atz_get_streams.argtypes = [C.c_void_p, C.POINTER(Stream), C.c_uint64]
        L.atz_get_diffs.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_get_nested.argtypes = [C.c_void_p, C.POINTER(Nested), C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_get_inflated.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]
        L.atz_get_inflated_recomp.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_get_inflated_list.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.atz_timer_start.argtypes = [C.c_void_p]
        L.atz_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.atz_inflate_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.atz_deflate_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.atz_deflate_batch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.atz_trial.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.POINTER(Options), C.POINTER(TrialResult)]
        _lib = L
    return _lib


EXPORTS = ["atz_version", "atz_last_error", "atz_ctx_create", "atz_ctx_destroy", "atz_ctx_set_budget", "atz_ctx_set_scan_flags", "atz_load", "atz_load_device",
           "atz_scan", "atz_attach", "atz_scan_shard", "atz_probe_export", "atz_probe_import", "atz_scan_finish", "atz_host_partition", "atz_search", "atz_search_shard", "atz_get_streams", "atz_get_owners", "atz_get_pieces", "atz_get_framing", "atz_get_diffs", "atz_get_nested", "atz_get_inflated", "atz_get_inflated_recomp", "atz_get_inflated_list", "atz_get_stats", "atz_timer_start", "atz_timer_stop",
           "atz_inflate_stream", "atz_deflate_stream", "atz_deflate_batch", "atz_trial", "atz_host_fdat_run"]


def _buf(b):
    """bytes / bytearray / numpy uint8 array -> (address, length, keepalive)"""
    if isinstance(b, (bytes, bytearray)):
        arr = (C.c_uint8 * max(len(b), 1)).from_buffer_copy(bytes(b) if len(b) else b"\0")
        return C.addressof(arr), len(b), arr
    import numpy as np  # numpy arrays are passed without a copy
    a = np.ascontiguousarray(b, dtype=np.uint8)
    return a.ctypes.data, a.size, a


class Context:
    """One GPU context (one per process/GPU).  Mirrors the reference's ATZcreator phases:
    load + scan = Phase1 (main.cpp:260), search = Phase3 (main.cpp:286); results feed the ATZ1 writer."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        rc = lib().atz_ctx_create(device, C.byref(self._h))
        if rc != ATZ_OK:
            raise AtzError(rc, "atz_ctx_create failed (no sm_100a CUDA device?) - there is no CPU fallback")

    def close(self):
        if self._h:
            lib().atz_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != ATZ_OK:
            raise AtzError(rc, lib().atz_last_error(self._h).decode(errors="replace"))

    def set_budget(self, nbytes):
        self._ck(lib().atz_ctx_set_budget(self._h, nbytes))

    def set_scan_flags(self, flags):
        """the header set of the scan (ATZ_SCAN_* bits); only before the first load() / load_device() / attach()"""
        self._ck(lib().atz_ctx_set_scan_flags(self._h, flags))

    def load(self, data):
        addr, n, keep = _buf(data)
        self._ck(lib().atz_load(self._h, addr, n))

    def load_device(self, dev_ptr, n):
        self._ck(lib().atz_load_device(self._h, dev_ptr, n))

    def scan(self, chunksize=524288):
        n = C.c_uint64()
        self._ck(lib().atz_scan(self._h, chunksize, C.byref(n)))
        return n.value

    # ---- one container over several GPUs (include/antiz_b200.h, SURVEY.md 8e) ----
    def attach(self, data):
        """like load(), but the bytes stay on the host (the buffer is kept alive by this object) and only what this shard needs is uploaded"""
        addr, n, keep = _buf(data)
        self._attached = keep
        self._ck(lib().atz_attach(self._h, addr, n))

    def attach_ptr(self, addr, n):
        self._ck(lib().atz_attach(self._h, addr, n))

    def scan_shard(self, chunksize, shard, nshards):
        self._ck(lib().atz_scan_shard(self._h, chunksize, shard, nshards))

    def probe_export(self):
        n = C.c_uint64()
        lib().atz_probe_export(self._h, None, 0, C.byref(n))
        out = (C.c_uint8 * max(n.value, 1))()
        self._ck(lib().atz_probe_export(self._h, out, n.value, C.byref(n)))
        return bytes(memoryview(out)[:n.value])

    def probe_import(self, shard, blob):
        addr, n, keep = _buf(blob)
        self._ck(lib().atz_probe_import(self._h, shard, addr, n))

    def scan_finish(self):
        n = C.c_uint64()
        self._ck(lib().atz_scan_finish(self._h, C.byref(n)))
        return n.value

    def search(self, opt=None, shard=0, nshards=1):
        opt = opt or Options()
        self._ck(lib().atz_search_shard(self._h, C.byref(opt), shard, nshards))

    def timer_start(self):
        self._ck(lib().atz_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_double()
        self._ck(lib().atz_timer_stop(self._h, C.byref(ms)))
        return ms.value

    def inflated_recomp_into(self, addr, cap):
        """all recompressed streams' payloads, concatenated, into caller memory (e.g. a pinned buffer)"""
        n = C.c_uint64()
        self._ck(lib().atz_get_inflated_recomp(self._h, addr, cap, C.byref(n)))
        return n.value

    def load_ptr(self, addr, n):
        self._ck(lib().atz_load(self._h, addr, n))

    def stats(self):
        st = Stats()
        self._ck(lib().atz_get_stats(self._h, C.byref(st)))
        return st

    def streams(self):
        n = self.stats().n_streams
        arr = (Stream * max(n, 1))()
        self._ck(lib().atz_get_streams(self._h, arr, n))
        return [arr[i] for i in range(n)]

    def owners(self):
        """owner shard of every stream (atz_get_owners)"""
        import numpy as np
        n = self.stats().n_streams
        ow = np.zeros(max(n, 1), dtype=np.uint32)
        self._ck(lib().atz_get_owners(self._h, ow.ctypes.data_as(C.POINTER(C.c_uint32)), n))
        return ow[:n].tolist()

    def pieces(self, i):
        """the piece lengths of stream i in the file: [] for an ordinary stream, >= 2 for one split over PNG IDAT or APNG fdAT chunks
        (atz_get_pieces)"""
        n = C.c_uint64()
        rc = lib().atz_get_pieces(self._h, i, None, 0, C.byref(n))     # the size query: ATZ_E_SMALL for a split stream
        if rc not in (ATZ_OK, ATZ_E_SMALL):
            self._ck(rc)
        out = (C.c_uint32 * max(n.value, 1))()
        if n.value:
            self._ck(lib().atz_get_pieces(self._h, i, out, n.value, C.byref(n)))
        return list(out[:n.value])

    def framing(self, i):
        """the bytes between two pieces of stream i in the file: 0 for an ordinary stream, 12 for IDAT chunks, 16 for fdAT chunks
        (atz_get_framing)"""
        b = C.c_uint32()
        self._ck(lib().atz_get_framing(self._h, i, C.byref(b)))
        return b.value

    def stream_table(self):
        """the same records as one numpy structured array (field names of Stream), without a Python object per stream"""
        import numpy as np
        n = self.stats().n_streams
        arr = (Stream * max(n, 1))()
        self._ck(lib().atz_get_streams(self._h, arr, n))
        dt = np.dtype({"names": [f[0] for f in Stream._fields_], "formats": [np.dtype(f[1]) for f in Stream._fields_],
                       "offsets": [getattr(Stream, f[0]).offset for f in Stream._fields_], "itemsize": C.sizeof(Stream)})
        return np.frombuffer(arr, dtype=dt, count=n).copy()

    def diffs(self):
        n = C.c_uint64()
        rc = lib().atz_get_diffs(self._h, None, None, 0, C.byref(n))
        if n.value == 0:
            return [], b""
        offs = (C.c_uint64 * n.value)()
        vals = (C.c_uint8 * n.value)()
        self._ck(lib().atz_get_diffs(self._h, offs, vals, n.value, C.byref(n)))
        return list(offs), bytes(vals)

    def nested(self):
        """the nested streams of the last search (atz_get_nested): Nested records, level by level, then by parent, then by offset; the
        payload of entry j is inflated(n_streams + j, ...)"""
        n = C.c_uint64()
        rc = lib().atz_get_nested(self._h, None, 0, C.byref(n))
        if rc not in (ATZ_OK, ATZ_E_SMALL):
            self._ck(rc)
        arr = (Nested * max(n.value, 1))()
        if n.value:
            self._ck(lib().atz_get_nested(self._h, arr, n.value, C.byref(n)))
        return [arr[i] for i in range(n.value)]

    def inflated(self, i, length):
        out = (C.c_uint8 * max(length, 1))()
        self._ck(lib().atz_get_inflated(self._h, i, out, length))
        return bytes(out[:length]) if length else b""

    def inflated_recomp(self):
        n = C.c_uint64()
        lib().atz_get_inflated_recomp(self._h, None, 0, C.byref(n))
        out = (C.c_uint8 * max(n.value, 1))()
        if n.value:
            self._ck(lib().atz_get_inflated_recomp(self._h, out, n.value, C.byref(n)))
        return bytes(memoryview(out)[:n.value])

    def inflate_stream(self, data, cap):
        addr, n, keep = _buf(data)
        out = (C.c_uint8 * max(cap, 1))()
        olen, used = C.c_uint64(), C.c_uint64()
        rc = lib().atz_inflate_stream(self._h, addr, n, out, cap, C.byref(olen), C.byref(used))
        return rc, bytes(memoryview(out)[:min(olen.value, cap)]) if rc == ATZ_OK else b"", used.value

    def deflate_stream(self, data, clevel, window, memlevel, cap=None):
        addr, n, keep = _buf(data)
        cap = cap if cap is not None else n + n // 8 + 1024
        out = (C.c_uint8 * max(cap, 1))()
        olen = C.c_uint64()
        self._ck(lib().atz_deflate_stream(self._h, addr, n, clevel, window, memlevel, out, cap, C.byref(olen)))
        return bytes(memoryview(out)[:olen.value])

    def deflate_batch(self, items):
        """items: list of (plaintext bytes, clevel, window, memlevel) -> list of zlib streams (one kernel launch per group)."""
        n = len(items)
        if n == 0:
            return []
        blob = b"".join(it[0] for it in items)
        addr, _, keep = _buf(blob)
        in_off = (C.c_uint64 * n)(); in_len = (C.c_uint64 * n)(); out_off = (C.c_uint64 * n)(); out_cap = (C.c_uint64 * n)(); out_len = (C.c_uint64 * n)()
        lv = (C.c_uint8 * n)(); wb = (C.c_uint8 * n)(); ml = (C.c_uint8 * n)()
        o = oo = 0
        for i, (d, c, w, m) in enumerate(items):
            in_off[i] = o; in_len[i] = len(d); o += len(d)
            out_off[i] = oo; out_cap[i] = len(d) + len(d) // 8 + 1024; oo += out_cap[i]
            lv[i] = c; wb[i] = w; ml[i] = m
        out = (C.c_uint8 * oo)()
        self._ck(lib().atz_deflate_batch(self._h, addr, in_off, in_len, lv, wb, ml, n, out, out_off, out_cap, out_len))
        mv = memoryview(out)
        return [bytes(mv[out_off[i]:out_off[i] + out_len[i]]) for i in range(n)]

    def trial(self, plain, orig, clevel, window, memlevel, opt=None):
        opt = opt or Options()
        a1, n1, k1 = _buf(plain)
        a2, n2, k2 = _buf(orig)
        r = TrialResult()
        self._ck(lib().atz_trial(self._h, a1, n1, a2, n2, clevel, window, memlevel, C.byref(opt), C.byref(r)))
        return r


def partition(inflated_lengths, nshards, probed_by=None):
    """owner shard of every accepted stream (atz_host_partition); probed_by: the shard whose chunk range each stream starts in"""
    import numpy as np
    ul = np.ascontiguousarray(inflated_lengths, dtype=np.uint64)
    n = int(ul.size)
    ow = np.zeros(max(n, 1), dtype=np.uint32)
    pb = None
    if probed_by is not None:
        pb = np.ascontiguousarray(probed_by, dtype=np.uint32)
        assert pb.size == n
    rc = lib().atz_host_partition(ul.ctypes.data_as(C.POINTER(C.c_uint64)), pb.ctypes.data_as(C.POINTER(C.c_uint32)) if pb is not None else None, n, nshards,
                                  ow.ctypes.data_as(C.POINTER(C.c_uint32)))
    if rc != ATZ_OK:
        raise AtzError(rc, "atz_host_partition")
    return ow[:n].tolist()
