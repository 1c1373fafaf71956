"""Host logic of the product pinned on the CPU: the reference's candidate order (SURVEY.md A.2), chunk list and the
ZBuffSearcher accept logic (A.1).  The accept logic is driven with probe records from the CPU oracle and compared with
what the reference binary (oracle/_ref/uncomp_ref) finds on the same file - or, where it has not been built, with the stored
record of what it finds (tests/golden/atz_reference.json)."""
import ctypes as C
import hashlib
import json
import os
import random
import struct
import subprocess
import tempfile

import pytest

import antiz_b200 as az
import corpus
import zref


def seq(ot, brute):
    L = az.lib()
    c = (C.c_uint8 * 512)(); w = (C.c_uint8 * 512)(); m = (C.c_uint8 * 512)()
    n = L.atz_host_candidate_sequence(ot, brute, c, w, m, 512)
    return [(c[i], w[i], m[i]) for i in range(n)]


def test_candidate_order_counts_and_heads():
    for ot in range(24):
        w = 10 + ot // 4
        s = seq(ot, 0)
        assert len(s) == (82 if ot % 4 == 0 else 81)
        assert len(set(s)) == len(s) and all(x[1] == w for x in s)
        assert {(c, m) for c, _, m in s} >= {(c, m) for c in range(1, 10) for m in range(1, 10)}
        b = seq(ot, 1)
        assert len(b) == 405 and len(set(b)) == 405 and all(x[1] != w for x in b)
    assert seq(20, 0)[:4] == [(0, 15, 8), (1, 15, 8), (1, 15, 9), (1, 15, 7)]          # main.cpp:489-503
    assert seq(21, 0)[:5] == [(5, 15, 8), (4, 15, 8), (3, 15, 8), (2, 15, 8), (5, 15, 7)]  # main.cpp:514-520
    assert seq(22, 0)[:4] == [(6, 15, 8), (6, 15, 9), (6, 15, 7), (6, 15, 6)]          # main.cpp:528-540
    assert seq(23, 0)[:4] == [(9, 15, 8), (8, 15, 8), (7, 15, 8), (9, 15, 7)]          # main.cpp:550-556
    assert seq(22, 1)[0] == (9, 14, 9) and seq(22, 1)[-1] == (1, 10, 1)                # main.cpp:595
    assert seq(2, 1)[0] == (9, 15, 9) and seq(2, 1)[-1] == (1, 11, 1)                  # main.cpp:592
    mid = seq(14, 1)                                                                   # window 13: 12..10 then 15..14 (main.cpp:597-598)
    assert [x[1] for x in mid[::81]] == [12, 11, 10, 15, 14]
    # measured trials-to-first-match of SURVEY.md A.2 follow from the order
    assert seq(21, 0).index((2, 15, 9)) + 1 == 36 and seq(22, 0).index((6, 15, 5)) + 1 == 5


def test_chunk_list():
    L = az.lib()

    def chunks(n, s):
        a = (C.c_uint64 * 4096)(); b = (C.c_uint64 * 4096)()
        k = L.atz_host_chunks(n, s, a, b, 4096)
        return [(a[i], b[i]) for i in range(k)]
    assert chunks(10, 100) == [(0, 10)]
    assert chunks(100, 100) == [(0, 100), (99, 1)]            # a read that exactly fills the buffer does not set eof (main.cpp:410)
    assert chunks(101, 100) == [(0, 100), (99, 2)]
    assert chunks(298, 100) == [(0, 100), (99, 100), (198, 100), (297, 1)]
    assert chunks(250, 100) == [(0, 100), (99, 100), (198, 52)]


def test_header_closed_form_equals_the_reference_switch():
    """K1's closed form (csrc/scan.cu is_magic + the type formula; SURVEY.md 8 a1) against parseOffsetType's 24-way switch
    (main.cpp:168-203), over all 65,536 byte pairs"""
    table = [0x2815, 0x2853, 0x2891, 0x28cf, 0x3811, 0x384f, 0x388d, 0x38cb, 0x480d, 0x484b, 0x4889, 0x48c7,
             0x5809, 0x5847, 0x5885, 0x58c3, 0x6805, 0x6843, 0x6881, 0x68de, 0x7801, 0x785e, 0x789c, 0x78da]
    want = {h: i for i, h in enumerate(table)}
    for b0 in range(256):
        for b1 in range(256):
            hit = (b0 & 0x8f) == 0x08 and b0 >= 0x28 and (b1 & 0x20) == 0 and ((b0 << 8) | b1) % 31 == 0
            # the 4-bytes-at-a-time prefilter of the kernel must never drop a header
            pre = (b0 & 0x8f) == 0x08 and b0 >= 0x28
            assert hit == (((b0 << 8) | b1) in want) and (pre or not hit)
            if hit:
                assert 4 * ((b0 >> 4) - 2) + (b1 >> 6) == want[(b0 << 8) | b1]


def test_strategy_sequence_extension():
    """ATZ_F_STRATEGIES: 54 Z_FILTERED (levels 9..4) + 81 Z_FIXED + 9 Z_RLE + 9 Z_HUFFMAN_ONLY candidates at the header's window"""
    L = az.lib()
    c = (C.c_uint8 * 600)(); w = (C.c_uint8 * 600)(); m = (C.c_uint8 * 600)()
    for ty in (0, 9, 22):
        n = L.atz_host_candidate_sequence(ty, 2, c, w, m, 600)
        assert n == 153
        seq = [(c[i] & 15, c[i] >> 4, w[i], m[i]) for i in range(n)]
        assert all(x[2] == 10 + ty // 4 for x in seq) and len(set(seq)) == n
        assert [x[1] for x in seq] == [1] * 54 + [4] * 81 + [3] * 9 + [2] * 9
        assert seq[0] == (9, 1, 10 + ty // 4, 9) and min(x[0] for x in seq[:54]) == 4


def _magic_positions(data):
    ok = {0x2815, 0x2853, 0x2891, 0x28cf, 0x3811, 0x384f, 0x388d, 0x38cb, 0x480d, 0x484b, 0x4889, 0x48c7,
          0x5809, 0x5847, 0x5885, 0x58c3, 0x6805, 0x6843, 0x6881, 0x68de, 0x7801, 0x785e, 0x789c, 0x78da}
    return [i for i in range(len(data) - 1) if (data[i] << 8 | data[i + 1]) in ok]


def _fold_with_oracle(data, S):
    """what atz_scan does, with the CPU oracle standing in for the K1/K2 kernels - including the reference's overlap-byte quirk
    (searchInfile keeps rBuffer[gcount - 1], main.cpp:408-413: the first byte of chunk k >= 2 is file[start_k - 1])"""
    L = az.lib(); o = zref.oracle()
    n = len(data)
    a = (C.c_uint64 * 65536)(); b = (C.c_uint64 * 65536)()
    nch = L.atz_host_chunks(n, S, a, b, 65536)
    cstart = [a[i] for i in range(nch)]; clen = [b[i] for i in range(nch)]
    ok = set(_magic_positions(data))
    special = set()
    for k in range(2, nch):
        p = cstart[k]
        ok.discard(p)
        if p + 1 < n and _magic_positions(bytes([data[p - 1], data[p + 1]])):
            ok.add(p); special.add(p)
    cand = sorted(ok)
    buf = C.create_string_buffer(data, n + 1)
    base = C.addressof(buf)

    def chunk_segs(j, first):
        """(ptr, n) pieces of chunk j as the reference's buffer holds it; `first`: start at this file position instead of the chunk start"""
        if first is not None:
            if first in special:
                return [(base + first - 1, 1), (base + first + 1, cstart[j] + clen[j] - first - 1)]
            return [(base + first, cstart[j] + clen[j] - first)]
        head = cstart[j] - 1 if j >= 2 else cstart[j]
        return [(base + head, 1), (base + cstart[j] + 1, clen[j] - 1)]

    def run(pieces, first_cap):
        pieces = [p for p in pieces if p[1] > 0]
        segs = (zref.OISeg * len(pieces))()
        for i, (ptr, ln) in enumerate(pieces):
            segs[i].p = ptr; segs[i].n = ln
        r = zref.OIResult()
        o.oracle_inflate_segs(segs, len(pieces), None, C.c_uint64(0), C.c_uint64(first_cap), C.byref(r))
        return r

    probe = []; avail = []; cont_of = []; cont = []
    for f in cand:
        c = f // (S - 1)
        av = cstart[c] + clen[c] - f
        r = run(chunk_segs(c, f), S)
        probe += [r.status, r.total_in, r.total_out, r.in_at_outcap]; avail.append(av)
        if r.status == zref.OI_NEED_INPUT and r.in_at_outcap > 16:
            pieces = chunk_segs(c, f)
            for j in range(c + 1, nch):
                pieces += chunk_segs(j, None)
            r2 = run(pieces, 0)
            cont_of.append(len(cont) // 4); cont += [r2.status, r2.total_in, r2.total_out, r2.in_at_outcap]
        else:
            cont_of.append(-1)
    nc = len(cand)
    out = (C.c_uint64 * (3 * (nc + 8)))()
    k = L.atz_host_scan_fold(n, S, (C.c_uint32 * max(nc, 1))(*cand), nc, (C.c_uint64 * max(4 * nc, 1))(*probe), (C.c_uint64 * max(nc, 1))(*avail),
                             (C.c_int32 * max(nc, 1))(*cont_of), (C.c_uint64 * max(len(cont), 1))(*cont), len(cont) // 4, out, nc + 8)
    return [(out[3 * i], out[3 * i + 1], out[3 * i + 2]) for i in range(k)]


GOLDEN_ATZ = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "atz_reference.json")


def atz_streams(exe, data, S, tmp):
    """(headers found, [(offset, streamLength, inflatedLength) of every recompressed stream]) of `exe -i file --notest --chunksize S`"""
    f = os.path.join(tmp, "in.bin")
    open(f, "wb").write(data)
    out = subprocess.check_output([exe, "-i", f, "--notest", "--chunksize", str(S)]).decode()
    found = int([l for l in out.splitlines() if l.startswith("Total zlib headers found")][0].split(":")[1])
    atz = open(f + ".atz", "rb").read()
    nrec = struct.unpack_from("<Q", atz, 20)[0]
    pos = 28; recs = []
    for _ in range(nrec):
        off, c, u = struct.unpack_from("<QQQ", atz, pos); nd = struct.unpack_from("<Q", atz, pos + 27)[0]
        recs.append((off, c, u)); pos += 35 + (8 + 9 * nd if nd else 0) + u
    return found, recs


def _reference_streams(key, data, S, tmp):
    if os.path.exists(zref.REF_BIN):
        return atz_streams(zref.REF_BIN, data, S, tmp)
    g = json.load(open(GOLDEN_ATZ))[key]
    assert g["chunksize"] == S and g["input_sha256"] == hashlib.sha256(data).hexdigest(), f"{key}: not the input the stored record was made for"
    return g["found"], [tuple(r) for r in g["records"]]


FOLD_SIZES = [524288, 40000, 4099, 1000]
QUIRK_CASES = [(5000, 91), (3000, 92), (20000, 93), (4099, 94)]


def fold_input(S):
    R = random.Random(S)
    streams = [zref.ref_deflate(corpus.text(R.randint(300, 30000), 100 + i, 400), R.randint(0, 9), 15, 8) for i in range(40)]
    streams += [zref.ref_deflate(b"tiny", 6, 15, 8), zref.ref_deflate(bytes(R.randint(1, 20000)), 9, 15, 8)]
    data, _ = corpus.container(streams, S)
    return data + b"\x78\x9c" + R.randbytes(300)   # false candidates, one of them at the very end


def fold_inputs():
    """key -> (input, chunk size) of every comparison with the reference binary in this module"""
    d = {f"scan_fold_{S}": (fold_input(S), S) for S in FOLD_SIZES}
    d.update({f"overlap_quirk_{S}_{seed}": (corpus.at_chunk_starts(S, seed), S) for S, seed in QUIRK_CASES})
    return d


@pytest.mark.parametrize("S", FOLD_SIZES)
def test_scan_fold_matches_reference_binary(S):
    data = fold_input(S)
    with tempfile.TemporaryDirectory() as tmp:
        found, recs = _reference_streams(f"scan_fold_{S}", data, S, tmp)
    got = _fold_with_oracle(data, S)
    assert len(got) == found
    assert [g for g in got if g in set(recs)] == recs   # every stream the reference recompressed, in order
    assert found < 42 or S == 524288                     # small chunks really lose boundary-crossing streams (A.1)


@pytest.mark.parametrize("S,seed", QUIRK_CASES)
def test_scan_fold_reproduces_the_overlap_byte_quirk(S, seed):
    """streams that start exactly on a chunk start k(S-1), k >= 2 (found at full size: one of configs[3]'s 50,000 streams)"""
    data = corpus.at_chunk_starts(S, seed)
    with tempfile.TemporaryDirectory() as tmp:
        found, recs = _reference_streams(f"overlap_quirk_{S}_{seed}", data, S, tmp)
    got = _fold_with_oracle(data, S)
    assert len(got) == found and [g for g in got if g in set(recs)] == recs
    # the quirk really decides something here: the plain "repeat the last byte" model finds a different number of streams
    starts = {k * (S - 1) for k in range(2, len(data) // (S - 1) + 1)}
    assert any(g[0] in starts for g in got) or found > 0


def _lanes(ulen, forced=0):
    n = len(ulen)
    out = (C.c_uint32 * max(n, 1))()
    nl = az.lib().atz_host_lane_partition((C.c_uint64 * max(n, 1))(*ulen), n, forced, out)
    return nl, list(out)[:n]


def test_lane_partition():
    """how a search splits its streams over lanes (api.cu lane_partition): every stream in exactly one lane, the longest streams in
    lane 0, byte shares as designed, one lane for long-stream containers and for tiny ones"""
    import random
    R = random.Random(5)
    # long streams (mean >= 32 KiB): a single lane unless forced
    big = [R.randrange(1 << 10, 256 << 10) for _ in range(500)]
    nl, lane = _lanes(big)
    assert nl == 1 and set(lane) == {0}
    # many small streams: four lanes
    small = [R.randrange(512, 8192) for _ in range(5000)]
    nl, lane = _lanes(small)
    assert nl == 4 and len(lane) == len(small) and set(lane) == {0, 1, 2, 3}
    by = [[u for u, l in zip(small, lane) if l == k] for k in range(4)]
    assert all(min(by[k]) >= max(by[k + 1]) for k in range(3))                   # sorted by length across lanes, the longest first
    tot = sum(small); cum = 0
    for k, want in enumerate((0.15, 0.4, 0.7, 1.0)):                              # cumulative byte shares
        cum += sum(by[k])
        assert abs(cum / tot - want) < 0.01, (k, cum / tot)
    # few streams: one lane per 16 streams at most; none: nothing to do
    assert _lanes([1000] * 15)[0] == 1 and _lanes([1000] * 40)[0] == 2 and _lanes([])[0] == 1
    # forced counts (ATZ_LANES) are clamped to 1..4 and still cover every stream once
    for forced in (1, 2, 3, 4, 9):
        nl, lane = _lanes(big, forced)
        assert nl == min(forced, 4) and len(lane) == len(big) and max(lane) == nl - 1
    nl, lane = _lanes([7, 7, 7], 4)                                               # more lanes than streams: some stay empty
    assert nl == 4 and len(lane) == 3 and all(0 <= l < 4 for l in lane)
