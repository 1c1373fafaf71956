"""-m gpu: ATZ_SCAN_SMALL_WINDOWS (uncomp --small-windows).  Streams with CINFO 0 and 1 headers (256- and 512-byte windows) are found
by the scan and searched at windowBits 9, where MAX_DIST (250) is below MAX_MATCH (258) and MIN_LOOKAHEAD (262) and the window slides
every 512 bytes.  Every trial path must stay bit-exact with zlib there; the ATZ file stays readable by the reference's reconstructor."""
import hashlib
import os
import random
import struct
import subprocess
import tempfile

import pytest

import antiz_b200 as az
import corpus
import test_host_logic
import zref

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")
SW = az.ATZ_SCAN_SMALL_WINDOWS
REFERENCE_24 = {0x2815, 0x2853, 0x2891, 0x28cf, 0x3811, 0x384f, 0x388d, 0x38cb, 0x480d, 0x484b, 0x4889, 0x48c7,
                0x5809, 0x5847, 0x5885, 0x58c3, 0x6805, 0x6843, 0x6881, 0x68de, 0x7801, 0x785e, 0x789c, 0x78da}
SMALL_8 = {0x081d, 0x085b, 0x0899, 0x08d7, 0x1819, 0x1857, 0x1895, 0x18d3}


@pytest.fixture(scope="module")
def ctx():
    c = az.Context(0)
    yield c
    c.close()


def grid_inputs():
    """the inputs of test_gpu_kernels.test_deflate_full_parameter_grid"""
    R = random.Random(1)
    return {"text70k": corpus.text(70000, 2), "bin": corpus.binaryish(60000, 9),
            "mixed": corpus.text(20000, 5) + R.randbytes(3000) + bytes(5000) + corpus.text(40000, 6)}


def cinfo0(z):
    """the header of a window-9 stream rewritten to CINFO 0 (what libpng's optimize_cmf does for small data): FLEVEL kept, FCHECK
    recomputed; the body is zlib's at window 9"""
    flg = z[1] & 0xc0
    flg |= (31 - ((0x0800 | flg) % 31)) % 31
    return bytes([0x08, flg]) + z[2:]


def small_stream(r, k, S):
    """stream k of the small-window corpora: reference headers, windowBits 8 and 9 (CINFO 1), and CINFO 0 rewrites, in turn"""
    n = r.randint(200, 2 * S)
    d = corpus.text(n, 500 + k, 300) if k % 3 else corpus.binaryish(n, 500 + k)
    m = r.randint(1, 9)
    kind = k % 4
    if kind == 0:
        return zref.ref_deflate(d, r.randint(0, 9), r.choice([10, 12, 15]), m)
    if kind == 2:     # zlib 1.2.8 turns windowBits 8 into 9 (the oracle, which stands in for level 0, takes 9..15 only)
        return zref.ref_deflate(d, r.randint(1, 9), 8, m)
    lvl = r.randint(0, 9)
    z = zref.ref_deflate(d, lvl, 9, 8 if lvl == 0 else m)    # (stored blocks depend on memLevel; the reference tries level 0 at memLevel 8 only)
    return cinfo0(z) if kind == 3 else z


def small_window_container(S, seed, nstreams):
    """small-window and reference streams, some exactly on the chunk starts k(S-1), k >= 2 (where the reference's reader sees
    file[start - 1] in place of the first byte: the byte before is made the stream's own first byte, so it is found), some one byte
    after them, some split around a boundary (a header pair (file[start - 1], file[start + 1]) that is not in the file), and the
    rest anywhere; streams of up to 2S bytes run across chunk boundaries"""
    r = random.Random(seed)
    out = bytearray(corpus.junk(r.randint(100, 300), seed))
    for k in range(nstreams):
        z = small_stream(r, k, S)
        mode = r.randrange(4)
        if mode < 3:
            c = max(2, (len(out) + 40) // (S - 1) + 1)
            start = c * (S - 1) + (1 if mode == 1 else 0)
            out += corpus.junk(start - len(out), seed * 31 + k)
            if mode == 0:
                out[-1] = z[0]
            elif mode == 2:
                out[-1] = z[0]; out += b"Q" + bytes([z[1]]) + corpus.junk(40, seed + k)
        else:
            out += corpus.junk(r.randint(20, 200), seed * 7 + k)
        out += z
    out += corpus.junk(300, seed)
    return bytes(out)


def fold(data, S, accepted):
    """ZBuffSearcher restated over the header set `accepted` (test_host_logic._fold_with_oracle with its header list swapped)"""
    orig = test_host_logic._magic_positions
    test_host_logic._magic_positions = lambda d: [i for i in range(len(d) - 1) if (d[i] << 8 | d[i + 1]) in accepted]
    try:
        return test_host_logic._fold_with_oracle(data, S)
    finally:
        test_host_logic._magic_positions = orig


def scanned(data, S, flags):
    c = az.Context(0)
    if flags:
        c.set_scan_flags(flags)
    c.load(data)
    c.scan(S)
    return c


# ---------------------------------------------------------------------------------------------------------------------------------
def test_deflate_window9_grid(ctx):
    """K5 at window 9: levels 0..9 x memLevel 1..9, batch and single-stream entry points, byte for byte against zlib"""
    for name, d in grid_inputs().items():
        items = [(d, lvl, 9, m) for lvl in range(10) for m in range(1, 10)]
        outs = ctx.deflate_batch(items)
        for (dd, lvl, w, m), o in zip(items, outs):
            want = zref.ref_deflate(dd, lvl, 9, m)
            assert o == want, (name, lvl, m)
            if m in (1, 5, 9) or lvl in (1, 4):
                assert ctx.deflate_stream(dd, lvl, 9, m) == want, (name, lvl, m)


def test_trials_window9_grid(ctx):
    """atz_trial's {status, C', ident} at window 9 against zlib's output, every level x memLevel against originals made at window 9
    (deflate_fast under the original's token hypothesis and after it breaks, deflate_slow with rows and resolved tables)"""
    exact = az.Options(flags=az.ATZ_F_EXACT_RECORDS)
    short = az.Options(shortcutLength=100, recompTresh=10, sizediffTresh=10, flags=az.ATZ_F_EXACT_RECORDS)
    for name, d in grid_inputs().items():
        cache = {(lvl, m): zref.ref_deflate(d, lvl, 9, m) for lvl in range(10) for m in range(1, 10)}
        for ol, om in ((6, 8), (1, 4), (9, 9)):
            orig = cache[(ol, om)]
            for o in (orig, cinfo0(orig)):
                for lvl in range(10):
                    for m in range(1, 10):
                        for opt in ((exact, short) if (lvl, m) == (ol, om) or m == om else (exact,)):
                            cp = cache[(lvl, m)]; C_, Cp = len(o), len(cp)
                            S, R_, SD = opt.shortcutLength, opt.recompTresh, opt.sizediffTresh
                            if C_ > S and sum(1 for i in range(min(S, Cp)) if cp[i] == o[i]) < S - R_:
                                want = (az.TR_BAILED, None, None)
                            elif abs(Cp - C_) > SD:
                                want = (az.TR_SIZE, None, None)
                            else:
                                want = (az.TR_COMPARED, Cp, sum(1 for a, b in zip(cp, o) if a == b))
                            r = ctx.trial(d, o, lvl, 9, m, opt)
                            got = (r.status, r.out_len, r.ident) if r.status == az.TR_COMPARED else (r.status, None, None)
                            assert got == want, (name, ol, om, lvl, m, opt.shortcutLength)
            # the original itself is reproduced; its CINFO 0 rewrite up to the two header bytes
            assert ctx.trial(d, orig, ol, 9, om, exact).ident == len(orig)
            assert ctx.trial(d, cinfo0(orig), ol, 9, om, exact).ident == len(orig) - 2


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,seed", [(524288, 11), (5000, 12), (3001, 13)])
def test_scan_small_window_headers(S, seed):
    """K1 + K2 + the accept logic with and without the flag, against ZBuffSearcher restated over the 32- and the 24-pair set"""
    data = small_window_container(min(S, 6000), seed, 24) if S != 524288 else small_window_container(4000, seed, 24)
    for flags, accepted in ((SW, REFERENCE_24 | SMALL_8), (0, REFERENCE_24)):
        c = scanned(data, S, flags)
        ss = c.streams()
        assert c.stats().n_candidates >= len(ss)
        want = fold(data, S, accepted)
        assert [(s.offset, s.streamLength, s.inflatedLength) for s in ss] == want, flags
        starts = {k * (S - 1) for k in range(2, len(data) // (S - 1) + 1)}
        for s in ss:
            b0 = data[s.offset - 1] if s.offset in starts else data[s.offset]      # the reference's overlap-byte quirk
            assert s.offsetType == az.lib().atz_host_header_type(flags, b0, data[s.offset + 1])
        c.close()
    # the flag finds the small-window streams (and keeps every one the reference finds)
    assert len(fold(data, S, REFERENCE_24 | SMALL_8)) > len(fold(data, S, REFERENCE_24))


def test_scan_without_flag_matches_reference_binary():
    """flag off: the ATZ file is the reference's (where its binary has been built)"""
    if not os.path.exists(zref.REF_BIN):
        pytest.skip("the reference binary is not built")
    data = small_window_container(6000, 21, 20)
    with tempfile.TemporaryDirectory() as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        assert subprocess.run([zref.REF_BIN, "-i", f, "-o", f + ".ref", "--notest"], capture_output=True).returncode == 0
        assert subprocess.run([UNCOMP, "-i", f, "-o", f + ".gpu", "--notest"], capture_output=True).returncode == 0
        assert open(f + ".ref", "rb").read() == open(f + ".gpu", "rb").read()


def test_scan_flags_state_and_shard_mismatch():
    c = az.Context(0)
    with pytest.raises(az.AtzError) as e:
        c.set_scan_flags(2)
    assert e.value.code == az.ATZ_E_ARG
    c.set_scan_flags(SW); c.set_scan_flags(0); c.set_scan_flags(SW)
    c.load(b"x" * 1000)
    with pytest.raises(az.AtzError) as e:
        c.set_scan_flags(0)
    assert e.value.code == az.ATZ_E_STATE
    c.close()
    # shards that scanned with different sets refuse each other's records
    data = small_window_container(5000, 31, 10)
    a, b = az.Context(0), az.Context(0)
    a.set_scan_flags(SW)
    for g, x in enumerate((a, b)):
        x.attach(data); x.scan_shard(5000, g, 2)
    for g, x in enumerate((a, b)):
        with pytest.raises(az.AtzError) as e:
            x.probe_import(1 - g, (b, a)[g].probe_export())
        assert e.value.code == az.ATZ_E_STATE
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------------------------------------------
def read_atz(atz):
    """a short ATZ1 reader (the layout of the reference's writer, main.cpp:775-831): header, records, residue"""
    assert atz[:4] == b"ATZ\x01"
    total, origlen, nrec = struct.unpack_from("<QQQ", atz, 4)
    assert total == len(atz)
    pos = 28; recs = []
    for _ in range(nrec):
        off, c, u = struct.unpack_from("<QQQ", atz, pos); lvl, w, m = atz[pos + 24:pos + 27]; nd = struct.unpack_from("<Q", atz, pos + 27)[0]
        pos += 35; first = -1; doffs = []; dvals = b""
        if nd:
            first = struct.unpack_from("<q", atz, pos)[0]; doffs = list(struct.unpack_from(f"<{nd}Q", atz, pos + 8)); dvals = atz[pos + 8 + 8 * nd:pos + 8 + 9 * nd]
            pos += 8 + 9 * nd
        recs.append(dict(off=off, c=c, u=u, lvl=lvl, w=w, m=m, first=first, doffs=doffs, dvals=dvals, plain=atz[pos:pos + u])); pos += u
    return origlen, recs, atz[pos:]


def reconstruct_on_cpu(atz):
    """what the reference's reconstructor does (doDeflate = deflateInit2(level, 8, window, memLevel, 0), then the diff patch), with zlib"""
    origlen, recs, residue = read_atz(atz)
    out = bytearray(); ri = 0; end = 0
    for r in recs:
        gap = r["off"] - end; out += residue[ri:ri + gap]; ri += gap
        assert r["lvl"] >> 4 == 0          # plain levels only: what the reference can read
        z = bytearray(zref.ref_deflate(r["plain"], r["lvl"], r["w"], r["m"]))
        z += bytes(max(0, r["c"] - len(z)))
        s = 0
        for o, v in zip(r["doffs"], r["dvals"]):
            s += o; z[r["first"] + s] = v
        out += z[:r["c"]]; end = r["off"] + r["c"]
    out += residue[ri:]
    assert len(out) == origlen
    return bytes(out)


@pytest.mark.parametrize("flags", [[], ["--brute-window"], ["--strategies"]])
def test_uncomp_small_windows_end_to_end(flags):
    """every small-window stream is recompressed at window 9: CINFO 1 without diffs, CINFO 0 with exactly its two header bytes as
    diffs; uncomp -r and the reference's reconstructor (its binary where built, else the same steps on the CPU) restore the file"""
    r = random.Random(41)
    streams = [small_stream(r, k, 20000) for k in range(28)]
    data, offs = corpus.container(streams, 42)
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        p = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--small-windows"] + flags, capture_output=True, text=True)
        assert p.returncode == 0 and "OK! Restoration is bit by bit identical" in p.stdout, p.stdout + p.stderr
        atz = open(f + ".atz", "rb").read()
        _, recs, _ = read_atz(atz)
        by_off = {x["off"]: x for x in recs}
        nsmall = 0
        for off, z in zip(offs, streams):
            if (z[0] << 8 | z[1]) not in SMALL_8:
                continue
            nsmall += 1
            x = by_off[off]
            assert x["w"] == 9 and x["c"] == len(z), (off, x["w"])
            if z[0] == 0x18:
                assert x["doffs"] == [], off
            else:
                assert x["first"] == 0 and x["doffs"] == [0, 1] and x["dvals"] == z[:2], (off, x["doffs"])
        assert nsmall >= 18
        rec = subprocess.run([UNCOMP, "-r", "-i", f + ".atz", "-o", f + ".rec"], capture_output=True, text=True)
        assert rec.returncode == 0 and open(f + ".rec", "rb").read() == data
        if os.path.exists(zref.REF_BIN):
            r2 = subprocess.run([zref.REF_BIN, "-r", "-i", f + ".atz", "-o", f + ".rec2"], capture_output=True, text=True)
            assert r2.returncode == 0 and open(f + ".rec2", "rb").read() == data
        else:
            assert reconstruct_on_cpu(atz) == data


# ---------------------------------------------------------------------------------------------------------------------------------
def _rec(s):
    return (s.offset, s.streamLength, s.inflatedLength, s.offsetType, s.clevel, s.window, s.memlevel, s.identBytes, s.recomp, s.ndiff, s.firstDiffByte)


def _records(data, opt, budget=0, **env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        c = az.Context(0); c.set_scan_flags(SW)
        if budget:
            c.set_budget(budget)
        c.load(data); c.scan(); c.search(opt)
        recs = [_rec(s) for s in c.streams()]; diffs = c.diffs()
        c.close()
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
    return recs, diffs


def schedule_corpus(seed):
    """window-9 streams long enough for rows, resolved tables, the burst parse and several blocks, and some imperfect ones (made with
    deflateTune: no plain parameter set reproduces them, so the whole sequence and the brute grid run)"""
    r = random.Random(seed)
    ss = []
    for k in range(30):
        n = r.randint(3000, 120000)
        d = corpus.text(n, 900 + k, 400) if k % 2 else corpus.binaryish(n, 900 + k)
        lvl, m = r.randint(1, 9), r.randint(1, 9)
        z = zref.ref_deflate_ex(d, lvl, 9, m, tune=(4, 5, 16, 8)) if k % 7 == 6 else zref.ref_deflate(d, lvl, 9, m)
        ss.append(cinfo0(z) if k % 3 == 0 else z)
    return corpus.container(ss, seed)[0]


def test_search_schedule_does_not_change_window9_records():
    """test_gpu_e2e.test_search_schedule_does_not_change_records on window-9 streams, plus a small budget with deferrals"""
    exact = az.ATZ_F_EXACT_RECORDS
    for data, opt in ((schedule_corpus(51), az.Options(flags=exact)), (schedule_corpus(52), az.Options(bruteforceWindow=True, flags=exact))):
        base = _records(data, opt, ATZ_BURST=0, ATZ_LANES=1, ATZ_BG_B=0)
        assert sum(1 for x in base[0] if x[8] and x[5] == 9) >= 20 and all(x[3] >= 24 for x in base[0])
        for budget, env in ((0, dict(ATZ_BURST=1, ATZ_LANES=1, ATZ_BG_B=0)), (0, dict(ATZ_BURST=1, ATZ_LANES=3, ATZ_BG_B=1)),
                            (0, dict(ATZ_BURST=0, ATZ_LANES=1, ATZ_BG_B=1, ATZ_ALL_ROWS=1)), (0, dict(ATZ_FORCE_REC=0)), (0, dict(ATZ_FORCE_RES=0)),
                            (56 << 20, dict(ATZ_BATCH_SETS=1))):
            assert _records(data, opt, budget, **env) == base, (budget, env)


@pytest.mark.parametrize("nsh,chunksize", [(2, 524288), (3, 65536), (4, 20000), (5, 5000)])
def test_sharded_small_windows_equal_single(nsh, chunksize):
    """2..5 emulated shards with the flag: the same records, diffs and payloads as one context"""
    data = small_window_container(5000, 61, 30) + schedule_corpus(62)
    opt = az.Options(flags=az.ATZ_F_EXACT_RECORDS)
    one = az.Context(0); one.set_scan_flags(SW); one.load(data); n1 = one.scan(chunksize); one.search(opt)
    base = [_rec(s) for s in one.streams()]; bd = one.diffs()
    one.close()
    assert any(b[3] >= 24 for b in base)
    ctxs = [az.Context(0) for _ in range(nsh)]
    for g, c in enumerate(ctxs):
        c.set_scan_flags(SW); c.attach(data); c.scan_shard(chunksize, g, nsh)
    blobs = [c.probe_export() for c in ctxs]
    for g, c in enumerate(ctxs):
        for h in range(nsh):
            if h != g:
                c.probe_import(h, blobs[h])
        assert c.scan_finish() == n1
    for g, c in enumerate(ctxs):
        c.search(opt, g, nsh)
    own = ctxs[0].owners(); got = []; offs = []; vals = b""
    for i in range(n1):
        c = ctxs[own[i]]; s = c.streams()[i]
        got.append(_rec(s))
        o, v = c.diffs()
        offs += list(o[s.diff_index:s.diff_index + s.ndiff]); vals += bytes(v[s.diff_index:s.diff_index + s.ndiff])
    assert got == base and (offs, vals) == (list(bd[0]), bytes(bd[1]))
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("gpus", [2, 4])
def test_uncomp_gpus_small_windows(gpus):
    """uncomp --small-windows --gpus N writes the same ATZ file as --gpus 1 (the contexts share a device where there are fewer)"""
    import torch
    env = dict(os.environ)
    if torch.cuda.device_count() < gpus:
        env["ATZ_TEST_ONE_DEVICE"] = "1"
    data = small_window_container(6000, 71, 30) + schedule_corpus(72)
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        one = subprocess.run([UNCOMP, "-i", f, "-o", f + ".g1", "--notest", "--small-windows", "--chunksize", "65536"], capture_output=True, text=True)
        many = subprocess.run([UNCOMP, "-i", f, "-o", f + ".gn", "--small-windows", "--chunksize", "65536", "--gpus", str(gpus)], capture_output=True, text=True, env=env)
        assert one.returncode == 0 and many.returncode == 0, many.stdout + many.stderr
        assert "OK! Restoration is bit by bit identical" in many.stdout
        h = lambda p: hashlib.sha256(open(p, "rb").read()).hexdigest()
        assert h(f + ".g1") == h(f + ".gn")
