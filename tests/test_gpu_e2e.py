"""-m gpu: whole-path parity.  The emitted ATZ1 file must be byte-identical to the reference binary's
(oracle/_ref/uncomp_ref, the unmodified main.cpp + zlib 1.2.8) for the same flags, and reconstruction must be bit-exact.
Where the reference has not been built, its .atz files are known by their sha256 and summary lines, stored for every input of
this module in tests/golden/atz_reference.json (tests/golden/make_atz_golden.py)."""
import hashlib
import json
import os
import subprocess
import tempfile

import pytest

import antiz_b200 as az
import corpus
import zref
from test_host_logic import _magic_positions

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")
GOLDEN_ATZ = os.path.join(ROOT, "tests", "golden", "atz_reference.json")
KEEP = ("Total zlib headers found", "recompressed:", "Total bytes written")

CASES = [
    ("c1_single_1MiB_text", lambda: corpus.c1(), []),
    ("c2_pdf_like", lambda: corpus.c2(40, 2), []),
    ("c2_small_chunks", lambda: corpus.c2(40, 22), ["--chunksize", "65536"]),
    ("c2_tiny_chunks", lambda: corpus.c2(30, 23, 1 << 10, 16 << 10), ["--chunksize", "5000"]),
    ("c3_png_like_brute_window", lambda: corpus.c3(8, 3), ["--brute-window"]),
    ("c4_jar_like", lambda: corpus.c4(1200, 4), ["--shortcut-len", "512", "--mismatch-tol", "2"]),
    ("c4_options", lambda: corpus.c4(300, 44), ["--mismatch-tol", "0", "--shortcut-len", "256", "--recomp-tresh", "16", "--sizediff-tresh", "4"]),
    ("c3_tol0_brute", lambda: corpus.c3(4, 33, 3000, 20000), ["--brute-window", "--mismatch-tol", "0"]),
    ("fast_levels_strategies", lambda: corpus.fast_mix(36, 61), []),
    ("c5_mixed_brute_window", lambda: corpus.mixed(1200000, 5), ["--brute-window"]),
    ("extremes_zeros_stored_level0", lambda: corpus.extremes(), []),
    ("c2_shortcut_off", lambda: corpus.c2(14, 29), ["--shortcut-len", "60000"]),
    ("no_streams", lambda: corpus.junk(100000, 5), []),
    # streams exactly on chunk starts: the reference's reader keeps the wrong overlap byte from chunk 1 on (main.cpp:408-413)
    ("streams_at_chunk_starts", lambda: corpus.at_chunk_starts(5000, 91), ["--chunksize", "5000"]),
    ("streams_at_chunk_starts_b", lambda: corpus.at_chunk_starts(3000, 92, 14), ["--chunksize", "3000"]),
    # imperfect winners (SURVEY.md 8 a16; main.cpp:699-715, 916-926): 19 streams with 7-35 diff bytes incl. the tail when C' < C ...
    ("imperfect_tail_flush", lambda: corpus.imperfect(101), []),
    # ... diff lists of up to ~1000 entries, either sign of C' - C (thresholds raised; --shortcut-len above them, main.cpp:649) ...
    ("imperfect_long_diff_lists", lambda: corpus.imperfect(102, True), ["--recomp-tresh", "1000", "--sizediff-tresh", "1000", "--shortcut-len", "4000"]),
    # ... and with the --brute-window grid, a tight size gate and a mismatch tolerance that ends the search early
    ("imperfect_brute_window", lambda: corpus.imperfect(104, True), ["--recomp-tresh", "700", "--sizediff-tresh", "50", "--shortcut-len", "1024", "--brute-window"]),
    ("imperfect_mismatch_tol", lambda: corpus.imperfect(103, True), ["--recomp-tresh", "400", "--sizediff-tresh", "300", "--mismatch-tol", "40"]),
]


def _strategies_data():
    """streams made with Z_FILTERED / Z_FIXED / Z_RLE / Z_HUFFMAN_ONLY, which no candidate of the reference reproduces"""
    import random
    r = random.Random(77)
    ss = []
    for i in range(24):
        d = corpus.binaryish(r.randint(3000, 60000), 700 + i) if i % 2 else corpus.text(r.randint(3000, 90000), 700 + i, 300)
        strat = [1, 2, 3, 4][i % 4]
        lvl = r.randint(4, 9) if strat == 1 else r.randint(1, 9)
        ss.append(zref.ref_deflate(d, lvl, r.choice([12, 15]), r.choice([8, 9, 4]), strat))
    return corpus.container(ss, 78)[0]


def reference_inputs():
    """key -> (input maker, flags) of every comparison with the reference binary in this module"""
    d = {name: (make, flags) for name, make, flags in CASES}
    d["batched_probe"] = (lambda: corpus.c4(400, 45) + corpus.c2(6, 46), [])
    d["strategies"] = (_strategies_data, [])
    d["gpus_mixed_brute_window"] = (lambda: corpus.mixed(2500000, 91), ["--brute-window"])
    d["gpus_c2_chunks"] = (lambda: corpus.c2(60, 92, 1 << 10, 128 << 10), ["--chunksize", "100000"])
    return d


def sha256(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def reference_atz(key, f, flags):
    """(sha256 of the reference binary's .atz, its summary lines) for input file f: from the binary where it has been built (its
    .atz is left at f + ".ref.atz"), else from the stored record, which must be for the same input bytes"""
    if os.path.exists(zref.REF_BIN):
        ref = subprocess.run([zref.REF_BIN, "-i", f, "-o", f + ".ref.atz", "--notest"] + flags, capture_output=True, text=True)
        assert ref.returncode == 0, ref.stdout
        return sha256(f + ".ref.atz"), [l for l in ref.stdout.splitlines() if l.startswith(KEEP)]
    g = json.load(open(GOLDEN_ATZ))[key]
    assert g["flags"] == flags and g["input_sha256"] == sha256(f), f"{key}: the input is not the one the stored record was made for"
    return g["atz_sha256"], g["lines"]


@pytest.mark.parametrize("name,make,flags", CASES, ids=[c[0] for c in CASES])
def test_atz_identical_to_reference_binary(name, make, flags):
    data = make()
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        f = os.path.join(tmp, "in.bin")
        open(f, "wb").write(data)
        want, lines = reference_atz(name, f, flags)
        gpu = subprocess.run([UNCOMP, "-i", f, "-o", f + ".gpu.atz"] + flags, capture_output=True, text=True)
        assert gpu.returncode == 0, gpu.stdout + gpu.stderr
        assert "OK! Restoration is bit by bit identical" in gpu.stdout
        assert sha256(f + ".gpu.atz") == want, f"{name}: ATZ differs"
        assert lines == [l for l in gpu.stdout.splitlines() if l.startswith(KEEP)]
        # our reconstructor on the reference's ATZ (the same bytes as ours), and the reference's reconstructor on ours
        r1 = subprocess.run([UNCOMP, "-r", "-i", f + ".gpu.atz", "-o", f + ".rec1"], capture_output=True, text=True)
        assert r1.returncode == 0 and open(f + ".rec1", "rb").read() == data
        if os.path.exists(zref.REF_BIN):
            r2 = subprocess.run([zref.REF_BIN, "-r", "-i", f + ".gpu.atz", "-o", f + ".rec2"], capture_output=True, text=True)
            assert r2.returncode == 0 and open(f + ".rec2", "rb").read() == data


def test_batched_probe_equals_reference():
    """more candidates than slots (forced with ATZ_SLOT_BATCH): probed in batches, accepted streams inflated again"""
    make, flags = reference_inputs()["batched_probe"]
    data = make()
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        want, _ = reference_atz("batched_probe", f, flags)
        gpu = subprocess.run([UNCOMP, "-i", f, "-o", f + ".gpu.atz"] + flags, capture_output=True, text=True, env=dict(os.environ, ATZ_SLOT_BATCH="97"))
        assert gpu.returncode == 0, gpu.stdout + gpu.stderr
        assert sha256(f + ".gpu.atz") == want


def test_strategies_extension_recompresses_what_the_reference_cannot():
    """--strategies (SURVEY.md 8 f4): streams made with Z_FILTERED / Z_FIXED / Z_RLE / Z_HUFFMAN_ONLY, which no candidate of the
    reference reproduces, are recompressed and reconstruct bit-exactly; without the flag the ATZ file stays the reference's"""
    data = _strategies_data()
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        want, _ = reference_atz("strategies", f, [])
        plain = subprocess.run([UNCOMP, "-i", f, "-o", f + ".gpu.atz", "--notest"], capture_output=True, text=True)
        ext = subprocess.run([UNCOMP, "-i", f, "-o", f + ".ext.atz", "--strategies"], capture_output=True, text=True)
        assert plain.returncode == 0 and ext.returncode == 0, ext.stdout + ext.stderr
        assert sha256(f + ".gpu.atz") == want
        assert "OK! Restoration is bit by bit identical" in ext.stdout
        count = lambda out: [int(x) for x in [l for l in out.splitlines() if l.startswith("recompressed:")][0].split(":")[1].split("/")]
        got, found = count(ext.stdout)       # (a stream that crosses the 524,288-byte chunk boundary is not detected, as in the reference)
        assert got == found >= 22 and count(plain.stdout)[0] < 12
        rec = subprocess.run([UNCOMP, "-r", "-i", f + ".ext.atz", "-o", f + ".rec"], capture_output=True, text=True)
        assert rec.returncode == 0 and open(f + ".rec", "rb").read() == data


def test_scan_candidates_and_records():
    data = corpus.c2(25, 7, 1 << 10, 64 << 10)
    ctx = az.Context(0)
    ctx.load(data)
    n = ctx.scan(524288)
    st = ctx.stats()
    assert st.n_candidates == len(_magic_positions(data))
    ss = ctx.streams()
    assert n == len(ss) == 25
    for s in ss:
        z = data[s.offset:s.offset + s.streamLength]
        r, out = zref.oracle_inflate(z, s.inflatedLength)
        assert r.status == zref.OI_END and r.total_in == s.streamLength and r.total_out == s.inflatedLength
        assert ctx.inflated(ss.index(s), s.inflatedLength) == out
    ctx.search(az.Options(flags=az.ATZ_F_EXACT_RECORDS))
    for s in ctx.streams():
        assert s.recomp == 1 and s.identBytes == s.streamLength and s.ndiff == 0 and s.window == 15 and s.memlevel == 8
    ctx.close()


def _rec(s):
    return (s.offset, s.streamLength, s.inflatedLength, s.offsetType, s.clevel, s.window, s.memlevel, s.identBytes, s.recomp, s.ndiff, s.firstDiffByte)


def test_sharded_search_equals_single():
    """stream partition (SURVEY.md 8e) after a plain scan: the records gathered by owner equal the unsharded run"""
    data = corpus.c3(10, 8, 3000, 30000)
    opt = az.Options(bruteforceWindow=True)
    one = az.Context(0); one.load(data); one.scan(); one.search(opt)
    base = [_rec(s) for s in one.streams()]
    own = az.partition([b[2] for b in base], 3)
    assert sorted(set(own)) == [0, 1, 2]
    got = [None] * len(base)
    for sh in range(3):
        c = az.Context(0); c.load(data); c.scan(); c.search(opt, sh, 3)
        for i, s in enumerate(c.streams()):
            if own[i] == sh:
                got[i] = _rec(s)
        c.close()
    one.close()
    assert got == base


@pytest.mark.parametrize("nsh,chunksize", [(2, 524288), (3, 65536), (5, 5000), (4, 1 << 30)])
def test_sharded_scan_and_search_equal_single(nsh, chunksize):
    """one container over nsh contexts (emulated on one device): every shard attaches the host file, probes its own chunk range,
    the probe records are exchanged, every context folds the same stream list and keeps only the plaintext of the streams it owns;
    records, diffs and payloads gathered by owner equal the single-context run (streams crossing chunk and shard boundaries included)"""
    data = corpus.c2(30, 81, 1 << 10, 200 << 10) + corpus.c4(150, 82) + corpus.fast_mix(12, 83) + corpus.extremes(84)
    opt = az.Options(flags=az.ATZ_F_EXACT_RECORDS)
    one = az.Context(0); one.load(data); n1 = one.scan(chunksize); one.search(opt)
    base = [_rec(s) for s in one.streams()]; base_diffs = one.diffs()
    base_payload = [one.inflated(i, b[2]) for i, b in enumerate(base)]
    one.close()
    ctxs = [az.Context(0) for _ in range(nsh)]
    for g, c in enumerate(ctxs):
        c.attach(data); c.scan_shard(chunksize, g, nsh)
    blobs = [c.probe_export() for c in ctxs]
    for g, c in enumerate(ctxs):
        for h in range(nsh):
            if h != g:
                c.probe_import(h, blobs[h])
        assert c.scan_finish() == n1
    own = ctxs[0].owners()
    assert all(c.owners() == own for c in ctxs) and set(own) <= set(range(nsh))
    got = [None] * n1; offs = []; vals = b""
    for g, c in enumerate(ctxs):
        c.search(opt, g, nsh)
    for i in range(n1):
        c = ctxs[own[i]]; s = c.streams()[i]
        got[i] = _rec(s)
        o, v = c.diffs()
        offs += list(o[s.diff_index:s.diff_index + s.ndiff]); vals += bytes(v[s.diff_index:s.diff_index + s.ndiff])
        assert c.inflated(i, s.inflatedLength) == base_payload[i]
        other = ctxs[(own[i] + 1) % nsh]
        with pytest.raises(az.AtzError):      # a shard holds only what it owns
            other.inflated(i, s.inflatedLength)
    assert got == base and (offs, vals) == (list(base_diffs[0]), bytes(base_diffs[1]))
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("gpus", [2, 4, 8])
def test_uncomp_gpus_equals_reference(gpus):
    """`uncomp --gpus N`: one container sharded over N contexts in one process, .atz byte-identical to --gpus 1 and to uncomp_ref.
    On a box with fewer devices the contexts share device 0 (ATZ_TEST_ONE_DEVICE, a test hook of the host program): the sharding
    logic is the same, only the hardware concurrency is missing."""
    import torch
    ndev = torch.cuda.device_count()
    env = dict(os.environ)
    if ndev < gpus:
        env["ATZ_TEST_ONE_DEVICE"] = "1"
    for key in ("gpus_mixed_brute_window", "gpus_c2_chunks"):
        make, flags = reference_inputs()[key]
        with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
            f = os.path.join(tmp, "in.bin"); open(f, "wb").write(make())
            want, _ = reference_atz(key, f, flags)
            one = subprocess.run([UNCOMP, "-i", f, "-o", f + ".g1.atz", "--notest"] + flags, capture_output=True, text=True)
            many = subprocess.run([UNCOMP, "-i", f, "-o", f + ".gn.atz", "--gpus", str(gpus)] + flags, capture_output=True, text=True, env=env)
            assert one.returncode == 0 and many.returncode == 0, many.stdout + many.stderr
            assert "OK! Restoration is bit by bit identical" in many.stdout
            assert want == sha256(f + ".g1.atz") == sha256(f + ".gn.atz")


def test_small_budget_batches_and_deferrals_do_not_change_records():
    """the search runs in batches sized for a few sets of bucket lists per stream; a stream whose next candidates need lists the arena
    has no room for is deferred to a later batch.  With a budget of a few dozen MB that happens all the time; records must not change."""
    data = corpus.mixed(1500000, 67) + corpus.c3(6, 68, 20000, 90000)
    opt = az.Options(bruteforceWindow=True, flags=az.ATZ_F_EXACT_RECORDS)
    def run(budget, **env):
        old = {k: os.environ.get(k) for k in env}
        os.environ.update({k: str(v) for k, v in env.items()})
        try:
            c = az.Context(0)
            if budget:
                c.set_budget(budget)
            c.load(data); c.scan(); c.search(opt)
            out = ([_rec(s) for s in c.streams()], c.diffs()); c.close()
        finally:
            for k, v in old.items():
                if v is None:
                    del os.environ[k]
                else:
                    os.environ[k] = v
        return out
    base = run(0)
    assert any(r[8] for r in base[0])
    # (half the budget is the bucket-list arena; the longest stream here, 256 KB, needs 24 MB for its nine hash sizes)
    for budget, env in ((64 << 20, {}), (56 << 20, dict(ATZ_BATCH_SETS=1)), (96 << 20, dict(ATZ_BATCH_SETS=9, ATZ_BG_B=0)), (0, dict(ATZ_BATCH_SETS=1))):
        assert run(budget, **env) == base, (budget, env)


def test_phase_order_guard():
    ctx = az.Context(0)
    with pytest.raises(az.AtzError) as e:
        ctx.scan()
    assert e.value.code == az.ATZ_E_STATE == -10   # main.cpp:263
    ctx.load(b"x" * 100)
    with pytest.raises(az.AtzError):
        ctx.search()
    ctx.close()


def _records(data, opt, **env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        c = az.Context(0); c.load(data); c.scan(); c.search(opt)
        recs = [(s.offset, s.streamLength, s.inflatedLength, s.clevel, s.window, s.memlevel, s.identBytes, s.recomp, s.ndiff, s.firstDiffByte) for s in c.streams()]
        diffs = c.diffs()
        c.close()
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
    return recs, diffs


def test_search_schedule_does_not_change_records():
    """the burst parse (speculation on the original's token boundaries), the
    lane partition, phase B in the background and rows at every position are scheduling choices: every per-stream record,
    including those of streams that are not recompressed, equals the one of the plain serial single-lane foreground search
    (exact-records mode: no early cut)"""
    exact = az.ATZ_F_EXACT_RECORDS
    cases = [
        (corpus.fast_mix(36, 62) + corpus.c2(24, 63, 1 << 10, 96 << 10), az.Options(flags=exact)),
        (corpus.c3(6, 64, 3000, 40000), az.Options(bruteforceWindow=True, flags=exact)),
        (corpus.extremes(72) + corpus.c4(200, 65), az.Options(flags=exact, mismatchTol=0, recompTresh=16)),
        (corpus.mixed(900000, 66), az.Options(bruteforceWindow=True)),     # default mode: the early cut only ever hides records that are not written
    ]
    for data, opt in cases:
        base = _records(data, opt, ATZ_BURST=0, ATZ_LANES=1, ATZ_BG_B=0)
        assert any(r[7] for r in base[0]) or not base[0]
        for env in (dict(ATZ_BURST=1, ATZ_LANES=1, ATZ_BG_B=0), dict(ATZ_BURST=1, ATZ_LANES=3, ATZ_BG_B=1),
                    dict(ATZ_BURST=0, ATZ_LANES=1, ATZ_BG_B=1, ATZ_ALL_ROWS=1), dict(ATZ_BURST=1, ATZ_LANES=2, ATZ_BG_B=1),
                    dict(ATZ_BURST=1, ATZ_LANES=1, ATZ_WAVE_GROWTH=16, ATZ_BATCH_SETS=1)):
            got = _records(data, opt, **env)
            if opt.flags & exact:
                assert got == base, env
            else:   # recompressed streams and their diffs are what the ATZ file holds
                keep = lambda rr: [r for r in rr if r[7]]
                assert keep(got[0]) == keep(base[0]) and got[1] == base[1], env
