"""-m gpu: the trial kernel's block flush (K3, csrc/deflate.cu: key heap, gen_bitlen and its depth-limit repair, forced codes,
stored/static/dynamic choice, scan_tree / send_tree run limits) on the inputs of flushcorpus.py, which reach the branches ordinary
inputs never do (test_flush_coverage.py shows which).  Bit-exact against zlib 1.2.8 (zref; the oracle at window 9)."""
import os
import subprocess
import tempfile
import zlib

import pytest

import antiz_b200 as az
import corpus
import flushcorpus as fc
import zref
from test_gpu_kernels import _trial_expect, expect_deflate
from test_host_logic import seq

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")
GRID = [(lvl, w, m) for lvl in range(1, 10) for w in range(10, 16) for m in range(1, 10)]


@pytest.fixture(scope="module")
def ctx():
    c = az.Context(0)
    yield c
    c.close()


def _inputs():
    ins = {f"lit_overflow_m{m}": fc.lit_overflow(m, m) for m in (7, 8, 9)}
    ins["dist_overflow"] = fc.dist_overflow(1)
    ins["dist_overflow_tail"] = fc.dist_overflow(2, corpus.text(3000, 5))
    ins.update({f"forced_{i}": d for i, d in enumerate(fc.forced_lit())})
    ins.update({f"single_dist_{i}": d for i, d in enumerate(fc.single_distance_code(3))})
    ins.update({f"stored_tie_{i}": d for i, d in enumerate(fc.stored_ties(4)[:12])})
    ins.update({f"static_tie_{i}": d for i, d in enumerate(fc.static_ties(6))})
    ins.update({f"slid_w{w}": fc.slid_blocks(5, w) for w in (9, 10)})
    ins.update({f"runs_{i}": d for i, d in enumerate(fc.length_runs(6))})
    return ins


def _check(ctx, items, want):
    got = ctx.deflate_batch(items)
    bad = [(it[1], it[2], it[3], len(it[0])) for it, g, x in zip(items, got, want) if g != x]
    assert not bad, bad[:10]


def test_store_mode_grid(ctx):
    """every input at levels 1-9 x windows 10-15 x memLevels 1-9"""
    for name, d in _inputs().items():
        items = [(d, lvl, w, m) for lvl, w, m in GRID]
        _check(ctx, items, [expect_deflate(d, lvl, w, m) for _, lvl, w, m in items])


def test_store_mode_window_9_slid_blocks(ctx):
    for w in (9, 10):
        d = fc.slid_blocks(5, w)
        items = [(d, lvl, 9, m) for lvl in range(1, 10) for m in range(1, 10)]
        _check(ctx, items, [zref.oracle_deflate(d, lvl, 9, m) for _, lvl, _, m in items])


def test_store_mode_strategies(ctx):
    """every generator with Z_FILTERED at levels 4-9 (deflate_slow with short matches turned into literals), Z_HUFFMAN_ONLY and Z_RLE
    (a block's literal/length tree is its byte histogram) and Z_FIXED (static blocks whatever the trees).  The host's zlib writes
    zlib 1.2.8's bytes for the first three; for Z_FIXED only where it writes no stored block (zlib 1.2.12 lets Z_FIXED choose a stored
    block that 1.2.8 would have written static), so those items are left out."""
    items, want = [], []
    for d in _inputs().values():
        for lvl, w, m in ((4, 15, 8), (6, 15, 9), (9, 15, 9), (5, 12, 7), (8, 15, 1)):
            items.append((d, az.clevel(lvl, 1), w, m)); want.append(zref.ref_deflate(d, lvl, w, m, 1))
        for lvl, w, m in ((2, 15, 9), (6, 15, 8), (9, 13, 2)):
            for strat in (2, 3, 4):
                z = zref.ref_deflate(d, lvl, w, m, strat)
                if strat == 4 and not zref.have_ref() and any(b["type"] == 0 for b in fc.blocks(z)):
                    continue
                items.append((d, az.clevel(lvl, strat), w, m)); want.append(z)
    assert len(items) > 300
    _check(ctx, items, want)


def test_store_mode_chain_walk_fallback(ctx):
    """the overflow inputs with row tables off (ATZ_FORCE_REC=0) and with rows but no resolved tables (ATZ_FORCE_RES=0)"""
    items = [(fc.lit_overflow(m, m), lvl, 15, m) for m in (8, 9) for lvl in (2, 3, 4, 6, 9)]
    items += [(fc.dist_overflow(1), lvl, 15, 9) for lvl in (1, 3, 4, 9)]
    want = [expect_deflate(*it) for it in items]
    for var in ("ATZ_FORCE_REC", "ATZ_FORCE_RES"):
        os.environ[var] = "0"
        try:
            got = ctx.deflate_batch(items)
        finally:
            del os.environ[var]
        assert got == want, var


OVERFLOWS = {"lit_m8": (lambda: fc.lit_overflow(8, 8), 8, 0), "lit_m9": (lambda: fc.lit_overflow(9, 9), 9, 0),
             "dist_m9_tail": (lambda: fc.dist_overflow(2, corpus.text(3000, 5)), 9, 1)}


@pytest.mark.parametrize("name", sorted(OVERFLOWS))
def test_compare_mode_at_the_repaired_block(ctx, name):
    """atz_trial with the zlib stream as the original, and with originals changed at one byte in the dynamic-tree header of the
    block that needed the depth-limit repair, in its symbols, and after it (in the block that follows, or in the adler32 trailer when
    the repaired block is the last); --shortcut-len / --recomp-tresh placed so that the prefix test ends inside that block"""
    make, memlevel, kind = OVERFLOWS[name]
    d = make()
    z = expect_deflate(d, 6, 15, memlevel)
    bl = fc.blocks(z)
    k = max(i for i, b in enumerate(bl) if b["type"] == 2 and fc.max_code_length(b, kind) == 15)
    rep = bl[k]
    h0, h1, e = rep["start"] // 8, rep["header_end"] // 8, rep["end"] // 8      # byte offsets in z
    later = [(bl[k + 1]["start"] + bl[k + 1]["end"]) // 16] if k + 1 < len(bl) else []
    origs = [z]
    for at in [h0 + 3, (h0 + h1) // 2, h1 + 40, (h1 + e) // 2, e - 2] + later + [len(z) - 2]:
        b = bytearray(z); b[at] ^= 0x24; origs.append(bytes(b))
    exact = az.ATZ_F_EXACT_RECORDS
    opts = [az.Options(flags=exact), az.Options(shortcutLength=h1 + 100, recompTresh=2, flags=exact),
            az.Options(shortcutLength=(h1 + e) // 2, recompTresh=1, sizediffTresh=4, flags=exact),
            az.Options(shortcutLength=h0 + 8, recompTresh=0, flags=exact)]
    for o in origs:
        for lvl, w, m in ((6, 15, memlevel), (5, 15, memlevel), (6, 15, memlevel - 1), (2, 15, memlevel)):
            for opt in opts:
                st, cp, ident = _trial_expect(d, o, lvl, w, m, opt)
                r = ctx.trial(d, o, lvl, w, m, opt)
                assert r.status == st, (lvl, m, opt.shortcutLength, r.status, st)
                if st == az.TR_COMPARED:
                    assert (r.out_len, r.ident) == (cp, ident), (lvl, m, opt.shortcutLength)
    r = ctx.trial(d, z, 6, 15, memlevel, az.Options(flags=exact))
    assert r.status == az.TR_COMPARED and r.out_len == len(z) == r.ident


def _container():
    ss = [expect_deflate(fc.lit_overflow(m, m), lvl, 15, m) for m in (7, 8, 9) for lvl in (2, 9)]
    ss += [expect_deflate(fc.dist_overflow(3, corpus.text(2000, 7)), lvl, 15, 9) for lvl in (3, 6)]
    ss += [expect_deflate(d, 6, 15, 1) for d in fc.static_ties(3)]
    ss += [expect_deflate(fc.slid_blocks(5, 10), lvl, 10, 8) for lvl in (1, 4)]
    ss += [expect_deflate(d, 9, 15, 8) for d in fc.length_runs(6)[:3]]
    return corpus.container(ss, 31)[0], len(ss)


def _records(data, opt, **env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        c = az.Context(0); c.load(data); c.scan(); c.search(opt)
        recs = [(s.offset, s.streamLength, s.inflatedLength, s.clevel, s.window, s.memlevel, s.identBytes, s.recomp, s.ndiff, s.offsetType)
                for s in c.streams()]
        diffs = c.diffs()
        c.close()
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
    return recs, diffs


def _fold(data, rec, opt):
    """the reference's search for one stream, restated on the CPU (SURVEY.md A.2, A.3): candidates in atz_host_candidate_sequence
    order, each judged by _trial_expect; the best is replaced only on a strictly larger ident, fullmatch (ident + mismatchTol >= C) is
    looked at only on an improvement and ends the walk; with --brute-window the other windows follow when C - best >= mismatchTol"""
    off, C = rec[0], rec[1]
    orig = data[off:off + C]
    plain = zlib.decompress(orig)
    best = [0, None]

    def walk(cands):
        for prm in cands:
            st, _, ident = _trial_expect(plain, orig, *prm, opt)
            if st == az.TR_COMPARED and ident > best[0]:
                best[:] = [ident, prm]
                if ident + opt.mismatchTol >= C:
                    return
    walk(seq(rec[9], 0))
    if opt.bruteforceWindow and C - best[0] >= opt.mismatchTol:
        walk(seq(rec[9], 1))
    return best


def test_search_records_with_and_without_the_burst_parse():
    """load + scan + search over a container of these streams: every record equals the CPU restatement of the reference's fold, and
    the serial parse (ATZ_BURST=0) and the burst parse, whose scratch is the tree area of the flush, give equal records"""
    data, n = _container()
    for opt in (az.Options(flags=az.ATZ_F_EXACT_RECORDS), az.Options(bruteforceWindow=True, mismatchTol=0, flags=az.ATZ_F_EXACT_RECORDS)):
        base = _records(data, opt)
        assert len(base[0]) == n
        for r in base[0]:
            ident, prm = _fold(data, r, opt)
            assert (r[3], r[4], r[5], r[6]) == (*prm, ident) and r[7] == (r[1] - ident <= opt.recompTresh), r
        assert _records(data, opt, ATZ_BURST=0) == base


def test_whole_path_round_trip():
    data, n = _container()
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        f = os.path.join(tmp, "in.bin"); open(f, "wb").write(data)
        pre = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz"], capture_output=True, text=True)
        assert pre.returncode == 0 and "OK! Restoration is bit by bit identical" in pre.stdout, pre.stdout + pre.stderr
        line = [l for l in pre.stdout.splitlines() if l.startswith("recompressed:")][0]
        assert [int(x) for x in line.split(":")[1].split("/")] == [n, n], line
        rec = subprocess.run([UNCOMP, "-r", "-i", f + ".atz", "-o", f + ".rec"], capture_output=True, text=True)
        assert rec.returncode == 0 and open(f + ".rec", "rb").read() == data
