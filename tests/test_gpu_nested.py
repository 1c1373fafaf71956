"""-m gpu: ATZ_F_NESTED_DEPTH (uncomp --nested N).  Containers of zlib streams are wrapped in outer zlib streams (levels 0-9, and one
level deeper for a depth-2 set); the nested records are checked against a restatement of the inner scan over each recompressed parent's
plaintext, and the ATZ files round-trip through `uncomp -r`."""
import hashlib
import os
import random
import subprocess
import tempfile
import zlib

import pytest

import antiz_b200 as az
import corpus
import zref
from test_gpu_png_idat import Corpus as PngCorpus

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")
SW = az.ATZ_SCAN_SMALL_WINDOWS
TMP = "/dev/shm" if os.path.isdir("/dev/shm") else None
EXACT = az.ATZ_F_EXACT_RECORDS


def py_inner(P, flags=0):
    """the inner scan (include/antiz_b200.h ATZ_F_NESTED_DEPTH) restated with zlib: [(offset, C, plaintext)]"""
    out, p, n = [], 0, len(P)
    while p + 1 < n:
        if az.lib().atz_host_header_type(flags, P[p], P[p + 1]) >= 0:
            d = zlib.decompressobj()
            try:
                u = d.decompress(P[p:])
                ok = d.eof
            except zlib.error:
                ok = False
            if ok:
                c = n - p - len(d.unused_data)
                if c > 16:
                    out.append((p, c, u)); p += c
                    continue
        p += 1
    return out


def inner_streams(seed, k, umax=40000):
    r = random.Random(seed)
    return [zref.ref_deflate(corpus.text(r.randint(200, umax), seed * 1000 + i) if i % 3 else corpus.binaryish(r.randint(200, umax), seed * 1000 + i),
                             r.randint(1, 9), 15, 8) for i in range(k)]


def nested_corpus(seed, nouter=10, depth2=True):
    """outer streams at levels 0..9 around containers of zlib streams; with depth2, some inner streams hold containers themselves"""
    r = random.Random(seed)
    outers = []
    for i in range(nouter):
        parts = inner_streams(seed * 100 + i, r.randint(1, 6))
        if depth2 and i % 3 == 1:
            deep = corpus.container(inner_streams(seed * 100 + 50 + i, 3, 8000), seed + i)[0]
            parts.append(zref.ref_deflate(deep, r.choice([0, 1, 6, 9]), 15, 8))
        outers.append(zref.ref_deflate(corpus.container(parts, seed * 7 + i)[0], i % 10, 15, 8))
        if i % 4 == 3:
            outers.append(zref.ref_deflate(corpus.text(r.randint(500, 20000), seed + 99 * i), r.randint(1, 9), 15, 8))   # nothing inside
    return corpus.container(outers, seed)[0]


def rec(s):
    return (s.offset, s.streamLength, s.inflatedLength, s.offsetType, s.clevel, s.window, s.memlevel, s.identBytes, s.recomp, s.ndiff, s.firstDiffByte)


def search(data, depth, opt=None, flags=0, env=None, budget=None, chunksize=524288):
    """(top records, nested (parent, depth, record), diffs, nested payloads, the context's top-level payloads of recompressed streams)"""
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update({k: str(v) for k, v in (env or {}).items()})
    try:
        c = az.Context(0)
        if flags:
            c.set_scan_flags(flags)
        if budget:
            c.set_budget(budget)
        c.load(data); n = c.scan(chunksize)
        o = opt or az.Options(flags=EXACT)
        o.flags |= az.nested_depth(depth)
        c.search(o)
        top = c.streams(); nest = c.nested(); do, dv = c.diffs()
        out = dict(top=[rec(s) for s in top], nested=[(x.parent, x.depth, rec(x.s)) for x in nest], diffs=(do, dv),
                   ndiffs=[(list(do[x.s.diff_index:x.s.diff_index + x.s.ndiff]), bytes(dv[x.s.diff_index:x.s.diff_index + x.s.ndiff])) for x in nest],
                   payload=[c.inflated(n + j, x.s.inflatedLength) for j, x in enumerate(nest)],
                   plain={i: c.inflated(i, s.inflatedLength) for i, s in enumerate(top) if s.recomp}, stats=c.stats())
        c.close()
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
    return out


def expected(res, depth, flags=0):
    """the nested list restated from the top-level payloads and the nested payloads: (parent, depth, offset, C, U) in the API's order"""
    n = len(res["top"]); want = []; plains = []
    level = [(i, res["plain"][i]) for i in sorted(res["plain"])]
    for d in range(1, depth + 1):
        nxt = []
        for pid, P in level:
            for off, c, u in py_inner(P, flags):
                want.append((pid, d, off, c, len(u))); plains.append(u)
                j = len(want) - 1
                if j < len(res["nested"]) and res["nested"][j][2][8]:     # recompressed: its plaintext is entered at the next level
                    nxt.append((n + j, u))
        level = nxt
    return want, plains


def check_records(res, depth, flags=0):
    want, plains = expected(res, depth, flags)
    got = [(p, d, r[0], r[1], r[2]) for p, d, r in res["nested"]]
    assert got == want
    assert res["payload"] == plains
    return want


@pytest.fixture(scope="module")
def nc():
    return nested_corpus(5)


def test_records_match_the_restatement(nc):
    r1, r2 = search(nc, 1), search(nc, 2)
    w1 = check_records(r1, 1); w2 = check_records(r2, 2)
    assert r1["top"] == r2["top"] == search(nc, 0)["top"]
    assert len(w1) >= 20 and sum(1 for x in w2 if x[1] == 2) >= 6
    assert [x for x in r2["nested"] if x[1] == 1] == r1["nested"]      # --nested 1 stops at level 1
    assert all(x[2][8] for x in r1["nested"])                          # zlib's own streams with default memLevel: all recompressed
    # the parents: only recompressed streams are entered; the top level counts stay top-level
    top = r1["top"]
    assert all(top[p][8] for p, d, _ in r1["nested"])
    s0, s1 = search(nc, 0)["stats"], r1["stats"]
    assert (s0.n_streams, s0.n_recomp) == (s1.n_streams, s1.n_recomp) and s1.ref_trials > s0.ref_trials


def uncomp(data, args, name="f"):
    """uncomp (with its self test) then uncomp -r; returns (stdout, .atz bytes)"""
    with tempfile.TemporaryDirectory(dir=TMP) as tmp:
        f = os.path.join(tmp, name)
        open(f, "wb").write(data)
        p = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz"] + args, capture_output=True, text=True)
        assert p.returncode == 0 and "bit by bit identical" in p.stdout, (args, p.stdout[-2000:], p.stderr[-2000:])
        r = subprocess.run([UNCOMP, "-r", "-i", f + ".atz", "-o", f + ".rec"], capture_output=True, text=True)
        assert r.returncode == 0 and open(f + ".rec", "rb").read() == data, r.stdout
        return p.stdout, open(f + ".atz", "rb").read()


@pytest.mark.parametrize("args", [["--nested", "1"], ["--nested", "2"], ["--nested", "2", "--brute-window"], ["--nested", "2", "--strategies"],
                                  ["--nested", "2", "--small-windows"]])
def test_round_trip(nc, args):
    out, atz = uncomp(nc, args)
    line = [x for x in out.splitlines() if x.startswith("nested recompressed:")]
    assert len(line) == 1
    a, b = map(int, line[0].split(":")[1].split("/"))
    assert a >= 20 and a <= b
    plain = uncomp(nc, [])[1]
    assert len(atz) > len(plain)        # the inner streams' plaintext is stored in place of their compressed bytes


def test_small_windows_inside():
    """CINFO 1 inner streams are found with --small-windows only"""
    r = random.Random(3)
    parts = [zref.ref_deflate(corpus.text(r.randint(2000, 9000), 300 + i), 6, 9, 8) for i in range(4)] + inner_streams(31, 2)
    data = corpus.container([zref.ref_deflate(corpus.container(parts, 1)[0], 6, 15, 8)], 2)[0]
    a, b = search(data, 1), search(data, 1, flags=SW)
    check_records(a, 1); check_records(b, 1, SW)
    assert len(b["nested"]) == len(a["nested"]) + 4
    uncomp(data, ["--nested", "1", "--small-windows"])


def test_edge_cases():
    r = random.Random(9)
    z = inner_streams(77, 6, 20000)
    tiny = [zlib.compress(b""), zlib.compress(b"a"), zlib.compress(b"abcabc")]
    assert all(len(t) <= 16 for t in tiny)
    flipped = bytearray(z[3]); flipped[len(flipped) // 2] ^= 0x10
    imperfect = zref.ref_deflate_ex(corpus.text(30000, 5), 6, 15, 8, flushes=[(29990, 2)])
    j = lambda n: corpus.junk(n, r.randint(0, 1 << 30))
    P1 = z[0] + j(50) + z[1] + z[2] + j(30) + bytes(flipped) + j(40) + imperfect + j(20) + b"".join(tiny) + j(10) + z[4]   # offset 0, adjacent, last byte
    P2 = j(100) + z[5][:-5]                                                            # truncated at the end of P
    big = corpus.container(inner_streams(88, 24, 60000), 4)[0]
    assert len(big) > 2 * 65536                                                        # level 0: crosses stored-block boundaries
    bc = corpus.container(inner_streams(99, 3), 5)[0]
    bad_outer = zref.ref_deflate_ex(bc, 6, 15, 8, flushes=[(k, 2) for k in range(300, len(bc) - 100, 300)])   # no parameter set comes close
    data = corpus.container([zref.ref_deflate(P1, 6, 15, 8), zref.ref_deflate(P2, 9, 15, 8), zref.ref_deflate(big, 0, 15, 8), bad_outer], 6)[0]
    res = search(data, 2, az.Options(flags=EXACT, recompTresh=400))
    want = check_records(res, 2)
    top = res["top"]
    assert top[0][8] and top[1][8] and top[2][8] and not top[3][8]
    assert not [x for x in res["nested"] if x[0] == 3]                                 # not recompressed: not entered
    l0 = [x for x in want if x[0] == 0]
    assert l0[0][2] == 0 and l0[-1][2] + l0[-1][3] == len(P1)
    assert [x for x in want if x[0] == 1] == []
    assert len([x for x in want if x[0] == 2]) == 24
    ni = [x for x in res["nested"] if x[2][2] == 30000]
    assert len(ni) == 1 and ni[0][2][8] and ni[0][2][9] > 0                            # the imperfect stream: recompressed with diffs
    o, v = res["diffs"]
    assert len(o) == sum(x[2][9] for x in res["nested"]) + sum(t[9] for t in top)
    uncomp(data, ["--nested", "2", "--recomp-tresh", "400"])


@pytest.mark.parametrize("name", ["c2", "imperfect", "extremes", "mixed", "png"])
def test_no_nested_streams_same_atz(name):
    data = {"c2": lambda: corpus.c2(nstreams=60), "imperfect": corpus.imperfect, "extremes": corpus.extremes,
            "mixed": lambda: corpus.mixed(16 << 20), "png": lambda: PngCorpus(11).data}[name]()
    extra = ["--png"] if name == "png" else []
    a = uncomp(data, extra)[1]
    b = uncomp(data, extra + ["--nested", "3"])[1]
    assert a == b


def tree_key(nested, n, j):
    """a nested entry identified independently of list positions: (top-level parent, offsets down to it)"""
    p, d, r = nested[j]
    return (p,) + (r[0],) if p < n else tree_key(nested, n, p - n) + (r[0],)


@pytest.mark.parametrize("nsh", [2, 3, 5])
def test_shards_union_equals_one_context(nc, nsh):
    """emulated shards: the union of their nested lists, diffs and payloads is one context's"""
    one = search(nc, 2, chunksize=65536)
    n = len(one["top"])

    def items(res):
        return sorted((tree_key(res["nested"], n, j), x[1], x[2], res["ndiffs"][j], hashlib.sha1(res["payload"][j]).hexdigest())
                      for j, x in enumerate(res["nested"]))
    ctxs = [az.Context(0) for _ in range(nsh)]
    for g, c in enumerate(ctxs):
        c.attach(nc); c.scan_shard(65536, g, nsh)
    blobs = [c.probe_export() for c in ctxs]
    got = []
    for g, c in enumerate(ctxs):
        for h in range(nsh):
            if h != g:
                c.probe_import(h, blobs[h])
        assert c.scan_finish() == n
        c.search(az.Options(flags=EXACT | az.nested_depth(2)), g, nsh)
        ns = c.nested(); co, cv = c.diffs()
        got += items(dict(nested=[(x.parent, x.depth, rec(x.s)) for x in ns], payload=[c.inflated(n + j, x.s.inflatedLength) for j, x in enumerate(ns)],
                          ndiffs=[(list(co[x.s.diff_index:x.s.diff_index + x.s.ndiff]), bytes(cv[x.s.diff_index:x.s.diff_index + x.s.ndiff])) for x in ns]))
        assert all(ctxs[0].owners()[x.parent] == g for x in ns if x.parent < n)
    assert sorted(got) == items(one)
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("gpus", [2, 4])
def test_gpus_write_the_same_atz(nc, gpus):
    a = uncomp(nc, ["--nested", "2"])[1]
    env = dict(os.environ, ATZ_TEST_ONE_DEVICE="1")
    with tempfile.TemporaryDirectory(dir=TMP) as tmp:
        f = os.path.join(tmp, "f")
        open(f, "wb").write(nc)
        p = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--nested", "2", "--gpus", str(gpus), "--notest"], capture_output=True, text=True, env=env)
        assert p.returncode == 0, p.stdout
        assert open(f + ".atz", "rb").read() == a


def test_search_schedule_does_not_change_nested_records(nc):
    want = search(nc, 2, env=dict(ATZ_LANES=1))
    keys = ("top", "nested", "diffs", "ndiffs", "payload")
    # ATZ_NEST_BATCH: the byte limit of a scan batch and of a probe launch's output regions (1: one parent per batch, one candidate
    # per launch; 200000: several of each, grown regions split over launches)
    for kw in (dict(env=dict(ATZ_LANES=2)), dict(env=dict(ATZ_BURST=0)), dict(budget=64 << 20), dict(env=dict(ATZ_NEST_BATCH=1)),
               dict(env=dict(ATZ_NEST_BATCH=200000))):
        got = search(nc, 2, **kw)
        assert all(got[k] == want[k] for k in keys), kw


def test_depth_limit():
    c = az.Context(0)
    c.load(nested_corpus(8, nouter=2, depth2=False)); c.scan()
    for flags in (az.nested_depth(9), az.nested_depth(256), az.nested_depth(265), -1):     # refused, not wrapped to a smaller depth
        with pytest.raises(az.AtzError) as e:
            c.search(az.Options(flags=flags))
        assert e.value.code == az.ATZ_E_ARG
    c.search(az.Options(flags=az.nested_depth(8)))
    assert len(c.nested()) > 0
    c.close()
