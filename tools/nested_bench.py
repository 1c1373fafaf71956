"""Nested-stream measurement for ATZ_F_NESTED_DEPTH (uncomp --nested N).  A seeded corpus of outer zlib streams at levels 0-9, each
holding a corpus.container (64-256 KB of compressed streams: an outer stream that runs over several of the scan's 512 KB chunks is
lost to the reference's chunk-overlap quirk) of c2-style (text, 1-64 KB, levels 1-9) and c4-style (0.5-8 KB slices of one text, levels 1/6/9) streams;
every fifth container also holds a zlib stream around another such container (depth 2).  For --nested 0, 1 and 2 it reports:
  * the streams found and recompressed per depth;
  * the ATZ bytes (`uncomp --notest` writes the file) and the deflate bytes left in it: the compressed bytes of every known stream that
    the file still holds compressed (a top-level stream, or one inside a stored plaintext, that this depth did not recompress);
  * lzma of a 16 MB sample of the ATZ file (16 slices of 1 MB spread over it);
  * value MB/s, png_bench.py's definition: input bytes over device-resident load + scan + search (CUDA events, best of --steps after
    a warm-up);
  * the reconstruct time: the wall time of `uncomp -r`, context creation included.
Prints the card's name and power limit first.

--overhead: the default bench.py workload (configs[4], 1 GB, --brute-window) with depth 0 and depth 2, alternating, `--steps` timed runs
each, each on a fresh context after one warm-up run; the top-level records of the two must be identical.  Needs a B200."""
import argparse
import json
import lzma
import multiprocessing
import os
import random
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

import antiz_b200 as az  # noqa: E402
import corpus  # noqa: E402
import zref  # noqa: E402

UNCOMP = os.path.join(ROOT, "antiz_b200", "uncomp")


def _inner(seed, target):
    """c2- and c4-style zlib streams, about `target` compressed bytes of them"""
    r = random.Random(seed)
    big = corpus.text(1 << 20, seed)
    out, size, i = [], 0, 0
    while size < target:
        i += 1
        if r.random() < 0.5:
            s = zref.ref_deflate(corpus.text(r.randint(1 << 10, 64 << 10), seed * 100003 + i), r.randint(1, 9), 15, 8)
        else:
            u = r.randint(512, 8192); o = r.randint(0, len(big) - u)
            s = zref.ref_deflate(big[o:o + u], r.choice([1, 6, 6, 6, 9]), 15, 8)
        out.append(s); size += len(s)
    return out


def _outer(args):
    seed, k = args
    r = random.Random(seed * 7919 + k)
    parts = _inner(seed * 1000 + k, r.randint(64 << 10, 256 << 10))
    if k % 5 == 0:      # depth 2: a zlib stream around another container
        deep = corpus.container(_inner(seed * 1000 + k + 500, 64 << 10), seed + k)[0]
        parts.insert(len(parts) // 2, zref.ref_deflate(deep, r.choice([0, 1, 6, 9]), 15, 8))
    return zref.ref_deflate(corpus.container(parts, seed + k)[0], k % 10, 15, 8)


def nested_corpus(mb, seed=7):
    n = max(1, mb * 6)
    with multiprocessing.Pool(min(32, os.cpu_count() or 1)) as pool:
        outers = pool.map(_outer, [(seed, k) for k in range(n)])
    return corpus.container(outers, seed)[0]


def records(data, depth, dev, steps):
    """(value ms best, stats, top-level records, nested (parent, depth, C, recomp)) of one context"""
    ctx = az.Context(0)
    best = None
    opt = az.Options(flags=az.nested_depth(depth))
    for i in range(steps + 1):    # the first pass warms up
        ctx.timer_start()
        ctx.load_device(dev.data_ptr(), len(data)); ctx.scan(); ctx.search(opt)
        ms = ctx.timer_stop()
        if i:
            best = ms if best is None else min(best, ms)
    top = [(s.streamLength, s.recomp) for s in ctx.streams()]
    nest = [(x.parent, x.depth, x.s.streamLength, x.s.recomp) for x in ctx.nested()]
    st = ctx.stats()
    ctx.close()
    return best, st, top, nest


def deflate_left(top, nest, depth):
    """compressed bytes the file holds for the streams known from the deepest run (see the module's docstring)"""
    n = len(top)
    opened = [rc for _, rc in top]             # plaintext stored: recompressed at a depth this run searched
    left = sum(c for c, rc in top if not rc)
    nopen = []
    for p, d, c, rc in nest:
        parent_open = opened[p] if p < n else nopen[p - n]
        mine = bool(rc) and d <= depth
        nopen.append(parent_open and mine)
        if parent_open and not mine:
            left += c
    return left


def uncomp_sizes(data, depth, tmp):
    f = os.path.join(tmp, "in")
    with open(f, "wb") as fh:
        fh.write(data)
    p = subprocess.run([UNCOMP, "-i", f, "-o", f + ".atz", "--notest", "--nested", str(depth)], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-2000:]
    atz = open(f + ".atz", "rb").read()
    t0 = time.perf_counter()
    r = subprocess.run([UNCOMP, "-r", "-i", f + ".atz", "-o", f + ".rec"], capture_output=True, text=True)
    t_rec = time.perf_counter() - t0
    assert r.returncode == 0 and open(f + ".rec", "rb").read() == data, r.stdout[-2000:]
    step = max(1, len(atz) // 16)
    sample = b"".join(atz[i * step:i * step + (1 << 20)] for i in range(16))
    os.remove(f + ".rec"); os.remove(f + ".atz")
    return len(atz), len(lzma.compress(sample, preset=6)), len(sample), t_rec


def overhead(steps):
    import bench
    data = bench.make_container("c5", bench.C5_DEFAULT_MB, bench.SEED)
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    ms = {0: [], 2: []}
    recs = {}
    nested = {}
    for i in range(steps):     # one context at a time (each takes 60 % of the free memory as its budget): a warm-up run, then a timed one
        for d in (0, 2):
            ctx = az.Context(0)
            opt = az.Options(bruteforceWindow=True, flags=az.nested_depth(d))
            for _ in range(2):
                ctx.timer_start()
                ctx.load_device(dev.data_ptr(), len(data)); ctx.scan(bench.CHUNKSIZE); ctx.search(opt)
                t = ctx.timer_stop()
            ms[d].append(round(t, 1))
            recs[d] = ctx.stream_table()
            nested[d] = len(ctx.nested())
            st = ctx.stats()
            ctx.close()
    same = recs[0].tobytes() == recs[2].tobytes() and len(recs[0]) > 0
    plain = int(sum(int(x) for x in recs[0]["inflatedLength"][recs[0]["recomp"] == 1]))
    print(json.dumps(dict(workload="configs[4]", input_bytes=len(data), streams=len(recs[0]), records_identical=same, nested_found=nested[2],
                          plaintext_scanned_bytes=plain, ms_depth0=ms[0], ms_depth2=ms[2], value_MBps_depth0=[round(len(data) / 1e3 / t, 1) for t in ms[0]],
                          value_MBps_depth2=[round(len(data) / 1e3 / t, 1) for t in ms[2]], last_ms_scan=round(st.ms_scan, 1))), flush=True)
    if not same:
        sys.exit("the top-level records differ between depth 0 and depth 2")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--overhead", action="store_true")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--mb", type=int, default=256, help="approximate corpus size")
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps(dict(card=smi[0] if smi else "unknown")), flush=True)
    if a.overhead:
        return overhead(a.steps)
    data = nested_corpus(a.mb)
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    print(json.dumps(dict(input_bytes=len(data))), flush=True)
    runs = {d: records(data, d, dev, a.steps) for d in (0, 1, 2)}
    _, _, top2, nest2 = runs[2]
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        for d in (0, 1, 2):
            ms, st, top, nest = runs[d]
            per = {"0": [len(top), sum(rc for _, rc in top)]}
            for k in (1, 2):
                per[str(k)] = [sum(1 for x in nest if x[1] == k), sum(x[3] for x in nest if x[1] == k)]
            atz, lz, sample, t_rec = uncomp_sizes(data, d, tmp)
            print(json.dumps(dict(nested=d, found_recompressed_by_depth=per, atz_bytes=atz, deflate_bytes_left=deflate_left(top2, nest2, d),
                                  lzma_sample=lz, sample_bytes=sample, value_MBps=round(len(data) / 1e6 / (ms / 1e3), 2), ms_best=round(ms, 1),
                                  reconstruct_s=round(t_rec, 2))), flush=True)


if __name__ == "__main__":
    main()
