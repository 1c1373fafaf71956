"""PNG corpus measurement for ATZ_SCAN_PNG_IDAT (uncomp --png): configs[2]'s generator parameters (500 images, 20-200 KB of
plaintext, half Z_FILTERED) written as PNGs with 8 KB IDAT chunks, scanned and searched with the flag off, with --png and with
--png --strategies.  Value MB/s uses bench.py's definition: input bytes over device-resident load + scan + search (CUDA events).
Prints one JSON line per mode and the card's name and power limit.

--apng: the same for ATZ_SCAN_APNG_FDAT (uncomp --apng): the same draws written as APNGs of four streams each, the default image in
8 KB IDAT chunks and three frames in 4 KB or 8 KB fdAT chunks, with the flag off, with --png, with --png --apng and with --png --apng
--strategies.

--overhead: the default bench.py workload (configs[4], 1 GB, --brute-window) with the flag off and on, alternating, `--steps` timed runs
each, each on a fresh context after one warm-up run; the records of the two must be identical.  With --apng the flag is
ATZ_SCAN_APNG_FDAT instead of ATZ_SCAN_PNG_IDAT.  Needs a B200."""
import argparse
import json
import os
import random
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

import antiz_b200 as az  # noqa: E402
import corpus  # noqa: E402
import zref  # noqa: E402
from test_gpu_apng_fdat import apng_file  # noqa: E402
from test_gpu_png_idat import idat_sizes, png_image  # noqa: E402


def c3_streams(n, seed, umin, umax, filtered_frac):
    r = random.Random(seed)
    for i in range(n):       # corpus.c3's draws, in the same order
        u = r.randint(umin, umax)
        d = corpus.binaryish(u, seed * 100003 + i) if i % 2 else corpus.text(u, seed * 100003 + i)
        lvl, w, m = r.randint(1, 9), r.randint(10, 15), r.randint(1, 9)
        strat = 1 if (r.random() < filtered_frac and lvl >= 4) else 0
        yield r, zref.ref_deflate(d, lvl, w, m, strat)


def png_corpus(n=500, seed=3, umin=20_000, umax=200_000, filtered_frac=0.5):
    imgs = [png_image(z, idat_sizes(len(z), 8192, r), i)[0] for i, (r, z) in enumerate(c3_streams(n, seed, umin, umax, filtered_frac))]
    return corpus.container(imgs, seed)[0]


def apng_corpus(n=500, seed=3, umin=20_000, umax=200_000, filtered_frac=0.5):
    """APNGs of four c3 streams each: the default image in 8 KB IDATs, three frames in 4 KB (even APNGs) or 8 KB (odd) fdATs"""
    zs = [z for _, z in c3_streams(n, seed, umin, umax, filtered_frac)]
    r = random.Random(seed + 1)
    imgs = []
    for k in range(0, n, 4):
        dflt = (zs[k], idat_sizes(len(zs[k]), 8192, r))
        frames = [(z, idat_sizes(len(z), 4096 if k % 8 == 0 else 8192, r)) for z in zs[k + 1:k + 4]]
        imgs.append(apng_file(dflt, frames, k)[0])
    return corpus.container(imgs, seed)[0]


def measure(data, dev, flags, opt, steps=3):
    ctx = az.Context(0)
    if flags:
        ctx.set_scan_flags(flags)
    best = None
    for _ in range(steps + 1):    # the first pass warms up
        ctx.timer_start()
        ctx.load_device(dev.data_ptr(), len(data)); ctx.scan(); ctx.search(opt)
        ms = ctx.timer_stop()
        best = ms if best is None else min(best, ms)
    st = ctx.stats(); ss = ctx.streams()
    atz = 28; last = 0
    for i, s in enumerate(ss):
        pc = ctx.pieces(i); fr = ctx.framing(i); span = s.streamLength + fr * max(0, len(pc) - 1)
        atz += s.offset - last if s.offset >= last else 0
        atz += 35 + (8 + 9 * s.ndiff if s.ndiff else 0) + s.inflatedLength + (8 + 4 * len(pc) + fr * (len(pc) - 1) if pc else 0) if s.recomp else span
        last = s.offset + span
    atz += max(0, len(data) - last)
    out = dict(streams=len(ss), split=sum(1 for i in range(len(ss)) if ctx.pieces(i)), recompressed=int(st.n_recomp), atz_bytes=atz,
               value_MBps=round(len(data) / 1e6 / (best / 1e3), 2), ms_best=round(best, 1), ms_scan=round(st.ms_scan, 2), ms_probe=round(st.ms_inflate_probe, 2))
    ctx.close()
    return out


def overhead(steps, name="png", flag=az.ATZ_SCAN_PNG_IDAT):
    import bench
    data = bench.make_container("c5", bench.C5_DEFAULT_MB, bench.SEED)
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    opt = az.Options(bruteforceWindow=True)
    ms = {"off": [], name: []}
    recs = {}
    for i in range(steps):     # one context at a time (each takes 60 % of the free memory as its budget): a warm-up run, then a timed one
        for k, flags in (("off", 0), (name, flag)):
            ctx = az.Context(0)
            if flags:
                ctx.set_scan_flags(flags)
            for _ in range(2):     # the warm-up, then the timed run
                ctx.timer_start()
                ctx.load_device(dev.data_ptr(), len(data)); ctx.scan(bench.CHUNKSIZE); ctx.search(opt)
                t = ctx.timer_stop()
            ms[k].append(round(t, 1))
            recs[k] = ctx.stream_table()
            ctx.close()
    same = recs["off"].tobytes() == recs[name].tobytes() and len(recs["off"]) > 0
    print(json.dumps({"workload": "configs[4]", "input_bytes": len(data), "streams": len(recs["off"]), "records_identical": same,
                      "ms_off": ms["off"], "ms_" + name: ms[name], "value_MBps_off": [round(len(data) / 1e3 / t, 1) for t in ms["off"]],
                      "value_MBps_" + name: [round(len(data) / 1e3 / t, 1) for t in ms[name]]}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--overhead", action="store_true")
    ap.add_argument("--apng", action="store_true")
    ap.add_argument("--steps", type=int, default=3)
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps(dict(card=smi[0] if smi else "unknown")))
    if a.overhead:
        return overhead(a.steps, *(("apng", az.ATZ_SCAN_APNG_FDAT) if a.apng else ()))
    PNG, APNG, STRAT = az.ATZ_SCAN_PNG_IDAT, az.ATZ_SCAN_APNG_FDAT, az.Options(flags=az.ATZ_F_STRATEGIES)
    data = apng_corpus() if a.apng else png_corpus()
    dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    print(json.dumps(dict(input_bytes=len(data))))
    modes = ((("off", 0, az.Options()), ("png", PNG, az.Options()), ("png+apng", PNG | APNG, az.Options()), ("png+apng+strategies", PNG | APNG, STRAT))
             if a.apng else (("off", 0, az.Options()), ("png", PNG, az.Options()), ("png+strategies", PNG, STRAT)))
    for name, flags, opt in modes:
        print(json.dumps(dict(mode=name, **measure(data, dev, flags, opt))), flush=True)


if __name__ == "__main__":
    main()
