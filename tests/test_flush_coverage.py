"""The block-flush branches each generator of flushcorpus.py is there to reach, measured with the CPU oracle's branch counters
(zref.oracle_flush_counts): a generator that drifts away from its branch fails here instead of quietly testing nothing.  The
counts in the comments were measured with this oracle, which is pinned to zlib 1.2.8's output (test_oracle_deflate)."""
import random

import pytest

import corpus
import flushcorpus as fc
import zref

# (generator id, its inputs, the (level, window, memLevel) set it is run with, counters that must be nonzero over that set)
TARGETS = {
    # over_lit: levels 2-9 at each memLevel (8 of 9); level 1 and memLevels <= 6 cannot reach it (see fc.lit_overflow)
    "lit_overflow_m7": (lambda: [fc.lit_overflow(7, 7)], [(l, 15, 7) for l in range(2, 10)], ["over_lit"]),
    "lit_overflow_m8": (lambda: [fc.lit_overflow(8, 8)], [(l, 15, 8) for l in range(2, 10)], ["over_lit"]),
    "lit_overflow_m9": (lambda: [fc.lit_overflow(9, 9)], [(l, 15, 9) for l in range(2, 10)], ["over_lit"]),
    # over_dist: levels 1-9 at memLevel 9, window 15 (9 of 9), with and without a block after the repaired one (see fc.dist_overflow)
    "dist_overflow_m9": (lambda: [fc.dist_overflow(1), fc.dist_overflow(2, corpus.text(3000, 5))], [(l, 15, 9) for l in range(1, 10)],
                         ["over_dist"]),
    # force_lit_high: empty blocks (9 at levels 1-9); force_dist_low: blocks without matches (39)
    "forced_lit": (fc.forced_lit, [(l, 15, 8) for l in range(1, 10)], ["force_lit_high", "force_dist_low"]),
    # distance trees with the one code 0 or 1 (12), or one code >= 2 (18)
    "single_distance_code": (lambda: fc.single_distance_code(3), [(l, 15, 8) for l in range(1, 10)], ["force_dist_low", "force_dist_high"]),
    "stored_ties": (lambda: fc.stored_ties(4), [(l, w, m) for l in range(1, 10) for w in (10, 15) for m in (1, 8)], ["tie_stored"]),   # 108
    "static_ties": (fc.static_ties, [(l, 15, m) for l in (3, 4, 6, 9) for m in (1, 2)], ["tie_static"]),                            # 12
    "slid_blocks_w9": (lambda: [fc.slid_blocks(5, 9)], [(l, 9, m) for l in range(1, 10) for m in (1, 8, 9)], ["unstorable"]),        # 18
    "slid_blocks_w10": (lambda: [fc.slid_blocks(5, 10)], [(l, 10, m) for l in range(1, 10) for m in (1, 8, 9)], ["unstorable"]),     # 18
    "length_runs": (lambda: fc.length_runs(6), [(l, 15, 8) for l in (1, 6, 9)],
                    ["rep16_6", "rep17_3", "rep17_10", "rep18_11", "rep18_138", "zrun_split"]),
}


def counts_over(inputs, params):
    zref.oracle_flush_counts()
    for d in inputs:
        for lvl, w, m in params:
            zref.oracle_deflate(d, lvl, w, m)
    return zref.oracle_flush_counts()


@pytest.mark.parametrize("name", sorted(TARGETS))
def test_generator_reaches_its_branch(name):
    make, params, want = TARGETS[name]
    c = counts_over(make(), params)
    assert all(c[k] > 0 for k in want), (name, {k: c[k] for k in want})


@pytest.mark.parametrize("memlevel", [7, 8, 9])
def test_lit_overflow_last_block_is_a_fibonacci_chain(memlevel):
    """what the oracle's (= zlib 1.2.8's) last block holds: only length codes 258.., counts 1597, 987, ... 2, 1 plus END_BLOCK, and a
    literal/length tree clamped to 15 bits"""
    z = zref.oracle_deflate(fc.lit_overflow(memlevel, memlevel), 6, 15, memlevel)
    last = fc.blocks(z)[-1]
    assert last["type"] == 2 and last["lit"][:256].sum() == 0 and last["dist"].sum() == last["lit"][257:].sum()
    got = sorted(int(x) for x in last["lit"][257:] if x)
    want = [1, 2]
    while len(want) < 16:
        want.append(want[-1] + want[-2])
    assert got == want and fc.max_code_length(last, 0) == 15


def test_dist_overflow_repaired_block_is_a_fibonacci_chain():
    """the repaired block's distance codes 13-29 carry exactly 1, 1, 2, ... 987, 1597 and nothing else, and the distance tree is
    clamped to 15 bits; with a tail, a block of its own follows"""
    for d, last in ((fc.dist_overflow(1), -1), (fc.dist_overflow(2, corpus.text(3000, 5)), -2)):
        bl = fc.blocks(zref.oracle_deflate(d, 6, 15, 9))
        blk = bl[last]
        want = [1, 1]
        while len(want) < 17:
            want.append(want[-1] + want[-2])
        assert list(blk["dist"][13:]) == want and blk["dist"][:13].sum() == 0 and fc.max_code_length(blk, 1) == 15


def test_oracle_counts_every_block_once():
    """the block-kind counters add up to the blocks the decoder finds"""
    d = corpus.text(50000, 3) + random.Random(1).randbytes(5000)
    for lvl, w, m in ((1, 15, 1), (6, 12, 8), (9, 15, 2)):
        zref.oracle_flush_counts()
        z = zref.oracle_deflate(d, lvl, w, m)
        c = zref.oracle_flush_counts()
        kinds = [b["type"] for b in fc.blocks(z)]
        assert (c["stored"], c["static"], c["dynamic"]) == (kinds.count(0), kinds.count(1), kinds.count(2))


def test_coverage_of_the_existing_kernel_grid():
    """the inputs of test_gpu_kernels.test_deflate_full_parameter_grid at levels 1-9 (measured: no literal/length or distance
    overflow, 491 bit-length-tree overflows, no stored tie): the branches flushcorpus.py exists for"""
    R = random.Random(1)
    ins = [corpus.text(70000, 2), corpus.binaryish(60000, 9), corpus.text(20000, 5) + R.randbytes(3000) + bytes(5000) + corpus.text(40000, 6)]
    c = counts_over(ins, [(l, w, m) for l in range(1, 10) for w in range(10, 16) for m in range(1, 10)])
    assert (c["over_lit"], c["over_dist"], c["over_bl"], c["tie_stored"]) == (0, 0, 491, 0)
    assert (c["stored"], c["static"], c["dynamic"]) == (2200, 325, 85360)
