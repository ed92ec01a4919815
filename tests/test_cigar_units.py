"""The device keeps the CIGAR stream as 16-bit units (inq_device.cuh, "CIGAR units"): H, P and the invalid op codes are
dropped, long M/N/=/X are split, long I/D/S become a head with the full length beside it. These tests put every op code
at the lengths around the unit limits into reads, at positions that straddle lanes, warp tiles and push chunks, and
check medians against the oracle and the event lists against a CIGAR walk, bit for bit. The statistics keep counting
BAM words."""
import os
import re

import numpy as np
import pytest

from oracle import oracle as O
from oracle.oracle import Reads, cigar_ref_len
from tests.datagen import expected_events, make_case, random_cigar

LENS = (0, 1, 4094, 4095, 4096, 8191, 65535, (1 << 28) - 1)
MINLENS = (0, 5, 4094, 4095, 4096, (1 << 28) - 1)


def stage_words() -> int:
    """BAM words per encoding chunk of a push, as the library defines it (kPushChunkWords in inq_capi.cu)"""
    src = open(os.path.join(os.path.dirname(__file__), "..", "inquistr_b200", "csrc", "inq_capi.cu")).read()
    m = re.search(r"constexpr uint64_t kPushChunkWords = 1ull << (\d+);", src)
    assert m, "kPushChunkWords not found in inq_capi.cu"
    return 1 << int(m.group(1))


def walk_events(reads: Reads, minlen: int):
    """expected_events, vectorised: (pos1, val) per event in CIGAR order, first event of every read"""
    w = reads.cigar.astype(np.int64)
    op, ln = w & 15, w >> 4
    n = len(w)
    rid = np.repeat(np.arange(reads.n), np.diff(reads.cigar_off.astype(np.int64)))
    cons = np.where(np.isin(op, [0, 2, 3, 7, 8]), ln, 0)
    before = np.cumsum(cons) - cons                                          # consumed before each word, stream-wide
    start = before[reads.cigar_off[:-1].astype(np.int64).clip(max=max(n - 1, 0))] if n else np.zeros(reads.n, np.int64)
    ev = np.isin(op, [1, 2, 4]) & (ln > minlen)
    pos = (reads.ref_start.astype(np.int64)[rid] + 1 + before - start[rid]) & 0xFFFFFFFF
    val = (np.where(op == 2, -ln, ln) << 1) | (op == 4)
    off = np.concatenate([[0], np.cumsum(np.bincount(rid[ev], minlength=reads.n))])
    return pos[ev].astype(np.uint32), val[ev].astype(np.int32), off.astype(np.uint32)


def joined_words(reads: Reads, case, unphased: bool) -> int:
    """BAM words of the reads that land at least one call in a bucket"""
    ls = case["locus_start"].astype(np.int64)[None, :]
    le = case["locus_end"].astype(np.int64)[None, :]
    lc = case["locus_contig"][None, :]
    rs = reads.ref_start.astype(np.int64)[:, None]
    re = reads.ref_end.astype(np.int64)[:, None]
    start_ext, end_ext = (ls - 10) & 0xFFFFFFFF, le + 10
    if unphased:
        keep = ~((start_ext < rs) | (re < end_ext))
        ok = reads.mapq > 10
    else:
        keep = (rs < end_ext) & (re > start_ext) & ~((start_ext < rs) & (re < end_ext))
        ok = (reads.mapq > 10) & ((reads.hp == 1) | (reads.hp == 2))
    joined = ok & ((reads.contig[:, None] == lc) & keep).any(axis=1)
    return int(np.diff(reads.cigar_off.astype(np.int64))[joined].sum())


def long_case(seed, filler_words=0, n_reads=400, n_lens=LENS):
    """make_case reads plus reads aimed at loci that carry one special word (every op code 0..15 at every length of
    n_lens) behind a random number of short filler ops, a few reads whose whole CIGAR is dropped ops, and optionally a
    first read of `filler_words` words that moves everything after it across a push chunk boundary"""
    base = make_case(seed, n_contigs=2, contig_len=60_000, n_loci=60, n_reads=n_reads, max_read=3000)
    rng = np.random.default_rng(seed + 1000)
    r0 = base["reads"]
    contig, rs, re, mq, hp, fl, cig = [], [], [], [], [], [], []

    def add(c, start, words, h=1):
        rlen = cigar_ref_len(words)
        contig.append(c); rs.append(start); re.append(start + max(rlen, 1))
        mq.append(60); hp.append(h); fl.append(0); cig.append(np.asarray(words, np.uint32))

    if filler_words:
        add(0, 100, np.full(filler_words, (1 << 4) | 1, np.uint32))          # 1I x filler_words: no consumption
    for r in range(r0.n):
        a, b = int(r0.cigar_off[r]), int(r0.cigar_off[r + 1])
        contig.append(int(r0.contig[r])); rs.append(int(r0.ref_start[r])); re.append(int(r0.ref_end[r]))
        mq.append(int(r0.mapq[r])); hp.append(int(r0.hp[r])); fl.append(int(r0.flags[r])); cig.append(r0.cigar[a:b])
    n_loci = len(base["locus_start"])
    for code in range(16):
        for ln in n_lens:
            for rep in range(2):
                k = int(rng.integers(0, n_loci))
                c, s = int(base["locus_contig"][k]), int(base["locus_start"][k])
                left = int(rng.integers(20, 400))
                # a random count of filler ops (1I: one unit; 0X and 3H: dropped) puts the special word at every offset
                # of a lane and of a warp tile
                pad = rng.choice(np.asarray([(1 << 4) | 1, 8, (3 << 4) | 5], np.uint32), int(rng.integers(0, 2100 if rep else 70)))
                pre = random_cigar(rng, left, exotic=True, clip_rate=0.0)
                post = random_cigar(rng, int(rng.integers(50, 400)), exotic=True, clip_rate=0.0)
                add(c, max(0, s - left), np.concatenate([pad, pre, [np.uint32((ln << 4) | code)], post]), h=1 + rep)
    for dropped in ([5, 6], [9, 10, 11, 12, 13, 14, 15], [5]):
        k = int(rng.integers(0, n_loci))
        add(int(base["locus_contig"][k]), max(0, int(base["locus_start"][k]) - 20),
            np.asarray([(int(rng.integers(1, 4096)) << 4) | d for d in dropped], np.uint32))
    off = np.concatenate([[0], np.cumsum([len(w) for w in cig])]).astype(np.uint64)
    reads = Reads(np.asarray(contig), np.asarray(rs), np.asarray(re), np.asarray(mq), np.asarray(hp), np.asarray(fl), off,
                  np.concatenate(cig).astype(np.uint32))
    return dict(base, reads=reads)


def test_walk_events_matches_cigar_walk():
    case = make_case(5, n_reads=300)
    for minlen in (0, 5):
        got, exp = walk_events(case["reads"], minlen), expected_events(case["reads"], minlen)
        assert all(np.array_equal(a, b) for a, b in zip(got, exp))


@pytest.fixture(scope="module")
def ctx():
    import inquistr_b200 as q
    c = q.Context(0)
    yield c
    c.close()


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def push_chunked(ctx, rd, chunks):
    cuts = np.linspace(0, rd.n, chunks + 1).astype(int)
    for a, b in zip(cuts[:-1], cuts[1:]):
        if b > a:
            base = rd.cigar_off[a]
            ctx.push_reads(rd.contig[a:b], rd.ref_start[a:b], rd.ref_end[a:b], rd.mapq[a:b], rd.hp[a:b], rd.flags[a:b],
                           rd.cigar_off[a:b + 1] - base, rd.cigar[int(base):int(rd.cigar_off[b])])


def check(ctx, case, minlen, unphased, all_reads=True):
    """all_reads: the context holds every read of the case (not only those a routed push keeps)"""
    rd = case["reads"]
    res = ctx.genotype(minlen, 3, unphased)
    rc, p1, p2, visits = O.genotype_loci(rd, case["n_contigs"], case["locus_contig"], case["locus_start"],
                                         case["locus_end"], minlen, 3, unphased, threads=4)
    assert rc == 0
    assert same(res.phase1, p1) and same(res.phase2, p2), minlen
    st = res.stats
    assert st["op_visits"] == visits
    if not all_reads:
        return res
    assert st["n_cigar_words"] == len(rd.cigar)
    assert st["n_cigar_words_joined"] == joined_words(rd, case, unphased)
    epos, eval_, eoff = walk_events(rd, minlen)
    assert st["n_events"] == len(epos)
    pos, val, off = ctx.debug_events()
    assert np.array_equal(off, eoff) and np.array_equal(pos, epos) and np.array_equal(val, eval_), minlen
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("unphased", [False, True])
def test_every_op_and_length_every_minlen(ctx, unphased):
    case = long_case(1)
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    ctx.push(case["reads"])
    for minlen in MINLENS:
        check(ctx, case, minlen, unphased)


@pytest.mark.gpu
def test_chunked_and_routed_pushes_and_reserve(ctx):
    case = long_case(2)
    rd = case["reads"]
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    expect = None
    for mode in ("chunked", "routed", "reserved"):
        ctx.clear_reads()
        if mode == "chunked":
            push_chunked(ctx, rd, 7)
        elif mode == "routed":
            assert 0 < ctx.push_routed(rd) <= rd.n        # keeps the reads that can reach a locus
        else:
            ctx.reserve_reads(rd.n, len(rd.cigar) // 4)   # far fewer units than the long ops expand to
            push_chunked(ctx, rd, 3)
        res = check(ctx, case, 5, False, all_reads=mode != "routed")
        if expect is None:
            expect = res
        assert same(res.phase1, expect.phase1) and same(res.phase2, expect.phase2)


@pytest.mark.gpu
def test_clear_reads_cycles(ctx):
    a, b = long_case(3, n_lens=(4095, 65535)), long_case(4)
    ctx.set_loci(a["contig_off"], a["locus_start"], a["locus_end"])
    for case in (a, b, a):
        ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
        ctx.clear_reads()
        ctx.push(case["reads"])
        check(ctx, case, 4095, False)
        check(ctx, case, 0, True)


@pytest.mark.gpu
def test_long_ops_straddle_push_chunks(ctx):
    # the filler read moves the special reads to the end of the first encoding chunk and into the second
    chunk = stage_words()
    case = long_case(5, filler_words=chunk - 60_000, n_reads=200)
    w = case["reads"].cigar
    op, ln = w & 15, w >> 4
    long_at = np.flatnonzero((ln >= 4095) & ((op <= 4) | (op == 7) | (op == 8)))      # words that expand or become heads
    assert long_at.min() < chunk <= long_at.max(), (long_at.min(), long_at.max(), chunk)
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    ctx.push(case["reads"])
    for minlen in (5, 4095):
        check(ctx, case, minlen, False)
