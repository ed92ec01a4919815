"""Call-key width: the pass runs on 32-bit call keys while every call of the reads fits [-2^29, 2^29) and repeats
itself with 64-bit keys when one does not. Either way the medians equal the CPU oracle bit for bit."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.datagen import OPS, make_case

pytestmark = pytest.mark.gpu

MAX_OP = (1 << 28) - 1                       # longest BAM op


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def with_long_insertions(case, lens, n_reads=6, locus=None):
    """the case's reads plus n_reads reads spanning one locus of contig 0, each with insertions of `lens` at one
    position inside the locus window: their calls are sum(lens). HP alternates 1 / 2."""
    ls, le = case["locus_start"], case["locus_end"]
    k = int(np.flatnonzero(case["locus_contig"] == 0)[0]) if locus is None else locus
    rd = case["reads"]
    contig, rs, re_, mq, hp, fl = (list(a) for a in (rd.contig, rd.ref_start, rd.ref_end, rd.mapq, rd.hp, rd.flags))
    words = [rd.cigar[int(rd.cigar_off[i]):int(rd.cigar_off[i + 1])] for i in range(rd.n)]
    for i in range(n_reads):
        start = max(0, int(ls[k]) - 400 - 7 * i)
        left = int(ls[k]) + 1 - start                    # anchor inside (ls - 10, le + 10)
        right = int(le[k]) - int(ls[k]) + 300
        w = np.asarray([(left << 4) | OPS["M"]] + [(int(n) << 4) | OPS["I"] for n in lens] + [(right << 4) | OPS["M"]],
                       np.uint32)
        contig.append(0); rs.append(start); re_.append(start + left + right)
        mq.append(60); hp.append(1 + i % 2); fl.append(0)
        words.append(w)
    off = np.concatenate([[0], np.cumsum([len(w) for w in words])]).astype(np.uint64)
    out = dict(case)
    out["reads"] = O.Reads(np.asarray(contig), np.asarray(rs), np.asarray(re_), np.asarray(mq), np.asarray(hp),
                           np.asarray(fl), off, np.concatenate(words))
    return out


def expect(case, minlen, support, unphased):
    rc, p1, p2, visits = O.genotype_loci(case["reads"], case["n_contigs"], case["locus_contig"], case["locus_start"],
                                         case["locus_end"], minlen, support, unphased, threads=4)
    assert rc == 0
    return p1, p2, visits


def check(res, want):
    p1, p2, visits = want
    assert same(res.phase1, p1) and same(res.phase2, p2)
    assert res.stats["op_visits"] == visits


@pytest.fixture(scope="module")
def ctx():
    import inquistr_b200 as q
    c = q.Context(0)
    yield c
    c.close()


def load(ctx, case):
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    ctx.push(case["reads"])


def test_wide_calls_repeat_the_pass_with_64bit_keys(ctx):
    case = with_long_insertions(make_case(301, n_reads=1200), [MAX_OP, MAX_OP, MAX_OP])
    load(ctx, case)
    res = ctx.genotype(5, 3, False)
    check(res, expect(case, 5, 3, False))
    assert res.stats["n_passes"] >= 2 and res.stats["key_bytes"] == 8
    # the switch holds for these reads: the next call goes straight to 64-bit keys, and so do other parameters
    res = ctx.genotype(5, 3, False)
    check(res, expect(case, 5, 3, False))
    assert res.stats["n_passes"] == 1 and res.stats["key_bytes"] == 8
    res = ctx.genotype(5, 3, True)
    check(res, expect(case, 5, 3, True))
    assert res.stats["key_bytes"] == 8
    # new reads start over with 32-bit keys
    plain = make_case(302, n_reads=1200)
    load(ctx, plain)
    res = ctx.genotype(5, 3, False)
    check(res, expect(plain, 5, 3, False))
    assert res.stats["key_bytes"] == 4


def test_widest_32bit_call_stays_32bit(ctx):
    # 2^29 - 1 is the largest call of the 32-bit layout; 2^29 is the smallest that is not
    for lens, key_bytes in (([MAX_OP, MAX_OP - 9, 10], 4), ([MAX_OP, MAX_OP - 8, 10], 8)):
        assert sum(lens) == (1 << 29) - (key_bytes == 4)
        case = with_long_insertions(make_case(303, n_reads=600), lens)
        load(ctx, case)
        for unphased in (False, True):
            res = ctx.genotype(5, 1, unphased)
            check(res, expect(case, 5, 1, unphased))
            assert res.stats["key_bytes"] == key_bytes, (lens, unphased)


@pytest.mark.parametrize("wide", [False, True])
def test_cta_path_both_widths(ctx, wide):
    # > 128 calls per locus (CTA sort in shared memory), > 4096 (in place in the call buffer), phased and unphased
    case = make_case(31, n_contigs=1, n_loci=6, n_reads=9000, dense_locus=True, max_read=3000)
    if wide:
        case = with_long_insertions(case, [MAX_OP, MAX_OP, MAX_OP], n_reads=8, locus=2)
    load(ctx, case)
    for minlen, support, unphased in ((5, 3, False), (5, 3, True), (0, 2000, True)):
        res = ctx.genotype(minlen, support, unphased)
        check(res, expect(case, minlen, support, unphased))
        assert res.stats["key_bytes"] == (8 if wide else 4)


def test_graph_replay_after_fallback():
    import inquistr_b200 as q
    case = with_long_insertions(make_case(304, n_contigs=3, contig_len=200_000, n_loci=700, n_reads=5000),
                                [MAX_OP, MAX_OP, MAX_OP])
    want = expect(case, 5, 3, False)
    with q.Context(0) as c:
        load(c, case)
        n = len(case["locus_start"])
        out = (q.pinned_empty(n, np.int64), q.pinned_empty(n, np.int64), q.pinned_empty(n, np.uint8))
        try:
            graphs = 0
            for it in range(4):
                out[0][:] = -1; out[1][:] = -1; out[2][:] = 0xFF
                res = c.genotype(5, 3, False, out=out)
                check(res, want)
                assert res.stats["key_bytes"] == 8
                assert res.stats["n_passes"] >= 2 if it == 0 else res.stats["n_passes"] == 1
                graphs += res.stats["used_graph"]
            assert graphs == 3                              # the first call direct, then capture + replay
            # back to 32-bit keys with new reads: the graph of the 64-bit pass is not replayed
            plain = make_case(305, n_contigs=3, contig_len=200_000, n_loci=700, n_reads=5000)
            c.set_loci(plain["contig_off"], plain["locus_start"], plain["locus_end"])
            c.clear_reads()
            c.push(plain["reads"])
            want = expect(plain, 5, 3, False)
            for it in range(3):
                res = c.genotype(5, 3, False, out=out)
                check(res, want)
                assert res.stats["key_bytes"] == 4 and res.stats["used_graph"] == (0 if it == 0 else 1)
        finally:
            for a in out:
                q.free_pinned(a)
