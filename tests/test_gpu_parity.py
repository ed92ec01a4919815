"""GPU parity: libinqcall.so (through the C ABI) against the CPU oracle on the same seeded inputs.
Integer/bit-exact: identical medians (as f64 bit patterns incl. NaN) for every locus."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.datagen import expected_events, make_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import inquistr_b200 as q
    c = q.Context(0)
    yield c
    c.close()


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def run_case(ctx, case, minlen, support, unphased, chunks=1):
    rd = case["reads"]
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    if chunks == 1:
        ctx.push(rd)
    else:
        cuts = np.linspace(0, rd.n, chunks + 1).astype(int)
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b <= a:
                continue
            base = rd.cigar_off[a]
            ctx.push_reads(rd.contig[a:b], rd.ref_start[a:b], rd.ref_end[a:b], rd.mapq[a:b], rd.hp[a:b],
                           rd.flags[a:b], rd.cigar_off[a:b + 1] - base,
                           rd.cigar[int(base):int(rd.cigar_off[b])])
    res = ctx.genotype(minlen, support, unphased)
    rc, p1, p2, visits = O.genotype_loci(rd, case["n_contigs"], case["locus_contig"], case["locus_start"],
                                         case["locus_end"], minlen, support, unphased, threads=4)
    assert rc == 0
    bad = np.flatnonzero(~((res.phase1 == p1) | (np.isnan(res.phase1) & np.isnan(p1))) |
                         ~((res.phase2 == p2) | (np.isnan(res.phase2) & np.isnan(p2))))
    assert len(bad) == 0, (bad[:10], res.phase1[bad[:10]], p1[bad[:10]], res.phase2[bad[:10]], p2[bad[:10]])
    assert res.stats["op_visits"] == visits
    return res


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("unphased", [False, True])
def test_random_small(ctx, seed, unphased):
    case = make_case(seed)
    run_case(ctx, case, 5, 3, unphased)


@pytest.mark.parametrize("minlen,support", [(0, 1), (1, 2), (5, 1), (12, 5), (3, 40), (10**9, 3)])
def test_parameters(ctx, minlen, support):
    case = make_case(100 + minlen % 97 + support, n_reads=1500)
    run_case(ctx, case, minlen, support, False)
    run_case(ctx, case, minlen, support, True)


def test_unsorted_reads_and_chunked_push(ctx):
    case = make_case(11, sort_reads=False, n_reads=2000)
    a = run_case(ctx, case, 5, 3, False, chunks=1)
    b = run_case(ctx, case, 5, 3, False, chunks=7)
    assert same(a.phase1, b.phase1) and same(a.phase2, b.phase2)


def test_events_match_cigar_walk(ctx):
    case = make_case(21, n_reads=1200)
    for minlen in (5, 0):
        run_case(ctx, case, minlen, 3, False)
        pos, val, off = ctx.debug_events()
        epos, eval_, eoff = expected_events(case["reads"], minlen)
        assert np.array_equal(off, eoff)
        assert np.array_equal(pos, epos)
        assert np.array_equal(val, eval_)


def test_deep_loci_take_the_cta_path(ctx):
    # > 128 calls per locus: CTA sort in shared memory; > 4096: in-place global sort
    case = make_case(31, n_contigs=1, n_loci=6, n_reads=9000, dense_locus=True, max_read=3000)
    run_case(ctx, case, 5, 3, False)
    run_case(ctx, case, 5, 3, True)
    run_case(ctx, case, 0, 2000, True)


def test_cta_path_guess_is_verified(ctx):
    """The CTA-path median kernel is only launched for catalog chunks that had deep loci in the last completed pass over
    the same reads; when other parameters make a locus deep (unphased counts the untagged and HP-0 reads too) the
    pass is repeated with the kernel. Same reads, alternating parameters, direct / captured / replayed."""
    case = make_case(77, n_contigs=1, n_loci=6, n_reads=330, dense_locus=True, max_read=3000,
                     hp_probs=(0.45, 0.05, 0.25, 0.25))
    rd = case["reads"]
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    ctx.push(rd)
    expect = {}
    for unphased in (False, True):
        rc, p1, p2, _ = O.genotype_loci(rd, case["n_contigs"], case["locus_contig"], case["locus_start"], case["locus_end"],
                                        5, 3, unphased, threads=2)
        assert rc == 0
        expect[unphased] = (p1, p2)
    # the case must straddle the 128-call limit of the warp path: per-locus pair counts of both modes
    per = {u: max(int(((rd.ref_start < e + 10) & (rd.ref_end > s - 10) & (rd.mapq > 10) & (u | (rd.hp <= 2))).sum())
                  for s, e in zip(case["locus_start"], case["locus_end"])) for u in (False, True)}
    assert per[True] > 128, per
    for unphased in (False, False, False, True, True, True, False, True, False):
        res = ctx.genotype(5, 3, unphased)
        assert same(res.phase1, expect[unphased][0]) and same(res.phase2, expect[unphased][1]), unphased


def test_long_reads_span_many_tiles(ctx):
    # reads with > 4096 CIGAR words cross tile boundaries of the scan kernel
    case = make_case(41, n_contigs=1, contig_len=3_000_000, n_loci=400, n_reads=300, max_read=900_000,
                     degenerate=True)
    res = run_case(ctx, case, 5, 3, False)
    assert res.stats["n_tiles"] > 50
    pos, val, off = ctx.debug_events()
    epos, eval_, eoff = expected_events(case["reads"], 5)
    assert np.array_equal(off, eoff) and np.array_equal(pos, epos) and np.array_equal(val, eval_)


def test_tiny_reads_many_starts_per_warp_tile(ctx):
    # reads of 1-40 CIGAR words: a 1024-word warp tile holds far more than 32 read starts, and with
    # minlen 0 most tiles hold several rounds of 32 events (the scan kernel's position-query pass loops)
    case = make_case(51, n_contigs=2, contig_len=40_000, n_loci=300, n_reads=12_000, max_read=400)
    assert case["reads"].n / (len(case["reads"].cigar) / 1024) > 40
    for minlen in (0, 5):
        run_case(ctx, case, minlen, 2, False)
        pos, val, off = ctx.debug_events()
        epos, eval_, eoff = expected_events(case["reads"], minlen)
        assert np.array_equal(off, eoff) and np.array_equal(pos, epos) and np.array_equal(val, eval_)
    run_case(ctx, case, 0, 2, True, chunks=5)


def test_event_dense_long_reads(ctx):
    # every second word is an event (minlen 0) in reads of tens of thousands of words: the pair kernel's
    # shared-memory event pool overflows and its warp-tile table does not fit -> global search paths
    case = make_case(61, n_contigs=1, contig_len=2_000_000, n_loci=600, n_reads=120, max_read=600_000)
    res = run_case(ctx, case, 0, 1, False)
    assert res.stats["n_events"] > 600 * 120
    run_case(ctx, case, 0, 1, True)


def test_empty_inputs(ctx):
    case = make_case(51, n_reads=50)
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    res = ctx.genotype(5, 3, False)
    assert np.all(res.valid == 0)
    ctx.set_loci(np.zeros(case["n_contigs"] + 1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.int32))
    ctx.push(case["reads"])
    res = ctx.genotype(5, 3, False)
    assert len(res.valid) == 0


def test_error_codes(ctx):
    import inquistr_b200 as q
    case = make_case(61, hp_values=(0xFF, 1, 2, 3), hp_probs=(0.1, 0.4, 0.4, 0.1))
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    ctx.push(case["reads"])
    with pytest.raises(q.InqError) as ei:
        ctx.genotype(5, 3, False)
    assert ei.value.code == -10                       # HP 3 on a read that passes the filter
    rc, *_ = O.genotype_loci(case["reads"], case["n_contigs"], case["locus_contig"], case["locus_start"],
                             case["locus_end"], 5, 3, False)
    assert rc == O.ORC_PANIC_BAD_HP
    ctx.genotype(5, 3, True)                          # unphased ignores HP (call.rs:297-300)
    with pytest.raises(q.InqError) as ei:
        ctx.genotype(5, 0, False)                     # support 0 -> some empty bucket -> panic in the reference
    assert ei.value.code in (-10, -11)
    with pytest.raises(q.InqError) as ei:
        ctx.set_loci([0, 1], [5], [50])
    assert ei.value.code == -12
    with pytest.raises(q.InqError) as ei:
        ctx.set_loci([0, 2], [500, 400], [550, 450])
    assert ei.value.code == -13
    with pytest.raises(q.InqError) as ei:
        ctx.set_loci([0, 1], [500], [450])
    assert ei.value.code == -13


@pytest.mark.parametrize("name", ["random_edge_cases", "expansion_panel"])
def test_golden_fixtures(ctx, name):
    """committed golden vectors (tests/golden/make_golden.py) through the C ABI"""
    from tests.test_cpu_suite import load_golden, parse_run
    z, rd, runs = load_golden(name)
    ctx.set_loci(z["contig_off"], z["locus_start"], z["locus_end"])
    ctx.clear_reads()
    ctx.push(rd)
    for key in runs:
        minlen, support, unphased = parse_run(key)
        res = ctx.genotype(minlen, support, unphased)
        assert same(res.phase1, z[key + "_p1"]) and same(res.phase2, z[key + "_p2"]), key
        assert res.stats["op_visits"] == int(z[key + "_visits"])


@pytest.mark.parametrize("cfg,scale", [(1, 1.0), (2, 0.02), (3, 0.004), (4, 1.0), (5, 0.002)])
def test_baseline_configs_small(ctx, cfg, scale):
    """every BASELINE.json configuration (shrunk) against the oracle, incl. the unphased run of each"""
    from synth.synth import make_workload
    w = make_workload(cfg, scale=scale, threads=4)
    ctx.set_loci(w.contig_locus_off, w.locus_start, w.locus_end)
    ctx.clear_reads()
    ctx.push(w.reads)
    for unphased in (w.unphased, not w.unphased):
        res = ctx.genotype(w.minlen, w.support, unphased)
        rc, p1, p2, visits = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig, w.locus_start.astype(np.uint32),
                                             w.locus_end.astype(np.uint32), w.minlen, w.support, unphased, threads=8)
        assert rc == 0 and same(res.phase1, p1) and same(res.phase2, p2)
        assert res.stats["op_visits"] == visits


def test_size_independent_properties(ctx):
    """properties that hold at any size: idempotence, permutation invariance of the read order,
    monotonicity in support (a valid median never appears when support grows)"""
    from synth.synth import make_workload
    from inquistr_b200 import shard as S
    w = make_workload(3, scale=0.01, threads=4)
    ctx.set_loci(w.contig_locus_off, w.locus_start, w.locus_end)
    ctx.clear_reads(); ctx.push(w.reads)
    a = ctx.genotype(5, 3, False)
    b = ctx.genotype(5, 3, False)
    assert same(a.phase1, b.phase1) and same(a.phase2, b.phase2)
    perm = np.random.default_rng(0).permutation(w.reads.n)
    mask = np.zeros(w.reads.n, bool); mask[:] = True
    sub = S.take_reads(w.reads, mask)
    rd = O.Reads(**sub)
    n_cig = (rd.cigar_off[1:] - rd.cigar_off[:-1]).astype(np.int64)
    off = np.zeros(rd.n + 1, np.uint64); off[1:] = np.cumsum(n_cig[perm])
    cig = np.concatenate([rd.cigar[int(rd.cigar_off[i]):int(rd.cigar_off[i + 1])] for i in perm])
    ctx.clear_reads()
    ctx.push_reads(rd.contig[perm], rd.ref_start[perm], rd.ref_end[perm], rd.mapq[perm], rd.hp[perm], rd.flags[perm], off, cig)
    c = ctx.genotype(5, 3, False)
    assert same(a.phase1, c.phase1) and same(a.phase2, c.phase2)
    d = ctx.genotype(5, 6, False)
    assert np.all((d.valid & ~a.valid) == 0)


# ------------------------------------------------------------------ range pipeline + CUDA graph
def _pinned_out(n):
    import inquistr_b200 as q
    return (q.pinned_empty(n, np.int64), q.pinned_empty(n, np.int64), q.pinned_empty(n, np.uint8))


@pytest.mark.parametrize("sort_reads", [True, False])
@pytest.mark.parametrize("ranges", [2, 3, 7, 16])
def test_range_pipeline_and_graph_replay(sort_reads, ranges):
    """the pass cut into `ranges` ranges of warp tiles (pair / median work of range k under the scan of
    range k+1), launched directly, captured, and replayed from the CUDA graph: same bits every time"""
    import inquistr_b200 as q
    case = make_case(70 + ranges, n_contigs=3, contig_len=200_000, n_loci=700, n_reads=5000, sort_reads=sort_reads)
    rd = case["reads"]
    assert len(rd.cigar) // 1024 >= 3 * ranges
    rc, p1, p2, visits = O.genotype_loci(rd, case["n_contigs"], case["locus_contig"], case["locus_start"],
                                         case["locus_end"], 5, 3, False, threads=4)
    assert rc == 0
    with q.Context(0) as c:
        c.set_option("ranges", ranges)
        c.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
        c.push(rd)
        out = _pinned_out(len(case["locus_start"]))
        graphs = 0
        for it in range(4):
            out[0][:] = -1; out[1][:] = -1; out[2][:] = 0xFF
            res = c.genotype(5, 3, False, out=out)
            assert same(res.phase1, p1) and same(res.phase2, p2), (it, res.stats)
            assert res.stats["op_visits"] == visits
            assert res.stats["n_ranges"] == ranges
            assert res.stats["reads_sorted"] == int(sort_reads)
            graphs += res.stats["used_graph"]
        assert graphs == 3                                  # first call direct, then capture + replay
        # other parameters: new key -> direct again, still right; unphased too
        rc, u1, u2, _ = O.genotype_loci(rd, case["n_contigs"], case["locus_contig"], case["locus_start"],
                                        case["locus_end"], 0, 2, True, threads=4)
        for it in range(3):
            res = c.genotype(0, 2, True, out=out)          # minlen 0: the event buffer regrows on the first of these
            assert same(res.phase1, u1) and same(res.phase2, u2)
        assert res.stats["used_graph"] == 1
        # pageable outputs: staged through the library's pinned buffer, no graph requirement on the caller
        res = c.genotype(5, 3, False)
        assert same(res.phase1, p1) and same(res.phase2, p2)
        # graph off
        c.set_option("graph", 0)
        for it in range(2):
            res = c.genotype(5, 3, False, out=out)
            assert res.stats["used_graph"] == 0 and same(res.phase1, p1) and same(res.phase2, p2)
        for a in out:
            q.free_pinned(a)


def test_sorted_reads_finish_loci_early():
    """coordinate-sorted reads: catalog chunks are reduced as soon as no later read can reach them"""
    import inquistr_b200 as q
    from synth.synth import make_workload
    w = make_workload(3, scale=0.02, threads=4, pack_filter=True)
    with q.Context(0) as c:
        c.set_option("ranges", 4)
        c.set_loci(w.contig_locus_off, w.locus_start, w.locus_end)
        c.push(w.reads)
        res = c.genotype(w.minlen, w.support, w.unphased)
        assert res.stats["reads_sorted"] == 1 and res.stats["n_median_chunks"] >= 4
        rc, p1, p2, visits = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig, w.locus_start.astype(np.uint32),
                                             w.locus_end.astype(np.uint32), w.minlen, w.support, w.unphased, threads=8)
        assert rc == 0 and same(res.phase1, p1) and same(res.phase2, p2) and res.stats["op_visits"] == visits


def test_reserve_after_push_keeps_padding_and_tile_table(ctx):
    """inq_reserve_reads between the last push and inq_genotype must not lose the zero padding of the
    CIGAR stream nor the tile_first entries of the last partial tiles"""
    case = make_case(81, n_reads=700)
    rd = case["reads"]
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    ctx.push(rd)
    a = ctx.genotype(5, 3, False)
    ctx.clear_reads()
    ctx.push(rd)
    ctx.reserve_reads(rd.n * 40, len(rd.cigar) * 40)        # grows every read buffer
    b = ctx.genotype(5, 3, False)
    assert same(a.phase1, b.phase1) and same(a.phase2, b.phase2)
    rc, p1, p2, _ = O.genotype_loci(rd, case["n_contigs"], case["locus_contig"], case["locus_start"], case["locus_end"], 5, 3, False)
    assert rc == 0 and same(b.phase1, p1) and same(b.phase2, p2)


@pytest.mark.parametrize("world", [2, 3, 5])
@pytest.mark.parametrize("cfg,scale", [(3, 0.01), (4, 1.0)])
def test_sharded_gpu_output_equals_unsharded_oracle(ctx, world, cfg, scale):
    """SURVEY 8e: contiguous catalog ranges, each shard's reads through the GPU, ordered concatenation
    == the oracle on the whole input"""
    from inquistr_b200 import shard as S
    from synth.synth import make_workload
    w = make_workload(cfg, scale=scale, threads=4)
    rc, p1, p2, visits = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig, w.locus_start.astype(np.uint32),
                                         w.locus_end.astype(np.uint32), w.minlen, w.support, w.unphased, threads=8)
    assert rc == 0
    g1, g2, tot_visits = [], [], 0
    for lo, hi in S.split_catalog(w.n_loci, world):
        s_off, s_start, s_end = S.shard_catalog(w.contig_locus_off, w.locus_start, w.locus_end, lo, hi)
        sub = S.take_reads(w.reads, S.reads_for_shard(w.reads.contig, w.reads.ref_start, w.reads.ref_end, s_off, s_start, s_end))
        ctx.set_loci(s_off, s_start, s_end)
        ctx.clear_reads()
        ctx.push_reads(**sub)
        res = ctx.genotype(w.minlen, w.support, w.unphased)
        g1.append(res.phase1); g2.append(res.phase2); tot_visits += res.stats["op_visits"]
    assert same(S.concat_ordered(g1), p1) and same(S.concat_ordered(g2), p2)
    assert tot_visits == visits


def test_sa_panic_flag_only_fires_when_the_read_pairs(ctx):
    """flags bit1 (INQ_FLAG_SA_PANIC): INQ_ERR_BAD_SA iff the oracle's walk would hit is_accidental_2d's panic"""
    import inquistr_b200 as q
    case = make_case(91, n_reads=600)
    rd = case["reads"]
    args = (case["n_contigs"], case["locus_contig"], case["locus_start"], case["locus_end"], 5, 3)
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    # flag only reads that can never pair in phased mode (mapq <= 10 or no HP): no error, same result
    quiet = (rd.mapq <= 10) | (rd.hp == 0xFF)
    assert quiet.sum() > 20
    fl = rd.flags.copy(); fl[quiet] |= 2
    rd2 = O.Reads(rd.contig, rd.ref_start, rd.ref_end, rd.mapq, rd.hp, fl, rd.cigar_off, rd.cigar)
    ctx.clear_reads(); ctx.push(rd2)
    res = ctx.genotype(5, 3, False)
    rc, p1, p2, _ = O.genotype_loci(rd2, *args, False)
    assert rc == 0 and same(res.phase1, p1) and same(res.phase2, p2)
    # unphased: the untagged ones now pair -> both sides report the SA panic
    rc, *_ = O.genotype_loci(rd2, *args, True)
    assert rc == O.ORC_PANIC_BAD_SA
    with pytest.raises(q.InqError) as ei:
        ctx.genotype(5, 3, True)
    assert ei.value.code == -17
    # flag one read that pairs in phased mode
    rc0, p1, p2, _ = O.genotype_loci(rd, *args, False)
    fl = rd.flags.copy()
    cand = np.flatnonzero((rd.mapq > 10) & (rd.hp != 0xFF) & (rd.hp <= 2))
    for r in cand[:50]:
        fl[:] = rd.flags; fl[r] |= 2
        rd3 = O.Reads(rd.contig, rd.ref_start, rd.ref_end, rd.mapq, rd.hp, fl, rd.cigar_off, rd.cigar)
        rc, *_ = O.genotype_loci(rd3, *args, False)
        ctx.clear_reads(); ctx.push(rd3)
        if rc == O.ORC_PANIC_BAD_SA:
            with pytest.raises(q.InqError) as ei:
                ctx.genotype(5, 3, False)
            assert ei.value.code == -17
        else:
            assert rc == 0
            res = ctx.genotype(5, 3, False)
            assert same(res.phase1, p1) and same(res.phase2, p2)


@pytest.mark.parametrize("sort_reads", [True, False])
def test_routed_push_over_catalog_shards(sort_reads):
    """inq_push_reads_routed: three contexts holding three contiguous catalog shards are each handed the WHOLE read
    set (in two batches) and keep what can reach them; concatenated output == oracle on the unsharded input.
    Sorted input takes the run path, shuffled input the gather path; the filter flags change nothing."""
    import inquistr_b200 as q
    from inquistr_b200 import shard as S
    case = make_case(95, n_contigs=3, contig_len=300_000, n_loci=400, n_reads=4000, sort_reads=sort_reads, max_read=6000)
    rd = case["reads"]
    n_loci = len(case["locus_start"])
    rc, p1, p2, visits = O.genotype_loci(rd, case["n_contigs"], case["locus_contig"], case["locus_start"], case["locus_end"], 5, 3, False, threads=4)
    assert rc == 0
    half = rd.n // 2
    parts = []
    for a, b in ((0, half), (half, rd.n)):
        base = rd.cigar_off[a]
        parts.append(O.Reads(rd.contig[a:b], rd.ref_start[a:b], rd.ref_end[a:b], rd.mapq[a:b], rd.hp[a:b], rd.flags[a:b],
                             rd.cigar_off[a:b + 1] - base, rd.cigar[int(base):int(rd.cigar_off[b])]))
    for drop in (False, True):
        g1, g2, tot_visits, tot_taken = [], [], 0, 0
        for lo, hi in S.split_catalog(n_loci, 3):
            s_off, s_start, s_end = S.shard_catalog(case["contig_off"], case["locus_start"], case["locus_end"], lo, hi)
            with q.Context(0) as c:
                c.set_loci(s_off, s_start, s_end)
                for p in parts:
                    tot_taken += c.push_routed(p, drop_low_mapq=drop, drop_no_hp=drop, host_threads=3)
                res = c.genotype(5, 3, False)
                g1.append(res.phase1); g2.append(res.phase2); tot_visits += res.stats["op_visits"]
        assert same(np.concatenate(g1), p1) and same(np.concatenate(g2), p2)
        assert tot_visits == visits
        assert tot_taken < 3 * rd.n                      # nobody takes everything


def test_bench_dump_outputs_are_the_timed_results(tmp_path):
    """bench.py --dump-outputs: the medians of the last timed step, as the caller of Context.genotype gets them,
    equal the oracle's on the same seeded workload; --steps is the number of timed steps"""
    import json
    import os
    import subprocess
    import sys
    from synth.synth import make_workload
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--scale", "0.002", "--steps", "2", "--warmup", "0",
                        "--no-cpu-baseline", "--no-e2e", "--no-cohort", "--bam-scale", "0", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    w = make_workload(3, scale=0.002, threads=2, pack_filter=True)
    rc, p1, p2, _ = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig, w.locus_start.astype(np.uint32),
                                    w.locus_end.astype(np.uint32), w.minlen, w.support, w.unphased, threads=4)
    assert rc == 0
    assert sorted(os.listdir(tmp_path)) == ["phase1.npy", "phase2.npy", "valid_mask.npy"]
    d1, d2, vm = (np.load(tmp_path / f) for f in ("phase1.npy", "phase2.npy", "valid_mask.npy"))
    assert d1.dtype == d2.dtype == vm.dtype == np.float64
    assert all(np.isfinite(a).all() for a in (d1, d2, vm))
    assert np.isnan(p1).any() and np.isnan(p2).any()              # the workload has loci without a call
    assert same(np.where(vm % 2 == 1, d1, np.nan), p1) and same(np.where(vm >= 2, d2, np.nan), p2)
