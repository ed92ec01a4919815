"""`inquistr-b200 call-cohort`: several BAMs against one catalog in one process. Its stdout must be the bytes of
`combine <(call BAM1) ... <(call BAMn)` with the same options; errors exit as that pipeline would fail, with
nothing on stdout. CLI behaviour without a GPU, byte parity with `call` + `combine` and the oracle with one."""
import json
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from tests import bamio
from tests.test_cli import expected_tsv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def cli():
    from inquistr_b200 import build
    build.build_libinqcall()
    return build.build_cli()


def run(cli, *args, env=None):
    return subprocess.run([cli, *args], capture_output=True, timeout=600, env={**os.environ, **(env or {})})


M, I = 0, 1
SPAN = np.asarray([(500 << 4) | M, (8 << 4) | I, (500 << 4) | M], np.uint32)


def tiny_bam(path, names, lens, n=6, hp=None, tid=0, pos=1000):
    recs = [bamio.encode_record(tid, pos, 60, 0, SPAN, name=b"r%d" % i, hp=(1 + i % 2) if hp is None else hp, end=pos + 1000)
            for i in range(n)]
    bamio.write_bam(path, names, lens, recs)
    return path


@pytest.fixture
def two_bams(tmp_path):
    a = tiny_bam(str(tmp_path / "a.bam"), ["chr1", "chr2"], [1_000_000, 500_000])
    b = tiny_bam(str(tmp_path / "b.bam"), ["chr1", "chr2"], [1_000_000, 500_000])
    return a, b


# ------------------------------------------------------------------------------------------- CPU
def test_usage_and_help(cli, two_bams):
    r = run(cli, "call-cohort")
    assert r.returncode == 2 and b"Usage: inquistr-b200 call-cohort" in r.stderr
    r = run(cli, "call-cohort", "--help")
    assert r.returncode == 0 and b"--region-file <REGION_FILE>" in r.stdout and b"17 bytes per locus and sample" in r.stdout
    a, b = two_bams
    for bad in (["--sample-name", "x"], ["--bogus"], ["--reference", "x.fa"], ["-x"]):
        r = run(cli, "call-cohort", "-r", "chr1:1490-1510", *bad, a, b)
        assert r.returncode == 2 and r.stdout == b"", bad
    r = run(cli, "call-cohort", "-r", "chr1:1490-1510")
    assert r.returncode == 2 and b"<BAM>..." in r.stderr
    r = run(cli, "help")
    assert r.returncode == 0 and b"call-cohort" in r.stdout
    r = run(cli, "nope")
    assert r.returncode == 2 and b"`call-cohort`" in r.stderr


def test_bad_inputs_exit_1_naming_the_bam(cli, two_bams, tmp_path):
    a, b = two_bams
    cram = tmp_path / "s3.cram"
    cram.write_bytes(b"CRAM")
    for bad, msg in ((str(tmp_path / "missing.bam"), b"is not valid"), (str(cram), b"CRAM input"),
                     ("https://example.org/x.bam", b"not supported")):
        r = run(cli, "call-cohort", "-r", "chr1:1490-1510", a, bad, b)
        assert r.returncode == 1 and msg in r.stderr and bad.encode() in r.stderr and r.stdout == b"", r.stderr
    r = run(cli, "call-cohort", a, b)
    assert r.returncode == 1 and b"Specify a region string (-r) or a region_file (-R)!" in r.stderr


def test_catalog_checked_against_every_header(cli, tmp_path):
    """a locus that only the second BAM's header cannot hold, or a contig it lacks: `call` on that BAM panics"""
    a = tiny_bam(str(tmp_path / "a.bam"), ["chr1", "chr2"], [1_000_000, 500_000])
    short = tiny_bam(str(tmp_path / "short.bam"), ["chr1", "chr2"], [1_000_000, 300_000])
    lacks = tiny_bam(str(tmp_path / "lacks.bam"), ["chr1"], [1_000_000])
    bed = tmp_path / "loci.bed"
    bed.write_text("chr1\t1490\t1510\nchr2\t400000\t400100\n")
    for second in (short, lacks):
        r = run(cli, "call-cohort", "-R", str(bed), a, second, a)
        assert r.returncode == 101 and r.stdout == b""
        assert b"Chromosome chr2 is not in the fasta file or the end coordinate is out of bounds" in r.stderr
        r = run(cli, "call", "-R", str(bed), second)             # the same message from `call`
        assert r.returncode == 101 and b"Chromosome chr2 is not in the fasta file" in r.stderr
    r = run(cli, "call-cohort", "-r", "chr1:5-100", a, a)
    assert r.returncode == 101 and r.stdout == b""


def test_fails_loudly_without_gpu(cli, two_bams):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    a, b = two_bams
    r = run(cli, "call-cohort", "-r", "chr1:1490-1510", a, b)
    assert r.returncode == 1 and b"no CPU fallback" in r.stderr and r.stdout == b""


# ------------------------------------------------------------------------------------------- GPU
def write_cohort(tmp_path, cfg, scale, seeds, index=True):
    """one catalog (config cfg, seed of the first sample), reads of each sample from its own seed"""
    from synth import synth as S
    bams, ws = [], []
    for k in seeds:
        w = S.make_workload(cfg, scale=scale, seed=seeds[0], read_seed=k, threads=4)
        bam = str(tmp_path / f"s{k}.bam")
        S.write_bam(w, bam)
        if index:
            bamio.index_bam(bam)
        bams.append(bam)
        ws.append(w)
    rows = S.write_bed(ws[0], str(tmp_path / "loci.bed"), shuffle_seed=11)
    return bams, ws, rows, str(tmp_path / "loci.bed")


def call_then_combine(cli, tmp_path, bams, opts, env=None):
    outs = []
    for k, bam in enumerate(bams):
        r = run(cli, "call", *opts, bam, env=env)
        assert r.returncode == 0, r.stderr
        p = tmp_path / f"call_{k}.tsv"
        p.write_bytes(r.stdout)
        outs.append(str(p))
    r = run(cli, "combine", *outs)
    assert r.returncode == 0, r.stderr
    return r.stdout


def oracle_table(bams, ws, rows, unphased, threads):
    sel = np.asarray([i for *_, i in rows])
    loci = [(c, s, e) for c, s, e, _ in rows]
    cols = None
    for bam, w in zip(bams, ws):
        rc, p1, p2, _ = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig[sel], w.locus_start[sel].astype(np.uint32),
                                        w.locus_end[sel].astype(np.uint32), 5, 3, unphased)
        assert rc == 0
        lines = expected_tsv(os.path.basename(bam)[:-4], None, loci, p1, p2, threads).decode().splitlines()
        cols = [ln.split("\t") for ln in lines] if cols is None else [c + ln.split("\t")[3:] for c, ln in zip(cols, lines)]
    return ("\n".join("\t".join(c) for c in cols) + "\n").encode()


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,scale,n,modes", [
    (4, 1.0, 8, [(1, False, "1"), (4, True, "0")]),
    (4, 1.0, 1, [(4, False, "1")]),
    (3, 0.002, 3, [(4, False, "0"), (1, True, "1")]),
])
def test_equals_combine_of_calls(cli, tmp_path, cfg, scale, n, modes):
    bams, ws, rows, bed = write_cohort(tmp_path, cfg, scale, list(range(1, n + 1)))
    for threads, unphased, idx in modes:
        opts = ["-R", bed, "-t", str(threads), *(["-u"] if unphased else [])]
        env = {"INQ_BAM_INDEX": idx}
        exp = call_then_combine(cli, tmp_path, bams, opts, env)
        stats = str(tmp_path / "st.json")
        r = run(cli, "call-cohort", *opts, "--stats-json", stats, *bams, env=env)
        assert r.returncode == 0, r.stderr
        assert r.stdout == exp, (threads, unphased, idx)
        assert r.stdout == oracle_table(bams, ws, rows, unphased, threads)
        st = json.load(open(stats))
        assert set(st) == {"n_samples", "n_contexts", "n_loci", "s_ctx_create_set_loci", "s_total", "samples"}
        assert all(set(s) == {"bam", "context", "used_index", "records", "records_pushed", "records_unpairable", "bytes_inflated",
                              "n_pairs", "ms_total", "s_bam_scan", "s_genotype"} for s in st["samples"])
        assert st["n_samples"] == n and st["n_contexts"] == 1 and len(st["samples"]) == n
        assert all(s["used_index"] == int(idx) for s in st["samples"])
        assert all(s["records_pushed"] > 0 and s["ms_total"] > 0 for s in st["samples"])


@pytest.mark.gpu
def test_devices_spread_samples_not_the_catalog(cli, tmp_path):
    bams, _, _, bed = write_cohort(tmp_path, 4, 1.0, [1, 2, 3, 4, 5])
    outs = {}
    for devs, n_ctx in (("0", 1), ("0,0,0", 3), (",".join(["0"] * 9), 5)):
        stats = str(tmp_path / "st.json")
        r = run(cli, "call-cohort", "-R", bed, "--devices", devs, "--stats-json", stats, *bams)
        assert r.returncode == 0, r.stderr
        outs[devs] = r.stdout
        st = json.load(open(stats))
        assert st["n_contexts"] == n_ctx and st["n_samples"] == 5
        assert all(0 <= s["context"] < n_ctx for s in st["samples"])
    assert len(set(outs.values())) == 1
    assert outs["0"] == call_then_combine(cli, tmp_path, bams, ["-R", bed])


@pytest.mark.gpu
def test_headers_in_other_orders_and_extra_contigs(cli, tmp_path):
    """contigs mapped by name: the same reads under a permuted header, and under a header with one more contig that
    carries reads, give the oracle's columns"""
    from tests.datagen import make_case
    case = make_case(31, n_contigs=3, n_loci=80, n_reads=1200)
    names = ["chr3", "chr1", "chr2"]
    rd = case["reads"]
    cat = [(names[int(case["locus_contig"][i])], int(case["locus_start"][i]), int(case["locus_end"][i])) for i in range(len(case["locus_start"]))]
    bed = tmp_path / "loci.bed"
    bed.write_text("".join(f"{c}\t{s}\t{e}\n" for c, s, e in cat))

    def as_bam(path, header_names, tid_of, extra=None):
        contig = np.asarray([tid_of[int(c)] for c in rd.contig], np.int32)
        r2 = O.Reads(contig, rd.ref_start, rd.ref_end, rd.mapq, rd.hp, rd.flags, rd.cigar_off, rd.cigar)
        if extra is not None:       # the same reads once more on the extra contig: nothing of the catalog is there
            r2 = O.Reads(np.concatenate([contig, np.full(rd.n, extra, np.int32)]), np.tile(rd.ref_start, 2), np.tile(rd.ref_end, 2),
                         np.tile(rd.mapq, 2), np.tile(rd.hp, 2), np.tile(rd.flags, 2),
                         np.concatenate([rd.cigar_off[:-1], rd.cigar_off + rd.cigar_off[-1]]), np.tile(rd.cigar, 2))
        bamio.reads_to_bam(path, header_names, [60_000] * len(header_names), r2)
        return path

    b0 = as_bam(str(tmp_path / "plain.bam"), names, {0: 0, 1: 1, 2: 2})
    b1 = as_bam(str(tmp_path / "permuted.bam"), ["chr2", "chr3", "chr1"], {0: 1, 1: 2, 2: 0})
    b2 = as_bam(str(tmp_path / "extra.bam"), ["chrX", "chr1", "chr2", "chr3"], {0: 3, 1: 1, 2: 2}, extra=0)
    for unphased in (False, True):
        rc, p1, p2, _ = O.genotype_loci(rd, 3, case["locus_contig"], case["locus_start"].astype(np.uint32),
                                        case["locus_end"].astype(np.uint32), 5, 3, unphased)
        assert rc == 0
        col = [ln.split("\t") for ln in expected_tsv("x", None, cat, p1, p2, 4).decode().splitlines()]
        exp = "\n".join("\t".join(c[:3] + (["plain_H1", "plain_H2", "permuted_H1", "permuted_H2", "extra_H1", "extra_H2"] if k == 0 else c[3:] * 3))
                        for k, c in enumerate(col)) + "\n"
        opts = ["-R", str(bed), "-t", "4", *(["-u"] if unphased else [])]
        r = run(cli, "call-cohort", *opts, b0, b1, b2, env={"INQ_BAM_INDEX": "0"})
        assert r.returncode == 0, r.stderr
        assert r.stdout == exp.encode()
        assert r.stdout == call_then_combine(cli, tmp_path, [b0, b1, b2], opts, {"INQ_BAM_INDEX": "0"})


@pytest.mark.gpu
def test_repeated_empty_and_header_only_samples(cli, tmp_path):
    bams, ws, rows, bed = write_cohort(tmp_path, 4, 1.0, [1])
    far = tiny_bam(str(tmp_path / "far.bam"), ws[0].contig_names, list(ws[0].contig_len), tid=0, pos=10)  # reads near no locus
    bamio.write_bam(str(tmp_path / "hdr.bam"), ws[0].contig_names, list(ws[0].contig_len), [])
    hdr = str(tmp_path / "hdr.bam")
    r = run(cli, "call-cohort", "-R", bed, bams[0], far, bams[0], hdr)
    assert r.returncode == 0, r.stderr
    lines = [ln.split(b"\t") for ln in r.stdout.splitlines()]
    assert lines[0][3:] == [b"s1_H1", b"s1_H2", b"far_H1", b"far_H2", b"s1_H1", b"s1_H2", b"hdr_H1", b"hdr_H2"]
    assert all(ln[3:5] == ln[7:9] and ln[5:7] == [b"NaN", b"NaN"] and ln[9:11] == [b"NaN", b"NaN"] for ln in lines[1:])
    assert any(ln[3] != b"NaN" for ln in lines[1:])
    assert r.stdout == call_then_combine(cli, tmp_path, [bams[0], far, bams[0], hdr], ["-R", bed])


@pytest.mark.gpu
def test_panic_in_third_sample_leaves_stdout_empty(cli, tmp_path):
    """HP 3 on a read that pairs (call.rs:358) in the third of four samples: exit 101, nothing printed"""
    names, lens = ["chr1"], [1_000_000]
    good = [tiny_bam(str(tmp_path / f"g{k}.bam"), names, lens) for k in range(3)]
    bad = tiny_bam(str(tmp_path / "bad.bam"), names, lens, hp=3)
    assert run(cli, "call", "-r", "chr1:1490-1510", "-s", "2", bad).returncode == 101
    for devs in ("0", "0,0,0"):
        r = run(cli, "call-cohort", "-r", "chr1:1490-1510", "-s", "2", "--devices", devs, good[0], good[1], bad, good[2])
        assert r.returncode == 101 and r.stdout == b"", (devs, r.stderr)
    r = run(cli, "call-cohort", "-r", "chr1:1490-1510", "-s", "2", "--devices", "0,0", *good)
    assert r.returncode == 0, r.stderr
    assert r.stdout == call_then_combine(cli, tmp_path, good, ["-r", "chr1:1490-1510", "-s", "2"])
    assert r.stdout.splitlines()[1].split(b"\t")[3] != b"NaN"
