"""`inquistr-b200 call` (C++ host above the C ABI): CLI behaviour without a GPU, and byte-for-byte
TSV parity against the oracle with a GPU. Mirrors the reference's own call tests
(call.rs:525-605): region, region file, unphased, wrong chromosome (should panic), header length."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O
from tests import bamio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "inquistr_b200", "bin", "inquistr-b200")


@pytest.fixture(scope="module")
def cli():
    from inquistr_b200 import build
    build.build_libinqcall()
    return build.build_cli()


def run(cli, *args, **kw):
    return subprocess.run([cli, *args], capture_output=True, timeout=300, **kw)


@pytest.fixture(scope="module")
def chr7_bam(tmp_path_factory):
    """stand-in for test-data/small-test.bam: chr7 (159,345,973 bp) with reads around test.bed's locus"""
    from synth.synth import make_workload
    w = make_workload(1, threads=2)
    d = tmp_path_factory.mktemp("cli")
    path = str(d / "small-test.sorted.bam")
    bamio.reads_to_bam(path, ["chr6", "chr7"], [170805979, 159345973],
                       O.Reads(w.reads.contig + 1, w.reads.ref_start, w.reads.ref_end, w.reads.mapq, w.reads.hp,
                               w.reads.flags, w.reads.cigar_off, w.reads.cigar))
    bed = str(d / "test.bed")
    open(bed, "w").write("chr7\t154778571\t154779363\n")
    return path, bed, w


def test_help_and_usage(cli):
    r = run(cli, "call")
    assert r.returncode == 2 and b"Usage: inquistr-b200 call [OPTIONS] <BAM>" in r.stderr     # arg_required_else_help
    r = run(cli, "call", "--help")
    assert r.returncode == 0 and b"--region-file <REGION_FILE>" in r.stdout and b"[default: 5]" in r.stdout
    r = run(cli, "call", "--bogus", "x.bam")
    assert r.returncode == 2


def test_invalid_bam_path_exits_1(cli):
    r = run(cli, "call", "-r", "chr7:100-200", "/nonexistent/x.bam")
    assert r.returncode == 1 and b"is not valid" in r.stderr and r.stdout == b""          # call.rs:87-90


def test_needs_region_or_bed(cli, chr7_bam):
    bam, bed, _ = chr7_bam
    r = run(cli, "call", bam)
    assert r.returncode == 1 and b"Specify a region string (-r) or a region_file (-R)!" in r.stderr   # call.rs:197-200
    r = run(cli, "call", "-r", "chr7:154778571-154779363", "-R", bed, bam)
    assert r.returncode == 1


def test_wrong_chromosome_panics(cli, chr7_bam):
    bam, _, _ = chr7_bam
    r = run(cli, "call", "-r", "7:154778571-154779363", bam)                              # call.rs:584-598
    assert r.returncode == 101 and b"is not in the fasta file or the end coordinate is out of bounds" in r.stderr
    r = run(cli, "call", "-r", "chr7:154778571-159345973", bam)                           # end must be < LN (call.rs:600-605)
    assert r.returncode == 101
    r = run(cli, "call", "-r", "chr7:200-100", bam)
    assert r.returncode == 101 and b"End coordinate is smaller than start coordinate" in r.stderr
    r = run(cli, "call", "-r", "chr7:5-100", bam)
    assert r.returncode == 101                                                            # start - 10 underflows u32


def test_unsupported_inputs_say_so(cli, tmp_path):
    p = tmp_path / "x.cram"
    p.write_bytes(b"CRAM")
    r = run(cli, "call", "-r", "chr7:100-200", str(p))
    assert r.returncode == 1 and b"CRAM input is not supported" in r.stderr
    r = run(cli, "call", "-r", "chr7:100-200", "https://example.org/x.bam")
    assert r.returncode == 1 and b"not supported" in r.stderr
    q = tmp_path / "bad.bam"
    q.write_bytes(b"not a bam at all, definitely")
    r = run(cli, "call", "-r", "chr7:100-200", str(q))
    assert r.returncode == 101 and b"Error opening local BAM" in r.stderr


def test_fails_loudly_without_gpu(cli, chr7_bam):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    bam, bed, _ = chr7_bam
    r = run(cli, "call", "-R", bed, bam)
    assert r.returncode == 1 and b"no CPU fallback" in r.stderr and r.stdout == b""


# ------------------------------------------------------------------------------------------- GPU
def expected_tsv(sample, names, loci, p1, p2, threads):
    """loci: list of (chrom, start, end) in BED order; -t 1 keeps it, -t >1 sorts (call.rs:137-157)"""
    idx = list(range(len(loci)))
    if threads > 1:
        def cmp(a, b):
            c = O.human_compare(loci[a][0], loci[b][0])
            return c if c else (loci[a][1] > loci[b][1]) - (loci[a][1] < loci[b][1])
        idx.sort(key=functools.cmp_to_key(cmp))
    lines = [f"chromosome\tbegin\tend\t{sample}_H1\t{sample}_H2"]
    lines += [O.format_row(loci[i][0], loci[i][1], loci[i][2], p1[i], p2[i]) for i in idx]
    return ("\n".join(lines) + "\n").encode()


@pytest.mark.gpu
def test_reference_smoke_cases_tsv(cli, chr7_bam):
    """the reference's test_region / test_region_bed / test_unphased, with the bytes checked"""
    bam, bed, w = chr7_bam
    rd = O.Reads(w.reads.contig + 1, w.reads.ref_start, w.reads.ref_end, w.reads.mapq, w.reads.hp, w.reads.flags,
                 w.reads.cigar_off, w.reads.cigar)
    for unphased in (False, True):
        rc, p1, p2, _ = O.genotype_loci(rd, 2, [1], [154778571], [154779363], 5, 3, unphased)
        exp = expected_tsv("small-test.sorted", None, [("chr7", 154778571, 154779363)], p1, p2, 4)
        for args in (["-r", "chr7:154778571-154779363", "-t", "4"], ["-R", bed], ["-R", bed, "-t", "4", "-m", "5", "-s", "3"]):
            r = run(cli, "call", *args, *(["-u"] if unphased else []), bam)
            assert r.returncode == 0, r.stderr
            assert r.stdout == exp
    r = run(cli, "call", "-R", bed, "--sample-name", "NA12878", bam)
    assert r.stdout.startswith(b"chromosome\tbegin\tend\tNA12878_H1\tNA12878_H2\n")


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [1, 4])
def test_multi_contig_bed_ordering_and_2d(cli, tmp_path, threads):
    """unsorted multi-contig BED: BED order for -t 1, human-sorted for -t 4; SA-derived 2D flags; HP:i"""
    from tests.datagen import make_case
    case = make_case(77, n_contigs=4, n_loci=150, n_reads=1500)
    names = ["chr10", "chr2", "chrX", "chr1_KI270706v1_random"]
    lens = [60_000] * 4
    rd = case["reads"]
    order = np.lexsort((rd.ref_start, rd.contig))                       # coordinate-sorted file
    off = np.zeros(rd.n + 1, np.uint64)
    n_cig = (rd.cigar_off[1:] - rd.cigar_off[:-1]).astype(np.int64)
    off[1:] = np.cumsum(n_cig[order])
    cig = np.concatenate([rd.cigar[int(rd.cigar_off[i]):int(rd.cigar_off[i + 1])] for i in order])
    srd = O.Reads(rd.contig[order], rd.ref_start[order], rd.ref_end[order], rd.mapq[order], rd.hp[order], rd.flags[order], off, cig)
    bam = str(tmp_path / "multi.bam")
    bamio.reads_to_bam(bam, names, lens, srd, hp_type="i")
    perm = np.random.default_rng(5).permutation(len(case["locus_start"]))
    loci = [(names[int(case["locus_contig"][i])], int(case["locus_start"][i]), int(case["locus_end"][i])) for i in perm]
    bed = str(tmp_path / "loci.bed")
    with open(bed, "w") as f:
        f.write("# comment line\n")
        for c, s, e in loci:
            f.write(f"{c}\t{s}\t{e}\tsome\textra\n")
    for unphased in (False, True):
        rc, p1, p2, _ = O.genotype_loci(srd, 4, case["locus_contig"][perm], case["locus_start"][perm].astype(np.uint32),
                                        case["locus_end"][perm].astype(np.uint32), 5, 3, unphased)
        assert rc == 0
        r = run(cli, "call", "-R", bed, "-t", str(threads), *(["-u"] if unphased else []), bam)
        assert r.returncode == 0, r.stderr
        assert r.stdout == expected_tsv("multi", names, loci, p1, p2, threads)


@pytest.mark.gpu
def test_long_cigar_cg_tag_and_bad_hp(cli, tmp_path):
    # one read with > 65535 CIGAR ops goes through the CG:B,I convention
    n = 70_000
    words = np.empty(2 * n + 1, np.uint32)
    words[0::2] = (3 << 4) | 0
    words[1::2] = (1 << 4) | 1
    words[2001] = (9 << 4) | 1                                  # the only insertion longer than 5
    rlen = 3 * (n + 1)
    recs = [bamio.encode_record(0, 1000, 60, 0, words, name=b"long%d" % i, hp=1 + (i % 2), end=1000 + rlen) for i in range(8)]
    bam = str(tmp_path / "long.bam")
    bamio.write_bam(bam, ["chr1"], [1_000_000], recs)
    r = run(cli, "call", "-r", "chr1:4000-4010", "-s", "2", bam)        # insertion anchored at 1000+3*1001+1 = 4004
    assert r.returncode == 0, r.stderr
    assert r.stdout.splitlines()[1] == b"chr1\t4000\t4010\t9\t9"
    # HP outside {0,1,2} on a read that passes the filter: the reference panics (call.rs:358)
    recs = [bamio.encode_record(0, 1000, 60, 0, words[:200], name=b"x%d" % i, hp=3, end=1000 + 3 * 100) for i in range(4)]
    bad = str(tmp_path / "badhp.bam")
    bamio.write_bam(bad, ["chr1"], [1_000_000], recs)
    r = run(cli, "call", "-r", "chr1:1100-1110", bad)
    assert r.returncode == 101
    r = run(cli, "call", "-r", "chr1:1100-1110", "-u", bad)             # unphased never looks at HP
    assert r.returncode == 0
    # HP stored as an int16: rust-htslib yields Aux::I16 and the reference panics (call.rs:487)
    recs = [bamio.encode_record(0, 1000, 60, 0, words[:200], name=b"y", hp=1, hp_type="s", end=1300)]
    bamio.write_bam(bad, ["chr1"], [1_000_000], recs)
    assert run(cli, "call", "-r", "chr1:1100-1110", bad).returncode == 101


def test_host_bam_reader_matches_workload(cli, tmp_path):
    """the BGZF/BAM reader alone (no GPU): record, CIGAR-word, HP, SA and accidental-2D counts of a
    synthetic BAM (with SEQ/QUAL, multi-batch, multi-threaded inflate) equal those of its SoA source"""
    import json
    from synth import synth as S
    w = S.make_workload(3, scale=0.0008, threads=2)
    for with_seq in (False, True):
        bam = str(tmp_path / f"s{int(with_seq)}.bam")
        assert S.write_bam(w, bam, with_seq=with_seq) > 0
        r = run(cli, "bamstat", bam)
        assert r.returncode == 0, r.stderr
        st = json.loads(r.stdout)
        assert st["refs"] == w.n_contigs and st["records"] == w.reads.n
        assert st["cigar_words"] == len(w.reads.cigar)
        assert st["hp_tagged"] == int((w.reads.hp != 0xFF).sum())
        assert st["accidental_2d"] == int((w.reads.flags & 1).sum()) == st["sa_tagged"]
        # the call driver's parallel parse (no device needed): every record seen, the CIGARs of the records that can
        # pair somewhere (mapq > 10) kept
        r = run(cli, "bamstat", bam, "--parsed")
        assert r.returncode == 0, r.stderr
        sp = json.loads(r.stdout)
        n_cig = (w.reads.cigar_off[1:] - w.reads.cigar_off[:-1]).astype(np.int64)
        assert sp["records"] == w.reads.n and sp["cigar_words"] == int(n_cig[w.reads.mapq > 10].sum())


def test_own_deflate_decoder_equals_zlib_on_every_block(cli, tmp_path):
    """`bgzf-check`: the host ingest's own DEFLATE decoder against zlib, block by block, bytes compared -- stored blocks
    (level 0), the match-heavy streams of level 1, the literal-heavy ones of level 6 (with SEQ/QUAL: long dynamic
    codes, two-level tables), and a plain gzip file like the reference's `file1.inq.gz`. A declined block would fall
    back to zlib in the product; here it fails the test."""
    import gzip
    import json
    from synth import synth as S
    w = S.make_workload(3, scale=0.0006, threads=2)
    for level, with_seq in ((0, False), (1, True), (6, True), (9, False)):
        bam = str(tmp_path / f"l{level}.bam")
        assert S.write_bam(w, bam, with_seq=with_seq, level=level) > 0
        r = run(cli, "bgzf-check", bam)
        assert r.returncode == 0, r.stderr
        st = json.loads(r.stdout)
        assert st["blocks"] > 1 and st["mismatch"] == 0 and st["fast_declined"] == 0, (level, st)
    plain_gz = str(tmp_path / "file1.inq.gz")       # plain gzip is not BGZF: the walker says so
    with gzip.open(plain_gz, "wt") as f:
        f.write("".join(f"chr7\t{154778571 + i}\t{154779363 + i}\t{i}.0\t{2 * i}.5\n" for i in range(50)))
    r = run(cli, "bgzf-check", plain_gz)
    assert r.returncode == 1 and b"not a BGZF member" in r.stdout


def test_clmul_crc32_equals_zlib(tmp_path):
    """csrc/host/crc32_fast.hpp: every BGZF block's CRC-32 goes through it (PCLMULQDQ where the CPU has it)"""
    exe = str(tmp_path / "crc32_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "inquistr_b200", "csrc", "host"), "-o", exe,
                    os.path.join(ROOT, "tests", "crc32_check.cpp"), "-lz"], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == "bad 0", r.stdout


def test_own_deflate_decoder_survives_corrupted_blocks(tmp_path):
    """tests/fuzz_inflate.cpp under ASan + UBSan: bit flips, random spans, damaged headers, truncated input, output
    buffers that are too small or too large -- the decoder declines or decodes, and never reads outside
    [in, in + in_len + 8) or writes outside [out, out + out_len). (In the product a declined block goes to zlib and
    every block is CRC-checked.)"""
    from synth import synth as S
    exe = str(tmp_path / "fuzz_inflate")
    cc = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                         "-I", os.path.join(ROOT, "inquistr_b200", "csrc", "host"), "-o", exe,
                         os.path.join(ROOT, "tests", "fuzz_inflate.cpp")], capture_output=True, text=True)
    if cc.returncode != 0:
        pytest.skip("no sanitizer runtime for g++ here: " + cc.stderr[-300:])
    w = S.make_workload(3, scale=0.0005, threads=2)
    for level, with_seq in ((1, True), (6, False)):
        bam = str(tmp_path / f"f{level}.bam")
        assert S.write_bam(w, bam, with_seq=with_seq, level=level) > 0
        r = subprocess.run([exe, bam, "4000"], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "fuzz: 4000 cases" in r.stdout, (r.stdout[-500:], r.stderr[-2000:])


@pytest.mark.gpu
def test_cli_on_synthetic_bam_with_seq(cli, tmp_path):
    """tools/bench_bam.py path: config 3 (shrunk) written as a BAM with SEQ/QUAL, shuffled BED, -t 8"""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_bam.py"), "--scale", "0.003", "--with-seq",
                          "--keep", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    res = json.loads(out.stdout.strip().splitlines()[-1])
    assert res["tsv_identical_to_oracle"] is True
    assert res["cli_stats"]["records"] == res["reads"]


@pytest.fixture(scope="module")
def panel_bam(tmp_path_factory):
    from synth import synth as S
    w = S.make_workload(4, threads=2)
    d = tmp_path_factory.mktemp("panel")
    bam = str(d / "panel.bam")
    S.write_bam(w, bam)
    bamio.index_bam(bam)
    rows = S.write_bed(w, str(d / "panel.bed"), shuffle_seed=3)
    return bam, str(d / "panel.bed"), rows, w


def test_bai_fetch_matches_htslib_overlap_rule(cli, panel_bam):
    """indexed random access (no GPU): records with pos < end && endpos > beg on the contig, in file order"""
    import json
    bam, _, _, w = panel_bam
    rd = w.reads
    n_cig = (rd.cigar_off[1:] - rd.cigar_off[:-1]).astype(np.int64)
    for k in (0, 13, 41, 59):
        c = int(w.locus_contig[k]); b = int(w.locus_start[k]) - 10; e = int(w.locus_end[k]) + 10
        m = (rd.contig == c) & (rd.ref_start < e) & (rd.ref_end > b)
        r = run(cli, "bamstat", bam, f"{w.contig_names[c]}:{b}-{e}")
        assert r.returncode == 0, r.stderr
        st = json.loads(r.stdout)
        assert st["records"] == int(m.sum()) and st["cigar_words"] == int(n_cig[m].sum())
        assert st["bytes_inflated"] < 0.3 * os.path.getsize(bam) * 4     # a fraction of the file, not all of it
    r = run(cli, "bamstat", bam, "chr1:1-2")                              # nothing there
    assert json.loads(r.stdout)["records"] == 0


@pytest.mark.gpu
def test_panel_with_and_without_index(cli, panel_bam, tmp_path):
    """config 4 (expansion panel): the .bai path and the sequential scan print the same bytes"""
    import json
    bam, bed, rows, w = panel_bam
    sel = np.asarray([i for *_, i in rows])
    rc, p1, p2, _ = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig[sel], w.locus_start[sel].astype(np.uint32),
                                    w.locus_end[sel].astype(np.uint32), 5, 3, False)
    exp = expected_tsv("panel", None, [(c, s, e) for c, s, e, _ in rows], p1, p2, 1)
    outs = {}
    for mode in ("1", "0"):
        stats = str(tmp_path / f"st{mode}.json")
        r = subprocess.run([cli, "call", "-R", bed, "--stats-json", stats, bam], capture_output=True, timeout=300,
                           env={**os.environ, "INQ_BAM_INDEX": mode})
        assert r.returncode == 0, r.stderr
        assert r.stdout == exp
        outs[mode] = json.load(open(stats))
    assert outs["1"]["used_index"] == 1 and outs["0"]["used_index"] == 0
    assert outs["1"]["records"] <= outs["0"]["records"]          # only records near the loci are decoded
    assert outs["1"]["records_pushed"] == outs["0"]["records_pushed"]
    # single region (-r) picks the index on its own
    stats = str(tmp_path / "st_r.json")
    c, s, e, _ = rows[0]
    r = run(cli, "call", "-r", f"{c}:{s}-{e}", "--stats-json", stats, bam)
    assert r.returncode == 0 and json.load(open(stats))["used_index"] == 1
    assert r.stdout.splitlines()[1] == exp.splitlines()[1]


@pytest.mark.gpu
def test_aux_panics_fire_only_for_reads_that_pair(cli, tmp_path):
    """is_accidental_2d (SA) and the HP bucket lookup only run for reads that passed the filter of some locus
    (call.rs:350-358,394,431): a low-mapq or untagged read with a malformed SA / HP 255 is skipped silently,
    the same tags on a read that pairs abort with a panic (exit 101)"""
    import struct
    M, S, I = 0, 4, 1
    spanning = np.asarray([(20 << 4) | S, (500 << 4) | M, (8 << 4) | I, (500 << 4) | M], np.uint32)
    noclip = np.asarray([(500 << 4) | M, (8 << 4) | I, (500 << 4) | M], np.uint32)
    sa_int = b"SAi" + struct.pack("<i", 7)                      # SA present but not a string: Aux::I32 -> panic at call.rs:431

    def bam_of(recs, name):
        p = str(tmp_path / name)
        bamio.write_bam(p, ["chr1"], [1_000_000], recs)
        return p

    good = [bamio.encode_record(0, 1000, 60, 0, spanning, name=b"g%d" % i, hp=1 + i % 2, end=2000) for i in range(6)]
    region = ["-r", "chr1:1490-1510", "-s", "2"]
    # harmless carriers: mapq 10, no HP tag (phased), or no soft clip at all
    quiet = [bamio.encode_record(0, 1000, 10, 0, spanning, name=b"q1", hp=1, end=2000, extra_aux=sa_int),
             bamio.encode_record(0, 1000, 60, 0, spanning, name=b"q2", end=2000, sa="chr1,100"),
             bamio.encode_record(0, 1000, 60, 0, noclip, name=b"q3", hp=2, end=2000, extra_aux=sa_int),
             bamio.encode_record(0, 1000, 5, 0, spanning, name=b"q4", hp=255, end=2000)]
    r = run(cli, "call", *region, bam_of(good + quiet, "quiet.bam"))
    assert r.returncode == 0, r.stderr
    base = run(cli, "call", *region, bam_of(good + quiet[2:3], "base.bam"))
    assert base.returncode == 0 and r.stdout.splitlines()[1] == base.stdout.splitlines()[1]
    # the same tags on reads that pair
    for k, bad in enumerate([bamio.encode_record(0, 1000, 60, 0, spanning, name=b"b1", hp=1, end=2000, extra_aux=sa_int),
                             bamio.encode_record(0, 1000, 60, 0, spanning, name=b"b2", hp=1, end=2000, sa="chr1,100"),
                             bamio.encode_record(0, 1000, 60, 16, spanning, name=b"b3", hp=1, end=2000, sa="chr1,100,+"),
                             bamio.encode_record(0, 1000, 60, 0, spanning, name=b"b4", hp=255, end=2000)]):
        r = run(cli, "call", *region, bam_of(good + [bad], f"bad{k}.bam"))
        assert r.returncode == 101, (k, r.stderr)
    # same strand: sa_entry[3] is never touched (call.rs:441-443), no panic although the entry has only 3 fields
    ok = bamio.encode_record(0, 1000, 60, 0, spanning, name=b"ok", hp=1, end=2000, sa="chr1,100,+")
    assert run(cli, "call", *region, bam_of(good + [ok], "ok.bam")).returncode == 0
    # unphased: q2 (no HP) now pairs and its SA panics; q4 (HP 255, mapq 5) stays quiet
    assert run(cli, "call", *region, "-u", bam_of(good + quiet[1:2], "u1.bam")).returncode == 101
    assert run(cli, "call", *region, "-u", bam_of(good + quiet[3:4], "u2.bam")).returncode == 0


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,scale", [(3, 0.004), (4, 1.0)])
def test_devices_sharding_prints_the_same_bytes(cli, tmp_path, cfg, scale):
    """`--devices 0,0,0`: the catalog cut into three contiguous shards, three contexts on three host threads
    (here all on GPU 0), reads routed to every shard they can reach, ordered concatenation -- byte-identical TSV
    to one context, for the genome-wide config and the expansion panel, with and without the .bai"""
    import json
    from synth import synth as S
    w = S.make_workload(cfg, scale=scale, threads=4)
    bam = str(tmp_path / "in.bam")
    S.write_bam(w, bam)
    bamio.index_bam(bam)
    rows = S.write_bed(w, str(tmp_path / "loci.bed"), shuffle_seed=9)
    sel = np.asarray([i for *_, i in rows])
    rc, p1, p2, _ = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig[sel], w.locus_start[sel].astype(np.uint32),
                                    w.locus_end[sel].astype(np.uint32), 5, 3, w.unphased)
    assert rc == 0
    for threads in (1, 4):
        exp = expected_tsv("in", None, [(c, s, e) for c, s, e, _ in rows], p1, p2, threads)
        for idx_mode in ("0", "1"):
            outs = {}
            for devs in ("0", "0,0,0", "0,0,0,0,0,0,0"):
                stats = str(tmp_path / f"st_{devs.count(',')}.json")
                r = subprocess.run([cli, "call", "-R", str(tmp_path / "loci.bed"), "-t", str(threads), "--devices", devs,
                                    "--stats-json", stats, *(["-u"] if w.unphased else []), bam],
                                   capture_output=True, timeout=600, env={**os.environ, "INQ_BAM_INDEX": idx_mode})
                assert r.returncode == 0, r.stderr
                assert r.stdout == exp, (devs, idx_mode, threads)
                outs[devs] = json.load(open(stats))
            assert outs["0"]["n_shards"] == 1 and outs["0,0,0"]["n_shards"] == 3
            assert outs["0,0,0"]["records_routed"] >= outs["0,0,0"]["records_pushed"]      # reads at a cut go to both sides
            assert outs["0,0,0"]["n_loci"] == w.n_loci
    # errors raised inside a shard keep the reference's exit behaviour: HP 3 on a read that pairs -> panic, exit 101
    r = run(cli, "call", "-r", "chr1:5-100", "--devices", "0,0", bam)
    assert r.returncode == 101
