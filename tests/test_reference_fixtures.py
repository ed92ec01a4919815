"""Known-answer tests on fixtures shaped like the reference's own test-data, which is not part of this
repository: an index in the layout htslib writes for `small-test.bam.bai` (195 references in hg38 order,
only chr7 populated, metadata pseudo-bin, n_no_coor trailer) pins the BAI reader
(`BamIndexedReader::load_index` / `query_chunks`, SURVEY 8f rank 2), and three call outputs like
`file{1,2,3}.inq[.gz]` -- the inputs of the reference's own `combine` tests (combine.rs:61-78), including
the line of `file1.inq` with spaces where a tab should be -- pin `inquistr-b200 combine`. The fixtures are
generated from fixed seeds (the index by tests/bamio.py, from a BAM whose records are known). CPU only."""
import gzip
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from tests import bamio

TEST_BED = ("chr7", 154778571, 154779363)                                   # test-data/test.bed:1


@pytest.fixture(scope="module")
def cli():
    from inquistr_b200 import build
    build.build_libinqcall()
    return build.build_cli()


@pytest.fixture(scope="module")
def indexed_bam(tmp_path_factory):
    """195 references (hg38 chr1-22,X,Y first, so chr7 is tid 6), reads only on chr7 around the test.bed locus:
    mapped reads of 0.5-60 kb, placed unmapped reads, and unplaced reads at the end of the file.
    Returns (bam, bai, n_mapped, n_unmapped, n_no_coor)."""
    from synth.synth import HG38
    names = [n for n, _ in HG38] + [f"chrUn_{i:03d}" for i in range(195 - len(HG38))]
    lens = [ln for _, ln in HG38] + [50_000] * (195 - len(HG38))
    rng = np.random.default_rng(8105)
    n_mapped, n_unmapped, n_no_coor = 3000, 40, 25
    pos = rng.integers(TEST_BED[1] - 200_000, TEST_BED[2] + 200_000, n_mapped + n_unmapped)
    rlen = np.where(rng.random(len(pos)) < 0.1, rng.integers(20_000, 60_000, len(pos)), rng.integers(500, 15_000, len(pos)))
    placed = []
    for i, (p, ln) in enumerate(zip(pos.tolist(), rlen.tolist())):
        if i < n_mapped:
            placed.append((p, bamio.encode_record(6, p, 60, 0, [(ln << 4) | 0], name=b"m%d" % i, end=p + ln)))
        else:
            placed.append((p, bamio.encode_record(6, p, 0, 4, [], name=b"u%d" % i)))
    placed.sort(key=lambda t: t[0])
    recs = [r for _, r in placed] + [bamio.encode_record(-1, -1, 0, 4, [], name=b"n%d" % i) for i in range(n_no_coor)]
    bam = str(tmp_path_factory.mktemp("bai") / "small-test.bam")
    bamio.write_bam(bam, names, lens, recs)
    return bam, bamio.index_bam(bam, meta=True), n_mapped, n_unmapped, n_no_coor


@pytest.fixture(scope="module")
def inq_files(tmp_path_factory):
    """three call outputs over the same loci, each as plain text and gzip; line 1 of the first has two spaces where
    the tab between H1 and H2 should be, as file1.inq:1 of the reference has. Returns the plain paths."""
    rng = np.random.default_rng(61)
    d = tmp_path_factory.mktemp("combine")
    loci = [(f"chr{1 + i // 10}", 10_000 + 731 * i, 10_040 + 731 * i) for i in range(30)]
    plain = []
    for k in (1, 2, 3):
        rows = []
        for c, b, e in loci:
            h = ["NaN" if rng.random() < 0.15 else f"{rng.integers(0, 400) / 2:.1f}" for _ in range(2)]
            rows.append(f"{c}\t{b}\t{e}\t{h[0]}\t{h[1]}")
        if k == 1:
            rows[0] = "\t".join(rows[0].split("\t")[:3]) + "\t4027.0  4081.0"
        p = d / f"file{k}.inq"
        p.write_text("\n".join(rows) + "\n")
        with gzip.open(str(p) + ".gz", "wb") as f:
            f.write(p.read_bytes())
        plain.append(str(p))
    return plain


# ---------------------------------------------------------------- independent BAI parse (SAM spec 5.2 / 5.3)
def parse_bai(path):
    b = open(path, "rb").read()
    assert b[:4] == b"BAI\x01"
    n_ref = struct.unpack_from("<i", b, 4)[0]
    p = 8
    refs = []
    for _ in range(n_ref):
        n_bin = struct.unpack_from("<i", b, p)[0]; p += 4
        bins, meta = {}, None
        for _ in range(n_bin):
            bin_, n_chunk = struct.unpack_from("<Ii", b, p); p += 8
            ch = [struct.unpack_from("<QQ", b, p + 16 * i) for i in range(n_chunk)]; p += 16 * n_chunk
            if bin_ == 37450:
                meta = ch
            else:
                bins[bin_] = ch
        n_intv = struct.unpack_from("<i", b, p)[0]; p += 4
        lin = list(struct.unpack_from(f"<{n_intv}Q", b, p)); p += 8 * n_intv
        refs.append((bins, lin, meta))
    n_no_coor = struct.unpack_from("<Q", b, p)[0] if p + 8 <= len(b) else 0
    return refs, n_no_coor


def reg2bins(beg, end):
    end -= 1
    out = [0]
    for shift, base in ((26, 1), (23, 9), (20, 73), (17, 585), (14, 4681)):
        out += list(range(base + (beg >> shift), base + (end >> shift) + 1))
    return out


def expected_chunks(ref, beg, end):
    bins, lin, _ = ref
    min_off = (lin[beg >> 14] if (beg >> 14) < len(lin) else lin[-1]) if lin else 0
    ch = sorted(c for b in reg2bins(beg, end) for c in bins.get(b, []) if c[1] > min_off)
    merged = []
    for a, e in ch:
        if merged and a <= merged[-1][1]:
            merged[-1][1] = max(merged[-1][1], e)
        else:
            merged.append([a, e])
    return merged


def test_reference_bai_loads_and_answers_the_test_bed_window(cli, indexed_bam):
    bam, bai, n_mapped, n_unmapped, n_no_coor_written = indexed_bam
    _, s, e = TEST_BED
    beg, end = s - 10, e + 10                                               # the fetch window of call.rs:285-288
    refs, n_no_coor = parse_bai(bai)
    populated = [t for t, r in enumerate(refs) if r[0]]
    assert len(refs) == 195 and populated == [6]                            # hg38 order: chr7 is tid 6
    assert n_no_coor == n_no_coor_written
    r = subprocess.run([cli, "baistat", bai, f"6:{beg}-{end}"], capture_output=True, timeout=60)
    assert r.returncode == 0, r.stderr
    got = json.loads(r.stdout)
    assert got["refs"] == 195 and got["n_no_coor"] == n_no_coor
    assert got["mapped"] == {"6": [n_mapped, n_unmapped]}                   # metadata pseudo-bin
    assert refs[6][2][1] == (n_mapped, n_unmapped)
    exp = expected_chunks(refs[6], beg, end)
    assert got["chunks"] == exp and len(exp) > 0
    # every chunk lies inside the BAM: below the largest virtual offset the index mentions
    max_voff = max(c[1] for ch in refs[6][0].values() for c in ch)
    assert (max_voff >> 16) < os.path.getsize(bam)
    assert all(a < b <= max_voff for a, b in got["chunks"])
    # a window on an unpopulated reference, and one far from any read, yield nothing
    r = subprocess.run([cli, "baistat", bai, "3:1000-2000"], capture_output=True, timeout=60)
    assert json.loads(r.stdout)["chunks"] == []
    r = subprocess.run([cli, "baistat", bai, "6:1000-2000"], capture_output=True, timeout=60)
    assert json.loads(r.stdout)["chunks"] == expected_chunks(refs[6], 1000, 2000)


def test_bai_rejects_garbage(cli, indexed_bam, tmp_path):
    p = tmp_path / "x.bai"
    p.write_bytes(b"BAM\x01" + b"\0" * 32)
    assert subprocess.run([cli, "baistat", str(p)], capture_output=True).returncode == 1
    good = open(indexed_bam[1], "rb").read()
    assert len(good) > 5000
    p.write_bytes(good[:5000])                                               # truncated
    assert subprocess.run([cli, "baistat", str(p)], capture_output=True).returncode == 1


# ---------------------------------------------------------------- combine on the reference's own fixtures
def py_combine(texts):
    """combine.rs:40-58: the first file's line in full, then columns 4.. (split on tab) of every other file"""
    lines = [t.split("\n")[:-1] if t.endswith("\n") else t.split("\n") for t in texts]
    out = []
    for i, first in enumerate(lines[0]):
        row = [first]
        for other in lines[1:]:
            row += other[i].split("\t")[3:]
        out.append("\t".join(row))
    return "\n".join(out) + "\n"


def test_combine_on_reference_fixtures_plain_and_gz(cli, inq_files):
    plain = inq_files                                                        # combine.rs:61-68
    gz = [p + ".gz" for p in plain]                                          # combine.rs:70-78
    texts = [open(p).read() for p in plain]
    assert "4027.0  4081.0" in texts[0].split("\n")[0]                       # file1.inq:1 has spaces where a tab should be
    a = subprocess.run([cli, "combine", *plain], capture_output=True, timeout=60)
    b = subprocess.run([cli, "combine", *gz], capture_output=True, timeout=60)
    assert a.returncode == 0 and b.returncode == 0, (a.stderr, b.stderr)
    assert a.stdout.decode() == py_combine(texts)
    gz_texts = [gzip.open(p, "rt").read() for p in gz]
    assert b.stdout.decode() == py_combine(gz_texts)
    assert gz_texts == texts and a.stdout == b.stdout
    # mixed plain / gz and a different first file
    c = subprocess.run([cli, "combine", gz[1], plain[0], gz[2]], capture_output=True, timeout=60)
    assert c.returncode == 0 and c.stdout.decode() == py_combine([gz_texts[1], texts[0], gz_texts[2]])
