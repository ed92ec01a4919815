"""`call` and `call-cohort` run through one driver: one option parser, one input check. A malformed line gives the same
exit code and the same first stderr line from both subcommands, and every input message names the file. No GPU is
needed: every case fails before a context is made."""
import pytest

from tests.test_cohort_call import cli, run, tiny_bam  # noqa: F401  (cli is a fixture)

REGION = ["-r", "chr1:1490-1510"]


@pytest.fixture
def bams(tmp_path):
    return [tiny_bam(str(tmp_path / f"{k}.bam"), ["chr1", "chr2"], [1_000_000, 500_000]) for k in "ab"]


def first_line(r):
    return r.stderr.splitlines()[0] if r.stderr else b""


@pytest.mark.parametrize("opts,code", [
    (REGION + ["--bogus"], 2),                      # an unknown long option at the end of the line takes no value
    (REGION + ["--bogus", "x"], 2),
    (REGION + ["--bogus=x"], 2),
    (REGION + ["-x"], 2),
    (REGION + ["-um"], 2),                          # a missing value
    (REGION + ["--support"], 2),
    (REGION + ["--minlen", "4294967296"], 2),
    (REGION + ["--threads=-1"], 2),
    (REGION + ["--devices", "0,,1"], 2),
    (REGION + ["-R", "loci.bed"], 1),               # neither only -r nor only -R
    ([], 1),
])
def test_malformed_lines_fail_alike(cli, bams, opts, code):
    a, b = bams
    one = run(cli, "call", a, *opts)
    many = run(cli, "call-cohort", a, b, *opts)
    assert one.returncode == many.returncode == code, (one.stderr, many.stderr)
    assert first_line(one) == first_line(many) and first_line(one).startswith(b"error: " if code == 2 else b"ERROR: ")
    assert one.stdout == many.stdout == b""


@pytest.mark.parametrize("opt", [["--sample-name", "x"], ["--reference", "ref.fa"], ["--device", "0"], ["--sample-name=x"]])
def test_call_only_options(cli, tmp_path, opt):
    missing = str(tmp_path / "missing.bam")
    r = run(cli, "call", *REGION, *opt, missing)
    assert r.returncode == 1 and b"is not valid" in r.stderr          # accepted: the input check is what fails
    r = run(cli, "call-cohort", *REGION, *opt, missing, missing)
    name = opt[0].split("=")[0].encode()
    assert r.returncode == 2 and first_line(r) == b"error: unexpected argument '" + name + b"' found"


def test_input_checks_name_the_file(cli, bams, tmp_path):
    cram = tmp_path / "x.cram"
    cram.write_bytes(b"CRAM")
    for bad, msg in ((str(tmp_path / "missing.bam"), b"is not valid"), (str(cram), b"CRAM input is not supported"),
                     ("https://example.org/x.bam", b"is not supported"), ("s3://bucket/x.bam", b"is not supported")):
        one = run(cli, "call", *REGION, bad)
        many = run(cli, "call-cohort", *REGION, bams[0], bad)
        assert one.returncode == many.returncode == 1
        assert one.stderr == many.stderr and msg in one.stderr and bad.encode() in one.stderr, (one.stderr, many.stderr)
