"""`assoc --traits` / inq_assoc_traits: several traits against one table in one run (DESIGN.md 5e, Several traits).
The contract: trait t's results are bit for bit those of the single-trait path over the samples that have trait t.
CPU: the contract restated on the oracle (reference_traits), the CLI's usage, input and count lines, the ABI's argument errors.
GPU: bit-identity with cohort.assoc per trait, parity with the oracle, and the CLI against `assoc --trait`."""
import ctypes as C

import numpy as np
import pytest

from oracle import assoc as A
from tests.test_assoc import check_parity, cli, make_cohort, run, small, write_table  # noqa: F401 (fixtures)

ERR_CUDA, ERR_ARG = -1, -2
HEAD_T = b"chromosome\tbegin\tend\ttrait\tn\tbeta\tse\tstat\tp\tstatus\n"


@pytest.fixture()
def multi(tmp_path):
    samples = ["a", "b", "c", "d", "e"]
    rows = [["chr1", "100", "120", "10", "12", "11", "NaN", "20", "22", "13", "14", "9", "9"],
            ["chr1", "200", "230", "5", "5", "6", "7", "NaN", "NaN", "8", "9", "4", "6"]]
    table = write_table(tmp_path / "t.tsv", samples, rows)
    ph = tmp_path / "p.tsv"
    # b: no bmi; d: no status; e: missing age (left out for every trait); f: only in the phenotype table
    ph.write_text("id\tstatus\tbmi\tage\na\t1\t22.5\t40\nb\t0\tNA\t51\nc\t1\t30.1\t33\nd\t\t27\t60\ne\t0\t25\tNaN\nf\t1\t20\t44\n")
    return tmp_path, table, str(ph)


# ------------------------------------------------------------------ the contract, restated on the oracle
def reference_traits(haps, Y, cov=None, model="linear", predictor_mode="sum"):
    """Y is samples x T with NaN where a sample has no value for a trait. Trait t is oracle/assoc.py's assoc_matrix
    over the samples where Y[:, t] is not NaN. -> dict of rows x T arrays."""
    haps = np.asarray(haps, np.float64)
    Y = np.asarray(Y, np.float64)
    ns, nt = Y.shape
    cov = None if cov is None else np.asarray(cov, np.float64).reshape(ns, -1)
    cols = []
    for t in range(nt):
        use = np.flatnonzero(~np.isnan(Y[:, t]))
        hc = np.ravel(np.column_stack([2 * use, 2 * use + 1]))
        cols.append(A.assoc_matrix(haps[:, hc], Y[use, t], None if cov is None else cov[use], model, predictor_mode))
    return {k: np.stack([c[k] for c in cols], axis=1) for k in cols[0]}


def test_reference_traits_is_assoc_matrix_per_trait():
    haps, y, cov = make_cohort(5, 40, 30, 2, 0.2, False)
    rng = np.random.default_rng(1)
    Y = np.column_stack([y, rng.normal(size=30), (rng.random(30) < 0.5).astype(float)])
    Y[rng.random(30) < 0.3, 1] = np.nan
    got = reference_traits(haps, Y, cov, "linear", "max")
    for t in range(3):
        use = ~np.isnan(Y[:, t])
        cols = np.ravel([[2 * i, 2 * i + 1] for i in np.flatnonzero(use)])
        ref = A.assoc_matrix(haps[:, cols], Y[use, t], cov[use], "linear", "max")
        for k in ref:
            assert np.array_equal(got[k][:, t], ref[k], equal_nan=True), (t, k)
    assert got["n"][:, 1].max() <= use.size


# ------------------------------------------------------------------ CLI without a device
def test_traits_usage_errors(cli, multi):
    d, table, ph = multi
    base = ["assoc", "--phenotype", ph, "--model", "linear"]
    cases = [
        (base + ["--trait", "status", "--traits", "status,bmi", table], b"cannot be used with '--trait"),
        (base + [table], b"--trait <COL>"),
        (base + ["--traits", "status,,bmi", table], b"an empty column name"),
        (base + ["--traits", "", table], b"an empty column name"),
        (base + ["--traits", "status,bmi,status", table], b"trait 'status' is listed twice"),
        (base + ["--traits", "status,bmi", "--covariates", "age,bmi", table], b"the trait 'bmi' is also listed as a covariate"),
    ]
    for args, msg in cases:
        r = run(cli, *args)
        assert r.returncode == 2 and r.stdout == b"", args
        assert msg in r.stderr, (args, r.stderr)
    r = run(cli, "assoc", "--help")
    assert r.returncode == 0 and b"--traits <A,B,...>" in r.stdout and b"chromosome begin end trait n beta se stat" in r.stdout


def test_traits_input_errors(cli, multi):
    d, table, ph = multi

    def fails(args, *msgs):
        r = run(cli, "assoc", "--phenotype", *args, table)
        assert r.returncode == 1, (args, r.stderr)
        for m in msgs:
            assert m.encode() in r.stderr, (args, m, r.stderr)

    p = d / "bad.tsv"
    p.write_text("id\tstatus\tbmi\na\t1\t22\nb\t0\theavy\n")
    fails([str(p), "--traits", "status,bmi", "--model", "linear"], "bad.tsv:3:", "column 'bmi'", "'heavy' is not a number")
    p.write_text("id\tstatus\tcase2\na\t1\t0\nb\t0\t2\n")
    fails([str(p), "--traits", "status,case2", "--model", "logistic"], "bad.tsv:3:", "column 'case2'", "'2' is not 0 or 1")
    fails([ph, "--traits", "status,height", "--model", "linear"], "p.tsv:1:", "column 'height' is not in the header")
    # a trait whose values are all on samples that are not in the table
    p.write_text("id\tstatus\tonly_f\na\t1\tNA\nb\t0\t\nf\t1\t3.5\n")
    fails([str(p), "--traits", "status,only_f", "--model", "linear"], "trait 'only_f': no sample is in both")


def test_traits_count_lines_equal_single_trait_runs(cli, multi):
    d, table, ph = multi
    r = run(cli, "assoc", "--phenotype", ph, "--traits", "status,bmi", "--model", "linear", "--covariates", "age", table)
    lines = [l for l in r.stderr.decode().splitlines() if l.startswith("assoc: trait")]
    assert len(lines) == 2
    for t, line in zip(("status", "bmi"), lines):
        s = run(cli, "assoc", "--phenotype", ph, "--trait", t, "--model", "linear", "--covariates", "age", table)
        single = s.stderr.decode().splitlines()[0]
        assert line == single.replace("assoc: ", f"assoc: trait '{t}': ", 1), (line, single)
    assert lines[0] == ("assoc: trait 'status': 3 samples used, 2 in the table only, 1 in the phenotype table only "
                        "(2 phenotype rows with a missing value left out)"), lines[0]


def test_traits_fail_loudly_without_gpu(cli, multi):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from inquistr_b200 import cohort
    from inquistr_b200.api import InqError
    with pytest.raises(InqError) as e:
        cohort.assoc_traits(np.ones((2, 8)), np.arange(8.0).reshape(4, 2))
    assert e.value.code == ERR_CUDA
    d, table, ph = multi
    r = run(cli, "assoc", "--phenotype", ph, "--traits", "status,bmi", "--model", "linear", table)
    assert r.returncode == 1 and r.stdout == HEAD_T and b"inquistr-b200:" in r.stderr


def test_traits_abi_argument_errors():
    """Returned before any device call, so they are the same with and without a GPU."""
    from inquistr_b200 import cohort
    from inquistr_b200.api import InqError
    haps = np.ones((3, 8))
    cases = [
        (dict(Y=np.array([[1.0, np.nan], [0.0, np.nan], [1.0, np.nan], [0.0, np.nan]])), "trait 1 has no value"),
        (dict(Y=np.array([[1.0, 2.0], [np.inf, 1.0], [1.0, 1.0], [0.0, 1.0]])), "trait 0 of sample 1 is not a finite number"),
        (dict(Y=np.array([[1.0, 2.0], [0.0, 1.0], [1.0, 1.0], [0.0, 1.0]]), model="logistic"), "logistic trait 1 of sample 0 is not 0 or 1"),
        (dict(Y=np.ones((4, 1)), cov=np.array([1.0, np.nan, 2.0, 3.0])), "covariate 0 of sample 1"),
        (dict(Y=np.ones((4, 1)), cov=np.ones((4, 31))), "31 covariates"),
    ]
    for kw, msg in cases:
        with pytest.raises(InqError) as e:
            cohort.assoc_traits(haps, **kw)
        assert e.value.code == ERR_ARG and msg in str(e.value), (kw, str(e.value))
    L = cohort._lib()
    z = np.zeros(64)
    rc = L.inq_assoc_traits(0, 0, 0, 3, 4, haps.ctypes.data, 0, z.ctypes.data, 0, None, *(z.ctypes.data,) * 4,
                            z.ctypes.data, z.ctypes.data, None, None)
    assert rc == ERR_ARG and b"no traits" in L.inq_cohort_last_error()
    rc = L.inq_assoc_traits(0, 0, 0, 1 << 62, 4, haps.ctypes.data, 64, z.ctypes.data, 0, None, *(z.ctypes.data,) * 4,
                            z.ctypes.data, z.ctypes.data, None, C.POINTER(C.c_float)())
    assert rc == -14                                                        # INQ_ERR_TOO_LARGE: rows x traits


# ------------------------------------------------------------------ GPU: bit-identity with the single-trait path
def traits_matrix(seed, samples, T, pattern, model, n_cov):
    """T traits: linear normal, or 0/1; pattern none (no NaN), shared (one NaN pattern for all) or distinct (per trait).
    Adds a constant linear trait / a one-class logistic trait, and a trait present in fewer samples than the rank."""
    rng = np.random.default_rng(seed)
    Y = (rng.random((samples, T)) < 0.4).astype(float) if model != "linear" else rng.normal(3, 1, (samples, T))
    if T > 1:
        Y[:, 1] = 0.0 if model != "linear" else 7.25
    if pattern == "shared":
        Y[rng.random(samples) < 0.25] = np.nan
    elif pattern == "distinct":
        for t in range(T):
            m = rng.random(samples) < 0.1 + 0.5 * rng.random()
            Y[m, t] = np.nan
        if T > 2:
            Y[:, 2] = np.nan
            few = rng.choice(samples, min(samples, max(1, n_cov)), replace=False)    # n <= rank
            Y[few, 2] = rng.integers(0, 2, len(few)) if model != "linear" else rng.normal(size=len(few))
    for t in range(T):                                            # every trait keeps a value
        if np.isnan(Y[:, t]).all():
            Y[0, t] = 1.0
    return Y


def check_identity(haps, Y, cov, model, pred, label):
    from inquistr_b200 import cohort
    got = cohort.assoc_traits(haps, Y, cov, model, pred)
    for t in range(Y.shape[1]):
        use = ~np.isnan(Y[:, t])
        cols = np.ravel([[2 * i, 2 * i + 1] for i in np.flatnonzero(use)])
        one = cohort.assoc(haps[:, cols], Y[use, t], None if cov is None else cov[use], model, pred)
        for k in ("beta", "se", "stat", "p", "n", "status", "n_iter"):
            assert np.array_equal(got[k][:, t], one[k], equal_nan=True), (label, t, k)
    return got


GRID = [(5, 0, 0.0), (268, 12, 0.3), (2100, 1, 0.0), (268, 30, 0.3), (268, 0, 0.3), (2100, 12, 0.3)]


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["linear", "logistic", "firth"])
@pytest.mark.parametrize("T", [1, 2, 5, 33])
@pytest.mark.parametrize("pattern", ["none", "shared", "distinct"])
def test_gpu_traits_bit_identical_to_single_trait(model, T, pattern):
    for gi, (samples, n_cov, missing) in enumerate(GRID):
        if model == "firth" and T == 33 and samples == 2100:
            continue                                               # the Firth cost of 33 x 2100 samples: covered by 268
        seed = 1000 + T * 17 + gi * 7 + len(pattern) + len(model)
        rows = 200 if samples < 2100 else 60
        haps, _, cov = make_cohort(seed, rows, samples, n_cov, missing, False)
        Y = traits_matrix(seed, samples, T, pattern, model, n_cov)
        for pred in ("sum", "max"):
            check_identity(haps, Y, cov if n_cov else None, model, pred, (model, T, pattern, samples, n_cov, missing, pred))


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["linear", "logistic", "firth"])
def test_gpu_traits_match_oracle(model):
    from inquistr_b200 import cohort
    haps, _, cov = make_cohort(77, 150, 120, 3, 0.2, False)
    Y = traits_matrix(77, 120, 5, "distinct", model, 3)
    for pred in ("sum", "max"):
        got = cohort.assoc_traits(haps, Y, cov, model, pred)
        ref = reference_traits(haps, Y, cov, model, pred)
        for t in range(Y.shape[1]):
            if model == "linear" and t == 1:
                continue                       # constant trait: beta is 0 up to rounding, with no relative precision
            g = {k: got[k][:, t] for k in ("beta", "se", "stat", "p", "n", "status", "n_iter")}
            r = {k: ref[k][:, t] for k in ref}
            check_parity(g, r, "logistic" if model != "linear" else "linear", (model, pred, t))


# ------------------------------------------------------------------ GPU: the CLI against `assoc --trait`
def cli_tables(tmp_path, gz, model):
    rng = np.random.default_rng(41 + gz)
    samples = [f"S{i}" for i in range(120)]
    haps, _, _ = make_cohort(98, 300, len(samples), 0, 0.1, False)
    text_rows = [[f"chr{1 + i // 100}", str(1000 + 50 * i), str(1030 + 50 * i)] + ["NaN" if np.isnan(v) else repr(float(v)) for v in haps[i]]
                 for i in range(len(haps))]
    table = write_table(tmp_path / ("c.tsv.gz" if gz else "c.tsv"), samples, text_rows)
    ph_samples = samples[10:] + [f"X{i}" for i in range(7)]
    lines = ["sample\tage\tA\tB\tpc1\tC"]
    for s in ph_samples:
        tv = [str(int(rng.random() < 0.45)) if model != "linear" else f"{rng.normal(3, 1):.6f}" for _ in range(3)]
        tv = ["NA" if rng.random() < 0.1 else v for v in tv]
        age = "" if rng.random() < 0.05 else f"{rng.normal(50, 12):.2f}"
        lines.append(f"{s}\t{age}\t{tv[0]}\t{tv[1]}\t{rng.normal():.5f}\t{tv[2]}")
    ph = tmp_path / "pheno.tsv"
    ph.write_text("\n".join(lines) + "\n")
    return table, str(ph)


@pytest.mark.gpu
@pytest.mark.parametrize("gz", [False, True])
@pytest.mark.parametrize("model", ["linear", "logistic", "firth"])
def test_gpu_cli_traits_equal_single_trait_runs(cli, tmp_path, gz, model):
    table, ph = cli_tables(tmp_path, gz, model)
    flags = ["--model", "logistic", "--firth"] if model == "firth" else ["--model", model]
    common = [*flags, "--covariates", "age,pc1", "--predictor", "max" if gz else "sum", table]
    r = run(cli, "assoc", "--phenotype", ph, "--traits", "A,B,C", *common)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.decode().split("\n")
    assert lines[0] + "\n" == HEAD_T.decode() and lines[-1] == ""
    body = [l.split("\t") for l in lines[1:-1]]
    assert [b[3] for b in body[:6]] == ["A", "B", "C"] * 2
    counts = r.stderr.decode().splitlines()
    for i, t in enumerate("ABC"):
        s = run(cli, "assoc", "--phenotype", ph, "--trait", t, *common)
        assert s.returncode == 0, s.stderr
        mine = "".join("\t".join(b[:3] + b[4:]) + "\n" for b in body if b[3] == t)
        assert mine == s.stdout.decode().split("\n", 1)[1], t
        assert counts[i] == s.stderr.decode().splitlines()[0].replace("assoc: ", f"assoc: trait '{t}': ", 1)


@pytest.mark.gpu
def test_gpu_cli_traits_rows_before_a_bad_line(cli, multi):
    d, table, ph = multi
    good = open(table).read()
    for name, extra in (("short.tsv", "chr2\t5\t9\t1\t2\n"), ("bad.tsv", "chr2\t5\t9\t1\t2\t3\t4\t5\tx7\t1\t2\t3\t4\n")):
        p = d / name
        p.write_text(good + extra + "chr3\t1\t2\t1\t2\t3\t4\t5\t6\t7\t8\t9\t10\n")
        r = run(cli, "assoc", "--phenotype", ph, "--traits", "status,bmi", "--model", "linear", str(p))
        assert r.returncode == 1 and f"{name}:4:".encode() in r.stderr, r.stderr
        for t in ("status", "bmi"):
            s = run(cli, "assoc", "--phenotype", ph, "--trait", t, "--model", "linear", str(p))
            assert s.returncode == 1 and s.stderr.splitlines()[-1] == r.stderr.splitlines()[-1]
            rows = [l.split("\t") for l in r.stdout.decode().split("\n")[1:-1]]
            mine = "".join("\t".join(b[:3] + b[4:]) + "\n" for b in rows if b[3] == t)
            assert mine == s.stdout.decode().split("\n", 1)[1]
            assert mine.count("\n") == 2
