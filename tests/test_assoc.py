"""`assoc`: per-locus association of STR length with a phenotype (DESIGN.md 5e).
CPU: the numpy oracle (oracle/assoc.py) pinned by closed-form answers and scipy, and the CLI's error paths.
GPU: inq_assoc (include/inqcohort.h) against the oracle over a grid of shapes, and the CLI end to end."""
import gzip
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

from oracle import assoc as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------ oracle, pinned independently of it
def test_linear_closed_form():
    r = A.fit_locus([1, 2, 3, 4, 5], [2, 4, 5, 4, 5])
    assert r["status"] == A.OK and r["n"] == 5
    assert r["beta"] == pytest.approx(0.6, rel=1e-12)
    assert r["se"] == pytest.approx(np.sqrt(0.08), rel=1e-12) and r["se"] == pytest.approx(0.28284271, abs=1e-8)
    assert r["stat"] == pytest.approx(2.12132034, abs=1e-8)
    assert r["p"] == pytest.approx(0.12402706, abs=1e-8)


def test_linear_matches_linregress():
    rng = np.random.default_rng(3)
    for _ in range(50):
        n = int(rng.integers(4, 300))
        x = rng.gamma(2, 15, n)
        y = 0.02 * x + rng.normal(size=n)
        x[rng.random(n) < 0.2] = np.nan
        use = ~np.isnan(x)
        if use.sum() < 3:
            continue
        ref = stats.linregress(x[use], y[use])
        r = A.fit_locus(x, y)
        assert r["status"] == A.OK and r["n"] == use.sum()
        assert r["beta"] == pytest.approx(ref.slope, rel=1e-9)
        assert r["se"] == pytest.approx(ref.stderr, rel=1e-9)
        assert r["p"] == pytest.approx(ref.pvalue, rel=1e-7)


def test_logistic_two_by_two_table():
    # x = 1: 12 cases / 5 controls, x = 0: 7 cases / 14 controls
    x = np.r_[np.ones(17), np.zeros(21)]
    y = np.r_[np.ones(12), np.zeros(5), np.ones(7), np.zeros(14)]
    r = A.fit_locus(x, y, model="logistic")
    assert r["status"] == A.OK and r["n"] == 38 and r["n_iter"] == 4
    assert r["beta"] == pytest.approx(np.log(12 * 14 / (5 * 7)), rel=1e-9)
    assert r["beta"] == pytest.approx(1.56861592, abs=1e-8)
    # The se comes from the weights of the last weighted solve (one iteration before the returned beta), as
    # summary.glm reports it, so it meets the closed form sqrt(1/12 + 1/5 + 1/7 + 1/14) only to the convergence level.
    assert r["se"] == pytest.approx(np.sqrt(1 / 12 + 1 / 5 + 1 / 7 + 1 / 14), rel=1e-6)
    assert r["se"] == pytest.approx(0.70542118, rel=1e-6)
    assert r["p"] == pytest.approx(0.02617142, rel=1e-5)


def test_logistic_score_is_zero_at_the_solution():
    rng = np.random.default_rng(11)
    for _ in range(20):
        n = 200
        cov = np.column_stack([rng.normal(50, 15, n), rng.integers(0, 2, n), rng.normal(size=n)])
        x = rng.gamma(2, 15, n)
        eta = -1 + 0.02 * (x - 30) + 0.3 * cov[:, 2]
        y = (rng.random(n) < 1 / (1 + np.exp(-eta))).astype(float)
        r = A.fit_locus(x, y, cov, "logistic")
        assert r["status"] == A.OK and r["coef"][-1] == r["beta"]
        X = np.column_stack([np.ones(n), cov, x])
        score = X.T @ (y - A.linkinv(X @ r["coef"]))
        assert np.all(np.abs(score) <= 1e-6 * np.abs(X).sum(axis=0)), score


def test_constant_covariate_is_dropped():
    rng = np.random.default_rng(5)
    n = 80
    x = rng.gamma(2, 15, n)
    x[:10] = np.nan
    age = rng.normal(50, 10, n)
    const = np.full(n, 3.7)
    const[:10] = 99.0                                   # constant over the samples used (x missing on the others)
    for model, y in (("linear", rng.normal(size=n)), ("logistic", (rng.random(n) < 0.4).astype(float))):
        a = A.fit_locus(x, y, np.column_stack([age, const]), model)
        b = A.fit_locus(x, y, age[:, None], model)
        assert a["status"] == b["status"] == A.OK
        for k in ("beta", "se", "stat", "p"):
            assert a[k] == pytest.approx(b[k], rel=1e-9), k


def test_constant_x_is_singular():
    y = np.arange(10.0)
    for model, yy in (("linear", y), ("logistic", (y > 4).astype(float))):
        r = A.fit_locus(np.full(10, 31.0), yy, None, model)
        assert r["status"] == A.SINGULAR and np.isnan(r["beta"]) and np.isnan(r["p"])


def test_separation_is_flagged():
    x = np.r_[np.arange(10.0), np.arange(10.0) + 20]
    y = np.r_[np.zeros(10), np.ones(10)]
    r = A.fit_locus(x, y, None, "logistic")
    assert r["status"] in (A.SEPARATION, A.NO_CONVERGENCE)
    assert np.isfinite(r["beta"]) and r["beta"] > 0
    # the clamps keep mu inside (0, 1) and mu_eta positive far outside +-30
    assert 0 < A.linkinv(np.array([-1e3]))[0] < 1e-15 and 1 - 1e-15 < A.linkinv(np.array([1e3]))[0] < 1
    assert A.mu_eta(np.array([40.0]))[0] == np.finfo(float).eps


def test_empty_and_one_class_loci():
    y = np.r_[np.zeros(5), np.ones(5)]
    r = A.fit_locus(np.full(10, np.nan), y)
    assert r["status"] == A.FEW_SAMPLES and r["n"] == 0 and np.isnan(r["beta"])
    x = np.r_[np.full(5, np.nan), np.arange(5.0)]                # only cases have a call
    r = A.fit_locus(x, y, None, "logistic")
    assert r["status"] == A.FEW_SAMPLES and r["n"] == 5
    r = A.fit_locus(np.r_[3.0, np.full(9, np.nan)], y)            # one sample: n <= rank
    assert r["status"] == A.FEW_SAMPLES and r["n"] == 1


def test_predictor_modes():
    h1 = np.array([1.0, np.nan, np.nan, 4.0])
    h2 = np.array([2.0, 5.0, np.nan, 3.0])
    assert np.array_equal(A.predictor(h1, h2, "sum"), [3.0, np.nan, np.nan, 7.0], equal_nan=True)
    assert np.array_equal(A.predictor(h1, h2, "max"), [2.0, 5.0, np.nan, 4.0], equal_nan=True)


# ------------------------------------------------------------------ CLI
@pytest.fixture(scope="module")
def cli():
    from inquistr_b200 import build
    build.build_libinqcall()
    return build.build_cli()


def run(cli, *args):
    return subprocess.run([cli, *args], capture_output=True, timeout=600)


def write_table(path, samples, rows):
    head = "chromosome\tbegin\tend\t" + "\t".join(f"{s}_H1\t{s}_H2" for s in samples)
    text = head + "\n" + "".join("\t".join(r) + "\n" for r in rows)
    if str(path).endswith(".gz"):
        with gzip.open(path, "wt") as f:
            f.write(text)
    else:
        open(path, "w").write(text)
    return str(path)


@pytest.fixture()
def small(tmp_path):
    samples = ["a", "b", "c", "d"]
    rows = [["chr1", "100", "120", "10", "12", "11", "NaN", "20", "22", "13", "14"],
            ["chr1", "200", "230", "5", "5", "6", "7", "NaN", "NaN", "8", "9"]]
    table = write_table(tmp_path / "t.tsv", samples, rows)
    ph = tmp_path / "p.tsv"
    ph.write_text("id\tstatus\tage\tsex\na\t1\t40\t0\nb\t0\t51\t1\nc\t1\t33\t1\nd\t0\t60\t0\n")
    return tmp_path, table, str(ph)


def test_cli_help_and_usage_errors(cli, small):
    d, table, ph = small
    r = run(cli, "assoc", "--help")
    assert r.returncode == 0 and b"[possible values: linear, logistic]" in r.stdout and b"[possible values: sum, max]" in r.stdout
    r = run(cli, "--help")
    assert r.returncode == 0 and b"assoc" in r.stdout
    base = ["assoc", "--phenotype", ph, "--trait", "status"]
    cases = [
        (base + ["--model", "linear", "--covariates", ",".join(f"c{i}" for i in range(31)), table], b"at most 30"),
        (base + ["--model", "linear", "--covariates", "age,status", table], b"also listed as a covariate"),
        (base + ["--model", "probit", table], b"invalid value 'probit' for '--model"),
        (base + ["--model", "linear", "--predictor", "min", table], b"invalid value 'min' for '--predictor"),
        (["assoc", "--phenotype", ph, "--model", "linear", table], b"--trait <COL>"),
        (["assoc", "--trait", "status", "--model", "linear", table], b"--phenotype <TSV>"),
        (base + [table], b"--model <MODEL>"),
        (base + ["--model", "linear"], b"<COMBINED>"),
    ]
    for args, msg in cases:
        r = run(cli, *args)
        assert r.returncode == 2 and r.stdout == b"", args
        assert msg in r.stderr, (args, r.stderr)


def test_cli_input_errors(cli, small):
    d, table, ph = small
    base = ["--phenotype", ph, "--trait", "status", "--model", "linear"]

    def fails(args, *msgs):
        r = run(cli, "assoc", *args)
        assert r.returncode == 1, (args, r.stderr)
        for m in msgs:
            assert m.encode() in r.stderr, (args, m, r.stderr)
        return r

    # combined table
    odd = d / "odd.tsv"
    odd.write_text("chromosome\tbegin\tend\ta_H1\ta_H2\tb_H1\n")
    fails(base + [str(odd)], "odd.tsv:1:", "pairs")
    mism = d / "mism.tsv"
    mism.write_text("chromosome\tbegin\tend\ta_H1\tb_H2\n")
    fails(base + [str(mism)], "mism.tsv:1:", "'a_H1', 'b_H2'")
    dup = write_table(d / "dup.tsv", ["a", "b", "a"], [])
    fails(base + [dup], "dup.tsv:1:", "sample 'a' appears twice")
    # the bad row comes first: nothing is pending, so the message is the same with or without a device
    head = open(table).read().split("\n")[0]
    short = d / "short.tsv"
    short.write_text(head + "\nchr2\t5\t9\t1\t2\n")
    r = fails(base + [str(short)], "short.tsv:2:", "2 values, the header has 8")
    assert r.stdout == b"chromosome\tbegin\tend\tn\tbeta\tse\tstat\tp\tstatus\n"
    bad = d / "bad.tsv"
    bad.write_text(head + "\nchr2\t5\t9\t1\t2\t3\t4\t5\tx7\t1\t2\n")
    fails(base + [str(bad)], "bad.tsv:2:", "column 9: 'x7' is not a number")
    fails(base + [str(d / "missing.tsv")], "missing.tsv")
    # phenotype table
    fails(["--phenotype", ph, "--trait", "height", "--model", "linear", table], "p.tsv:1:", "column 'height' is not in the header")
    fails(base + ["--covariates", "age,pc1", table], "p.tsv:1:", "column 'pc1'")
    p2 = d / "p2.tsv"
    p2.write_text("id\tstatus\tage\na\t1\t40\nb\t0\tforty\n")
    fails(["--phenotype", str(p2), "--trait", "status", "--model", "linear", "--covariates", "age", table], "p2.tsv:3:", "column 'age'", "'forty' is not a number")
    p3 = d / "p3.tsv"
    p3.write_text("id\tstatus\na\t1\nb\t0\na\t1\n")
    fails(["--phenotype", str(p3), "--trait", "status", "--model", "linear", table], "p3.tsv:4:", "column 'id'", "sample 'a' appears twice")
    p4 = d / "p4.tsv"
    p4.write_text("id\tstatus\na\t1\nb\t2\n")
    fails(["--phenotype", str(p4), "--trait", "status", "--model", "logistic", table], "p4.tsv:3:", "column 'status'", "'2' is not 0 or 1")
    p5 = d / "p5.tsv"
    p5.write_text("id\tstatus\nx\t1\ny\t0\n")
    fails(["--phenotype", str(p5), "--trait", "status", "--model", "linear", table], "no sample is in both")


def test_cli_sample_counts(cli, small):
    d, table, ph = small
    p = d / "partial.tsv"
    # a: used; b: missing trait; d: NA covariate; e, f: only in the phenotype table; c: only in the table
    p.write_text("id\tstatus\tage\na\t1\t40\nb\tNA\t51\nd\t0\t\ne\t1\t20\nf\t0\tNaN\n")
    r = run(cli, "assoc", "--phenotype", str(p), "--trait", "status", "--model", "linear", "--covariates", "age", table)
    line = r.stderr.decode().splitlines()[0]
    assert line == "assoc: 1 samples used, 3 in the table only, 2 in the phenotype table only (3 phenotype rows with a missing value left out)", line


def test_assoc_fails_loudly_without_gpu(cli, small):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from inquistr_b200 import cohort
    from inquistr_b200.api import InqError
    with pytest.raises(InqError) as e:
        cohort.assoc(np.ones((2, 8)), np.arange(4.0))
    assert e.value.code == -1                                            # INQ_ERR_CUDA: no CPU implementation behind the ABI
    d, table, ph = small
    r = run(cli, "assoc", "--phenotype", ph, "--trait", "status", "--model", "linear", table)
    assert r.returncode == 1 and r.stdout == b"chromosome\tbegin\tend\tn\tbeta\tse\tstat\tp\tstatus\n" and b"inquistr-b200:" in r.stderr


# ------------------------------------------------------------------ GPU parity through the C ABI
def make_cohort(seed, rows, samples, n_cov, missing, logistic):
    """Heavy-tailed lengths, some constant loci, covariates of mixed scale (age, sex, PCs), a seeded trait."""
    rng = np.random.default_rng(seed)
    haps = np.round(rng.gamma(2.0, 12.0, (rows, 2 * samples)) * 2) / 2
    big = rng.random((rows, 2 * samples)) < 0.03
    haps[big] = rng.integers(200, 3000, big.sum())
    const = rng.random(rows) < 0.05
    haps[const] = 30.0
    if missing:
        haps[rng.random(haps.shape) < missing] = np.nan
    cov = np.empty((samples, n_cov))
    for c in range(n_cov):
        kind = c % 3
        cov[:, c] = rng.normal(50, 15, samples) if kind == 0 else (rng.integers(0, 2, samples) if kind == 1 else rng.normal(0, 1, samples))
    lin = 0.3 * (cov[:, 2] if n_cov > 2 else 0) + rng.normal(size=samples)
    y = (rng.random(samples) < 1 / (1 + np.exp(-(lin - 0.4)))).astype(float) if logistic else 5 + 0.01 * (cov[:, 0] if n_cov else 0) + lin
    return haps, y, cov


def close(a, b, rtol):
    return np.abs(a - b) <= rtol * np.abs(b)


def check_parity(got, ref, model, label):
    st, gs = ref["status"], got["status"].astype(np.int64)
    bad = np.flatnonzero(gs != st)                                              # the status matches on every locus
    assert len(bad) == 0, (label, [(int(i), int(gs[i]), int(st[i]), int(got["n_iter"][i]), int(ref["n_iter"][i])) for i in bad[:10]])
    assert np.array_equal(got["n"], ref["n"]), label
    na = (gs == A.FEW_SAMPLES) | (gs == A.SINGULAR)
    for k in ("beta", "se", "stat", "p"):
        assert np.isnan(got[k][na]).all(), (label, k)
    # Values are compared where the fit is ok: a separated or unconverged logistic fit walks beta towards infinity,
    # and two correct implementations agree on the status there but not on where the walk stopped.
    ok = (st == A.OK) & (gs == A.OK)
    if model == "logistic":
        same = ok & (got["n_iter"] == ref["n_iter"])
        off = ok & (got["n_iter"] != ref["n_iter"])
        assert np.all(np.abs(got["n_iter"][off].astype(int) - ref["n_iter"][off]) == 1), label
        assert off.sum() <= 0.001 * len(st), (label, off.sum())                 # at most 0.1 % of the loci
        gb, rb, rs = got["beta"][off], ref["beta"][off], ref["se"][off]
        assert np.all(np.abs(gb - rb) <= 1e-6 * (np.abs(rb) + rs)), label
        ok = same
    tol = 1e-9
    # A coefficient near zero has no relative precision of its own: its rounding error scales with se, so beta and the
    # statistic are held to the tolerance of (|value| + its standard scale) rather than of |value| alone.
    b, s = ref["beta"][ok], ref["se"][ok]
    assert np.all(np.abs(got["beta"][ok] - b) <= tol * (np.abs(b) + s)), (label, np.max(np.abs(got["beta"][ok] - b) / (np.abs(b) + s) / tol))
    assert np.all(np.abs(got["se"][ok] - s) <= tol * s), (label, np.max(np.abs(got["se"][ok] / s - 1) / tol))
    t = ref["stat"][ok]
    assert np.all(np.abs(got["stat"][ok] - t) <= tol * (np.abs(t) + 1)), label
    gp, rp = np.maximum(got["p"][ok], 1e-300), np.maximum(ref["p"][ok], 1e-300)
    assert np.all(np.abs(np.log10(gp) - np.log10(rp)) <= 1e-6), (label, np.max(np.abs(np.log10(gp) - np.log10(rp))))


@pytest.mark.gpu
@pytest.mark.parametrize("rows,samples", [(1, 5), (1000, 268), (300, 2100), (5000, 40)])
@pytest.mark.parametrize("n_cov", [0, 1, 12, 30])
@pytest.mark.parametrize("missing", [0.0, 0.3])
@pytest.mark.parametrize("model", ["linear", "logistic"])
def test_gpu_assoc_matches_oracle(rows, samples, n_cov, missing, model):
    from inquistr_b200 import cohort
    seed = rows * 7 + samples * 13 + n_cov * 101 + int(missing * 10) + (model == "logistic") * 5
    haps, y, cov = make_cohort(seed, rows, samples, n_cov, missing, model == "logistic")
    for pred in ("sum", "max"):
        got = cohort.assoc(haps, y, cov if n_cov else None, model, pred)
        ref = A.assoc_matrix(haps, y, cov if n_cov else None, model, pred)            # every locus
        check_parity(got, ref, model, (rows, samples, n_cov, missing, model, pred))


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["linear", "logistic"])
def test_gpu_assoc_edge_loci(model):
    from inquistr_b200 import cohort
    rng = np.random.default_rng(21)
    ns = 60
    y = (rng.random(ns) < 0.5).astype(float) if model == "logistic" else rng.normal(size=ns)
    y[:2] = [0.0, 1.0]
    age = rng.normal(50, 10, ns)
    flag = np.where(np.arange(ns) < 20, 1.0, 0.0)                 # constant on samples 20.. (aliased where 0..19 miss)
    cov = np.column_stack([age, flag])
    rows = []
    rows.append(np.full(2 * ns, 25.0))                                  # constant x: singular
    h = rng.gamma(2, 12, 2 * ns)
    h[:40] = np.nan                                                      # samples 0..19 missing: flag constant
    rows.append(h)
    # separates the classes (logistic), cases spread over 80..160: far cases pass the +-30 clamps before convergence
    sep = np.where(np.repeat(y, 2) > 0, 40.0 + 40.0 * rng.random(2 * ns), 10.0 + rng.random(2 * ns))
    rows.append(sep)
    one = np.full(2 * ns, np.nan)
    one[10:12] = [12.0, 13.0]                                            # one sample
    rows.append(one)
    rows.append(np.full(2 * ns, np.nan))                                 # all NaN
    haps = np.stack(rows)
    for pred in ("sum", "max"):
        got = cohort.assoc(haps, y, cov, model, pred)
        ref = A.assoc_matrix(haps, y, cov, model, pred)
        check_parity({k: v for k, v in got.items() if k != "ms_kernel"}, ref, model, (model, pred))
        assert got["status"][0] == A.SINGULAR
        assert got["status"][1] == A.OK
        assert list(got["status"][3:]) == [A.FEW_SAMPLES, A.FEW_SAMPLES] and list(got["n"][3:]) == [1, 0]
        if model == "logistic":
            assert got["status"][2] in (A.SEPARATION, A.NO_CONVERGENCE)
    # the aliased covariate (constant over the samples used) leaves the fit without it
    a = cohort.assoc(haps[1:2], y, cov, model)
    b = cohort.assoc(haps[1:2], y, age[:, None], model)
    for k in ("beta", "se", "p"):
        assert a[k][0] == pytest.approx(b[k][0], rel=1e-9)


# ------------------------------------------------------------------ GPU, CLI end to end
def parse_output(text):
    lines = text.split("\n")
    assert lines[0] == "chromosome\tbegin\tend\tn\tbeta\tse\tstat\tp\tstatus" and lines[-1] == ""
    return [l.split("\t") for l in lines[1:-1]]


@pytest.mark.gpu
@pytest.mark.parametrize("gz", [False, True])
@pytest.mark.parametrize("model", ["linear", "logistic"])
def test_gpu_cli_end_to_end(cli, tmp_path, gz, model):
    rng = np.random.default_rng(31 + gz)
    samples = [f"S{i}" for i in range(150)]
    rows = 700
    haps, _, _ = make_cohort(99, rows, len(samples), 0, 0.1, False)
    loci = [(f"chr{1 + i // 300}", 1000 + 50 * i, 1030 + 50 * i) for i in range(rows)]
    text_rows = [[c, str(b), str(e)] + ["NaN" if np.isnan(v) else repr(float(v)) for v in haps[i]] for i, (c, b, e) in enumerate(loci)]
    table = write_table(tmp_path / ("c.tsv.gz" if gz else "c.tsv"), samples, text_rows)
    # phenotype: 20 table samples absent, 15 extra samples, NA in the trait and in a covariate
    ph_samples = samples[20:] + [f"X{i}" for i in range(15)]
    rng.shuffle(ph_samples)
    lines = ["sample\tage\ttrait\tpc1\tsex"]
    for s in ph_samples:
        trait = str(int(rng.random() < 0.45)) if model == "logistic" else f"{rng.normal(3, 1):.6f}"
        age = f"{rng.normal(50, 12):.2f}"
        if rng.random() < 0.05:
            trait = "NA"
        if rng.random() < 0.05:
            age = ""
        lines.append(f"{s}\t{age}\t{trait}\t{rng.normal():.5f}\t{rng.integers(0, 2)}")
    ph = tmp_path / "pheno.tsv"
    ph.write_text("\n".join(lines) + "\n")
    for pred in ("sum", "max"):
        r = run(cli, "assoc", "--phenotype", str(ph), "--trait", "trait", "--model", model, "--covariates", "age,pc1,sex",
                "--predictor", pred, table)
        assert r.returncode == 0, r.stderr
        out = parse_output(r.stdout.decode())
        assert [tuple(o[:3]) for o in out] == [(c, str(b), str(e)) for c, b, e in loci]
        # the oracle on the same selection of samples, in table order
        pht = {l.split("\t")[0]: l.split("\t")[1:] for l in lines[1:]}
        used = [i for i, s in enumerate(samples) if s in pht and "" not in pht[s] and "NA" not in pht[s]]
        y = np.array([float(pht[samples[i]][1]) for i in used])
        cov = np.array([[float(pht[samples[i]][0]), float(pht[samples[i]][2]), float(pht[samples[i]][3])] for i in used])
        cols = np.ravel([[2 * i, 2 * i + 1] for i in used])
        ref = A.assoc_matrix(haps[:, cols], y, cov, model, pred)
        assert r.stderr.decode().startswith(f"assoc: {len(used)} samples used, {len(samples) - len(used)} in the table only, 15 in the phenotype table only")
        got = {k: np.array([float(o[j]) for o in out]) for j, k in ((4, "beta"), (5, "se"), (6, "stat"), (7, "p"))}
        got["n"] = np.array([int(o[3]) for o in out])
        got["status"] = np.array([A.STATUS_NAMES.index(o[8]) for o in out])
        got["n_iter"] = ref["n_iter"]                                   # not printed: iteration differences show in the values
        check_parity(got, ref, model, (gz, model, pred))


@pytest.mark.gpu
def test_gpu_cli_prints_rows_before_a_bad_line(cli, small):
    d, table, ph = small
    for name, extra in (("short.tsv", "chr2\t5\t9\t1\t2\n"), ("bad.tsv", "chr2\t5\t9\t1\t2\t3\t4\t5\tx7\t1\t2\n")):
        p = d / name
        p.write_text(open(table).read() + extra + "chr3\t1\t2\t1\t2\t3\t4\t5\t6\t7\t8\n")
        r = run(cli, "assoc", "--phenotype", ph, "--trait", "status", "--model", "linear", str(p))
        assert r.returncode == 1 and f"{name}:4:".encode() in r.stderr, r.stderr
        out = parse_output(r.stdout.decode())
        assert [o[:3] for o in out] == [["chr1", "100", "120"], ["chr1", "200", "230"]]
