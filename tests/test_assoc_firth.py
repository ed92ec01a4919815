"""`assoc --firth`: Firth-penalized logistic regression with a penalized likelihood-ratio test (DESIGN.md 5e, Firth).
CPU: the numpy restatement (oracle/assoc.py, model "firth") pinned by the closed forms of 2x2 tables, its modified
score and its invariance under a change of x's scale; the CLI's and the ABI's error paths.
GPU: inq_assoc with INQ_ASSOC_FIRTH against the restatement over a grid of shapes with case-only expansions, the
closed forms through the kernel, edge loci, and the CLI end to end."""
import subprocess

import numpy as np
import pytest

from oracle import assoc as A
from tests.test_assoc import make_cohort, parse_output, run, write_table

TABLES = [(12, 5, 7, 14), (9, 0, 4, 11), (3, 0, 0, 8), (40, 0, 0, 300), (1, 0, 30, 237)]


def two_by_two(a, b, c, d):
    """x = 1000 on a cases and b controls, 0 on c cases and d controls -> (x, y)."""
    x = np.r_[np.ones(a + b), np.zeros(c + d)] * 1000.0
    y = np.r_[np.ones(a), np.zeros(b), np.ones(c), np.zeros(d)]
    return x, y


def closed_form(a, b, c, d):
    """Firth fit of a 2x2 table: (beta per unit of x in {0, 1}, its se, the penalized likelihood ratio)."""
    n1, n0 = a + b, c + d
    m1, m0 = (a + 0.5) / (n1 + 1), (c + 0.5) / (n0 + 1)
    beta = np.log((a + 0.5) * (d + 0.5) / ((b + 0.5) * (c + 0.5)))
    se = np.sqrt(1 / (n1 * m1 * (1 - m1)) + 1 / (n0 * m0 * (1 - m0)))

    def ll(k, n, m):
        return k * np.log(m) + (n - k) * np.log(1 - m)

    d_full = -2 * (ll(a, n1, m1) + ll(c, n0, m0)) - np.log(n1 * m1 * (1 - m1) * n0 * m0 * (1 - m0))
    mu0 = (a + c + 1) / (n1 + n0 + 2)
    d_null = -2 * ll(a + c, n1 + n0, mu0) - np.log(n1 * n0 * (mu0 * (1 - mu0)) ** 2)
    return beta, se, d_null - d_full


def check_closed_form(r, table):
    beta, se, lr = closed_form(*table)
    assert r["status"] == A.OK, table
    assert abs(r["beta"] * 1000 - beta) <= 1e-5 * se, (table, r["beta"] * 1000, beta)
    assert r["se"] * 1000 == pytest.approx(se, rel=1e-5), table
    assert abs(r["stat"] - lr) <= 1e-8 * (1 + lr), (table, r["stat"], lr)


def separated_edge_loci(ns=60):
    """The loci of test_assoc.py's edge test: constant x, covariate aliased by missing calls, separated classes,
    one sample, all NaN."""
    rng = np.random.default_rng(21)
    y = (rng.random(ns) < 0.5).astype(float)
    y[:2] = [0.0, 1.0]
    age = rng.normal(50, 10, ns)
    flag = np.where(np.arange(ns) < 20, 1.0, 0.0)
    cov = np.column_stack([age, flag])
    rows = [np.full(2 * ns, 25.0)]
    h = rng.gamma(2, 12, 2 * ns)
    h[:40] = np.nan
    rows.append(h)
    rows.append(np.where(np.repeat(y, 2) > 0, 40.0 + 40.0 * rng.random(2 * ns), 10.0 + rng.random(2 * ns)))
    one = np.full(2 * ns, np.nan)
    one[10:12] = [12.0, 13.0]
    rows.append(one)
    rows.append(np.full(2 * ns, np.nan))
    return np.stack(rows), y, cov


# ------------------------------------------------------------------ the restatement, pinned independently of it
def test_two_by_two_closed_forms():
    for table in TABLES:
        x, y = two_by_two(*table)
        check_closed_form(A.fit_locus(x, y, model="firth"), table)
    r = A.fit_locus(*two_by_two(*TABLES[0]), model="firth")
    assert r["stat"] == pytest.approx(5.061824, abs=1e-6) and r["p"] == pytest.approx(0.0244585, abs=1e-7)


def test_modified_score_is_zero_at_the_solution():
    rng = np.random.default_rng(13)
    for i in range(12):
        n = 150
        cov = np.column_stack([rng.normal(50, 15, n), rng.integers(0, 2, n), rng.normal(size=n)])
        x = rng.gamma(2, 15, n)
        y = (rng.random(n) < 1 / (1 + np.exp(-(-1.5 + 0.3 * cov[:, 2])))).astype(float)
        if i % 2:
            x[np.flatnonzero(y)[:3]] = 2000.0 + 1000 * i                    # case-only expansions: separated
        r = A.fit_locus(x, y, cov, "firth")
        assert r["status"] == A.OK and r["stat"] >= 0 and np.isfinite(r["beta"])
        X = np.column_stack([np.ones(n), cov, x])
        mu = A.linkinv(X @ r["coef"])
        w = mu * (1 - mu)
        info = X.T @ (w[:, None] * X)
        h = w * np.einsum("ij,ij->i", X, np.linalg.solve(info, X.T).T)
        score = X.T @ (y - mu + h * (0.5 - mu))
        hess = X.T @ ((w * (1 + h))[:, None] * X)
        # converged: U*' H^-1 U* < 1e-10, so |U*_j| <= 1e-5 sqrt(H_jj) (Cauchy-Schwarz); 10 % slack for rounding
        assert np.all(np.abs(score) <= 1.1e-5 * np.sqrt(np.diag(hess))), (i, score)


def test_invariant_under_a_change_of_scale_of_x():
    rng = np.random.default_rng(17)
    n = 120
    cov = rng.normal(size=(n, 2))
    x = rng.gamma(2, 0.5, n)
    y = (rng.random(n) < 0.3).astype(float)
    x[np.flatnonzero(y)[:2]] = 9.0
    a = A.fit_locus(x, y, cov, "firth")
    b = A.fit_locus(1000 * x + 7, y, cov, "firth")
    assert a["status"] == b["status"] == A.OK and a["n_iter"] == b["n_iter"]
    assert b["stat"] == pytest.approx(a["stat"], rel=1e-7) and b["p"] == pytest.approx(a["p"], rel=1e-6)
    assert b["beta"] * 1000 == pytest.approx(a["beta"], rel=1e-7) and b["se"] * 1000 == pytest.approx(a["se"], rel=1e-7)


def test_separated_locus_gets_a_finite_answer():
    haps, y, cov = separated_edge_loci()
    for pred in ("sum", "max"):
        x = A.predictor(haps[2, 0::2], haps[2, 1::2], pred)
        ml = A.fit_locus(x, y, cov, "logistic")
        assert ml["status"] in (A.SEPARATION, A.NO_CONVERGENCE)
        r = A.fit_locus(x, y, cov, "firth")
        assert r["status"] == A.OK and np.isfinite(r["beta"]) and r["beta"] > 0 and np.isfinite(r["se"])
        assert 0 < r["p"] < 1e-6                                          # a separated locus is strong evidence
    ref = A.assoc_matrix(haps, y, cov, "firth")
    assert list(ref["status"]) == [A.SINGULAR, A.OK, A.OK, A.FEW_SAMPLES, A.FEW_SAMPLES]


# ------------------------------------------------------------------ CLI and ABI
@pytest.fixture(scope="module")
def cli():
    from inquistr_b200 import build
    build.build_libinqcall()
    return build.build_cli()


@pytest.fixture()
def small(tmp_path):
    rows = [["chr1", "100", "120", "10", "12", "11", "NaN", "20", "22", "13", "14"],
            ["chr1", "200", "230", "5", "5", "6", "7", "NaN", "NaN", "8", "9"]]
    table = write_table(tmp_path / "t.tsv", ["a", "b", "c", "d"], rows)
    ph = tmp_path / "p.tsv"
    ph.write_text("id\tstatus\tage\na\t1\t40\nb\t0\t51\nc\t1\t33\nd\t0\t60\n")
    return table, str(ph)


def test_cli_firth_usage(cli, small):
    table, ph = small
    r = run(cli, "assoc", "--help")
    assert r.returncode == 0 and b"--firth" in r.stdout and b"penalized likelihood-ratio" in r.stdout
    for model in ("linear",):
        r = run(cli, "assoc", "--phenotype", ph, "--trait", "status", "--model", model, "--firth", table)
        assert r.returncode == 2 and r.stdout == b"" and b"'--firth' requires '--model logistic'" in r.stderr, r.stderr
    r = run(cli, "assoc", "--phenotype", ph, "--trait", "age", "--model", "logistic", "--firth", table)
    assert r.returncode == 1 and b"'40' is not 0 or 1 (--model logistic)" in r.stderr, r.stderr


def test_firth_fails_loudly_without_gpu(cli, small):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from inquistr_b200 import cohort
    from inquistr_b200.api import InqError
    with pytest.raises(InqError) as e:
        cohort.assoc(np.ones((2, 8)), np.r_[0.0, 1.0, 1.0, 0.0], model="firth")
    assert e.value.code == -1                                            # INQ_ERR_CUDA: no CPU implementation
    table, ph = small
    r = run(cli, "assoc", "--phenotype", ph, "--trait", "status", "--model", "logistic", "--firth", table)
    assert r.returncode == 1 and r.stdout == b"chromosome\tbegin\tend\tn\tbeta\tse\tstat\tp\tstatus\n" and b"inquistr-b200:" in r.stderr


def test_abi_checks_the_firth_trait_before_the_device():
    import ctypes as C
    from inquistr_b200 import cohort
    from inquistr_b200.api import InqError
    with pytest.raises(InqError) as e:                                   # INQ_ERR_ARG, whether or not a GPU is present
        cohort.assoc(np.ones((2, 8)), np.r_[0.0, 1.0, 2.0, 0.0], model="firth")
    assert e.value.code == -2 and "is not 0 or 1" in str(e.value)
    L = cohort._lib()
    h, y = np.ones((1, 8)), np.r_[0.0, 1.0, 1.0, 0.0]
    out = [np.zeros(1) for _ in range(4)] + [np.zeros(1, np.uint32), np.zeros(1, np.uint8)]
    rc = L.inq_assoc(0, 3, cohort.PRED_SUM, 1, 4, h.ctypes.data, y.ctypes.data, 0, None, *[o.ctypes.data for o in out], None,
                     C.POINTER(C.c_float)())
    assert rc == -2 and b"unknown model 3" in L.inq_cohort_last_error()


# ------------------------------------------------------------------ GPU parity through the C ABI
def add_expansions(seed, haps, y, frac=0.1):
    """Rows where 1-5 cases carry a 400-6000 bp allele and every other call is in the normal range."""
    rng = np.random.default_rng(seed)
    rows, ns = haps.shape[0], haps.shape[1] // 2
    cases = np.flatnonzero(y)
    picked = rng.choice(rows, max(1, int(frac * rows)), replace=False) if len(cases) else []
    for i in picked:
        miss = np.isnan(haps[i])
        haps[i] = np.round(rng.gamma(2.0, 12.0, 2 * ns) * 2) / 2
        haps[i][miss] = np.nan
        for s in rng.choice(cases, min(len(cases), int(rng.integers(1, 6))), replace=False):
            haps[i, 2 * s] = float(rng.integers(400, 6001))
            if np.isnan(haps[i, 2 * s + 1]):
                haps[i, 2 * s + 1] = 20.0
    return np.asarray(picked, np.int64)


def check_firth_parity(got, ref, label):
    st, gs = ref["status"], got["status"].astype(np.int64)
    bad = np.flatnonzero(gs != st)
    assert len(bad) == 0, (label, [(int(i), int(gs[i]), int(st[i]), int(got["n_iter"][i]), int(ref["n_iter"][i])) for i in bad[:10]])
    assert np.array_equal(got["n"], ref["n"]), label
    na = (gs == A.FEW_SAMPLES) | (gs == A.SINGULAR)
    for k in ("beta", "se", "stat", "p"):
        assert np.isnan(got[k][na]).all(), (label, k)
    fit = ~na
    off = fit & (got["n_iter"] != ref["n_iter"])
    assert np.all(np.abs(got["n_iter"][off].astype(int) - ref["n_iter"][off]) == 1), label
    assert off.sum() <= 0.001 * len(st), (label, off.sum())                    # at most 0.1 % of the loci
    ok = (st == A.OK) & ~off
    tol = 1e-9
    b, s = ref["beta"][ok], ref["se"][ok]
    assert np.all(np.abs(got["beta"][ok] - b) <= tol * (np.abs(b) + s)), (label, np.max(np.abs(got["beta"][ok] - b) / (np.abs(b) + s) / tol))
    assert np.all(np.abs(got["se"][ok] - s) <= tol * s), (label, np.max(np.abs(got["se"][ok] / s - 1) / tol))
    t = ref["stat"][ok]
    assert np.all(np.abs(got["stat"][ok] - t) <= 1e-8 * (t + 1)), (label, np.max(np.abs(got["stat"][ok] - t) / (t + 1) / 1e-8))
    gp, rp = np.maximum(got["p"][ok], 1e-300), np.maximum(ref["p"][ok], 1e-300)
    assert np.all(np.abs(np.log10(gp) - np.log10(rp)) <= 1e-6), (label, np.max(np.abs(np.log10(gp) - np.log10(rp))))


@pytest.mark.gpu
@pytest.mark.parametrize("rows,samples", [(1, 5), (400, 268), (150, 2100), (2000, 40)])
@pytest.mark.parametrize("n_cov", [0, 1, 12, 30])
@pytest.mark.parametrize("missing", [0.0, 0.3])
def test_gpu_firth_matches_oracle(rows, samples, n_cov, missing):
    from inquistr_b200 import cohort
    seed = rows * 7 + samples * 13 + n_cov * 101 + int(missing * 10) + 3
    haps, y, cov = make_cohort(seed, rows, samples, n_cov, missing, True)
    exp_rows = add_expansions(seed, haps, y)
    c = cov if n_cov else None
    for pred in ("sum", "max"):
        got = cohort.assoc(haps, y, c, "firth", pred)
        ref = A.assoc_matrix(haps, y, c, "firth", pred)                        # every locus
        label = (rows, samples, n_cov, missing, pred)
        check_firth_parity(got, ref, label)
        if samples in (268, 2100):
            assert not (got["status"] == A.NO_CONVERGENCE).any(), label
            assert (got["status"][exp_rows] == A.OK).all(), label          # expansion loci get an answer


@pytest.mark.gpu
def test_gpu_firth_two_by_two_closed_forms():
    from inquistr_b200 import cohort
    for table in TABLES:
        x, y = two_by_two(*table)
        haps = np.zeros((1, 2 * len(y)))
        haps[0, 0::2] = x
        got = cohort.assoc(haps, y, None, "firth", "sum")
        check_closed_form({k: v[0] for k, v in got.items() if k != "ms_kernel"}, table)


@pytest.mark.gpu
def test_gpu_firth_edge_loci():
    from inquistr_b200 import cohort
    haps, y, cov = separated_edge_loci()
    one_class = np.full((1, haps.shape[1]), np.nan)
    five = 2 * np.flatnonzero(y)[:5]
    one_class[0, five] = one_class[0, five + 1] = 30.0                     # calls on five cases only
    haps = np.vstack([haps, one_class])
    for pred in ("sum", "max"):
        got = cohort.assoc(haps, y, cov, "firth", pred)
        ref = A.assoc_matrix(haps, y, cov, "firth", pred)
        check_firth_parity({k: v for k, v in got.items() if k != "ms_kernel"}, ref, pred)
        assert list(got["status"]) == [A.SINGULAR, A.OK, A.OK, A.FEW_SAMPLES, A.FEW_SAMPLES, A.FEW_SAMPLES], got["status"]
        assert list(got["n"][3:]) == [1, 0, 5]
        assert np.isfinite(got["beta"][2]) and np.isfinite(got["p"][2])
        ml = cohort.assoc(haps[2:3], y, cov, "logistic", pred)
        assert ml["status"][0] in (A.SEPARATION, A.NO_CONVERGENCE)


# ------------------------------------------------------------------ GPU, CLI end to end
@pytest.mark.gpu
@pytest.mark.parametrize("gz", [False, True])
def test_gpu_firth_cli_end_to_end(cli, tmp_path, gz):
    rng = np.random.default_rng(41 + gz)
    samples = [f"S{i}" for i in range(150)]
    rows = 500
    haps, _, _ = make_cohort(77, rows, len(samples), 0, 0.1, False)
    ph_samples = samples[20:] + [f"X{i}" for i in range(15)]
    rng.shuffle(ph_samples)
    lines = ["sample\tage\ttrait\tpc1\tsex"]
    for s in ph_samples:
        trait = str(int(rng.random() < 0.3))
        age = f"{rng.normal(50, 12):.2f}"
        if rng.random() < 0.05:
            trait = "NA"
        if rng.random() < 0.05:
            age = ""
        lines.append(f"{s}\t{age}\t{trait}\t{rng.normal():.5f}\t{rng.integers(0, 2)}")
    pht = {l.split("\t")[0]: l.split("\t")[1:] for l in lines[1:]}
    used = [i for i, s in enumerate(samples) if s in pht and "" not in pht[s] and "NA" not in pht[s]]
    y = np.array([float(pht[samples[i]][1]) for i in used])
    cov = np.array([[float(pht[samples[i]][0]), float(pht[samples[i]][2]), float(pht[samples[i]][3])] for i in used])
    cols = np.ravel([[2 * i, 2 * i + 1] for i in used])
    sub = haps[:, cols]
    add_expansions(5, sub, y)                                              # case-only expansions among the used samples
    haps[:, cols] = sub
    loci = [(f"chr{1 + i // 200}", 1000 + 50 * i, 1030 + 50 * i) for i in range(rows)]
    text_rows = [[c, str(b), str(e)] + ["NaN" if np.isnan(v) else repr(float(v)) for v in haps[i]] for i, (c, b, e) in enumerate(loci)]
    table = write_table(tmp_path / ("c.tsv.gz" if gz else "c.tsv"), samples, text_rows)
    ph = tmp_path / "pheno.tsv"
    ph.write_text("\n".join(lines) + "\n")
    for pred in ("sum", "max"):
        r = run(cli, "assoc", "--phenotype", str(ph), "--trait", "trait", "--model", "logistic", "--firth",
                "--covariates", "age,pc1,sex", "--predictor", pred, table)
        assert r.returncode == 0, r.stderr
        out = parse_output(r.stdout.decode())
        assert [tuple(o[:3]) for o in out] == [(c, str(b), str(e)) for c, b, e in loci]
        ref = A.assoc_matrix(haps[:, cols], y, cov, "firth", pred)
        got = {k: np.array([float(o[j]) for o in out]) for j, k in ((4, "beta"), (5, "se"), (6, "stat"), (7, "p"))}
        got["n"] = np.array([int(o[3]) for o in out])
        got["status"] = np.array([A.STATUS_NAMES.index(o[8]) for o in out])
        got["n_iter"] = ref["n_iter"]                                       # not printed
        check_firth_parity(got, ref, (gz, pred))
        assert (got["status"] == A.OK).sum() > 0.7 * rows
