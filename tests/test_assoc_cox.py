"""`assoc --model cox` / inq_assoc_cox: Cox proportional-hazards regression of age at onset on STR length, with
censoring and tied times (DESIGN.md 5e, Cox).
CPU: the restatement (tests/cox_reference.py fit_locus_cox) pinned by R's documented `aml` fit and by direct maximisation of
the partial likelihood written here, its invariances and edge statuses, the CLI's usage and data errors and the ABI's
argument errors. GPU: inq_assoc_cox against the restatement over a grid of shapes, ties and censoring, the edge and
overflow loci, and the CLI end to end."""
import numpy as np
import pytest
from scipy import optimize, stats

from oracle import assoc as A
from tests import cox_reference as C
from tests.test_assoc import check_parity, cli, make_cohort, run, write_table  # noqa: F401 (fixtures)

ERR_CUDA, ERR_ARG = -1, -2
HEAD = b"chromosome\tbegin\tend\tn\tbeta\tse\tstat\tp\tstatus\n"

# R survival's `aml`: Maintained (x = 0) and Nonmaintained (x = 1); event 0 = censored ("+")
AML_TIME = np.array([9, 13, 13, 18, 23, 28, 31, 34, 45, 48, 161, 5, 5, 8, 8, 12, 16, 23, 27, 30, 33, 43, 45], float)
AML_EVENT = np.array([1, 1, 0, 1, 1, 0, 1, 1, 0, 1, 0, 1, 1, 1, 1, 1, 0, 1, 1, 1, 1, 1, 1], float)
AML_X = np.r_[np.zeros(11), np.ones(12)]


def partial_loglik(b, x, time, event, ties):
    """The partial log-likelihood of one covariate, one loop over the event times: the independent check."""
    ll = 0.0
    for tau in np.unique(time[event != 0]):
        dead = (time == tau) & (event != 0)
        risk = time >= tau
        m = dead.sum()
        ll += b * x[dead].sum()
        for k in range(m):
            f = k / m if ties == "efron" else 0.0
            ll -= np.log(np.exp(b * x[risk]).sum() - f * np.exp(b * x[dead]).sum())
    return ll


def direct_fit(x, time, event, ties):
    r = optimize.minimize_scalar(lambda b: -partial_loglik(b, x, time, event, ties), bracket=(0, 1), tol=1e-12)
    h = 1e-4
    d2 = (partial_loglik(r.x + h, x, time, event, ties) - 2 * partial_loglik(r.x, x, time, event, ties)
          + partial_loglik(r.x - h, x, time, event, ties)) / h ** 2
    return r.x, 1 / np.sqrt(-d2)


def score_loop(U, time, event, beta, ties):
    """The score of the partial likelihood at beta, one sample at a time."""
    s = np.zeros(U.shape[1])
    for tau in np.unique(time[event != 0]):
        dead = np.flatnonzero((time == tau) & (event != 0))
        risk = np.flatnonzero(time >= tau)
        m = len(dead)
        for k in range(m):
            f = k / m if ties == "efron" else 0.0
            d0, d1 = 0.0, np.zeros(U.shape[1])
            for i in risk:
                w = np.exp(U[i] @ beta) * (1 - f * (i in dead))
                d0 += w
                d1 += w * U[i]
            s -= d1 / d0
        s += U[dead].sum(axis=0)
    return s


# ------------------------------------------------------------------ the restatement, pinned independently of it
def test_aml_efron_as_r_prints_it():
    r = C.fit_locus_cox(AML_X, AML_TIME, AML_EVENT, None, "efron")
    assert r["status"] == A.OK and r["n"] == 23
    assert round(r["beta"], 4) == 0.9155 and round(r["se"], 4) == 0.5119
    assert round(r["stat"], 3) == 1.788 and round(r["p"], 4) == 0.0737


@pytest.mark.parametrize("ties,coef,se", [("efron", 0.915533, 0.511934), ("breslow", 0.904220, 0.512248)])
def test_aml_direct_maximisation(ties, coef, se):
    b, s = direct_fit(AML_X, AML_TIME, AML_EVENT, ties)
    assert b == pytest.approx(coef, abs=1e-6) and s == pytest.approx(se, abs=1e-6)
    r = C.fit_locus_cox(AML_X, AML_TIME, AML_EVENT, None, ties)
    assert r["status"] == A.OK
    assert r["beta"] == pytest.approx(b, abs=1e-6) and r["se"] == pytest.approx(s, abs=1e-5)
    assert r["p"] == pytest.approx(2 * stats.norm.sf(abs(r["beta"] / r["se"])), rel=1e-12)


def onset_cohort(seed, n, n_cov=3, cens=0.5, years=True):
    rng = np.random.default_rng(seed)
    cov = np.column_stack([rng.normal(50, 15, n), rng.integers(0, 2, n), rng.normal(size=n)])[:, :n_cov]
    x = rng.gamma(2, 15, n)
    t = 60 * rng.weibull(2.0, n) * np.exp(-0.01 * (x - 30))
    if years:
        t = np.round(t)
    ev = (rng.random(n) >= cens).astype(float)
    return x, t, ev, cov


@pytest.mark.parametrize("ties", ["efron", "breslow"])
def test_score_is_zero_at_the_solution(ties):
    for seed in range(4):
        x, t, ev, cov = onset_cohort(seed, 60)
        r = C.fit_locus_cox(x, t, ev, cov, ties)
        assert r["status"] == A.OK
        U = np.column_stack([cov, x])
        s = score_loop(U, t, ev, r["coef"], ties)
        assert np.all(np.abs(s) <= 1e-6 * np.abs(U).sum(axis=0)), s


def test_monotone_time_transform_changes_nothing():
    x, t, ev, cov = onset_cohort(5, 80)
    for ties in ("efron", "breslow"):
        a = C.fit_locus_cox(x, t, ev, cov, ties)
        b = C.fit_locus_cox(x, np.exp(t / 20) + 3, ev, cov, ties)
        for k in ("beta", "se", "stat", "p", "status", "n_iter"):
            assert a[k] == b[k], k


def test_scale_and_shift_of_x():
    x, t, ev, cov = onset_cohort(6, 90)
    a = C.fit_locus_cox(x, t, ev, cov)
    for c, shift in ((2.5, 0.0), (0.1, -40.0), (7.0, 1000.0)):
        b = C.fit_locus_cox(c * x + shift, t, ev, cov)
        assert b["status"] == a["status"] == A.OK
        assert b["beta"] * c == pytest.approx(a["beta"], rel=1e-9)
        assert b["stat"] == pytest.approx(a["stat"], rel=1e-9) and b["p"] == pytest.approx(a["p"], rel=1e-9)


def test_without_ties_efron_is_breslow():
    x, t, ev, cov = onset_cohort(7, 70, years=False)
    assert len(np.unique(t)) == len(t)
    a = C.fit_locus_cox(x, t, ev, cov, "efron")
    b = C.fit_locus_cox(x, t, ev, cov, "breslow")
    for k in ("beta", "se", "stat", "p"):
        assert a[k] == pytest.approx(b[k], rel=1e-12), k


def test_edge_statuses():
    x, t, ev, cov = onset_cohort(8, 50)
    with_const = C.fit_locus_cox(x, t, ev, np.column_stack([cov, np.full(50, 4.2)]))
    without = C.fit_locus_cox(x, t, ev, cov)
    assert with_const["status"] == without["status"] == A.OK
    for k in ("beta", "se", "stat", "p"):
        assert with_const[k] == pytest.approx(without[k], rel=1e-9), k
    r = C.fit_locus_cox(np.full(50, 31.0), t, ev, cov)
    assert r["status"] == A.SINGULAR and np.isnan(r["beta"])
    r = C.fit_locus_cox(x, t, np.zeros(50), cov)
    assert r["status"] == A.FEW_SAMPLES and r["n"] == 50 and np.isnan(r["p"])


def test_case_only_expansions_at_the_earliest_onsets():
    x, t, ev, _ = onset_cohort(9, 100, cens=0.3, years=False)
    order = np.argsort(t, kind="stable")
    x[:] = 30.0
    ev[order[:4]] = 1
    x[order[:4]] = [6000.0, 4000.0, 3100.0, 2500.0]           # the four earliest onsets carry the expansions
    r = C.fit_locus_cox(x, t, ev)
    assert r["status"] == A.SEPARATION and np.isfinite(r["beta"]) and r["beta"] > 0 and np.isfinite(r["se"])


# ------------------------------------------------------------------ CLI and ABI without a device
@pytest.fixture()
def onset(tmp_path):
    samples = ["a", "b", "c", "d", "e"]
    rows = [["chr1", "100", "120", "10", "12", "11", "NaN", "20", "22", "13", "14", "9", "9"],
            ["chr1", "200", "230", "5", "5", "6", "7", "NaN", "NaN", "8", "9", "4", "6"]]
    table = write_table(tmp_path / "t.tsv", samples, rows)
    ph = tmp_path / "p.tsv"
    # b: no onset age; d: no event; f: only in the phenotype table
    ph.write_text("id\tonset\taffected\tsex\na\t41.5\t1\t0\nb\tNA\t0\t1\nc\t55\t0\t1\nd\t38\t\t0\ne\t47\t1\t1\nf\t50\t1\t0\n")
    return tmp_path, table, str(ph)


def test_cox_usage_errors(cli, onset):
    d, table, ph = onset
    base = ["assoc", "--phenotype", ph, "--trait", "onset"]
    cases = [
        (base + ["--model", "linear", "--event", "affected", table], b"'--event <COL>' requires '--model cox'"),
        (base + ["--model", "logistic", "--ties", "breslow", table], b"'--ties <TIES>' requires '--model cox'"),
        (base + ["--model", "cox", table], b"--event <COL>"),
        (base + ["--model", "cox", "--event", "affected", "--firth", table], b"'--firth' requires '--model logistic'"),
        (["assoc", "--phenotype", ph, "--traits", "onset,sex", "--model", "cox", "--event", "affected", table],
         b"'--traits <A,B,...>' cannot be used with '--model cox'"),
        (base + ["--model", "cox", "--event", "onset", table], b"the event column 'onset' is also the time column"),
        (base + ["--model", "cox", "--event", "affected", "--covariates", "sex,affected", table],
         b"the event column 'affected' is also listed as a covariate"),
        (base + ["--model", "cox", "--event", "affected", "--ties", "exact", table], b"invalid value 'exact' for '--ties"),
    ]
    for args, msg in cases:
        r = run(cli, *args)
        assert r.returncode == 2 and r.stdout == b"", args
        assert msg in r.stderr, (args, r.stderr)
    r = run(cli, "assoc", "--help")
    assert r.returncode == 0 and b"--event <COL>" in r.stdout and b"[possible values: efron, breslow]" in r.stdout


def test_cox_data_errors(cli, onset):
    d, table, ph = onset

    def fails(text, *msgs):
        p = d / "bad.tsv"
        p.write_text(text)
        r = run(cli, "assoc", "--phenotype", str(p), "--trait", "onset", "--model", "cox", "--event", "affected", table)
        assert r.returncode == 1 and r.stdout == b"", r.stderr
        for m in msgs:
            assert m.encode() in r.stderr, (m, r.stderr)

    fails("id\tonset\taffected\na\t40\t1\nb\t51\t2\n", "bad.tsv:3:", "column 'affected'", "'2' is not 0 or 1 (--event)")
    fails("id\tonset\taffected\na\t40\t1\nb\tforty\t0\n", "bad.tsv:3:", "column 'onset'", "'forty' is not a number")
    fails("id\tonset\taffected\na\t40\t1\nb\tinf\t0\n", "bad.tsv:3:", "'inf' is not a number")
    fails("id\tonset\n", "bad.tsv:1:", "column 'affected' is not in the header")


def test_cox_sample_counts_and_no_gpu(cli, onset):
    import torch
    d, table, ph = onset
    r = run(cli, "assoc", "--phenotype", ph, "--trait", "onset", "--model", "cox", "--event", "affected", table)
    line = r.stderr.decode().splitlines()[0]
    assert line == ("assoc: 3 samples used, 2 in the table only, 1 in the phenotype table only "
                    "(2 phenotype rows with a missing value left out)"), line
    if torch.cuda.is_available():
        return
    assert r.returncode == 1 and r.stdout == HEAD and b"inquistr-b200:" in r.stderr
    from inquistr_b200 import cohort
    from inquistr_b200.api import InqError
    with pytest.raises(InqError) as e:
        cohort.assoc_cox(np.ones((2, 8)), np.arange(4.0), np.ones(4))
    assert e.value.code == ERR_CUDA


def test_cox_abi_argument_errors():
    """Returned before any device call, so they are the same with and without a GPU."""
    from inquistr_b200 import cohort
    from inquistr_b200.api import InqError
    haps = np.ones((3, 8))
    t, ev = np.array([40.0, 50, 60, 70]), np.array([1.0, 0, 1, 0])
    cases = [
        (dict(time=np.array([40.0, np.nan, 60, 70]), event=ev), "time of sample 1 is not a finite number"),
        (dict(time=np.array([40.0, 50, np.inf, 70]), event=ev), "time of sample 2 is not a finite number"),
        (dict(time=t, event=np.array([1.0, 0, 0.5, 0])), "event of sample 2 is not 0 or 1"),
        (dict(time=t, event=np.array([1.0, 0, 1, 2])), "event of sample 3 is not 0 or 1"),
        (dict(time=t, event=ev, cov=np.array([1.0, 2, np.nan, 3])), "covariate 0 of sample 2"),
        (dict(time=t, event=ev, cov=np.ones((4, 31))), "31 covariates"),
    ]
    for kw, msg in cases:
        with pytest.raises(InqError) as e:
            cohort.assoc_cox(haps, **kw)
        assert e.value.code == ERR_ARG and msg in str(e.value), (kw, str(e.value))
    L = cohort._lib()
    z = np.zeros(64)
    e8 = np.zeros(4, np.uint8)
    rc = L.inq_assoc_cox(0, 2, 0, 3, 4, haps.ctypes.data, t.ctypes.data, e8.ctypes.data, 0, None, *(z.ctypes.data,) * 4,
                         z.ctypes.data, z.ctypes.data, None, None)
    assert rc == ERR_ARG and b"unknown ties method 2" in L.inq_cohort_last_error()
    rc = L.inq_assoc_cox(0, 0, 0, 1 << 40, 4, haps.ctypes.data, t.ctypes.data, e8.ctypes.data, 0, None, *(z.ctypes.data,) * 4,
                         z.ctypes.data, z.ctypes.data, None, None)
    assert rc == -14                                                        # INQ_ERR_TOO_LARGE


# ------------------------------------------------------------------ GPU parity through the C ABI
def onset_times(seed, n, pattern, cens):
    """Seeded Weibull onset ages; pattern: none (distinct), years (rounded), straddle (40 samples share one time that
    spans the first tile boundary of the time order), all (one time). cens: share of censored samples."""
    rng = np.random.default_rng(seed)
    t = 30 + 25 * rng.weibull(2.5, n)
    if pattern == "years":
        t = np.round(t)
    elif pattern == "straddle":
        order = np.argsort(t, kind="stable")
        t[order[min(12, n - 1):52]] = t[order[min(12, n - 1)]]
    elif pattern == "all":
        t[:] = 47.0
    ev = (rng.random(n) >= cens).astype(float)
    return t, ev


COX_GRID = [(5, 0, 0.0, 0.0, "sum", 40), (33, 1, 0.5, 0.1, "max", 60), (100, 3, 0.95, 0.0, "sum", 40),
            (100, 12, 0.5, 0.1, "sum", 30), (268, 12, 0.5, 0.1, "max", 20), (268, 0, 0.0, 0.0, "sum", 20),
            (268, 30, 0.5, 0.1, "sum", 8), (1000, 3, 0.5, 0.1, "max", 4), (1000, 12, 0.95, 0.0, "sum", 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("ties", ["efron", "breslow"])
@pytest.mark.parametrize("pattern", ["none", "years", "straddle", "all"])
def test_gpu_cox_matches_oracle(ties, pattern):
    from inquistr_b200 import cohort
    for gi, (n, n_cov, cens, missing, pred, rows) in enumerate(COX_GRID):
        seed = 500 + gi * 31 + len(pattern) * 7 + len(ties)
        haps, _, cov = make_cohort(seed, rows, n, n_cov, missing, False)
        t, ev = onset_times(seed, n, pattern, cens)
        c = cov if n_cov else None
        got = cohort.assoc_cox(haps, t, ev, c, ties, pred)
        ref = C.assoc_cox_matrix(haps, t, ev, c, ties, pred)
        check_parity(got, ref, "logistic", (ties, pattern, n, n_cov, cens, missing, pred))


@pytest.mark.gpu
def test_gpu_cox_monotone_time_transform_is_bit_identical():
    from inquistr_b200 import cohort
    haps, _, cov = make_cohort(71, 200, 150, 3, 0.1, False)
    t, ev = onset_times(71, 150, "years", 0.5)
    for ties in ("efron", "breslow"):
        a = cohort.assoc_cox(haps, t, ev, cov, ties, "sum")
        b = cohort.assoc_cox(haps, np.log(t) * 3 - 1, ev, cov, ties, "sum")
        for k in ("beta", "se", "stat", "p", "n", "status", "n_iter"):
            assert np.array_equal(a[k], b[k], equal_nan=True), (ties, k)


@pytest.mark.gpu
@pytest.mark.parametrize("ties", ["efron", "breslow"])
def test_gpu_cox_edge_loci(ties):
    from inquistr_b200 import cohort
    rng = np.random.default_rng(23)
    ns = 60
    t, ev = onset_times(23, ns, "years", 0.5)
    age = rng.normal(50, 10, ns)
    flag = np.where(np.arange(ns) < 20, 1.0, 0.0)                  # constant on samples 20.. (aliased where 0..19 miss)
    cov = np.column_stack([age, flag])
    rows = [np.full(2 * ns, 25.0)]                                 # constant x: singular
    h = rng.gamma(2, 12, 2 * ns)
    h[:40] = np.nan                                                # samples 0..19 missing: flag constant
    rows.append(h)
    one = np.full(2 * ns, np.nan)
    one[10:12] = [12.0, 13.0]                                      # one sample
    rows.append(one)
    rows.append(np.full(2 * ns, np.nan))                           # all NaN
    h = rng.gamma(2, 12, 2 * ns)
    h[np.repeat(ev, 2) > 0] = np.nan                               # only censored samples have a call: no event
    rows.append(h)
    haps = np.stack(rows)
    for pred in ("sum", "max"):
        got = cohort.assoc_cox(haps, t, ev, cov, ties, pred)
        ref = C.assoc_cox_matrix(haps, t, ev, cov, ties, pred)
        check_parity({k: v for k, v in got.items() if k != "ms_kernel"}, ref, "logistic", (ties, pred))
        assert list(got["status"]) == [A.SINGULAR, A.OK, A.FEW_SAMPLES, A.FEW_SAMPLES, A.FEW_SAMPLES]
        assert list(got["n"][2:4]) == [1, 0]
    a = cohort.assoc_cox(haps[1:2], t, ev, cov, ties)
    b = cohort.assoc_cox(haps[1:2], t, ev, age[:, None], ties)
    for k in ("beta", "se", "p"):
        assert a[k][0] == pytest.approx(b[k][0], rel=1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("ties", ["efron", "breslow"])
def test_gpu_cox_overflow_loci_stay_finite(ties):
    """Expansions of up to 6,000 bp on the earliest onsets: beta walks far out, and exp(eta) of a plain sum would
    overflow (or underflow to an empty late risk set)."""
    from inquistr_b200 import cohort
    rng = np.random.default_rng(17)
    ns, rows = 268, 64
    t, ev = onset_times(17, ns, "years", 0.5)
    order = np.argsort(t, kind="stable")
    haps = np.round(rng.gamma(2.0, 12.0, (rows, 2 * ns)) * 2) / 2
    for i in range(rows):
        k = 1 + i % 6
        carriers = order[:k] if i % 2 else rng.choice(ns, k, replace=False)
        haps[i, 2 * carriers] = rng.uniform(1500, 6000, k)
        if i % 4 == 3:                                                   # the latest samples carry it: beta -> -inf
            haps[i, 2 * order[-k:]] = rng.uniform(1500, 6000, k)
    for pred in ("sum", "max"):
        got = cohort.assoc_cox(haps, t, ev, None, ties, pred)
        for k in ("beta", "se", "stat", "p"):
            assert np.all(np.isfinite(got[k])), (pred, k, got["status"])
        assert np.all(got["status"] != A.FEW_SAMPLES)
        ref = C.assoc_cox_matrix(haps, t, ev, None, ties, pred)
        check_parity(got, ref, "logistic", (ties, pred))


# ------------------------------------------------------------------ GPU, CLI end to end
@pytest.mark.gpu
@pytest.mark.parametrize("gz", [False, True])
def test_gpu_cli_cox_prints_the_binding(cli, tmp_path, gz):
    from inquistr_b200 import cohort
    rng = np.random.default_rng(61 + gz)
    samples = [f"S{i}" for i in range(150)]
    haps, _, _ = make_cohort(97, 500, len(samples), 0, 0.1, False)
    text_rows = [[f"chr{1 + i // 200}", str(1000 + 50 * i), str(1030 + 50 * i)] + ["NaN" if np.isnan(v) else repr(float(v)) for v in haps[i]]
                 for i in range(len(haps))]
    table = write_table(tmp_path / ("c.tsv.gz" if gz else "c.tsv"), samples, text_rows)
    ph_samples = samples[20:] + [f"X{i}" for i in range(15)]
    rng.shuffle(ph_samples)
    t, ev = onset_times(61 + gz, len(ph_samples), "years", 0.5)
    lines = ["sample\tage\tonset\taffected\tpc1"]
    for i, s in enumerate(ph_samples):
        onset = "NA" if rng.random() < 0.05 else f"{t[i]:g}"
        aff = "" if rng.random() < 0.05 else str(int(ev[i]))
        lines.append(f"{s}\t{rng.normal(50, 12):.2f}\t{onset}\t{aff}\t{rng.normal():.5f}")
    ph = tmp_path / "pheno.tsv"
    ph.write_text("\n".join(lines) + "\n")
    pht = {l.split("\t")[0]: l.split("\t")[1:] for l in lines[1:]}
    used = [i for i, s in enumerate(samples) if s in pht and "" not in pht[s] and "NA" not in pht[s]]
    tt = np.array([float(pht[samples[i]][1]) for i in used])
    ee = np.array([float(pht[samples[i]][2]) for i in used])
    cov = np.array([[float(pht[samples[i]][0]), float(pht[samples[i]][3])] for i in used])
    cols = np.ravel([[2 * i, 2 * i + 1] for i in used])
    for ties, pred in (("efron", "sum"), ("breslow", "max")):
        r = run(cli, "assoc", "--phenotype", str(ph), "--trait", "onset", "--model", "cox", "--event", "affected",
                "--ties", ties, "--covariates", "age,pc1", "--predictor", pred, table)
        assert r.returncode == 0, r.stderr
        missing = sum(1 for s in ph_samples if "" in pht[s] or "NA" in pht[s])
        assert r.stderr.decode().splitlines()[0] == (f"assoc: {len(used)} samples used, {len(samples) - len(used)} in the table only, "
                                                     f"15 in the phenotype table only ({missing} phenotype rows with a missing value left out)")
        lines_out = r.stdout.decode().split("\n")
        assert lines_out[0] + "\n" == HEAD.decode() and lines_out[-1] == ""
        out = [l.split("\t") for l in lines_out[1:-1]]
        want = cohort.assoc_cox(haps[:, cols], tt, ee, cov, ties, pred)
        assert [o[:3] for o in out] == [r_[:3] for r_ in text_rows]
        assert [int(o[3]) for o in out] == list(want["n"])
        assert [o[8] for o in out] == [A.STATUS_NAMES[s] for s in want["status"]]
        for j, k in ((4, "beta"), (5, "se"), (6, "stat"), (7, "p")):
            assert np.array_equal(np.array([float(o[j]) for o in out]), want[k], equal_nan=True), (ties, k)
