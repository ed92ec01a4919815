#!/usr/bin/env python
"""Measures `assoc` (include/inqcohort.h inq_assoc) at the scale the reference's R script reports: 654,000 loci x 268
samples, 12 covariates, 10 % missing calls, about 20 % constant loci, seeded. Prints one JSON line per model x
predictor with the kernel time (CUDA events, H2D excluded; median of --reps runs after a warm-up), loci/s, the f64
FMAs the fits need (from shapes and iteration counts) and GFLOP/s, and parity of --parity random loci against the
numpy restatement (oracle/assoc.py, not R or logistf) with its host time. `firth` lines (the case/control trait,
`--firth`) report the steps of the full fit over every locus and of both fits on the parity loci instead of FMAs.
Then one line per model for the CLI on the same table written as TSV: wall time with text parse, device and output
time separated (`--stats-json`). With --traits, `assoc_traits` lines: the kernel time of one inq_assoc_traits call
for 1, 8 and 32 linear traits and for 8 logistic and 8 Firth traits (seeded extra traits; the last quarter of them
share one distinct NaN pattern, so they form a second sample set) against that many times the single-trait kernel
of the same run, and the CLI wall time of `--traits` with 8 traits against 8 `--trait` runs on the same TSV.
With --cox, only the Cox lines (and the logistic `sum` kernel on the same loci, for comparison): seeded Weibull onset
ages rounded to whole years (so times are tied) with about half of them censored; per ties method (Efron, Breslow)
with `sum`, the kernel time (median of --reps after a warm-up), loci/s, mean and max Newton iterations and status
counts, parity of --parity random loci against tests/cox_reference.py's assoc_cox_matrix (run on every host core; its wall
time and the worker count are reported), and the CLI (`--model cox --stats-json`) on the same table as TSV.
The card's name and power limit are read in the same run.
Temporary files go to a temporary directory."""
import argparse
import concurrent.futures
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def workload(rows, samples, n_cov, seed=2024):
    rng = np.random.default_rng(seed)
    haps = np.round(rng.gamma(2.0, 12.0, (rows, 2 * samples)) * 2) / 2
    big = rng.random(haps.shape) < 0.02
    haps[big] = np.round(rng.pareto(1.5, big.sum()) * 100 + 100)    # heavy tail: expansions
    haps = np.minimum(haps, 3000.0)
    haps[rng.random(rows) < 0.2] = 30.0                                # constant loci
    haps[rng.random(haps.shape) < 0.1] = np.nan
    cov = np.empty((samples, n_cov))
    for c in range(n_cov):
        cov[:, c] = rng.normal(50, 15, samples) if c == 0 else (rng.integers(0, 2, samples) if c == 1 else rng.normal(0, 1, samples))
    y_lin = 3 + (0.01 * cov[:, 0] if n_cov else 0.0) + rng.normal(size=samples)
    y_bin = (rng.random(samples) < 0.4).astype(float)
    return haps, cov, y_lin, y_bin


def onsets(samples, seed=2025):
    """Onset ages: Weibull(shape 3, scale 55) rounded to whole years; about half the samples censored."""
    rng = np.random.default_rng(seed)
    t = np.round(55 * rng.weibull(3.0, samples))
    ev = (rng.random(samples) < 0.5).astype(float)
    return t, ev


def _cox_oracle(job):
    from tests import cox_reference
    haps, t, ev, cov, ties = job
    return cox_reference.assoc_cox_matrix(haps, t, ev, cov, ties, "sum")


def cox_bench(args, name, haps, cov, y_bin):
    from inquistr_b200 import cohort
    from oracle import assoc as A
    t, ev = onsets(args.samples)
    res = cohort.assoc(haps, y_bin, cov, "logistic", "sum")
    lms = float(np.median([cohort.assoc(haps, y_bin, cov, "logistic", "sum")["ms_kernel"] for _ in range(args.reps)]))
    print(json.dumps({"bench": "assoc_kernel", "card": name, "model": "logistic", "predictor": "sum", "loci": args.rows,
                      "samples": args.samples, "covariates": args.cov, "kernel_ms_median": lms}), flush=True)
    sel = np.sort(np.random.default_rng(7).choice(args.rows, min(args.parity, args.rows), replace=False))
    workers = os.cpu_count() or 1
    for ties in ("efron", "breslow"):
        cohort.assoc_cox(haps, t, ev, cov, ties, "sum")                   # warm-up
        ms = []
        for _ in range(args.reps):
            res = cohort.assoc_cox(haps, t, ev, cov, ties, "sum")
            ms.append(res["ms_kernel"])
        med = float(np.median(ms))
        t0 = time.perf_counter()
        chunks = np.array_split(sel, workers * 4)
        with concurrent.futures.ProcessPoolExecutor(workers) as ex:
            parts = list(ex.map(_cox_oracle, [(haps[c], t, ev, cov, ties) for c in chunks if len(c)]))
        ref = {k: np.concatenate([q[k] for q in parts]) for k in parts[0]}
        oracle_s = time.perf_counter() - t0
        st = res["status"][sel]
        ok = (ref["status"] == A.OK) & (st == A.OK) & (res["n_iter"][sel] == ref["n_iter"])
        rb = np.abs(res["beta"][sel][ok] - ref["beta"][ok]) / (np.abs(ref["beta"][ok]) + ref["se"][ok])
        rs = np.abs(res["se"][sel][ok] / ref["se"][ok] - 1)
        lp = np.abs(np.log10(np.maximum(res["p"][sel][ok], 1e-300)) - np.log10(np.maximum(ref["p"][ok], 1e-300)))
        fitted = ~np.isin(res["status"], (1, 2))
        print(json.dumps({
            "bench": "assoc_cox_kernel", "card": name, "ties": ties, "predictor": "sum", "loci": args.rows,
            "samples": args.samples, "covariates": args.cov, "events": int(ev.sum()), "distinct_times": int(len(np.unique(t))),
            "kernel_ms_median": med, "kernel_ms_all": ms, "loci_per_s": args.rows / (med * 1e-3),
            "logistic_sum_kernel_ms": lms, "ratio_to_logistic": med / lms,
            "mean_iterations": float(res["n_iter"][fitted].mean()), "max_iterations": int(res["n_iter"][fitted].max()),
            "status_counts": {A.STATUS_NAMES[k]: int((res["status"] == k).sum()) for k in range(5)},
            "parity": {"loci": int(len(sel)), "status_equal": bool(np.array_equal(st, ref["status"])),
                       "iter_equal": bool(np.array_equal(res["n_iter"][sel], ref["n_iter"])), "compared": int(ok.sum()),
                       "max_beta_err_rel_to_abs_beta_plus_se": float(rb.max()) if ok.any() else None,
                       "max_se_rel_err": float(rs.max()) if ok.any() else None, "max_dlog10_p": float(lp.max()) if ok.any() else None},
            "numpy_oracle_wall_s": oracle_s, "numpy_oracle_workers": workers}), flush=True)
    if args.no_cli:
        return
    from inquistr_b200 import build
    exe = os.path.join(os.path.dirname(build.__file__), "bin", "inquistr-b200")
    with tempfile.TemporaryDirectory() as d:
        samples = [f"S{i}" for i in range(args.samples)]
        table = write_table(d, haps, samples)
        ph = os.path.join(d, "pheno.tsv")
        with open(ph, "w") as f:
            f.write("sample\tonset\taffected\t" + "\t".join(f"c{c}" for c in range(args.cov)) + "\n")
            for i, s in enumerate(samples):
                f.write(f"{s}\t{t[i]:g}\t{int(ev[i])}\t" + "\t".join(repr(float(v)) for v in cov[i]) + "\n")
        for ties in ("efron", "breslow"):
            sj = os.path.join(d, "stats.json")
            t0 = time.perf_counter()
            r = subprocess.run([exe, "assoc", "--phenotype", ph, "--trait", "onset", "--model", "cox", "--event", "affected",
                                "--ties", ties, "--covariates", ",".join(f"c{c}" for c in range(args.cov)), "--stats-json", sj, table],
                               stdout=subprocess.PIPE, stderr=subprocess.PIPE)
            wall = time.perf_counter() - t0
            st = json.load(open(sj)) if r.returncode == 0 else {}
            print(json.dumps({"bench": "assoc_cox_cli", "card": name, "ties": ties, "predictor": "sum", "rc": r.returncode,
                              "table_bytes": os.path.getsize(table), "wall_s": wall, "rows_out": r.stdout.count(b"\n") - 1,
                              **st, "stderr_tail": r.stderr.decode()[-300:]}), flush=True)


def write_table(d, haps, samples):
    lut = np.array([f"{v / 2:g}" for v in range(0, 6001)] + ["NaN"], dtype=object)
    idx = np.where(np.isnan(haps), 6001, np.nan_to_num(haps * 2).astype(np.int64))
    table = os.path.join(d, "cohort.tsv")
    with open(table, "w") as f:
        f.write("chromosome\tbegin\tend\t" + "\t".join(f"{s}_H1\t{s}_H2" for s in samples) + "\n")
        for i in range(len(haps)):
            f.write(f"chr{1 + i // 30000}\t{1000 + 100 * i}\t{1040 + 100 * i}\t" + "\t".join(lut[idx[i]]) + "\n")
    return table


def traits_matrix(y0, T, model, seed=99):
    """T traits for --traits: y0 first, then seeded ones of the same kind; the last T // 4 share one NaN pattern."""
    rng = np.random.default_rng(seed)
    n = len(y0)
    Y = np.empty((n, T))
    Y[:, 0] = y0
    for t in range(1, T):
        Y[:, t] = rng.normal(3, 1, n) if model == "linear" else (rng.random(n) < 0.4).astype(float)
    if T >= 4:
        Y[rng.random(n) < 0.1, T - T // 4:] = np.nan
    return Y


def fmas(res, p, model):
    """f64 FMAs of the passes over the samples, n samples used and p design columns per locus:
    linear   one Gram pass, n * (p^2 + p) for G and X'y, and one residual pass, n * p for eta: n * (p^2 + 2p);
    logistic n_iter + 1 passes, each n * p for eta and n * (p^2 + p) for G and X'Wz (the last pass's G is accumulated
             and not solved): (n_iter + 1) * n * (p^2 + 2p).
    few_samples loci (no solve) count nothing; the elimination (about p^3 / 3 per solve) is small next to these."""
    n = res["n"].astype(np.float64)
    fit = res["status"] != 1                                           # few_samples
    if model == "linear":
        return float(np.sum(n[fit] * (p * p + 2 * p)))
    passes = res["n_iter"].astype(np.float64) + 1
    return float(np.sum(n[fit] * passes[fit] * (p * p + 2 * p)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=654_000)
    ap.add_argument("--samples", type=int, default=268)
    ap.add_argument("--cov", type=int, default=12)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parity", type=int, default=2000)
    ap.add_argument("--no-cli", action="store_true")
    ap.add_argument("--traits", action="store_true")
    ap.add_argument("--cox", action="store_true")
    args = ap.parse_args()
    from inquistr_b200 import cohort
    from oracle import assoc as A
    name = card()
    haps, cov, y_lin, y_bin = workload(args.rows, args.samples, args.cov)
    if args.cox:
        cox_bench(args, name, haps, cov, y_bin)
        return
    p = args.cov + 2
    sel = np.sort(np.random.default_rng(7).choice(args.rows, min(args.parity, args.rows), replace=False))
    single_ms = {}
    for model in ("linear", "logistic", "firth"):
        y = y_lin if model == "linear" else y_bin
        for pred in ("sum", "max"):
            res = cohort.assoc(haps, y, cov, model, pred)                # warm-up
            ms = []
            for _ in range(args.reps):
                res = cohort.assoc(haps, y, cov, model, pred)
                ms.append(res["ms_kernel"])
            med = float(np.median(ms))
            single_ms[model, pred] = med
            f = fmas(res, p, model) if model != "firth" else None
            t0 = time.perf_counter()
            ref = A.assoc_matrix(haps[sel], y, cov, model, pred)
            oracle_s = time.perf_counter() - t0
            st = res["status"][sel]
            ok = (ref["status"] == A.OK) & (st == A.OK)
            if model != "linear":
                ok &= res["n_iter"][sel] == ref["n_iter"]
            rb = np.abs(res["beta"][sel][ok] - ref["beta"][ok]) / (np.abs(ref["beta"][ok]) + ref["se"][ok])
            rs = np.abs(res["se"][sel][ok] / ref["se"][ok] - 1)
            lp = np.abs(np.log10(np.maximum(res["p"][sel][ok], 1e-300)) - np.log10(np.maximum(ref["p"][ok], 1e-300)))
            steps = {}
            if model == "firth":                                        # over the loci with a fit (not few_samples / singular)
                fitted, rf = ~np.isin(res["status"], (1, 2)), ~np.isin(ref["status"], (1, 2))
                steps = {"full_steps_mean": float(res["n_iter"][fitted].mean()), "full_steps_max": int(res["n_iter"][fitted].max()),
                         "parity_full_steps_mean": float(ref["n_iter"][rf].mean()), "parity_full_steps_max": int(ref["n_iter"][rf].max()),
                         "parity_null_steps_mean": float(ref["n_iter_null"][rf].mean()),
                         "parity_null_steps_max": int(ref["n_iter_null"][rf].max())}
            print(json.dumps({
                "bench": "assoc_kernel", "card": name, "model": model, "predictor": pred, "loci": args.rows,
                "samples": args.samples, "covariates": args.cov, "kernel_ms_median": med, "kernel_ms_all": ms,
                "loci_per_s": args.rows / (med * 1e-3), "f64_fma": f, "gflops": 2 * f / (med * 1e-3) / 1e9 if f else None, **steps,
                "status_counts": {A.STATUS_NAMES[k]: int((res["status"] == k).sum()) for k in range(5)},
                "mean_iterations": float(res["n_iter"][res["status"] != 1].mean()) if model == "logistic" else 0.0,
                "parity": {"loci": int(len(sel)), "status_equal": bool(np.array_equal(st, ref["status"])),
                           "iter_equal": bool(np.array_equal(res["n_iter"][sel], ref["n_iter"])),
                           "compared": int(ok.sum()), "max_beta_err_rel_to_abs_beta_plus_se": float(rb.max()) if ok.any() else None,
                           "max_se_rel_err": float(rs.max()) if ok.any() else None, "max_dlog10_p": float(lp.max()) if ok.any() else None},
                "numpy_oracle_s": oracle_s, "numpy_oracle_loci_per_s": len(sel) / oracle_s}), flush=True)
    if args.traits:
        for model, T in (("linear", 1), ("linear", 8), ("linear", 32), ("logistic", 8), ("firth", 8)):
            Y = traits_matrix(y_lin if model == "linear" else y_bin, T, model)
            cohort.assoc_traits(haps, Y, cov, model, "sum")               # warm-up
            ms = [cohort.assoc_traits(haps, Y, cov, model, "sum")["ms_kernel"] for _ in range(args.reps)]
            med = float(np.median(ms))
            groups = len({tuple(np.isnan(Y[:, t])) for t in range(T)})
            print(json.dumps({"bench": "assoc_traits_kernel", "card": name, "model": model, "predictor": "sum", "traits": T,
                              "groups": groups, "loci": args.rows, "samples": args.samples, "covariates": args.cov,
                              "kernel_ms_median": med, "kernel_ms_all": ms, "single_trait_kernel_ms": single_ms[model, "sum"],
                              "traits_x_single_ms": T * single_ms[model, "sum"],
                              "speedup": T * single_ms[model, "sum"] / med}), flush=True)
    if args.no_cli:
        return
    from inquistr_b200 import build
    exe = os.path.join(os.path.dirname(build.__file__), "bin", "inquistr-b200")
    with tempfile.TemporaryDirectory() as d:
        samples = [f"S{i}" for i in range(args.samples)]
        t0 = time.perf_counter()
        table = write_table(d, haps, samples)
        write_s = time.perf_counter() - t0
        ph = os.path.join(d, "pheno.tsv")
        with open(ph, "w") as f:
            f.write("sample\tlin\tbin\t" + "\t".join(f"c{c}" for c in range(args.cov)) + "\n")
            for i, s in enumerate(samples):
                f.write(f"{s}\t{float(y_lin[i])!r}\t{int(y_bin[i])}\t" + "\t".join(repr(float(v)) for v in cov[i]) + "\n")
        for model, trait in (("linear", "lin"), ("logistic", "bin"), ("firth", "bin")):
            sj = os.path.join(d, "stats.json")
            flags = ["--model", "logistic", "--firth"] if model == "firth" else ["--model", model]
            t0 = time.perf_counter()
            r = subprocess.run([exe, "assoc", "--phenotype", ph, "--trait", trait, *flags, "--covariates",
                                ",".join(f"c{c}" for c in range(args.cov)), "--stats-json", sj, table],
                               stdout=subprocess.PIPE, stderr=subprocess.PIPE)
            wall = time.perf_counter() - t0
            st = json.load(open(sj)) if r.returncode == 0 else {}
            out_rows = r.stdout.count(b"\n") - 1
            print(json.dumps({"bench": "assoc_cli", "card": name, "model": model, "predictor": "sum", "rc": r.returncode,
                              "table_bytes": os.path.getsize(table), "table_write_s": write_s, "wall_s": wall,
                              "rows_out": out_rows, **st, "stderr_tail": r.stderr.decode()[-300:]}), flush=True)
        if not args.traits:
            return
        Y = traits_matrix(y_lin, 8, "linear")
        ph8 = os.path.join(d, "pheno8.tsv")
        with open(ph8, "w") as f:
            f.write("sample\t" + "\t".join(f"t{t}" for t in range(8)) + "\t" + "\t".join(f"c{c}" for c in range(args.cov)) + "\n")
            for i, s in enumerate(samples):
                f.write(s + "\t" + "\t".join("NA" if np.isnan(v) else repr(float(v)) for v in Y[i]) + "\t" +
                        "\t".join(repr(float(v)) for v in cov[i]) + "\n")
        covs = ",".join(f"c{c}" for c in range(args.cov))

        def cli_run(*trait_args):
            sj = os.path.join(d, "stats.json")
            t0 = time.perf_counter()
            r = subprocess.run([exe, "assoc", "--phenotype", ph8, *trait_args, "--model", "linear", "--covariates", covs,
                                "--stats-json", sj, table], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
            return time.perf_counter() - t0, r.returncode, json.load(open(sj)) if r.returncode == 0 else {}

        wall, rc, st = cli_run("--traits", ",".join(f"t{t}" for t in range(8)))
        singles = [cli_run("--trait", f"t{t}") for t in range(8)]
        print(json.dumps({"bench": "assoc_traits_cli", "card": name, "model": "linear", "traits": 8, "rc": rc, "wall_s": wall, **st,
                          "single_runs_wall_s": sum(w for w, _, _ in singles), "single_runs_rc": [c for _, c, _ in singles],
                          "single_runs_s_parse": sum(x.get("s_parse", 0.0) for _, _, x in singles),
                          "single_runs_s_device": sum(x.get("s_device", 0.0) for _, _, x in singles)}), flush=True)


if __name__ == "__main__":
    main()
