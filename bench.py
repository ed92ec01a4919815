#!/usr/bin/env python
"""bench.py -- `inquiSTR call` hot path on B200: STR loci genotyped / s and CIGAR ops / s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 3] [--scale S] [--dump-outputs DIR]

A step = one pass of the hot path (join -> CIGAR scan -> pair sums -> medians) over the whole
workload. `value` is measured with the reads already resident in HBM (CUDA events on the library's
own stream); `e2e` is the same job through the C ABI from pinned HOST buffers (set_loci + push_reads
+ genotype, H2D and D2H inside the timed region). One process per GPU; for N > 1 the sorted locus
catalog is range-sharded across ranks (no collective on the data path; torch.distributed is used
for the barrier and the max-over-ranks only). Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, help="BASELINE.json configs[] index + 1 (default 3 = headline)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the genome and catalog (tests)")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pack-filter", action="store_true",
                    help="ship every generated read (also the ones with mapq <= 10 / without HP that can never pair)")
    ap.add_argument("--ranges", type=int, default=None, help="inq_set_option('ranges') (default: automatic)")
    ap.add_argument("--no-graph", action="store_true", help="inq_set_option('graph', 0)")
    ap.add_argument("--set", action="append", default=[], metavar="NAME=VALUE", help="inq_set_option(NAME, VALUE), repeatable (experiments)")
    ap.add_argument("--bam-scale", type=float, default=0.1,
                    help="e2e_bam: `inquistr-b200 call` on a synthetic BAM with SEQ/QUAL of config 3 at this scale (0 = skip)")
    ap.add_argument("--no-cohort", action="store_true", help="skip the extra.cohort_outlier block (SURVEY 8f rank 3 kernels)")
    ap.add_argument("--parity-seconds", type=float, default=6.0, help="budget of the per-rank oracle check at N > 1")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the medians of the last timed step as DIR/phase1.npy and DIR/phase2.npy (float64, 0 where no "
                         "call) and their valid_mask (include/inqcall.h) as DIR/valid_mask.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times a sample of the loci sized by the clock)")
    return args


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, phase1: np.ndarray, phase2: np.ndarray) -> None:
    """phase1 / phase2 as the caller of Context.genotype receives them, one value per catalog locus, written as finite
    arrays: the medians with 0 where there is no call (NaN in phase1 / phase2) and valid_mask, bit 0 = H1 called,
    bit 1 = H2 called. A catalog too large for DUMP_MAX_BYTES is cut to a fixed seeded sample of loci, whose catalog
    indices go to locus_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(phase1)
    ok1, ok2 = ~np.isnan(phase1), ~np.isnan(phase2)
    arrays = {"phase1": np.where(ok1, phase1, 0.0), "phase2": np.where(ok2, phase2, 0.0), "valid_mask": ok1 + 2.0 * ok2}
    if len(arrays) * 8 * n > DUMP_MAX_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_BYTES // ((len(arrays) + 1) * 8), replace=False))
        arrays = {name: a[keep] for name, a in arrays.items()}
        arrays["locus_index"] = keep.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


class Clocks:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, smax, reasons = [], [], set()
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons), samples=len(sm))
        return out


def algorithmic_bytes(st: dict) -> dict:
    """SURVEY.md 8(d): bytes_alg = 4*C_j + 24*R + 12*L + 16*P + 17*L (each CIGAR word counted once)."""
    Cj, R, L, P = st["n_cigar_words_joined"], st["n_reads"], st["n_loci"], st["n_pairs"]
    Rj = st["n_reads_joined"]
    return {
        "pipeline": 4 * Cj + 24 * R + 12 * L + 16 * P + 17 * L,
        # what the dominant kernel (k_cigar_scan) must touch: the joined reads' packed CIGAR words once,
        # plus cigar_off (8 B) and ref_start (4 B) of those reads
        "cigar_scan": 4 * Cj + 12 * Rj,
    }


def cpu_reference(w, threads: int, seconds: float):
    """Times the oracle (CPU restatement of call.rs:103-158,279-522; the reference itself is a Rust
    crate that cannot be built here) on a bounded sample of the workload's loci, all host threads."""
    from oracle import oracle as O
    n = w.n_loci
    lc = w.locus_contig
    ls = w.locus_start.astype(np.uint32)
    le = w.locus_end.astype(np.uint32)
    # probe on ~1% of the loci (evenly spaced), then size the sample to the time budget
    probe = np.unique(np.linspace(0, n - 1, max(1, min(n, n // 100 + 1))).astype(np.int64))
    t0 = time.perf_counter()
    O.genotype_loci(w.reads, w.n_contigs, lc[probe], ls[probe], le[probe], w.minlen, w.support, w.unphased, threads)
    t_probe = time.perf_counter() - t0          # includes building the read index (the oracle's "fetch")
    t1 = time.perf_counter()
    O.genotype_loci(w.reads, w.n_contigs, lc[probe], ls[probe], le[probe], w.minlen, w.support, w.unphased, threads)
    t_probe2 = time.perf_counter() - t1
    per_locus = max(t_probe2 / len(probe), 1e-9)
    m = int(min(n, max(len(probe), seconds / per_locus)))
    sel = np.unique(np.linspace(0, n - 1, m).astype(np.int64))
    t2 = time.perf_counter()
    rc, p1, p2, visits = O.genotype_loci(w.reads, w.n_contigs, lc[sel], ls[sel], le[sel], w.minlen, w.support,
                                         w.unphased, threads)
    dt = time.perf_counter() - t2
    return {
        "value": len(sel) / dt, "unit": "loci/s", "cores": threads, "kind": "port",
        "sample": f"{len(sel)} of {n} loci (evenly spaced) against all {w.reads.n} resident reads, "
                  f"{dt:.2f} s incl. in-memory read index build; per-locus fetch/BGZF inflate of the real "
                  f"reference is NOT included (oracle restatement of call.rs, reference is Rust and cannot be built here)",
        "op_visits_per_s": visits / dt, "seconds": dt, "rc": rc,
    }, (sel, p1, p2)


def cohort_outlier_block(peak_gbs: float) -> dict:
    """`inquistr-b200 outlier` kernels (include/inqcohort.h) on a 200,000 loci x 536 haplotype-column matrix (268 samples,
    the cohort size of the reference's README): kernel time by CUDA events (H2D excluded), algorithmic bytes = 4 B per
    value read once, parity of the first 2,000 rows against the oracle (outlier.rs restated)."""
    from inquistr_b200 import cohort
    from oracle import oracle as O
    rng = np.random.default_rng(9)
    rows, cols = 200_000, 536
    m = (np.round(rng.gamma(2.0, 15.0, (rows, cols)) * 2) / 2).astype(np.float32)
    m[rng.random(m.shape) < 0.05] = np.nan
    big = rng.random(rows) < 0.2
    m[big, rng.integers(0, cols, big.sum())] = rng.integers(150, 3000, big.sum())
    out = {"workload": f"{rows} x {cols} f32, 5% NaN, 20% of the rows carry one expansion", "bound": "hbm", "peak": peak_gbs, "unit": "GB/s"}
    for method, kernel in (("zscore", "k_outlier_zscore_warp"), ("dbscan", "k_outlier_dbscan")):
        best = None
        for _ in range(3):
            kept, hr, hc, ms = cohort.outlier(m, 10, 3.0, method)
            best = ms if best is None else min(best, ms)
        n = 2000
        k2, f2, _ = O.outlier_matrix(m[:n], 10, 3.0, method)
        er, ec = np.nonzero(f2)
        sel = hr < n
        ok = bool(np.array_equal(kept[:n], k2) and np.array_equal(hr[sel], er) and np.array_equal(hc[sel], ec))
        gbps = m.nbytes / (best * 1e-3) / 1e9
        out[method] = {"kernel": kernel, "kernel_ms": best, "achieved": gbps, "frac": gbps / peak_gbs, "rows_per_s": rows / (best * 1e-3),
                       "outliers": int(len(hr)), "parity_first_rows": {"rows": n, "bit_exact_vs_oracle": ok}}
    return out


def emit(line: dict) -> None:
    """The one JSON line goes to the real stdout; everything else this process (or NCCL) prints to fd 1
    was redirected to stderr in main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)               # libraries that print to stdout (e.g. "NCCL version ...") must not break the contract
    rank, local_rank, world = dist_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    threads = os.cpu_count() or 1
    affinity = None
    if world > 1 and args.impl == "ours" and hasattr(os, "sched_setaffinity"):
        # one process per GPU, each on its own slice of the host cores: the routing / packing threads of a rank and
        # its launch thread do not migrate onto another rank's cores
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = len(cores) // world
            if per >= 1:
                mine = cores[local_rank * per:(local_rank + 1) * per]
                os.sched_setaffinity(0, mine)
                affinity = f"{per} cores per rank"
                threads = len(cores)
        except OSError:
            affinity = None

    from synth.synth import make_workload

    config_desc = {
        "workload": None, "config_index": args.config, "scale": args.scale, "minlen": 5, "support": 3,
        "sharding": f"locus catalog range-sharded over {world} rank(s), no collective",
        "l2": "inputs (packed CIGAR stream) are far larger than the 126 MB L2; no flush needed",
        "timed_region": "per rank: barrier + synchronize, K calls, synchronize; the job's time is the max over ranks; the closing barrier follows the clock",
        "data_seed": args.config,
        "pack_filter": (not args.no_pack_filter),
        "pack_filter_note": "the host packer drops reads that fail the per-read part of call.rs:297-300/350-352 for every "
                            "locus (mapq <= 10; phased: no HP tag), like `inquistr-b200 call` does; both arms get the same reads",
    }

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        w = make_workload(args.config, scale=args.scale, threads=threads, pack_filter=not args.no_pack_filter)
        config_desc["workload"] = w.name
        config_desc["unphased"] = bool(w.unphased)
        vals = []
        base = None
        steps = max(1, args.steps)
        per_step = max(2.0, min(args.cpu_seconds, 120.0 / (steps + max(args.warmup, 0))))
        for i in range(max(args.warmup, 0) + steps):
            base, _ = cpu_reference(w, threads, per_step)
            if i >= args.warmup:
                vals.append(base["value"])
        v = float(np.mean(vals))
        line = {
            "impl": "reference", "metric": "str_loci_genotyped_per_s", "value": v, "unit": "loci/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * base["seconds"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic", "config": config_desc,
            "cpu_baseline": {**{k: base[k] for k in ("unit", "cores", "kind", "sample")}, "value": v},
            "e2e": {"value": v, "unit": "loci/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "cigar_op_visits_per_s": base["op_visits_per_s"], "gpu_launches": 0,
        }
        emit(line)
        return 0

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_ranks(x: float) -> list:
        if world == 1:
            return [x]
        t = torch.zeros(world, dtype=torch.float64, device="cuda")
        t[rank] = x
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    import inquistr_b200 as q

    t_gen = time.perf_counter()
    w = make_workload(args.config, scale=args.scale, threads=max(1, threads // max(1, world)), pinned=True,
                      shard=(rank, world), pack_filter=not args.no_pack_filter)
    t_gen = time.perf_counter() - t_gen
    rd = w.reads
    config_desc["workload"] = w.name
    config_desc["unphased"] = bool(w.unphased)

    ctx = q.Context(local_rank)
    if args.ranges is not None:
        ctx.set_option("ranges", args.ranges)
    if args.no_graph:
        ctx.set_option("graph", 0)
    for kv in args.set:
        name, _, val = kv.partition("=")
        ctx.set_option(name, int(val))
    ctx.set_loci(w.contig_locus_off, w.locus_start, w.locus_end)
    ctx.reserve_reads(rd.n, len(rd.cigar))

    def push_all():
        # N > 1: every rank hands its host-side slice of the input (a superset of what its shard needs: everything
        # that starts within one maximal read length of the shard) to the routed push, which keeps what htslib's
        # fetch would return for some locus of the shard -- the routing cost is inside the e2e timed region
        if world > 1:
            return ctx.push_routed(rd, host_threads=max(1, threads // world))
        ctx.push(rd)
        return rd.n

    n_pushed = push_all()
    # results land in pinned host memory (the D2H read of every step's result is inside both timed regions)
    out = (q.pinned_empty(w.n_loci, np.int64), q.pinned_empty(w.n_loci, np.int64), q.pinned_empty(w.n_loci, np.uint8))

    # warm-up (also sizes the speculative event / bucket buffers)
    res = None
    for _ in range(max(args.warmup, 3)):
        res = ctx.genotype(w.minlen, w.support, w.unphased, out=out)
    st0 = res.stats

    # ---- timed: device-resident inputs
    clocks = Clocks(local_rank) if rank == 0 else None
    barrier()
    dev_ms, cigar_ms, stage_ms = 0.0, 0.0, {}
    call, cst = ctx.genotype_fn(w.minlen, w.support, w.unphased, out)     # pre-bound C call: no Python work inside the timed loop
    stage_keys = ("ms_index", "ms_join", "ms_cigar", "ms_fixup", "ms_scan", "ms_pairs", "ms_median", "ms_d2h")
    acc = [0.0, 0.0]
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rc = call()
        if rc != 0:
            raise SystemExit(f"inq_genotype failed with {rc}")
        acc[0] += cst.ms_total
        acc[1] += cst.ms_cigar
    torch.cuda.synchronize()
    t_rank = time.perf_counter() - t0
    barrier()
    # every inq_genotype call ends with a synchronize of the library's streams, so each rank's bracket
    # barrier -> K calls -> synchronize is device time + launch gaps + the D2H of the results; the job's time is
    # the slowest rank's (the closing barrier's own NCCL latency is not part of any rank's K steps)
    wall_resident = max_over_ranks(t_rank)
    wall_per_rank = gather_ranks(t_rank / args.steps * 1e3)
    dev_ms = acc[0]
    cigar_ms = acc[1]
    dev_ms_max = max_over_ranks(dev_ms)
    dev_per_rank = gather_ranks(dev_ms / args.steps)
    st = cst.as_dict()
    res = q.GenotypeResult(out[0], out[1], out[2], st)
    # phase1 / phase2 are fresh arrays: the e2e and diagnostic passes below overwrite `out`
    last_step = (res.phase1, res.phase2) if args.dump_outputs else None

    # ---- timed: end to end from pinned host buffers through the C ABI
    e2e = None
    if not args.no_e2e:
        barrier()
        t1 = time.perf_counter()
        for _ in range(args.steps):
            ctx.set_loci(w.contig_locus_off, w.locus_start, w.locus_end)
            ctx.clear_reads()
            push_all()
            res2 = ctx.genotype(w.minlen, w.support, w.unphased, out=out)
        torch.cuda.synchronize()
        e2e_rank = time.perf_counter() - t1
        barrier()
        e2e_s = max_over_ranks(e2e_rank)
        h2d = rd.nbytes() + w.locus_start.nbytes + w.locus_end.nbytes + w.contig_locus_off.nbytes
        d2h = out[0].nbytes + out[1].nbytes + out[2].nbytes
        e2e = {"seconds_per_step": e2e_s / args.steps, "h2d_bytes_per_step": int(sum_over_ranks(h2d)),
               "d2h_bytes_per_step": int(sum_over_ranks(d2h)), "ms_h2d_last": res2.stats["ms_h2d"]}
    clk = clocks.stop() if clocks else None

    # ---- diagnostic, outside every timed region: the per-stage event records (timing level 2) cost ~5 us apiece on
    #      the chain of the replayed graph, so the timed steps run with the three records of level 1 only
    ctx.set_option("timing", 2)
    for _ in range(3):
        res = ctx.genotype(w.minlen, w.support, w.unphased, out=out)
    n_diag = 5
    acc2 = {k: 0.0 for k in stage_keys}
    for _ in range(n_diag):
        res = ctx.genotype(w.minlen, w.support, w.unphased, out=out)
        for k in stage_keys:
            acc2[k] += res.stats[k]
    stage_ms = {k: v / n_diag for k, v in acc2.items()}
    ctx.set_option("timing", 1)

    tot_loci = sum_over_ranks(st["n_loci"])
    cj_per_rank = [int(v) for v in gather_ranks(float(st["n_cigar_words_joined"]))]
    tot_words = sum_over_ranks(st["n_cigar_words"])
    tot_words_j = sum_over_ranks(st["n_cigar_words_joined"])
    tot_visits = sum_over_ranks(st["op_visits"])
    tot_pairs = sum_over_ranks(st["n_pairs"])
    tot_reads = sum_over_ranks(st["n_reads"])
    sec_per_step = wall_resident / args.steps                # whole call, max over ranks
    dev_sec_per_step = dev_ms_max / 1e3 / args.steps          # kernels only (CUDA events on the library's stream)
    value = tot_loci / sec_per_step

    # ---- roofline of the dominant kernel (rank 0's shard)
    peaks = {}
    peak_src = "fallback 6650 GB/s (B200_PROFILING.md)"
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak = float(peaks["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except Exception:
        peak = 6650.0
    ab = algorithmic_bytes(st)
    ms_cigar = cigar_ms / args.steps
    achieved = ab["cigar_scan"] / (ms_cigar * 1e-3) / 1e9 if ms_cigar > 0 else 0.0
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = f"config{args.config}_scale{args.scale:g}_gpus{world}" + ("" if not args.no_pack_filter else "_nofilter")
        ent = tj.get(key)
        if ent:
            traffic = ent["k_cigar_scan_dram_bytes_per_launch"]
    except Exception:
        pass
    step_ms = sec_per_step * 1e3
    roofline = {
        "kernel": "k_cigar_scan", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
        "formula": "achieved = (4*C_j + 12*R_j) / ms_per_launch: the packed CIGAR words of reads joined to >= 1 locus, once, "
                   "plus cig_off (8 B) and ref_start (4 B) of those reads; the other 12 B of SURVEY 8(d)'s 24 B read record "
                   "are read by k_join_ranges / k_pair_eval and count in pipeline_* only",
        "algorithmic_bytes_per_launch": ab["cigar_scan"], "ms_per_launch": ms_cigar,
        "launches_per_step": int(st["n_ranges"]),
        "ms_note": "one launch per range of the pass; ms_per_launch is the SUM over the ranges of a step (CUDA events on "
                   "the launching stream), i.e. the time to scan the whole stream once, while k_pair_eval / k_locus_median "
                   "of the previous range share the SMs",
        "bytes_streamed_per_launch": 4 * st["n_cigar_words"],
        "streamed_GBps": 4 * st["n_cigar_words"] / (ms_cigar * 1e-3) / 1e9 if ms_cigar > 0 else 0.0,
        "pipeline_algorithmic_bytes": ab["pipeline"],
        "pipeline_formula": "4*C_j + 24*R + 12*L + 16*P + 17*L (SURVEY 8d) / ms_per_step (the driver-timed step, not the device time)",
        "pipeline_GBps": ab["pipeline"] / (step_ms * 1e-3) / 1e9 if step_ms > 0 else 0.0,
        "pipeline_frac": (ab["pipeline"] / (step_ms * 1e-3) / 1e9 / peak) if step_ms > 0 else 0.0,
        "frac_of_nominal_8TBps": achieved / 8000.0,
    }

    # ---- CPU baseline (rank 0, N=1 only) + parity check of the GPU result against the oracle (every rank, every N)
    cpu = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        cpu, (sel, p1, p2) = cpu_reference(w, threads, args.cpu_seconds)
        g1, g2 = res.phase1[sel], res.phase2[sel]
        ok = bool(np.array_equal(g1, p1, equal_nan=True) and np.array_equal(g2, p2, equal_nan=True))
        parity = {"loci_checked": int(len(sel)), "bit_exact_vs_oracle": ok, "ranks_checked": 1}
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "op_visits_per_s")}
    elif world > 1:
        # every rank checks a bounded sample of ITS shard's GPU output against the oracle on its shard's reads
        _, (sel, p1, p2) = cpu_reference(w, max(1, threads // world), args.parity_seconds)
        g1, g2 = res.phase1[sel], res.phase2[sel]
        ok = bool(np.array_equal(g1, p1, equal_nan=True) and np.array_equal(g2, p2, equal_nan=True))
        n_bad = sum_over_ranks(0.0 if ok else 1.0)
        n_chk = sum_over_ranks(float(len(sel)))
        parity = {"loci_checked": int(n_chk), "bit_exact_vs_oracle": bool(n_bad == 0), "ranks_checked": world,
                  "note": "each rank: evenly spaced sample of its catalog shard, oracle on the shard's reads"}

    # ---- BAM -> TSV through the product CLI (rank 0; the other ranks idle at the barrier below)
    e2e_bam = None
    if rank == 0 and args.bam_scale > 0 and not args.no_e2e:
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_bam.py"), "--config", "3", "--scale", str(args.bam_scale),
                                "--with-seq", "-t", str(threads), "--devices", ",".join(str(i) for i in range(world))],
                               capture_output=True, text=True, timeout=900)
            if r.returncode == 0:
                e2e_bam = json.loads(r.stdout.strip().splitlines()[-1])
                e2e_bam.pop("cli_stats", None)
                e2e_bam["note"] = ("inquistr-b200 call -R loci.bed -t N --devices ... sample.bam: BGZF inflate (own decoder, zlib fallback) + "
                                   "record parse + routing + pinned pushes + kernels + TSV, one process, page-cache-warm file; "
                                   "loci_per_s is over the whole process wall time incl. CUDA context creation")
            else:
                e2e_bam = {"error": r.stderr[-400:]}
        except Exception as ex:          # the headline numbers do not depend on this leg
            e2e_bam = {"error": repr(ex)}
    # ---- cohort follow-on kernels (SURVEY 8f rank 3), so that the driver's record carries their numbers too
    cohort_block = None
    if rank == 0 and world == 1 and not args.no_cohort:
        try:
            cohort_block = cohort_outlier_block(peak)
        except Exception as ex:
            cohort_block = {"error": repr(ex)}
    if args.dump_outputs:
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, last_step)          # the ranks' catalog shards are contiguous, in rank order
            last_step = tuple(np.concatenate([p[k] for p in parts]) for k in (0, 1))
        if rank == 0:
            dump_outputs(args.dump_outputs, *last_step)
    if world > 1:
        dist.barrier()

    if rank == 0:
        line = {
            "metric": "str_loci_genotyped_per_s", "value": value, "unit": "loci/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": sec_per_step * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic", "config": config_desc,
            "cigar_ops_per_s": tot_words_j / sec_per_step,
            "cigar_op_visits_per_s_reference_equivalent": tot_visits / sec_per_step,
            "counts": {"loci": int(tot_loci), "reads": int(tot_reads), "cigar_words": int(tot_words),
                       "cigar_words_joined": int(tot_words_j), "pairs": int(tot_pairs),
                       "events_rank0": int(st["n_events"]), "tiles_rank0": int(st["n_tiles"])},
            "device_ms_per_step": dev_sec_per_step * 1e3,
            "per_rank": {"ms_per_step": [round(v, 4) for v in wall_per_rank], "device_ms_per_step": [round(v, 4) for v in dev_per_rank],
                         "cigar_words_joined": cj_per_rank},
            "stage_ms_rank0": stage_ms,
            "pipeline": {"ranges": int(st["n_ranges"]), "median_chunks": int(st["n_median_chunks"]),
                         "cuda_graph": bool(st["used_graph"]), "reads_sorted": bool(st["reads_sorted"]),
                         "note": "stage_ms: separate passes with one event record per stage (timing level 2, ~50 us slower than the timed steps); per-stage sums under overlap, they add up to more than the step"},
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": None if e2e is None else {
                "value": tot_loci / e2e["seconds_per_step"], "unit": "loci/s",
                "h2d_bytes_per_step": e2e["h2d_bytes_per_step"], "d2h_bytes_per_step": e2e["d2h_bytes_per_step"],
                "seconds_per_step": e2e["seconds_per_step"], "ms_h2d_rank0": e2e["ms_h2d_last"],
                "cigar_ops_per_s": tot_words_j / e2e["seconds_per_step"]},
            "e2e_bam": e2e_bam,
            "extra": {"cohort_outlier": cohort_block},
            "gpu_launches": int(st["n_kernel_launches"]) * args.steps,
            "clocks": clk,
            "parity": parity,
            "host": {"cores": threads, "affinity": affinity, "gen_seconds": t_gen, "wall_resident_s": wall_resident,
                     "reads_host_rank0": int(rd.n), "reads_pushed_rank0": int(n_pushed),
                     "push": "inq_push_reads_routed" if world > 1 else "inq_push_reads"},
        }
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
