#!/usr/bin/env python
"""`inquistr-b200 call-cohort` against the shell way of genotyping a cohort (one `call` process per BAM, then
`combine`), on two synthetic cohorts that share one catalog per workload:
  A  32 indexed panel BAMs (config 4 catalog of seed 1, reads of seeds 1..32)
  B   8 genome BAMs (config 3 at scale 0.05, catalog of seed 1, reads of seeds 1..8)
Records carry no SEQ/QUAL unless --with-seq (which makes workload A's files ~30x larger and slow to index here).
Per workload: wall time of `call-cohort` on one device and on every device, of the `call` loop run sequentially and
with one process per device in parallel (+ `combine`), the per-sample `s_bam_scan` / `ms_total` of the cohort run,
and whether every output is byte-identical. One JSON line, with the card's name and power limit. Usage:
  python tools/bench_cohort.py [--workloads A,B] [--reps 2] [--with-seq] [--keep DIR]"""
import argparse, json, os, shutil, statistics, subprocess, sys, tempfile, time
from concurrent.futures import ThreadPoolExecutor
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from synth import synth as S
from tests import bamio

ap = argparse.ArgumentParser()
ap.add_argument("--workloads", default="A,B")
ap.add_argument("--reps", type=int, default=2, help="each way is timed this many times, the ways alternating")
ap.add_argument("--with-seq", action="store_true")
ap.add_argument("--keep", default=None)
ap.add_argument("--gen-threads", type=int, default=0)
a = ap.parse_args()

from inquistr_b200 import build
cli = build.build_cli()
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
if smi.returncode != 0 or not smi.stdout.strip():
    raise SystemExit("bench_cohort.py needs a CUDA device (no CPU fallback)")
cards = [ln.strip() for ln in smi.stdout.strip().splitlines()]
n_gpus = len(cards)
all_devs = ",".join(str(g) for g in range(n_gpus))
root = a.keep or tempfile.mkdtemp(prefix="inqcohort")
os.makedirs(root, exist_ok=True)

WORKLOADS = {"A": dict(config=4, scale=1.0, n=32, index=True),
             "B": dict(config=3, scale=0.05, n=8, index=False)}


def timed(args, env=None):
    t0 = time.perf_counter()
    r = subprocess.run(args, capture_output=True, env={**os.environ, **(env or {})})
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        raise SystemExit(f"{' '.join(args[:3])} ... exited {r.returncode}: {r.stderr.decode()[-2000:]}")
    return r.stdout, dt


def call_loop(d, bams, bed, n_par):
    """one `call` per BAM (n_par at a time, process k on device k % n_par), then `combine`"""
    t0 = time.perf_counter()
    outs = [os.path.join(d, f"call_{k}.tsv") for k in range(len(bams))]

    def one(k):
        out, _ = timed([cli, "call", "-R", bed, "--devices", str(k % n_par), bams[k]])
        open(outs[k], "wb").write(out)
    with ThreadPoolExecutor(n_par) as ex:
        list(ex.map(one, range(len(bams))))
    table, _ = timed([cli, "combine", *outs])
    return table, time.perf_counter() - t0


res = {"cards": cards, "n_gpus": n_gpus, "workloads": {}}
for name in a.workloads.split(","):
    p = WORKLOADS[name]
    d = os.path.join(root, name)
    os.makedirs(d, exist_ok=True)
    t0 = time.perf_counter()
    bams, ws = [], []
    for k in range(1, p["n"] + 1):
        w = S.make_workload(p["config"], scale=p["scale"], seed=1, read_seed=k, threads=a.gen_threads)
        bam = os.path.join(d, f"s{k}.bam")
        S.write_bam(w, bam, with_seq=a.with_seq, threads=a.gen_threads)
        if p["index"]:
            bamio.index_bam(bam)
        bams.append(bam)
        ws.append(w)
    bed = os.path.join(d, "loci.bed")
    S.write_bed(ws[0], bed, shuffle_seed=1)
    gen_s = time.perf_counter() - t0

    ways = {"cohort_1_device": None, "call_loop_sequential": None}
    if n_gpus > 1:
        ways.update({f"cohort_{n_gpus}_devices": None, f"call_loop_{n_gpus}_parallel": None})
    walls = {k: [] for k in ways}
    stats = {}
    for rep in range(a.reps):
        for way in ways:
            if way.startswith("cohort"):
                devs = "0" if way == "cohort_1_device" else all_devs
                st = os.path.join(d, f"{way}.json")
                out, dt = timed([cli, "call-cohort", "-R", bed, "--devices", devs, "--stats-json", st, *bams])
                stats[way] = json.load(open(st))
            else:
                out, dt = call_loop(d, bams, bed, 1 if way == "call_loop_sequential" else n_gpus)
            walls[way].append(round(dt, 3))
            ways[way] = out if ways[way] is None or ways[way] == out else b"<differs between repetitions>"
    ref = ways["call_loop_sequential"]
    one = stats["cohort_1_device"]
    scan = [s["s_bam_scan"] for s in one["samples"]]
    dev_ms = [s["ms_total"] for s in one["samples"]]
    res["workloads"][name] = {
        "what": ws[0].name, "samples": len(bams), "loci": ws[0].n_loci, "reads_per_sample": ws[0].reads.n,
        "with_seq": a.with_seq, "indexed": p["index"], "bam_bytes_total": sum(os.path.getsize(b) for b in bams),
        "generate_s": round(gen_s, 1), "wall_s": walls,
        "speedup_cohort_1dev_vs_call_loop": round(min(walls["call_loop_sequential"]) / min(walls["cohort_1_device"]), 2),
        "byte_identical": all(v == ref for v in ways.values()) and not ref.startswith(b"<"),
        "table_bytes": len(ref),
        "cohort_1_device": {"s_total": one["s_total"], "s_ctx_create_set_loci": one["s_ctx_create_set_loci"],
                            "n_contexts": one["n_contexts"], "used_index": one["samples"][0]["used_index"],
                            "s_bam_scan_per_sample": {"median": round(statistics.median(scan), 4), "max": round(max(scan), 4)},
                            "ms_total_per_sample": {"median": round(statistics.median(dev_ms), 4), "max": round(max(dev_ms), 4)}},
    }
res["byte_identical"] = all(w["byte_identical"] for w in res["workloads"].values())
print(json.dumps(res))
if not a.keep:
    shutil.rmtree(root, ignore_errors=True)
