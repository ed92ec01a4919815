#!/usr/bin/env python
"""GPU box: one workload, many builds of libinqcall.so (variants/*.so, compiled on the CPU box with -D
switches by tools/build_variants.sh) x inq_set_option settings. Prints one line per combination:
step time (wall, K calls between synchronisations), per-stage CUDA-event sums, and whether the output
equals the first combination's (which is checked against the oracle on a sample)."""
import argparse
import glob
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--variants", default="variants/*.so")
    ap.add_argument("--graph", default="1", help="comma list of 0/1")
    ap.add_argument("--timing", default="1", help="comma list of 0/1")
    ap.add_argument("--no-pack-filter", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import inquistr_b200 as q
    from inquistr_b200 import api
    from oracle import oracle as O
    from synth.synth import make_workload

    threads = os.cpu_count() or 1
    w = make_workload(args.config, scale=args.scale, threads=threads, pinned=True, pack_filter=not args.no_pack_filter)
    rd = w.reads
    out = (q.pinned_empty(w.n_loci, np.int64), q.pinned_empty(w.n_loci, np.int64), q.pinned_empty(w.n_loci, np.uint8))
    ref = None
    rows = []
    libs = sorted(glob.glob(os.path.join(ROOT, args.variants))) or [api._LIB_PATH]
    for path in libs:
        lib = api.load_library(path)
        for graph in [int(x) for x in args.graph.split(",")]:
            for timing in [int(x) for x in args.timing.split(",")]:
                ctx = q.Context(0, lib=lib)
                ctx.set_option("graph", graph)
                ctx.set_option("timing", timing)
                ctx.set_loci(w.contig_locus_off, w.locus_start, w.locus_end)
                ctx.reserve_reads(rd.n, len(rd.cigar))
                ctx.push(rd)
                for _ in range(3):
                    res = ctx.genotype(w.minlen, w.support, w.unphased, out=out)
                t0 = time.perf_counter()
                stage = {}
                for _ in range(args.steps):
                    res = ctx.genotype(w.minlen, w.support, w.unphased, out=out)
                    for k, v in res.stats.items():
                        if k.startswith("ms_"):
                            stage[k] = stage.get(k, 0.0) + v / args.steps
                ms = (time.perf_counter() - t0) / args.steps * 1e3
                cur = (res.twice_h1.copy(), res.twice_h2.copy(), res.valid.copy())
                if ref is None:
                    ref = cur
                    n = w.n_loci
                    sel = np.unique(np.linspace(0, n - 1, min(n, 20000)).astype(np.int64))
                    rc, p1, p2, _ = O.genotype_loci(rd, w.n_contigs, w.locus_contig[sel], w.locus_start.astype(np.uint32)[sel],
                                                    w.locus_end.astype(np.uint32)[sel], w.minlen, w.support, w.unphased, threads)
                    same = bool(rc == 0 and np.array_equal(res.phase1[sel], p1, equal_nan=True) and
                                np.array_equal(res.phase2[sel], p2, equal_nan=True))
                    tag = "oracle_ok" if same else "ORACLE_MISMATCH"
                else:
                    okv = np.array_equal(ref[2], cur[2])
                    m1, m2 = (cur[2] & 1) != 0, (cur[2] & 2) != 0
                    same = bool(okv and np.array_equal(ref[0][m1], cur[0][m1]) and np.array_equal(ref[1][m2], cur[1][m2]))
                    tag = "same" if same else "DIFFERENT"
                row = {"lib": os.path.basename(path), "graph": res.stats["used_graph"], "timing": timing,
                       "ms_step": round(ms, 4), "chunks": res.stats["n_median_chunks"], "launches": res.stats["n_kernel_launches"],
                       **{k: round(v, 4) for k, v in stage.items() if k != "ms_h2d"}, "check": tag}
                rows.append(row)
                print(json.dumps(row), flush=True)
                ctx.close()
    if args.out:
        json.dump(rows, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
