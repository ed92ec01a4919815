"""CPU-only checks (-m "not gpu"): golden fixtures vs the oracle, C-ABI exports, the synthetic
generator, range-sharding (world_size 2 over gloo), the reference arm of bench.py and its output dump."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def load_golden(name):
    z = np.load(os.path.join(GOLD, name + ".npz"))
    rd = O.Reads(z["contig"], z["ref_start"], z["ref_end"], z["mapq"], z["hp"], z["flags"], z["cigar_off"], z["cigar"])
    runs = sorted({k[:-3] for k in z.files if k.endswith("_p1")})
    return z, rd, runs


def parse_run(key):
    m = re.match(r"m(\d+)_s(\d+)_u(\d)", key)
    return int(m.group(1)), int(m.group(2)), bool(int(m.group(3)))


@pytest.mark.parametrize("name", ["random_edge_cases", "expansion_panel"])
def test_oracle_matches_golden(name):
    z, rd, runs = load_golden(name)
    assert runs
    for key in runs:
        minlen, support, unphased = parse_run(key)
        rc, p1, p2, visits = O.genotype_loci(rd, int(z["n_contigs"]), z["locus_contig"], z["locus_start"].astype(np.uint32),
                                             z["locus_end"].astype(np.uint32), minlen, support, unphased, threads=3)
        assert rc == 0
        assert np.array_equal(p1, z[key + "_p1"], equal_nan=True)
        assert np.array_equal(p2, z[key + "_p2"], equal_nan=True)
        assert visits == int(z[key + "_visits"])


def test_golden_python_mirror_spot_check():
    z, rd, runs = load_golden("random_edge_cases")
    for key in runs[:2]:
        minlen, support, unphased = parse_run(key)
        for i in range(0, len(z["locus_start"]), 7):
            q1, q2 = O.py_genotype_locus(rd, int(z["locus_contig"][i]), int(z["locus_start"][i]), int(z["locus_end"][i]),
                                         minlen, support, unphased)
            for a, b in ((q1, z[key + "_p1"][i]), (q2, z[key + "_p2"][i])):
                assert (np.isnan(a) and np.isnan(b)) or a == b


def test_expansion_panel_has_clip_topup_and_kb_alleles():
    z, _, _ = load_golden("expansion_panel")
    assert np.nanmax(z["m5_s3_u0_p2"]) >= 1000        # H2 carries the 1-10 kb insertion


# ------------------------------------------------------------------------------------- C ABI
def test_cabi_exports_every_declared_symbol():
    import inquistr_b200 as q
    from inquistr_b200 import api
    from inquistr_b200 import cohort
    from inquistr_b200 import bgzf
    hdr = "".join(open(os.path.join(ROOT, "include", h)).read() for h in ("inqcall.h", "inqcohort.h", "inqbgzf.h"))
    declared = sorted(set(re.findall(r"\b(inq_[a-z0-9_]+)\s*\(", hdr)))
    assert set(declared) == set(api.EXPORTS) | set(cohort.EXPORTS) | set(bgzf.EXPORTS), (declared, api.EXPORTS, cohort.EXPORTS, bgzf.EXPORTS)
    lib = q.load_library()
    for name in declared:
        assert hasattr(lib, name), name
    assert b"sm_100a" in lib.inq_version()
    # plain C ABI: no C++ mangled inq_ symbols are exported
    out = subprocess.run(["nm", "-D", "--defined-only", os.path.join(ROOT, "inquistr_b200", "lib", "libinqcall.so")],
                         capture_output=True, text=True).stdout
    exported = [l.split()[-1] for l in out.splitlines() if " T " in l]
    assert all(not s.startswith("_Z") or "inq_" not in s for s in exported if "inq_ctx" in s)
    assert all(name in exported for name in declared)


def test_no_cpu_fallback_in_product_path():
    import torch
    import inquistr_b200 as q
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(q.InqError) as ei:
        q.Context(0)
    assert ei.value.code == -1 and "no CPU fallback" in str(ei.value)
    # nothing under inquistr_b200/ may reference the oracle
    for dirpath, _, files in os.walk(os.path.join(ROOT, "inquistr_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle" not in txt.replace("no CPU fallback", ""), os.path.join(dirpath, f)


def test_inq_stats_layout_matches_header():
    from inquistr_b200.api import Stats
    hdr = open(os.path.join(ROOT, "include", "inqcall.h")).read()
    body = hdr[hdr.index("typedef struct inq_stats {"):hdr.index("} inq_stats;")]
    fields = re.findall(r"^\s*(uint64_t|uint32_t|float)\s+([a-z0-9_]+);", body, flags=re.M)
    cmap = {"uint64_t": ctypes.c_uint64, "uint32_t": ctypes.c_uint32, "float": ctypes.c_float}
    assert [(n, cmap[t]) for t, n in fields] == list(Stats._fields_)


# ------------------------------------------------------------------------------------- synth
def test_synth_deterministic_and_sorted():
    from synth.synth import make_workload
    a = make_workload(3, scale=0.0005, threads=1)
    b = make_workload(3, scale=0.0005, threads=4)
    for name in ("contig", "ref_start", "ref_end", "mapq", "hp", "flags", "cigar_off", "cigar"):
        assert np.array_equal(getattr(a.reads, name), getattr(b.reads, name)), name
    key = a.reads.contig.astype(np.int64) * (1 << 32) + a.reads.ref_start
    assert np.all(np.diff(key) >= 0)
    lk = a.locus_contig.astype(np.int64) * (1 << 32) + a.locus_start
    assert np.all(np.diff(lk) >= 0) and np.all(a.locus_start >= 10)
    assert np.all(a.locus_end < a.contig_len[a.locus_contig])
    # ref_end is bam_endpos of the generated CIGAR
    ops = a.reads.cigar & 15
    cons = np.where(np.isin(ops, [0, 2, 3, 7, 8]), (a.reads.cigar >> 4).astype(np.int64), 0)
    cs = np.concatenate([[0], np.cumsum(cons)])
    rl = cs[a.reads.cigar_off[1:].astype(np.int64)] - cs[a.reads.cigar_off[:-1].astype(np.int64)]
    assert np.array_equal(a.reads.ref_start + np.maximum(rl, 1), a.reads.ref_end)


@pytest.mark.parametrize("cfg,scale", [(1, 1.0), (2, 0.004), (4, 1.0)])
def test_synth_configs_recover_planted_alleles(cfg, scale):
    from synth.synth import make_workload
    w = make_workload(cfg, scale=scale, threads=2)
    rc, p1, p2, _ = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig, w.locus_start.astype(np.uint32),
                                    w.locus_end.astype(np.uint32), w.minlen, w.support, w.unphased, threads=2)
    assert rc == 0
    if not w.unphased:
        big = np.abs(w.delta_h2) > 5
        assert np.mean(p2[big] == w.delta_h2[big]) > 0.9


def test_shard_helpers_cover_every_pair():
    from inquistr_b200 import shard as S
    from synth.synth import make_workload
    w = make_workload(3, scale=0.0006, threads=2)
    rc, g1, g2, _ = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig, w.locus_start.astype(np.uint32),
                                    w.locus_end.astype(np.uint32), 5, 3, False, threads=2)
    parts1, parts2 = [], []
    for lo, hi in S.split_catalog(w.n_loci, 3):
        off, ls, le = S.shard_catalog(w.contig_locus_off, w.locus_start, w.locus_end, lo, hi)
        sub = S.take_reads(w.reads, S.reads_for_shard(w.reads.contig, w.reads.ref_start, w.reads.ref_end, off, ls, le))
        rd = O.Reads(**sub)
        lc = np.repeat(np.arange(w.n_contigs, dtype=np.int32), np.diff(off))
        rc, p1, p2, _ = O.genotype_loci(rd, w.n_contigs, lc, ls.astype(np.uint32), le.astype(np.uint32), 5, 3, False, threads=2)
        assert rc == 0
        parts1.append(p1); parts2.append(p2)
    assert np.array_equal(S.concat_ordered(parts1), g1, equal_nan=True)
    assert np.array_equal(S.concat_ordered(parts2), g2, equal_nan=True)


# ------------------------------------------------------------------------------------- world_size 2 (gloo)
def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from synth.synth import make_workload
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    w = make_workload(3, scale=0.0006, threads=1, shard=(rank, world))       # what bench.py does per rank
    rc, p1, p2, _ = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig, w.locus_start.astype(np.uint32),
                                    w.locus_end.astype(np.uint32), 5, 3, False, threads=1)
    gathered = [None] * world
    dist.all_gather_object(gathered, (rank, w.locus_range, p1, p2, rc))
    dist.barrier()
    if rank == 0:
        q.put(gathered)
    dist.destroy_process_group()


def test_range_sharding_world_size_2_gloo():
    import torch.multiprocessing as mp
    from synth.synth import make_workload
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    gathered = q.get(timeout=180)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    gathered.sort(key=lambda t: t[0])
    assert all(g[4] == 0 for g in gathered)
    assert gathered[0][1][1] == gathered[1][1][0]                     # contiguous ranges
    w = make_workload(3, scale=0.0006, threads=2)
    rc, g1, g2, _ = O.genotype_loci(w.reads, w.n_contigs, w.locus_contig, w.locus_start.astype(np.uint32),
                                    w.locus_end.astype(np.uint32), 5, 3, False, threads=2)
    assert np.array_equal(np.concatenate([g[2] for g in gathered]), g1, equal_nan=True)
    assert np.array_equal(np.concatenate([g[3] for g in gathered]), g2, equal_nan=True)


# ------------------------------------------------------------------------------------- bench reference arm
def test_bench_reference_arm_prints_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--scale", "0.002",
                          "--steps", "1", "--warmup", "0", "--cpu-seconds", "1"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "loci/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_rejects_zero_steps_and_a_reference_dump(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=60)
        assert out.returncode == 2 and out.stdout == "", extra
    assert os.listdir(tmp_path) == []


def test_bench_dump_outputs_float64_and_size_cap(tmp_path, monkeypatch):
    import bench
    rng = np.random.default_rng(3)
    p1 = rng.integers(0, 400, 1000) / 2.0
    p2 = p1 + 1.5
    p1[::7] = np.nan
    p1[0] = 0.0                                     # a called median of 0 stays apart from "no call" through the mask
    p2[::11] = np.nan
    bench.dump_outputs(str(tmp_path / "all"), p1, p2)
    files = ["phase1.npy", "phase2.npy", "valid_mask.npy"]
    assert sorted(os.listdir(tmp_path / "all")) == files
    a1, a2, vm = (np.load(tmp_path / "all" / f) for f in files)
    assert a1.dtype == a2.dtype == vm.dtype == np.float64
    assert all(np.isfinite(a).all() for a in (a1, a2, vm))
    assert np.array_equal(vm, np.where(np.isnan(p1), 0, 1) + np.where(np.isnan(p2), 0, 2))
    assert np.array_equal(np.where(vm % 2 == 1, a1, np.nan), p1, equal_nan=True)
    assert np.array_equal(np.where(vm >= 2, a2, np.nan), p2, equal_nan=True)
    assert np.all(a1[np.isnan(p1)] == 0) and np.all(a2[np.isnan(p2)] == 0)
    # over the cap: a fixed seeded sample of the loci, the same on every run, with its catalog indices
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 4 * 8 * 100)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), p1, p2)
    files = ["locus_index.npy", "phase1.npy", "phase2.npy", "valid_mask.npy"]
    assert sorted(os.listdir(tmp_path / "s1")) == files
    assert sum(os.path.getsize(tmp_path / "s1" / f) for f in files) <= 4 * 8 * 100 + 4 * 128
    for f in files:
        a = np.load(tmp_path / "s1" / f)
        assert np.isfinite(a).all() and np.array_equal(a, np.load(tmp_path / "s2" / f))
    idx = np.load(tmp_path / "s1" / "locus_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 100 and np.all(np.diff(idx) > 0)
    k = idx.astype(np.int64)
    for f in ("phase1.npy", "phase2.npy", "valid_mask.npy"):
        assert np.array_equal(np.load(tmp_path / "s1" / f), np.load(tmp_path / "all" / f)[k])
