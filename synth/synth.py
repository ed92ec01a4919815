"""Seeded synthetic workloads for the BASELINE.json configurations (SURVEY.md 8d).

Benchmark / test infrastructure (ctypes front end of synth/libinqsynth.so); not on the product path.

  config 1  stand-in for `call -R test-data/test.bed test-data/small-test.bam` (the BAM is absent from
            the reference checkout): chr7, the single test.bed locus, 30x phased reads around it
  config 2  one 248,956,422 bp contig, 10k loci, 30x, run unphased (-u)
  config 3  hg38 chr1-22,X,Y, 1M loci, 30x, 85% HP-tagged, -m 5 -s 3      (headline)
  config 4  expansion panel: 60 loci, 100x, H2 carries a 1-10 kb insertion, 40% truncated into a clip
  config 5  config 3 at 60x
`scale` shrinks contig lengths and locus counts together (tests use scale << 1).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

HG38 = [
    ("chr1", 248956422), ("chr2", 242193529), ("chr3", 198295559), ("chr4", 190214555),
    ("chr5", 181538259), ("chr6", 170805979), ("chr7", 159345973), ("chr8", 145138636),
    ("chr9", 138394717), ("chr10", 133797422), ("chr11", 135086622), ("chr12", 133275309),
    ("chr13", 114364328), ("chr14", 107043718), ("chr15", 101991189), ("chr16", 90338345),
    ("chr17", 83257441), ("chr18", 80373285), ("chr19", 58617616), ("chr20", 64444167),
    ("chr21", 46709983), ("chr22", 50818468), ("chrX", 156040895), ("chrY", 57227415),
]

GAMMA_SHAPE = 1.3
GAMMA_SCALE = 20000.0 / 1.974      # N50 = median of the length-weighted Gamma(2.3) ~= 1.974 * scale -> 20 kb
MAX_READ = 300_000


class _Cfg(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("n_contigs", C.c_int32), ("threads", C.c_int32),
        ("contig_len", C.c_void_p), ("contig_locus_off", C.c_void_p), ("lstart", C.c_void_p),
        ("lend", C.c_void_p), ("delta_h1", C.c_void_p), ("delta_h2", C.c_void_p),
        ("n_regions", C.c_int64), ("reg_contig", C.c_void_p), ("reg_start", C.c_void_p),
        ("reg_end", C.c_void_p), ("depth", C.c_double), ("gamma_shape", C.c_double),
        ("gamma_scale", C.c_double), ("min_len", C.c_int32), ("max_len", C.c_int32),
        ("mrun_mean", C.c_double), ("indel_mean", C.c_double), ("clip_mean", C.c_double),
        ("p_ins", C.c_double), ("p_clip", C.c_double), ("p_tagged", C.c_double),
        ("p_supp", C.c_double), ("p_2d_given_supp", C.c_double), ("big_delta", C.c_int32),
        ("p_big_trunc", C.c_double), ("sel_lo", C.c_void_p), ("sel_hi", C.c_void_p),
    ]


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "libinqsynth.so")
    src = os.path.join(_HERE, "synth.cpp")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-o", so, src, "-lz"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.synth_loci.restype = C.c_int
        L.synth_loci.argtypes = [C.c_uint64, C.c_int32, C.c_void_p, C.c_int64, C.c_int] + [C.c_void_p] * 5
        L.synth_plan.restype = C.c_uint64
        L.synth_plan.argtypes = [C.POINTER(_Cfg), C.c_void_p]
        L.synth_selected.restype = C.c_uint64
        L.synth_selected.argtypes = [C.POINTER(_Cfg)]
        L.synth_headers.restype = C.c_int
        L.synth_headers.argtypes = [C.POINTER(_Cfg), C.c_uint64] + [C.c_void_p] * 7
        L.synth_cigars.restype = C.c_int
        L.synth_cigars.argtypes = [C.POINTER(_Cfg), C.c_uint64, C.c_void_p, C.c_void_p]
        L.synth_cigars_sel.restype = C.c_int
        L.synth_cigars_sel.argtypes = [C.POINTER(_Cfg), C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.synth_write_bam.restype = C.c_int64
        L.synth_write_bam.argtypes = [C.c_char_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint64] + [C.c_void_p] * 8 + [C.c_int, C.c_int, C.c_int]
        _LIB = L
    return _LIB


@dataclass
class ReadSet:
    contig: np.ndarray
    ref_start: np.ndarray
    ref_end: np.ndarray
    mapq: np.ndarray
    hp: np.ndarray
    flags: np.ndarray
    cigar_off: np.ndarray
    cigar: np.ndarray

    @property
    def n(self) -> int:
        return len(self.contig)

    def nbytes(self) -> int:
        return sum(a.nbytes for a in (self.contig, self.ref_start, self.ref_end, self.mapq, self.hp,
                                      self.flags, self.cigar_off, self.cigar))


@dataclass
class Workload:
    config: int
    name: str
    seed: int
    contig_names: list
    contig_len: np.ndarray           # int64
    contig_locus_off: np.ndarray     # int64 [n_contigs+1]
    locus_start: np.ndarray          # int32, sorted by (contig, start)
    locus_end: np.ndarray
    delta_h1: np.ndarray
    delta_h2: np.ndarray
    reads: ReadSet
    minlen: int = 5
    support: int = 3
    unphased: bool = False
    depth: float = 30.0
    shard: tuple = (0, 1)
    locus_range: tuple = (0, 0)      # [lo, hi) of the global sorted catalog this shard owns
    meta: dict = field(default_factory=dict)

    @property
    def n_contigs(self) -> int:
        return len(self.contig_len)

    @property
    def n_loci(self) -> int:
        return len(self.locus_start)

    @property
    def locus_contig(self) -> np.ndarray:
        return np.repeat(np.arange(self.n_contigs, dtype=np.int32), np.diff(self.contig_locus_off))


def _alloc(n, dtype, pinned):
    if pinned:
        from inquistr_b200.api import pinned_empty
        return pinned_empty(int(n), dtype)
    return np.empty(int(n), dtype=dtype)


def pack_keep_mask(mapq, hp, unphased: bool) -> np.ndarray:
    """The host packer's per-read predicate (`lite_record()` in csrc/host/bam_reader.cpp): a read with mapq <= 10
    fails both filters (call.rs:297-300,350-352), and without an HP tag it fails the phased one, for
    every locus -- such a read can never pair, so the host does not ship it. HP 0 and HP > 2 reads are
    kept: they pass the filter (the reference walks them / panics on them)."""
    keep = np.asarray(mapq) > 10
    if not unphased:
        keep &= np.asarray(hp) != 0xFF
    return keep


def make_workload(config: int, scale: float = 1.0, seed: int | None = None, threads: int = 0,
                  pinned: bool = False, shard: tuple = (0, 1), depth: float | None = None,
                  n_loci: int | None = None, pack_filter: bool = False, read_seed: int | None = None) -> Workload:
    """Build one of the BASELINE.json configurations. `shard=(rank, world)` keeps only the loci of
    the rank's contiguous slice of the sorted catalog and the reads that can overlap them.
    `pack_filter` applies the host packer's per-read predicate (pack_keep_mask) while packing: the same
    reads are drawn, the ones that can never pair are not emitted.
    `read_seed` draws the reads from their own seed over the catalog of `seed`: samples of one cohort."""
    L = lib()
    seed = config if seed is None else seed
    p_tagged, p_big_trunc, mode, unphased = 0.85, 0.0, 0, False
    panel = False
    if config == 1:
        names, lens = ["chr7"], [159345973]
        d, nl, name = 30.0, 1, "cfg1-standin chr7:154778571-154779363 30x phased"
        panel = True
    elif config == 2:
        names, lens = ["chr1"], [248956422]
        d, nl, name, unphased, p_tagged = 30.0, 10_000, "cfg2 1 contig 10k loci 30x unphased", True, 0.0
    elif config in (3, 5):
        names, lens = [n for n, _ in HG38], [l for _, l in HG38]
        d = 30.0 if config == 3 else 60.0
        nl, name = 1_000_000, f"cfg{config} hg38 1M loci {int(d)}x phased"
    elif config == 4:
        names, lens = [n for n, _ in HG38[:22]], [l for _, l in HG38[:22]]
        d, nl, name, mode, p_big_trunc = 100.0, 60, "cfg4 expansion panel 60 loci 100x", 1, 0.4
        panel = True
    else:
        raise ValueError(f"unknown config {config}")
    if depth is not None:
        d = depth
    if scale != 1.0 and not panel:
        lens = [max(int(l * scale), 400_000) for l in lens]
        nl = max(int(nl * scale), 1)
        name += f" (scale {scale:g})"
    if n_loci is not None:
        nl = n_loci
    nc = len(lens)
    contig_len = np.asarray(lens, dtype=np.int64)

    # ---- catalog
    off = np.zeros(nc + 1, np.int64)
    ls = np.zeros(nl, np.int32); le = np.zeros(nl, np.int32)
    d1 = np.zeros(nl, np.int32); d2 = np.zeros(nl, np.int32)
    if config == 1:
        off[:] = [0, 1]; ls[0], le[0] = 154778571, 154779363    # test-data/test.bed:1
        d1[0], d2[0] = 0, 36
    else:
        rc = L.synth_loci(seed, nc, contig_len.ctypes.data, nl, mode, off.ctypes.data, ls.ctypes.data,
                          le.ctypes.data, d1.ctypes.data, d2.ctypes.data)
        assert rc == 0

    # ---- shard: contiguous slice of the sorted catalog
    from inquistr_b200.shard import split_catalog
    rank, world = shard
    lo, hi = split_catalog(nl, world)[rank]
    lcontig = np.repeat(np.arange(nc, dtype=np.int32), np.diff(off))

    # ---- regions where reads are placed
    if panel:
        reg_c = lcontig.copy()
        reg_s = np.maximum(ls.astype(np.int64) - 40_000, 0)
        reg_e = np.minimum(le.astype(np.int64) + 2_000, contig_len[lcontig] - 1)
    else:
        reg_c = np.arange(nc, dtype=np.int32)
        reg_s = np.zeros(nc, np.int64)
        reg_e = contig_len - 1
    cfg = _Cfg()
    cfg.seed, cfg.n_contigs, cfg.threads = (seed if read_seed is None else read_seed), nc, threads
    cfg.contig_len = contig_len.ctypes.data
    cfg.contig_locus_off, cfg.lstart, cfg.lend = off.ctypes.data, ls.ctypes.data, le.ctypes.data
    cfg.delta_h1, cfg.delta_h2 = d1.ctypes.data, d2.ctypes.data
    reg_c = np.ascontiguousarray(reg_c, np.int32); reg_s = np.ascontiguousarray(reg_s, np.int64)
    reg_e = np.ascontiguousarray(reg_e, np.int64)
    cfg.n_regions = len(reg_c)
    cfg.reg_contig, cfg.reg_start, cfg.reg_end = reg_c.ctypes.data, reg_s.ctypes.data, reg_e.ctypes.data
    cfg.depth, cfg.gamma_shape, cfg.gamma_scale = d, GAMMA_SHAPE, GAMMA_SCALE
    cfg.min_len, cfg.max_len = 500, MAX_READ
    cfg.mrun_mean, cfg.indel_mean, cfg.clip_mean = 60.0, 1.8, 60.0
    cfg.p_ins, cfg.p_clip, cfg.p_tagged = 0.45, 0.055, p_tagged
    cfg.p_supp, cfg.p_2d_given_supp = 0.03, 0.5
    cfg.big_delta, cfg.p_big_trunc = 1000, p_big_trunc
    per = np.zeros(len(reg_c), np.uint64)
    L.synth_plan(C.byref(cfg), per.ctypes.data)

    sel_lo = sel_hi = None
    if world > 1:
        # reads of region g are stratified: read j starts in [s + j*span/n, s + (j+1)*span/n).
        # keep every read that can reach [first window start, last window end) of this shard.
        sel_lo = np.zeros(len(reg_c), np.uint64); sel_hi = np.zeros(len(reg_c), np.uint64)
        if hi > lo:
            c_first, c_last = int(lcontig[lo]), int(lcontig[hi - 1])
            for g in range(len(reg_c)):
                c = int(reg_c[g]); n = int(per[g])
                if c < c_first or c > c_last or n == 0:
                    continue
                span = float(reg_e[g] - reg_s[g])
                in_c = np.flatnonzero(lcontig[lo:hi] == c) + lo
                if len(in_c) == 0:
                    continue
                p_lo = int(ls[in_c].min()) - 10 - MAX_READ
                p_hi = int(le[in_c].max()) + 10
                j_lo = int(np.floor((p_lo - reg_s[g]) * n / span)) - 1
                j_hi = int(np.ceil((p_hi - reg_s[g]) * n / span)) + 1
                sel_lo[g] = min(max(j_lo, 0), n); sel_hi[g] = min(max(j_hi, 0), n)
        cfg.sel_lo, cfg.sel_hi = sel_lo.ctypes.data, sel_hi.ctypes.data
    R = int(L.synth_selected(C.byref(cfg)))

    hdr_pinned = pinned and not pack_filter
    contig = _alloc(R, np.int32, hdr_pinned); rs = _alloc(R, np.int32, hdr_pinned); re_ = _alloc(R, np.int32, hdr_pinned)
    mapq = _alloc(R, np.uint8, hdr_pinned); hp = _alloc(R, np.uint8, hdr_pinned); fl = _alloc(R, np.uint8, hdr_pinned)
    coff = _alloc(R + 1, np.uint64, hdr_pinned)
    rc = L.synth_headers(C.byref(cfg), R, contig.ctypes.data, rs.ctypes.data, re_.ctypes.data, mapq.ctypes.data,
                         hp.ctypes.data, fl.ctypes.data, coff.ctypes.data)
    assert rc == 0, rc
    n_generated, words_generated = R, (int(coff[R]) if R else 0)
    if pack_filter:
        keep = pack_keep_mask(mapq, hp, unphased)
        idx = np.flatnonzero(keep)
        ncw = (coff[1:] - coff[:-1])[idx]
        Rk = len(idx)
        dst = np.zeros(R, np.uint64)
        koff = _alloc(Rk + 1, np.uint64, pinned)
        koff[0] = 0
        np.cumsum(ncw, out=koff[1:])
        dst[idx] = koff[:-1]
        ncig = int(koff[Rk]) if Rk else 0
        cigar = _alloc(ncig, np.uint32, pinned)
        keep8 = np.ascontiguousarray(keep, np.uint8)
        rc = L.synth_cigars_sel(C.byref(cfg), R, coff.ctypes.data, keep8.ctypes.data, dst.ctypes.data, cigar.ctypes.data)
        assert rc == 0, rc

        def take(a, dt):
            out = _alloc(Rk, dt, pinned)
            out[:] = a[idx]
            return out
        contig, rs, re_ = take(contig, np.int32), take(rs, np.int32), take(re_, np.int32)
        mapq, hp, fl = take(mapq, np.uint8), take(hp, np.uint8), take(fl, np.uint8)
        coff = koff
    else:
        ncig = int(coff[R]) if R else 0
        cigar = _alloc(ncig, np.uint32, pinned)
        rc = L.synth_cigars(C.byref(cfg), R, coff.ctypes.data, cigar.ctypes.data)
        assert rc == 0, rc
    reads = ReadSet(contig, rs, re_, mapq, hp, fl, coff, cigar)

    # shard view of the catalog (offsets rebuilt for the slice)
    if world > 1:
        s_off = np.searchsorted(lcontig[lo:hi], np.arange(nc + 1)).astype(np.int64)
        ls_s, le_s, d1_s, d2_s = ls[lo:hi].copy(), le[lo:hi].copy(), d1[lo:hi].copy(), d2[lo:hi].copy()
    else:
        s_off, ls_s, le_s, d1_s, d2_s = off, ls, le, d1, d2
    return Workload(config=config, name=name, seed=seed, contig_names=names, contig_len=contig_len,
                    contig_locus_off=s_off, locus_start=ls_s, locus_end=le_s, delta_h1=d1_s, delta_h2=d2_s,
                    reads=reads, minlen=5, support=3, unphased=unphased, depth=d, shard=shard,
                    locus_range=(lo, hi), meta={"n_loci_global": nl, "scale": scale, "pack_filter": bool(pack_filter),
                                                "reads_generated": n_generated, "cigar_words_generated": words_generated})


def write_bam(w: Workload, path: str, with_seq: bool = False, level: int = 1, threads: int = 0) -> int:
    """Coordinate-sorted BAM of the workload's reads (HP:C, SA for accidental-2D reads, CG for long
    CIGARs); with_seq adds SEQ/QUAL of the query length so that records have realistic sizes."""
    names = (C.c_char_p * w.n_contigs)(*[n.encode() for n in w.contig_names])
    rd = w.reads
    n = lib().synth_write_bam(path.encode(), w.n_contigs, names, w.contig_len.ctypes.data, rd.n, rd.contig.ctypes.data,
                              rd.ref_start.ctypes.data, rd.ref_end.ctypes.data, rd.mapq.ctypes.data, rd.hp.ctypes.data,
                              rd.flags.ctypes.data, rd.cigar_off.ctypes.data, rd.cigar.ctypes.data, int(with_seq), level, threads)
    if n < 0:
        raise OSError(f"cannot write {path}")
    return int(n)


def write_bed(w: Workload, path: str, shuffle_seed: int | None = None):
    """BED of the workload's catalog; returns the loci in file order as (chrom, start, end, catalog index)."""
    idx = np.arange(w.n_loci)
    if shuffle_seed is not None:
        idx = np.random.default_rng(shuffle_seed).permutation(w.n_loci)
    lc = w.locus_contig
    rows = [(w.contig_names[int(lc[i])], int(w.locus_start[i]), int(w.locus_end[i]), int(i)) for i in idx]
    with open(path, "w") as f:
        f.write("".join(f"{c}\t{s}\t{e}\n" for c, s, e, _ in rows))
    return rows
