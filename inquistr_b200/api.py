"""ctypes binding of libinqcall.so (include/inqcall.h). No CPU fallback."""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "lib", "libinqcall.so")
_LIB = None

INQ_OK = 0
ERR_NAMES = {
    -1: "INQ_ERR_CUDA", -2: "INQ_ERR_ARG", -3: "INQ_ERR_NOMEM", -4: "INQ_ERR_STATE",
    -10: "INQ_ERR_BAD_HP", -11: "INQ_ERR_MEDIAN_EMPTY", -12: "INQ_ERR_LOCUS_START",
    -13: "INQ_ERR_LOCUS_ORDER", -14: "INQ_ERR_TOO_LARGE", -15: "INQ_ERR_NO_MODE", -16: "INQ_ERR_HITS_CAP", -17: "INQ_ERR_BAD_SA",
}
EXPORTS = [
    "inq_ctx_create", "inq_ctx_destroy", "inq_last_error", "inq_version", "inq_host_alloc",
    "inq_host_free", "inq_set_loci", "inq_push_reads", "inq_reserve_reads", "inq_clear_reads",
    "inq_genotype", "inq_debug_events", "inq_set_option", "inq_push_reads_routed",
]


class InqError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


class Stats(C.Structure):
    _fields_ = [
        ("n_loci", C.c_uint64), ("n_reads", C.c_uint64), ("n_cigar_words", C.c_uint64),
        ("n_cigar_words_joined", C.c_uint64), ("n_reads_joined", C.c_uint64),
        ("n_pairs", C.c_uint64), ("n_candidates", C.c_uint64), ("n_events", C.c_uint64),
        ("op_visits", C.c_uint64), ("n_kernel_launches", C.c_uint32), ("n_tiles", C.c_uint32),
        ("ms_total", C.c_float), ("ms_index", C.c_float), ("ms_join", C.c_float),
        ("ms_cigar", C.c_float), ("ms_fixup", C.c_float), ("ms_scan", C.c_float), ("ms_pairs", C.c_float),
        ("ms_median", C.c_float), ("ms_h2d", C.c_float), ("ms_d2h", C.c_float),
        ("n_ranges", C.c_uint32), ("used_graph", C.c_uint32), ("reads_sorted", C.c_uint32),
        ("n_median_chunks", C.c_uint32), ("n_passes", C.c_uint32), ("key_bytes", C.c_uint32),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


def load_library():
    """Load libinqcall.so; raises OSError if it has not been built (python -m inquistr_b200.build)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(_LIB_PATH):
        raise OSError(f"{_LIB_PATH} not found: build it with `python -m inquistr_b200.build` "
                      "(there is no CPU fallback)")
    L = C.CDLL(_LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32
    L.inq_ctx_create.restype = C.c_int
    L.inq_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.inq_ctx_destroy.restype = None
    L.inq_ctx_destroy.argtypes = [vp]
    L.inq_last_error.restype = C.c_char_p
    L.inq_last_error.argtypes = [vp]
    L.inq_version.restype = C.c_char_p
    L.inq_host_alloc.restype = C.c_int
    L.inq_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.inq_host_free.restype = C.c_int
    L.inq_host_free.argtypes = [vp]
    L.inq_set_loci.restype = C.c_int
    L.inq_set_loci.argtypes = [vp, i32, vp, vp, vp]
    L.inq_push_reads.restype = C.c_int
    L.inq_push_reads.argtypes = [vp, u64, vp, vp, vp, vp, vp, vp, vp, vp]
    L.inq_push_reads_routed.restype = C.c_int
    L.inq_push_reads_routed.argtypes = [vp, u64, vp, vp, vp, vp, vp, vp, vp, vp, u32, C.c_int, C.POINTER(u64)]
    L.inq_reserve_reads.restype = C.c_int
    L.inq_reserve_reads.argtypes = [vp, u64, u64]
    L.inq_clear_reads.restype = C.c_int
    L.inq_clear_reads.argtypes = [vp]
    L.inq_genotype.restype = C.c_int
    L.inq_genotype.argtypes = [vp, u32, u32, C.c_int, vp, vp, vp, C.POINTER(Stats)]
    L.inq_set_option.restype = C.c_int
    L.inq_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    L.inq_debug_events.restype = C.c_int
    L.inq_debug_events.argtypes = [vp, C.POINTER(u64), vp, vp, u64, vp]
    _LIB = L
    return L


def pinned_empty(n: int, dtype) -> np.ndarray:
    """numpy array backed by inq_host_alloc pinned memory. Released with free_pinned() or at exit."""
    L = load_library()
    dt = np.dtype(dtype)
    p = C.c_void_p()
    rc = L.inq_host_alloc(max(1, n * dt.itemsize), C.byref(p))
    if rc != INQ_OK:
        raise InqError(rc, "inq_host_alloc failed")
    buf = (C.c_char * max(1, n * dt.itemsize)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dt, count=n)
    _PINNED[p.value] = buf
    return arr


_PINNED: dict = {}


def free_pinned(arr: np.ndarray) -> None:
    """Release a pinned_empty() array; the caller must not touch it (or views of it) afterwards."""
    addr = arr.ctypes.data
    if _PINNED.pop(addr, None) is not None and _LIB is not None:
        _LIB.inq_host_free(C.c_void_p(addr))


@dataclass
class GenotypeResult:
    twice_h1: np.ndarray   # int64, 2 x median
    twice_h2: np.ndarray
    valid: np.ndarray      # uint8 bit0 H1, bit1 H2
    stats: dict

    @property
    def phase1(self) -> np.ndarray:
        """f64 the reference prints: twice/2.0 (call.rs:515-521), NaN where not valid."""
        out = self.twice_h1.astype(np.float64) / 2.0
        out[(self.valid & 1) == 0] = np.nan
        return out

    @property
    def phase2(self) -> np.ndarray:
        out = self.twice_h2.astype(np.float64) / 2.0
        out[(self.valid & 2) == 0] = np.nan
        return out


class Context:
    """One GPU context (inq_ctx). Mirrors the call order of the C ABI."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        h = C.c_void_p()
        rc = self._lib.inq_ctx_create(int(device), C.byref(h))
        if rc != INQ_OK:
            raise InqError(rc, self._lib.inq_last_error(None).decode())
        self._h = h
        self.n_loci = 0
        self.n_reads = 0

    def close(self):
        if getattr(self, "_h", None):
            self._lib.inq_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc != INQ_OK:
            raise InqError(rc, self._lib.inq_last_error(self._h).decode())

    def set_loci(self, contig_locus_offsets, start, end):
        off = np.ascontiguousarray(contig_locus_offsets, dtype=np.int64)
        s = np.ascontiguousarray(start, dtype=np.int32)
        e = np.ascontiguousarray(end, dtype=np.int32)
        assert len(s) == len(e) == int(off[-1])
        self._check(self._lib.inq_set_loci(self._h, len(off) - 1, off.ctypes.data, s.ctypes.data, e.ctypes.data))
        self.n_loci = len(s)

    def set_option(self, name: str, value: int):
        """inq_set_option: "graph" (0/1) or "timing" (0/1/2) (include/inqcall.h)."""
        self._check(self._lib.inq_set_option(self._h, name.encode(), int(value)))

    def reserve_reads(self, n_reads, n_words):
        self._check(self._lib.inq_reserve_reads(self._h, int(n_reads), int(n_words)))

    def clear_reads(self):
        self._check(self._lib.inq_clear_reads(self._h))
        self.n_reads = 0

    def push_reads(self, contig, ref_start, ref_end, mapq, hp, flags, cigar_off, cigar):
        def chk(a, dt):
            a = np.ascontiguousarray(a, dtype=dt)
            return a
        contig, ref_start, ref_end = chk(contig, np.int32), chk(ref_start, np.int32), chk(ref_end, np.int32)
        mapq, hp, flags = chk(mapq, np.uint8), chk(hp, np.uint8), chk(flags, np.uint8)
        cigar_off, cigar = chk(cigar_off, np.uint64), chk(cigar, np.uint32)
        n = len(contig)
        assert len(cigar_off) == n + 1 and all(len(a) == n for a in (ref_start, ref_end, mapq, hp, flags))
        self._check(self._lib.inq_push_reads(self._h, n, contig.ctypes.data, ref_start.ctypes.data,
                                             ref_end.ctypes.data, mapq.ctypes.data, hp.ctypes.data,
                                             flags.ctypes.data, cigar_off.ctypes.data, cigar.ctypes.data))
        self.n_reads += n

    def push_routed(self, reads, drop_low_mapq=False, drop_no_hp=False, host_threads=0) -> int:
        """inq_push_reads_routed: keep only the reads that can reach this context's catalog; returns how many"""
        def chk(a, dt):
            return np.ascontiguousarray(a, dtype=dt)
        contig, rs, re_ = chk(reads.contig, np.int32), chk(reads.ref_start, np.int32), chk(reads.ref_end, np.int32)
        mapq, hp, fl = chk(reads.mapq, np.uint8), chk(reads.hp, np.uint8), chk(reads.flags, np.uint8)
        off, cig = chk(reads.cigar_off, np.uint64), chk(reads.cigar, np.uint32)
        taken = C.c_uint64(0)
        self._check(self._lib.inq_push_reads_routed(self._h, len(contig), contig.ctypes.data, rs.ctypes.data, re_.ctypes.data,
                                                    mapq.ctypes.data, hp.ctypes.data, fl.ctypes.data, off.ctypes.data, cig.ctypes.data,
                                                    (1 if drop_low_mapq else 0) | (2 if drop_no_hp else 0), int(host_threads), C.byref(taken)))
        self.n_reads += int(taken.value)
        return int(taken.value)

    def push(self, reads):
        """reads: any object carrying the SoA attributes of include/inqcall.h:inq_push_reads."""
        self.push_reads(reads.contig, reads.ref_start, reads.ref_end, reads.mapq, reads.hp,
                        reads.flags, reads.cigar_off, reads.cigar)

    def genotype(self, minlen=5, support=3, unphased=False, out=None) -> GenotypeResult:
        n = self.n_loci
        if out is None:
            t1 = np.zeros(n, np.int64)
            t2 = np.zeros(n, np.int64)
            vm = np.zeros(n, np.uint8)
        else:
            t1, t2, vm = out
        st = Stats()
        self._check(self._lib.inq_genotype(self._h, int(minlen), int(support), int(bool(unphased)),
                                           t1.ctypes.data, t2.ctypes.data, vm.ctypes.data, C.byref(st)))
        return GenotypeResult(t1, t2, vm, st.as_dict())

    def genotype_fn(self, minlen, support, unphased, out):
        """Pre-bound inq_genotype call for tight loops (bench.py): returns (call, stats) where call() runs one pass
        into the `out` arrays and returns the error code, and stats is the ctypes struct it fills."""
        t1, t2, vm = out
        st = Stats()
        fn, h = self._lib.inq_genotype, self._h
        a = (h, C.c_uint32(int(minlen)), C.c_uint32(int(support)), C.c_int(int(bool(unphased))), C.c_void_p(t1.ctypes.data),
             C.c_void_p(t2.ctypes.data), C.c_void_p(vm.ctypes.data), C.byref(st))
        return (lambda: fn(*a)), st

    def debug_events(self):
        n = C.c_uint64(0)
        self._check(self._lib.inq_debug_events(self._h, C.byref(n), None, None, 0, None))
        E = int(n.value)
        pos = np.zeros(E, np.uint32)
        val = np.zeros(E, np.int32)
        off = np.zeros(self.n_reads + 1, np.uint32)
        self._check(self._lib.inq_debug_events(self._h, C.byref(n), pos.ctypes.data, val.ctypes.data, E, off.ctypes.data))
        return pos, val, off
