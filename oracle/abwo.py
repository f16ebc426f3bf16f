"""TEST INFRASTRUCTURE ONLY -- ctypes binding of oracle/libabw_oracle.so (the CPU restatement).

Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg.
The product (abawaca_b200/) never imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

NKMER = 180

READ_DTYPE = np.dtype([("scaf", "<u4"), ("pos0", "<u4"), ("len", "<u4"), ("flag_nsnps", "<u4")])


class Params(C.Structure):
    _fields_ = [("cluster_ndps_threshold", C.c_uint32), ("sensitivity_threshold", C.c_double), ("specificity_threshold", C.c_double),
                ("product_threshold", C.c_double), ("sum_threshold", C.c_double), ("scg_overlap_threshold", C.c_double),
                ("scg_min_size", C.c_uint64), ("fraction_dps_in", C.c_double), ("split_scaf_ratio_threshold", C.c_double),
                ("max_snps", C.c_uint32), ("window_size", C.c_uint32)]


class SearchData(C.Structure):
    _fields_ = [("values", C.c_void_p), ("N", C.c_uint64), ("D", C.c_uint32), ("dp2scaf", C.c_void_p), ("S", C.c_uint32),
                ("T", C.c_void_p), ("len", C.c_void_p), ("scgmask", C.c_void_p), ("W", C.c_uint32)]


class Best(C.Structure):
    _fields_ = [("found", C.c_int32), ("dim", C.c_uint32), ("value", C.c_double), ("a", C.c_double), ("b", C.c_double), ("legal", C.c_int32)]


class ClusterRec(C.Structure):
    _fields_ = [("id", C.c_uint32), ("parent", C.c_uint32), ("ndps", C.c_uint64), ("nscafs", C.c_uint32), ("split", C.c_int32),
                ("best", Best), ("child1", C.c_uint32), ("child2", C.c_uint32), ("child1_ndps", C.c_uint64), ("child2_ndps", C.c_uint64),
                ("child1_nscafs", C.c_uint32), ("child2_nscafs", C.c_uint32), ("child1_raw", C.c_uint64), ("child2_raw", C.c_uint64),
                ("total_size", C.c_uint64), ("scg_unique", C.c_uint32), ("scg_avg", C.c_double)]


def build():
    """Compile the C restatement (building the checker is not using it)."""
    subprocess.run(["make", "-s", "-C", _HERE, "oracle"], check=True)


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "libabw_oracle.so")
        if not os.path.exists(path):
            build()
        L = C.CDLL(path)
        L.abwo_segment.restype = C.c_uint64
        L.abwo_count_N.restype = C.c_uint64
        L.abwo_gc.restype = C.c_double
        L.abwo_trunc3.restype = C.c_double
        L.abwo_trunc3.argtypes = [C.c_double]
        L.abwo_validate_upper.restype = C.c_int64
        L.abwo_kmer_dim_name.restype = C.c_char_p
        L.abwo_build_features.restype = C.c_uint64
        L.abwo_run.restype = C.c_uint32
        _LIB = L
    return _LIB


def default_params():
    p = Params()
    lib().abwo_default_params(C.byref(p))
    return p


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def dim_names():
    return [lib().abwo_kmer_dim_name(i).decode() for i in range(NKMER)]


def validate_upper(seq: np.ndarray):
    out = np.array(seq, dtype=np.uint8, copy=True)
    bad = lib().abwo_validate_upper(_ptr(out), C.c_uint64(out.size))
    return out, int(bad)


def segment(seq: np.ndarray, window=2000):
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    n = lib().abwo_segment(_ptr(seq), C.c_uint64(seq.size), C.c_uint64(window), None, None, C.c_uint64(0))
    st = np.zeros(n, dtype=np.uint64)
    en = np.zeros(n, dtype=np.uint64)
    lib().abwo_segment(_ptr(seq), C.c_uint64(seq.size), C.c_uint64(window), _ptr(st), _ptr(en), C.c_uint64(n))
    return st, en


def kmer_features(seg: np.ndarray):
    seg = np.ascontiguousarray(seg, dtype=np.uint8)
    out = np.zeros(NKMER, dtype=np.float64)
    counts = np.zeros(340, dtype=np.uint32)
    totals = np.zeros(4, dtype=np.uint32)
    lib().abwo_kmer_features(_ptr(seg), C.c_uint64(seg.size), _ptr(out), _ptr(counts), _ptr(totals))
    return out, counts, totals


def build_features(seq, offsets, reads, this_sample=0, params=None, want_raw=False):
    """Whole feature stage.  Returns a dict with rows (truncated .lrn values, [nseg][179+nsamples]) etc."""
    L = lib()
    p = params or default_params()
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    nscaf = offsets.size - 1
    ns = len(reads)
    reads = [np.ascontiguousarray(r) for r in reads]
    rp = (C.c_void_p * max(ns, 1))(*[r.ctypes.data for r in reads])
    rn = np.array([r.size for r in reads] + [0], dtype=np.uint64)
    args_head = (_ptr(seq), _ptr(offsets), C.c_uint32(nscaf), C.byref(p), rp, _ptr(rn), C.c_uint32(ns), C.c_int(this_sample))
    nseg = L.abwo_build_features(*args_head, None, None, None, None, None, None, None, None, None)
    if nseg == 2 ** 64 - 1:
        raise ValueError("Illegal_DNAString: lower-case 'n' in sequence (String.cpp:47-49)")
    seg_scaf = np.zeros(nseg, dtype=np.uint32)
    seg_start = np.zeros(nseg, dtype=np.uint64)
    seg_end = np.zeros(nseg, dtype=np.uint64)
    seg_nonN = np.zeros(nseg, dtype=np.uint64)
    rows = np.zeros((nseg, NKMER - 1 + ns), dtype=np.float64)
    raw = np.zeros((nseg, NKMER + ns), dtype=np.float64) if want_raw else None
    cvg = np.zeros(nscaf, dtype=np.float64)
    gc = np.zeros(nscaf, dtype=np.float64)
    Ns = np.zeros(nscaf, dtype=np.uint64)
    L.abwo_build_features(*args_head, _ptr(seg_scaf), _ptr(seg_start), _ptr(seg_end), _ptr(seg_nonN), _ptr(rows),
                          _ptr(raw) if want_raw else None, _ptr(cvg), _ptr(gc), _ptr(Ns))
    return dict(nseg=int(nseg), seg_scaf=seg_scaf, seg_start=seg_start, seg_end=seg_end, seg_nonN=seg_nonN, rows=rows, raw=raw,
                info_cvg=cvg, info_gc=gc, info_Ns=Ns)


class Search:
    """Holds the flat arrays of one search problem (kept alive for the C struct)."""

    def __init__(self, values_colmajor, dp2scaf, T, length, scgmask):
        self.values = np.ascontiguousarray(values_colmajor, dtype=np.float64)  # [D][N]
        self.D, self.N = self.values.shape
        self.dp2scaf = np.ascontiguousarray(dp2scaf, dtype=np.uint32)
        self.T = np.ascontiguousarray(T, dtype=np.uint32)
        self.len = np.ascontiguousarray(length, dtype=np.uint64)
        self.scgmask = np.ascontiguousarray(scgmask, dtype=np.uint64)
        if self.scgmask.ndim == 1:
            self.scgmask = self.scgmask.reshape(-1, 1)
        self.S = self.T.size
        self.W = self.scgmask.shape[1]
        self.c = SearchData(self.values.ctypes.data, self.N, self.D, self.dp2scaf.ctypes.data, self.S, self.T.ctypes.data,
                            self.len.ctypes.data, self.scgmask.ctypes.data, self.W)

    def separate(self, dps, strategy=0, params=None):
        p = params or default_params()
        dps = np.ascontiguousarray(dps, dtype=np.uint32)
        b = Best()
        lib().abwo_separate(C.byref(self.c), C.byref(p), C.c_int(strategy), _ptr(dps), C.c_uint64(dps.size), C.byref(b))
        return b

    def children(self, dps, dim1, value, params=None):
        p = params or default_params()
        dps = np.ascontiguousarray(dps, dtype=np.uint32)
        side = np.zeros(dps.size, dtype=np.uint8)
        raw = np.zeros(dps.size, dtype=np.uint8)
        assigned = np.zeros(self.S + 1, dtype=np.uint8)
        n1 = C.c_uint64()
        n2 = C.c_uint64()
        ok = lib().abwo_children(C.byref(self.c), C.byref(p), _ptr(dps), C.c_uint64(dps.size), C.c_uint32(dim1), C.c_double(value),
                                 _ptr(side), _ptr(raw), _ptr(assigned), C.byref(n1), C.byref(n2))
        return int(ok), side, raw, assigned[:self.S], n1.value, n2.value

    def run(self, strategy=0, params=None, nthreads=0, cap=None):
        p = params or default_params()
        cap = cap or max(16, 2 * self.N // 100 + 16)
        recs = (ClusterRec * cap)()
        dp2c = np.zeros(self.N, dtype=np.uint32)
        s2c = np.zeros(self.S, dtype=np.uint32)
        n = lib().abwo_run(C.byref(self.c), C.byref(p), C.c_int(strategy), recs, C.c_uint32(cap), _ptr(dp2c), _ptr(s2c), C.c_int(nthreads))
        return [recs[i] for i in range(min(n, cap))], dp2c, s2c

    def cluster_scg(self, scafs):
        """(number of unique SCG names, average copies per unique name) of a scaffold list (abwo_cluster_scg)."""
        scafs = np.ascontiguousarray(scafs, dtype=np.uint32)
        u, avg = C.c_uint32(), C.c_double()
        lib().abwo_cluster_scg(C.byref(self.c), _ptr(scafs), C.c_uint32(scafs.size), C.byref(u), C.byref(avg))
        return u.value, avg.value
