"""ctypes binding of libabawaca_b200.so -- exactly the entry points declared in include/abawaca_b200.h.

There is no CPU fallback: `load()` raises if the shared library is missing, and `Context()` raises
if no CUDA device can be opened.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ABW_B200_LIB") or os.path.join(_HERE, "libabawaca_b200.so")      # the override is for A/B experiments with two builds
_LIB = None

NKMER = 180
SENS_SPEC, SPLIT_SCAFS = 0, 1
LAYOUT_COLMAJOR, LAYOUT_ROWMAJOR, LAYOUT_ROWMAJOR_MILLI32 = 0, 1, 2
FEAT_TRUNC3, FEAT_RAW = 0, 1
TEXT_3LF, TEXT_LF = 0, 1         # abw_format_lrn: "%.3lf" (abawaca.lrn), "%lf" (clusters/<id>.lrn)

READ_DTYPE = np.dtype([("scaf", "<u4"), ("pos0", "<u4"), ("len", "<u4"), ("flag_nsnps", "<u4")])
READ8_DTYPE = np.dtype([("scaf", "<u4"), ("pos0", "<u4")])      # abw_read8: reads the host parser already filtered
READ_RUN_DTYPE = np.dtype([("scaf", "<u4"), ("count", "<u4")])   # abw_read_run: `count` consecutive reads on scaffold `scaf` (sorted format)
READS_FULL, READS_COMPACT, READS_SORTED = 0, 1, 2
BASE_RUN_DTYPE = np.dtype([("scaf", "<u4"), ("start", "<u4"), ("len", "<u4"), ("kind", "<u4")])   # abw_base_run
BASE_N, BASE_OTHER = 0, 1


class AbwError(RuntimeError):
    pass


class Params(C.Structure):
    _fields_ = [("cluster_ndps_threshold", C.c_uint32), ("sensitivity_threshold", C.c_double), ("specificity_threshold", C.c_double),
                ("product_threshold", C.c_double), ("sum_threshold", C.c_double), ("scg_overlap_threshold", C.c_double),
                ("scg_min_size", C.c_uint64), ("fraction_dps_in", C.c_double), ("split_scaf_ratio_threshold", C.c_double),
                ("max_snps", C.c_uint32), ("window_size", C.c_uint32), ("min_reported_score", C.c_double)]


class Best(C.Structure):
    _fields_ = [("found", C.c_int32), ("dim", C.c_uint32), ("value", C.c_double), ("a", C.c_double), ("b", C.c_double), ("legal", C.c_int32)]


class ClusterRec(C.Structure):
    _fields_ = [("id", C.c_uint32), ("parent", C.c_uint32), ("ndps", C.c_uint64), ("nscafs", C.c_uint32), ("split", C.c_int32),
                ("best", Best), ("child1", C.c_uint32), ("child2", C.c_uint32), ("child1_ndps", C.c_uint64), ("child2_ndps", C.c_uint64),
                ("child1_nscafs", C.c_uint32), ("child2_nscafs", C.c_uint32), ("child1_raw", C.c_uint64), ("child2_raw", C.c_uint64),
                ("total_size", C.c_uint64), ("scg_unique", C.c_uint32), ("scg_avg", C.c_double),
                ("gc_avg", C.c_double), ("gc_sd", C.c_double), ("cvg_avg", C.c_double), ("cvg_sd", C.c_double)]


class Sample(C.Structure):
    """abw_sample"""
    _fields_ = [("reads", C.c_void_p), ("nreads", C.c_uint64), ("format", C.c_int32), ("len", C.c_uint32), ("len16", C.c_void_p), ("h2d_ticket", C.c_uint64),
                ("runs", C.c_void_p), ("nruns", C.c_uint64), ("exc", C.c_void_p), ("nexc", C.c_uint64)]


class TwoBitAssembly(C.Structure):
    """abw_2bit_assembly"""
    _fields_ = [("codes", C.c_void_p), ("nbytes", C.c_uint64), ("h_byte_off", C.c_void_p), ("h_len", C.c_void_p), ("runs", C.c_void_p), ("nruns", C.c_uint64),
                ("h2d_ticket", C.c_uint64)]


class SearchProfile(C.Structure):
    _fields_ = [("build_ms", C.c_float), ("sweep_ms", C.c_float), ("partition_ms", C.c_float), ("other_ms", C.c_float),
                ("sweep_elements", C.c_uint64), ("partition_elements", C.c_uint64), ("levels", C.c_uint32), ("sweep_launches", C.c_uint32)]


ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t)
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)


class Collectives(C.Structure):
    _fields_ = [("allgather", ALLGATHER_FN), ("allreduce_sum_i64", ALLREDUCE_FN), ("user", C.c_void_p), ("rank", C.c_int), ("world", C.c_int),
                ("stream_ordered", C.c_int)]


EXPORTS = [
    "abw_ctx_create", "abw_ctx_destroy", "abw_last_error", "abw_version", "abw_default_params", "abw_kernel_launches", "abw_arena_misses", "abw_redzone_violations", "abw_ctx_stream",
    "abw_ctx_synchronize", "abw_profile_enable", "abw_profile_report", "abw_pack_sequences", "abw_seqset_destroy", "abw_seqset_stats", "abw_segment", "abw_segments_destroy",
    "abw_segments_count", "abw_segments_get", "abw_segments_get_async", "abw_kmer_features", "abw_coverage", "abw_coverage_batch", "abw_rows_to_milli", "abw_device_alloc", "abw_device_free",
    "abw_copy_to_device", "abw_copy_to_host", "abw_memset_device", "abw_h2d_async", "abw_wait_h2d", "abw_d2h_async", "abw_search_create", "abw_search_create_from_features", "abw_search_destroy", "abw_search_run",
    "abw_search_set_shard", "abw_search_set_shard_strided", "abw_search_set_max_levels", "abw_search_run_sharded", "abw_search_get_profile", "abw_cluster_scg",
    "abw_names_create", "abw_names_destroy", "abw_parse_sam", "abw_fasta_scan", "abw_fasta_destroy", "abw_fasta_count", "abw_fasta_get", "abw_fasta_pack", "abw_nccl_unique_id", "abw_nccl_collectives_create", "abw_nccl_collectives_destroy", "abw_peer_buffer_create", "abw_peer_buffer_destroy", "abw_peer_group_create", "abw_peer_group_destroy",
    "abw_scatter_columns_milli", "abw_parse_lrn", "abw_gather_rows", "abw_format_lrn", "abw_search_set_scaffold_stats",
    "abw_pack_2bit", "abw_twobit_scan", "abw_twobit_destroy", "abw_twobit_count", "abw_twobit_get", "abw_twobit_decode", "abw_twobit_pack",
    "abw_fasta_format", "abw_twobit_format", "abw_fasta_base_counts", "abw_twobit_base_counts",
    "abw_bam_create", "abw_bam_feed", "abw_bam_finish", "abw_bam_destroy",
]


def load():
    """Load the CUDA library.  Fails loudly: the product has no other code path."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise AbwError(f"{LIB_PATH} is missing: build it with `make -C abawaca_b200/csrc` (or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    L.abw_last_error.restype = C.c_char_p
    L.abw_version.restype = C.c_char_p
    L.abw_kernel_launches.restype = C.c_uint64
    L.abw_arena_misses.restype = C.c_uint64
    L.abw_arena_misses.argtypes = [C.c_void_p]
    L.abw_redzone_violations.restype = C.c_uint64
    L.abw_redzone_violations.argtypes = []
    L.abw_ctx_stream.restype = C.c_void_p
    L.abw_segments_count.restype = C.c_uint64
    L.abw_segments_count.argtypes = [C.c_void_p]
    L.abw_ctx_destroy.argtypes = [C.c_void_p]
    L.abw_seqset_destroy.argtypes = [C.c_void_p]
    L.abw_segments_destroy.argtypes = [C.c_void_p]
    L.abw_search_destroy.argtypes = [C.c_void_p]
    L.abw_last_error.argtypes = [C.c_void_p]
    L.abw_kernel_launches.argtypes = [C.c_void_p]
    L.abw_ctx_stream.argtypes = [C.c_void_p]
    L.abw_ctx_synchronize.argtypes = [C.c_void_p]
    L.abw_profile_enable.argtypes = [C.c_void_p, C.c_int]
    L.abw_profile_report.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t]
    L.abw_profile_report.restype = C.c_size_t
    L.abw_pack_sequences.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.abw_seqset_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.abw_segment.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.abw_segments_get.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.abw_segments_get_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.abw_kmer_features.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_uint32]
    L.abw_coverage.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_uint32, C.c_int, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
    L.abw_coverage_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_void_p]
    L.abw_rows_to_milli.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
    L.abw_device_alloc.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.abw_device_free.argtypes = [C.c_void_p, C.c_void_p]
    L.abw_copy_to_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.abw_copy_to_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.abw_memset_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t]
    L.abw_h2d_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64)]
    L.abw_wait_h2d.argtypes = [C.c_void_p, C.c_uint64]
    L.abw_d2h_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.abw_search_create.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
    L.abw_search_create_from_features.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_int,
                                                  C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.c_void_p, C.POINTER(C.c_void_p)]
    L.abw_search_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p, C.c_void_p]
    L.abw_search_set_shard.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
    L.abw_search_set_shard_strided.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
    L.abw_search_set_max_levels.argtypes = [C.c_void_p, C.c_uint32]
    L.abw_search_run_sharded.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p, C.c_void_p]
    L.abw_search_get_profile.argtypes = [C.c_void_p, C.c_void_p]
    L.abw_names_create.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.abw_names_destroy.argtypes = [C.c_void_p]
    L.abw_parse_sam.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    L.abw_fasta_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]
    L.abw_fasta_destroy.argtypes = [C.c_void_p]
    L.abw_fasta_count.argtypes = [C.c_void_p]
    L.abw_fasta_count.restype = C.c_uint64
    L.abw_fasta_get.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.abw_fasta_pack.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.abw_pack_2bit.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.abw_twobit_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
    L.abw_twobit_destroy.argtypes = [C.c_void_p]
    L.abw_twobit_destroy.restype = None
    L.abw_twobit_count.argtypes = [C.c_void_p]
    L.abw_twobit_count.restype = C.c_uint64
    L.abw_twobit_get.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.abw_twobit_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    L.abw_twobit_pack.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.abw_fasta_format.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.abw_twobit_format.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64),
                                    C.POINTER(C.c_uint64)]
    L.abw_fasta_base_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.abw_twobit_base_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    L.abw_bam_create.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
    L.abw_bam_feed.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    L.abw_bam_finish.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    L.abw_bam_destroy.argtypes = [C.c_void_p]
    L.abw_bam_destroy.restype = None
    L.abw_nccl_unique_id.argtypes = [C.c_void_p, C.c_void_p]
    L.abw_nccl_collectives_create.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.abw_nccl_collectives_destroy.argtypes = [C.c_void_p]
    L.abw_peer_buffer_create.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.c_void_p]
    L.abw_peer_buffer_destroy.argtypes = [C.c_void_p, C.c_void_p]
    L.abw_peer_group_create.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    L.abw_peer_group_destroy.argtypes = [C.c_void_p]
    L.abw_peer_group_destroy.restype = None
    L.abw_scatter_columns_milli.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64, C.c_size_t, C.c_void_p]
    L.abw_parse_lrn.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    L.abw_gather_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64]
    L.abw_format_lrn.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64,
                                 C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.abw_search_set_scaffold_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.abw_cluster_scg.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_double)]
    _LIB = L
    return L


def default_params():
    p = Params()
    load().abw_default_params(C.byref(p))
    return p


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


class Context:
    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.abw_ctx_create(C.c_int(device), C.byref(h))
        if rc != 0:
            raise AbwError(f"abw_ctx_create(device={device}) failed with status {rc}: no usable CUDA device (there is no CPU fallback)")
        self.h = h
        self.device = device

    def close(self):
        if self.h:
            self.lib.abw_ctx_destroy(self.h)
            self.h = None

    def check(self, rc):
        if rc != 0:
            raise AbwError(f"status {rc}: {self.lib.abw_last_error(self.h).decode()}")

    @property
    def launches(self):
        return int(self.lib.abw_kernel_launches(self.h))

    @property
    def arena_misses(self):
        return int(self.lib.abw_arena_misses(self.h))

    @property
    def stream(self):
        return self.lib.abw_ctx_stream(self.h)

    def synchronize(self):
        self.check(self.lib.abw_ctx_synchronize(self.h))

    def profile(self, on=True):
        self.check(self.lib.abw_profile_enable(self.h, 1 if on else 0))

    def profile_report(self):
        """{kernel: (launches, total_ms)} accumulated since profile(True)"""
        n = self.lib.abw_profile_report(self.h, None, 0)
        buf = C.create_string_buffer(int(n) + 16)
        self.lib.abw_profile_report(self.h, buf, len(buf))
        out = {}
        for line in buf.value.decode().splitlines():
            k, c, ms = line.split("\t")
            out[k] = (int(c), float(ms))
        return out

    # raw device memory
    def alloc(self, nbytes):
        d = C.c_void_p()
        self.check(self.lib.abw_device_alloc(self.h, nbytes, C.byref(d)))
        return d.value

    def free(self, dptr):
        self.check(self.lib.abw_device_free(self.h, C.c_void_p(dptr)))

    def to_device(self, dptr, arr):
        arr = np.ascontiguousarray(arr)
        self.check(self.lib.abw_copy_to_device(self.h, C.c_void_p(dptr), _p(arr), arr.nbytes))

    def to_host(self, arr, dptr):
        self.check(self.lib.abw_copy_to_host(self.h, _p(arr), C.c_void_p(dptr), arr.nbytes))

    def h2d_async(self, dptr, arr):
        """enqueue a copy of a (pinned) numpy array on the copy stream; returns a ticket for wait_h2d"""
        t = C.c_uint64()
        self.check(self.lib.abw_h2d_async(self.h, C.c_void_p(dptr), _p(arr), arr.nbytes, C.byref(t)))
        return t.value

    def wait_h2d(self, ticket):
        self.check(self.lib.abw_wait_h2d(self.h, ticket))

    def d2h_async(self, arr, dptr, nbytes=None):
        """enqueue a copy into a (pinned) numpy array on the copy stream; complete after synchronize()"""
        self.check(self.lib.abw_d2h_async(self.h, _p(arr), C.c_void_p(dptr), arr.nbytes if nbytes is None else nbytes))

    def memset(self, dptr, byte, nbytes):
        self.check(self.lib.abw_memset_device(self.h, C.c_void_p(dptr), byte, nbytes))
