"""Host-side drivers over the C ABI, mirroring the two reference programs' hot paths.

`build_features`  ~ abawaca-build.cpp main(): FASTA -> windows -> k-mer signature + per-sample coverage rows
`search`          ~ abawaca.cpp main(): recursive split search from the all-inclusive cluster

Everything that computes goes through libabawaca_b200.so; numpy only carries buffers.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np

from . import capi


def _host_bytes(data):
    """bytes, bytearray, memoryview or array -> (contiguous uint8 array, its pointer for the C ABI or None when it is empty)"""
    arr = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else np.ascontiguousarray(data, dtype=np.uint8)
    return arr, capi._p(arr) if arr.size else None


def _first_of_each_name(ctx, data, h, n, get):
    """(names, record indices, lengths) of the scaffolds among the n records of `data`: the first of every name, in byte-wise name order (abawaca-build.cpp:482-490)"""
    name_off = np.zeros(n, dtype=np.uint64)
    name_len = np.zeros(n, dtype=np.uint32)
    seq_len = np.zeros(n, dtype=np.uint64)
    ctx.check(get(ctx.h, h, capi._p(name_off), capi._p(name_len), capi._p(seq_len)))
    first = {}
    for i in range(n):
        first.setdefault(bytes(data[int(name_off[i]):int(name_off[i]) + int(name_len[i])]), i)
    names = sorted(first)
    order = np.array([first[k] for k in names], dtype=np.uint32)
    return [k.decode() for k in names], order, seq_len[order]


class SamParser:
    """SAM text -> abw_read records on the device (abw_names_create / abw_parse_sam)."""

    def __init__(self, ctx, names):
        self.ctx = ctx
        blob = "".join(names).encode()
        off = np.zeros(len(names) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(n.encode()) for n in names])
        self._blob = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, dtype=np.uint8)
        h = C.c_void_p()
        ctx.check(ctx.lib.abw_names_create(ctx.h, capi._p(self._blob), capi._p(off), len(names), C.byref(h)))
        self.h = h

    def parse(self, text, d_reads, cap):
        """text: bytes or uint8 array (host), ending at a line boundary.  Returns the number of records written to d_reads."""
        arr, p = _host_bytes(text)
        n = C.c_uint64()
        self.ctx.check(self.ctx.lib.abw_parse_sam(self.ctx.h, self.h, p, arr.size, 0, C.c_void_p(d_reads), cap, C.byref(n)))
        return int(n.value)

    def parse_to_host(self, text):
        """convenience for tests: parse one chunk and fetch the records"""
        arr, _ = _host_bytes(text)
        cap = int(np.count_nonzero(arr == 10)) + 1
        d = self.ctx.alloc(max(cap, 1) * 16)
        try:
            n = self.parse(arr, d, cap)
            out = np.zeros(n, dtype=capi.READ_DTYPE)
            if n:
                self.ctx.to_host(out, d)
            return out
        finally:
            self.ctx.free(d)

    def close(self):
        if self.h:
            self.ctx.lib.abw_names_destroy(self.h)
            self.h = None


class BamReader:
    """BAM file -> abw_read records on the device (abw_bam_*), the counterpart of SamParser.  feed() takes the file's bytes in pieces split
    anywhere; finish() returns (device pointer, number of records) of the array the reader owns until close()."""

    def __init__(self, ctx, names):
        self.ctx = ctx
        self.names = SamParser(ctx, names)
        h = C.c_void_p()
        ctx.check(ctx.lib.abw_bam_create(ctx.h, self.names.h, C.byref(h)))
        self.h = h

    def feed(self, data):
        arr, p = _host_bytes(data)
        self.ctx.check(self.ctx.lib.abw_bam_feed(self.ctx.h, self.h, p, arr.size))

    def finish(self):
        d, n = C.c_void_p(), C.c_uint64()
        self.ctx.check(self.ctx.lib.abw_bam_finish(self.ctx.h, self.h, C.byref(d), C.byref(n)))
        return d.value, int(n.value)

    def to_host(self):
        """finish() and fetch the records"""
        d, n = self.finish()
        out = np.zeros(n, dtype=capi.READ_DTYPE)
        if n:
            self.ctx.to_host(out, d)
        return out

    def close(self):
        if self.h:
            self.ctx.lib.abw_bam_destroy(self.h)
            self.h = None
        self.names.close()


def parse_lrn_rows(ctx, text, D):
    """data lines of a .lrn file (bytes, after the four header lines) -> (keys uint64 [n], device pointer of the row-major [n][D] matrix, n).
    The caller frees the matrix with ctx.free()."""
    arr, p = _host_bytes(text)
    cap = int(np.count_nonzero(arr == 10)) + 1
    d_keys = ctx.alloc(cap * 8)
    d_vals = ctx.alloc(max(cap * D, 1) * 8)
    n = C.c_uint64()
    try:
        ctx.check(ctx.lib.abw_parse_lrn(ctx.h, p, arr.size, 0, D, C.c_void_p(d_keys), C.c_void_p(d_vals), cap, C.byref(n)))
    except Exception:
        ctx.free(d_keys); ctx.free(d_vals)
        raise
    keys = np.zeros(int(n.value), dtype=np.uint64)
    if keys.size:
        ctx.to_host(keys, d_keys)
    ctx.free(d_keys)
    return keys, d_vals, int(n.value)


def format_lrn_rows(ctx, d_values, ld, ncols, rows=None, nlines=None, fmt=capi.TEXT_3LF, col0=0, cap=64 << 20, rows_on_device=False) -> bytes:
    """.lrn data lines of a row-major device matrix (abw_format_lrn): line i is "<r+1>\\t<v_0>...\\n" with r = rows[i] (None: r = i, nlines lines).
    rows: uint64 numpy array, or a device pointer with rows_on_device.  The text is made in pieces of at most `cap` bytes and concatenated."""
    if rows is not None and not rows_on_device:
        rows = np.ascontiguousarray(rows, dtype=np.uint64)
        nlines = rows.size if nlines is None else nlines
    if nlines is None:
        raise ValueError("format_lrn_rows: nlines is required unless rows is a host array")
    d_text = ctx.alloc(max(cap, 1))
    out, line0 = [], 0
    done, nbytes = C.c_uint64(), C.c_uint64()
    try:
        while True:                  # at least one call, so that an empty range goes through abw_format_lrn too
            ctx.check(ctx.lib.abw_format_lrn(ctx.h, C.c_void_p(d_values), ld, col0, ncols, None if rows is None else (C.c_void_p(rows) if rows_on_device else capi._p(rows)),
                                             1 if rows_on_device else 0, line0, nlines, fmt, C.c_void_p(d_text), cap, C.byref(done), C.byref(nbytes)))
            buf = np.empty(int(nbytes.value), dtype=np.uint8)
            ctx.to_host(buf, d_text)
            out.append(buf.tobytes())
            line0 += int(done.value)
            if line0 >= nlines:
                break
    finally:
        ctx.free(d_text)
    return b"".join(out)


def fasta_to_seqset(ctx, text):
    """FASTA text (bytes) -> (seqset handle, names in scaffold order, lengths): records indexed on the device (abw_fasta_scan), packed by abw_fasta_pack"""
    L = ctx.lib
    arr, p = _host_bytes(text)
    f = C.c_void_p()
    ctx.check(L.abw_fasta_scan(ctx.h, p, arr.size, 0, C.byref(f)))
    try:
        names, order, lengths = _first_of_each_name(ctx, text, f, int(L.abw_fasta_count(f)), L.abw_fasta_get)
        ss = C.c_void_p()
        ctx.check(L.abw_fasta_pack(ctx.h, f, capi._p(order), order.size, C.byref(ss)))
        return ss, names, lengths
    finally:
        L.abw_fasta_destroy(f)


def twobit_to_seqset(ctx, data):
    """UCSC .2bit file image (bytes) -> (seqset handle, names in scaffold order, lengths), the counterpart of fasta_to_seqset: header and records
    parsed by abw_twobit_scan, the file copied to the device once as it is and decoded there (abw_twobit_pack)."""
    L = ctx.lib
    arr, p = _host_bytes(data)
    t = C.c_void_p()
    ctx.check(L.abw_twobit_scan(ctx.h, p, arr.size, C.byref(t)))
    d_file = None
    try:
        names, order, lengths = _first_of_each_name(ctx, data, t, int(L.abw_twobit_count(t)), L.abw_twobit_get)
        d_file = ctx.alloc(max(arr.size, 1))
        if arr.size:
            ctx.to_device(d_file, arr)
        ss = C.c_void_p()
        ctx.check(L.abw_twobit_pack(ctx.h, t, C.c_void_p(d_file), 0, capi._p(order), order.size, C.byref(ss)))
        ctx.synchronize()
        return ss, names, lengths
    finally:
        if d_file is not None:
            ctx.free(d_file)
        L.abw_twobit_destroy(t)


def is_twobit(data) -> bool:
    """a UCSC .2bit file starts with the signature 0x1A412743 in the byte order of the file"""
    return bytes(data[:4]) in (b"\x43\x27\x41\x1A", b"\x1A\x41\x27\x43")


class AssemblyFile:
    """An assembly file held on the device for the FASTA writer and the base counts: FASTA text indexed by abw_fasta_scan, or a UCSC .2bit image
    (told apart by its signature) parsed by abw_twobit_scan and copied to the device as it is.  d_text: the FASTA text is already in device memory
    there (data is its host copy, which only gives the ids); it must stay alive until close()."""

    def __init__(self, ctx, data, d_text=None):
        self.ctx, self.data = ctx, data
        L = ctx.lib
        arr, p = _host_bytes(data)
        self.twobit = is_twobit(arr)
        self.h = C.c_void_p()
        self.d_file = None
        if self.twobit:
            ctx.check(L.abw_twobit_scan(ctx.h, p, arr.size, C.byref(self.h)))
            self.d_file = ctx.alloc(max(arr.size, 1))
            ctx.to_device(self.d_file, arr)
            self.count = int(L.abw_twobit_count(self.h))
        else:
            ctx.check(L.abw_fasta_scan(ctx.h, p if d_text is None else C.c_void_p(d_text), arr.size, 0 if d_text is None else 1, C.byref(self.h)))
            self.count = int(L.abw_fasta_count(self.h))

    def records(self):
        """(ids as bytes, sequence lengths) per record in file order"""
        off, idl, sl = np.zeros(self.count, np.uint64), np.zeros(self.count, np.uint32), np.zeros(self.count, np.uint64)
        get = self.ctx.lib.abw_twobit_get if self.twobit else self.ctx.lib.abw_fasta_get
        self.ctx.check(get(self.ctx.h, self.h, capi._p(off), capi._p(idl), capi._p(sl)))
        return [bytes(self.data[int(a):int(a) + int(n)]) for a, n in zip(off, idl)], sl

    def format_window(self, recs, byte0, d_text, cap):
        """abw_*_format of the records `recs` (uint32 array): bytes [byte0, byte0 + cap) of their FASTA text to d_text -> (total bytes, bytes written)"""
        total, n = C.c_uint64(), C.c_uint64()
        L, ctx = self.ctx.lib, self.ctx
        pr = capi._p(recs) if recs.size else None
        if self.twobit:
            ctx.check(L.abw_twobit_format(ctx.h, self.h, C.c_void_p(self.d_file), 0, pr, recs.size, byte0, C.c_void_p(d_text), cap, C.byref(total), C.byref(n)))
        else:
            ctx.check(L.abw_fasta_format(ctx.h, self.h, pr, recs.size, byte0, C.c_void_p(d_text), cap, C.byref(total), C.byref(n)))
        return int(total.value), int(n.value)

    def close(self):
        if self.h:
            (self.ctx.lib.abw_twobit_destroy if self.twobit else self.ctx.lib.abw_fasta_destroy)(self.h)
            self.h = None
        if self.d_file is not None:
            self.ctx.free(self.d_file)
            self.d_file = None


def format_fasta(ctx, asm: AssemblyFile, recs, cap=64 << 20) -> bytes:
    """The FASTA text abawaca writes for the records `recs` (file-order indices, in list order) of an AssemblyFile, made on the device in windows of
    at most `cap` bytes (abw_fasta_format / abw_twobit_format) and concatenated."""
    recs = np.ascontiguousarray(recs, dtype=np.uint32)
    d_text = ctx.alloc(max(cap, 1))
    out, byte0 = [], 0
    try:
        while True:                  # at least one call, so that an empty list goes through the library too
            total, n = asm.format_window(recs, byte0, d_text, cap)
            buf = np.empty(n, dtype=np.uint8)
            if n:
                ctx.to_host(buf, d_text)
            out.append(buf.tobytes())
            byte0 += n
            if byte0 >= total:
                break
    finally:
        ctx.free(d_text)
    return b"".join(out)


def base_counts(ctx, asm: AssemblyFile):
    """(N, C+G) per record of an AssemblyFile in file order, uint64 arrays, after upper-casing (abw_fasta_base_counts / abw_twobit_base_counts)"""
    cn, cgc = np.zeros(max(asm.count, 1), np.uint64), np.zeros(max(asm.count, 1), np.uint64)
    if asm.twobit:
        ctx.check(ctx.lib.abw_twobit_base_counts(ctx.h, asm.h, C.c_void_p(asm.d_file), 0, capi._p(cn), capi._p(cgc)))
    else:
        ctx.check(ctx.lib.abw_fasta_base_counts(ctx.h, asm.h, capi._p(cn), capi._p(cgc)))
    return cn[:asm.count], cgc[:asm.count]


class PackedAssembly:
    """An assembly in 2 bits per base (abw_2bit_assembly): UCSC-order codes with every scaffold starting at a byte of its own, plus runs of the
    characters that are not A/C/G/T (capi.BASE_RUN_DTYPE, kind BASE_N for 'N', BASE_OTHER for the rest)."""

    def __init__(self, codes, byte_off, lengths, runs):
        self.codes, self.byte_off, self.lengths, self.runs = codes, byte_off, lengths, runs

    @property
    def nscaf(self):
        return int(self.lengths.size)

    @property
    def nbytes(self):
        """what crosses the host link: codes and runs"""
        return int(self.codes.nbytes + self.runs.nbytes)


_UCSC_CODE = np.zeros(256, dtype=np.uint8)           # T=0 C=1 A=2 G=3, either case; 0 for every other byte
_BASE_CLASS = np.full(256, 2, dtype=np.uint8)          # 0: A/C/G/T (either case), 1: 'N', 2: any other byte (quirk Q2)
for _i, _c in enumerate(b"TCAG"):
    _UCSC_CODE[_c] = _UCSC_CODE[_c | 0x20] = _i
    _BASE_CLASS[_c] = _BASE_CLASS[_c | 0x20] = 0
_BASE_CLASS[ord("N")] = 1


def packed_assembly(seq, offsets) -> PackedAssembly:
    """ASCII scaffolds (uint8 text, offsets [nscaf+1] delimit them) -> PackedAssembly, lossless with respect to abw_pack_sequences: A/C/G/T of
    either case become codes, maximal runs of 'N' and of any other character become runs.  Raises ValueError on a lower-case 'n', which the
    reference throws on (String.cpp:47-49) and which the encoding cannot carry."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64).astype(np.int64)
    lengths = np.diff(offsets)
    if (lengths < 0).any():
        raise ValueError("offsets must be non-decreasing")
    seq = seq[offsets[0]:offsets[-1]] if offsets.size else seq[:0]
    offsets = offsets - (offsets[0] if offsets.size else 0)
    nscaf = lengths.size
    # every scaffold padded to whole bytes: insert (-len) % 4 zero codes after it
    pad = (-lengths) % 4
    codes = np.insert(_UCSC_CODE[seq], np.repeat(offsets[1:], pad), 0) if pad.any() else _UCSC_CODE[seq]
    q = codes.reshape(-1, 4)
    packed = (q[:, 0] << 6) | (q[:, 1] << 4) | (q[:, 2] << 2) | q[:, 3]
    byte_off = np.zeros(nscaf, dtype=np.uint64)
    if nscaf > 1:
        byte_off[1:] = np.cumsum((lengths + 3) // 4)[:-1]
    # runs: maximal stretches of one non-ACGT class inside one scaffold
    cls = _BASE_CLASS[seq]
    nz = np.flatnonzero(cls)
    if nz.size and (seq[nz] == ord("n")).any():
        raise ValueError("lower-case 'n' in a sequence: the reference throws Illegal_DNAString (String.cpp:47-49)")
    scaf = np.searchsorted(offsets, nz, side="right") - 1
    c = cls[nz]
    new = np.ones(nz.size, dtype=bool)
    if nz.size > 1:
        new[1:] = (nz[1:] != nz[:-1] + 1) | (c[1:] != c[:-1]) | (scaf[1:] != scaf[:-1])
    first = np.flatnonzero(new)
    runs = np.empty(first.size, dtype=capi.BASE_RUN_DTYPE)
    runs["scaf"] = scaf[first]
    runs["start"] = nz[first] - offsets[scaf[first]]
    runs["len"] = np.diff(np.append(first, nz.size))
    runs["kind"] = np.where(c[first] == 1, capi.BASE_N, capi.BASE_OTHER)
    return PackedAssembly(np.ascontiguousarray(packed, dtype=np.uint8), byte_off, lengths.astype(np.uint64), runs)


def pack_2bit(ctx, pa: PackedAssembly, d_codes, d_runs, ticket=0):
    """abw_pack_2bit of a PackedAssembly whose codes and runs are in device memory already (possibly still in flight behind `ticket`)"""
    desc = capi.TwoBitAssembly(d_codes, pa.codes.nbytes, capi._p(pa.byte_off).value, capi._p(pa.lengths).value, d_runs if pa.runs.size else None,
                               pa.runs.size, ticket)
    ss = C.c_void_p()
    ctx.check(ctx.lib.abw_pack_2bit(ctx.h, C.byref(desc), pa.nscaf, C.byref(ss)))
    return ss


class FeatureBuild:
    """Device-resident result of the feature stage; `rows_host()` fetches the .lrn matrix."""

    def __init__(self, ctx, seqset, segs, d_rows, nseg, ncols, nscaf, d_nbps, nk=None):
        self.ctx, self.seqset, self.segs, self.d_rows, self.nseg, self.ncols, self.nscaf, self.d_nbps = ctx, seqset, segs, d_rows, nseg, ncols, nscaf, d_nbps
        self.nk = ncols if nk is None else nk              # k-mer columns; the remaining ncols - nk are coverage columns
        self._milli = None
        self._milli32 = None

    def rows_milli(self, out16=None, out32=None, wait=True):
        """The .lrn matrix as integer thousandths (abw_rows_to_milli): uint16 [nseg][nk] k-mer columns and uint32 [nseg][ncols - nk] coverage columns,
        a quarter of the bytes of the doubles.  out16 / out32: (pinned) buffers to fill; wait=False enqueues the copies on the copy stream
        (complete after ctx.synchronize(); milli_inexact() then tells whether every value was an exact multiple of 0.001)."""
        L, ctx = self.ctx.lib, self.ctx
        ns = self.ncols - self.nk
        n16, n32 = self.nseg * self.nk, self.nseg * ns
        if self._milli is None:
            self._milli = (ctx.alloc(max(n16, 1) * 2), ctx.alloc(max(n32, 1) * 4), ctx.alloc(16))
        d16, d32, dflag = self._milli
        ctx.memset(dflag, 0, 16)
        ctx.check(L.abw_rows_to_milli(ctx.h, C.c_void_p(self.d_rows), self.nseg, self.ncols, 0, self.nk, 16, C.c_void_p(d16), C.c_void_p(dflag)))
        ctx.check(L.abw_rows_to_milli(ctx.h, C.c_void_p(self.d_rows), self.nseg, self.ncols, self.nk, ns, 32, C.c_void_p(d32), C.c_void_p(dflag)))
        k16 = np.empty(n16, dtype=np.uint16) if out16 is None else out16.reshape(-1)[:n16]
        k32 = np.empty(n32, dtype=np.uint32) if out32 is None else out32.reshape(-1)[:n32]
        for arr, d in ((k16, d16), (k32, d32)):
            if arr.size:
                if wait:
                    ctx.to_host(arr, d)
                else:
                    ctx.d2h_async(arr, d)
        return k16.reshape(self.nseg, self.nk), k32.reshape(self.nseg, ns)

    def milli_inexact(self):
        flag = np.zeros(4, dtype=np.int32)
        self.ctx.to_host(flag, (self._milli or self._milli32)[2])
        return int(flag[0])

    def rows_milli32_device(self):
        """Device pointer of the whole matrix as uint32 thousandths [nseg][ncols] (abw_rows_to_milli, bits = 32): what abw_search_create reads with
        ABW_LAYOUT_ROWMAJOR_MILLI32, and what the ranks of a dimension-sharded search exchange instead of doubles.  Freed by close()."""
        L, ctx = self.ctx.lib, self.ctx
        if self._milli32 is None:
            self._milli32 = (ctx.alloc(max(self.nseg * self.ncols, 1) * 4), None, ctx.alloc(16))
        d32, _, dflag = self._milli32
        ctx.memset(dflag, 0, 16)
        ctx.check(L.abw_rows_to_milli(ctx.h, C.c_void_p(self.d_rows), self.nseg, self.ncols, 0, self.ncols, 32, C.c_void_p(d32), C.c_void_p(dflag)))
        return d32

    def rows_milli_host(self):
        k16, k32 = self.rows_milli()
        return k16, k32, self.milli_inexact()

    def rows_host(self, out=None, wait=True):
        """The .lrn matrix.  `out`: a (pinned) float64 buffer of at least nseg*ncols elements to fill instead of a fresh array;
        wait=False enqueues the copy on the copy stream (it overlaps later device work; complete after ctx.synchronize())."""
        if out is None:
            out = np.empty((self.nseg, self.ncols), dtype=np.float64)
        else:
            out = out.reshape(-1)[:self.nseg * self.ncols].reshape(self.nseg, self.ncols)
        if out.size:
            if wait:
                self.ctx.to_host(out, self.d_rows)
            else:
                self.ctx.d2h_async(out, self.d_rows)
        return out

    def seg_first_host(self):
        """first window of every scaffold (+ the total), uint64 [nscaf+1]"""
        seg_first = np.zeros(self.nscaf + 1, dtype=np.uint64)
        self.ctx.check(self.ctx.lib.abw_segments_get(self.ctx.h, self.segs, capi._p(seg_first), None, None, None, None))
        return seg_first

    def segments_host(self):
        seg_first = np.zeros(self.nscaf + 1, dtype=np.uint64)
        seg_scaf = np.zeros(self.nseg, dtype=np.uint32)
        seg_start = np.zeros(self.nseg, dtype=np.uint64)
        seg_end = np.zeros(self.nseg, dtype=np.uint64)
        seg_nonN = np.zeros(self.nseg, dtype=np.uint64)
        L = self.ctx.lib
        self.ctx.check(L.abw_segments_get(self.ctx.h, self.segs, capi._p(seg_first), capi._p(seg_scaf), capi._p(seg_start), capi._p(seg_end), capi._p(seg_nonN)))
        return dict(seg_first=seg_first, seg_scaf=seg_scaf, seg_start=seg_start, seg_end=seg_end, seg_nonN=seg_nonN)

    def segments_async(self, seg_scaf, seg_start, seg_end, seg_nonN):
        """the window table into pinned numpy buffers (uint32, 3 x uint64, at least nseg elements each) on the copy stream; complete after ctx.synchronize()"""
        self.ctx.check(self.ctx.lib.abw_segments_get_async(self.ctx.h, self.segs, capi._p(seg_scaf), capi._p(seg_start), capi._p(seg_end), capi._p(seg_nonN)))

    def scaffold_stats_host(self, lengths):
        """(.info columns) length-normalised coverage of the -c sample, GC and N count -- abawaca-build.cpp:597"""
        nN = np.zeros(self.nscaf, dtype=np.uint64)
        nGC = np.zeros(self.nscaf, dtype=np.uint64)
        self.ctx.check(self.ctx.lib.abw_seqset_stats(self.ctx.h, self.seqset, capi._p(nN), capi._p(nGC)))
        nbps = np.zeros(self.nscaf, dtype=np.uint64)
        if self.nscaf:
            self.ctx.to_host(nbps, self.d_nbps)
        lengths = np.asarray(lengths, dtype=np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            cvg = nbps.astype(np.float64) / lengths                               # Scaf::cvg, abawaca-build.cpp:57
            denom = lengths - nN.astype(np.float64)
            gc = np.where(denom == 0, 0.0, nGC.astype(np.float64) / np.where(denom == 0, 1.0, denom))   # Bio::gc, String.cpp:114-131
        trunc3 = lambda x: np.trunc(1000.0 * x) / 1000.0                         # noqa: E731  int(1000.0*x)/1000.0
        return dict(cvg=trunc3(cvg), gc=trunc3(gc), Ns=nN)

    def close(self):
        L = self.ctx.lib
        if self.d_rows:
            self.ctx.free(self.d_rows)
            self.d_rows = None
        if self.d_nbps:
            self.ctx.free(self.d_nbps)
            self.d_nbps = None
        if self._milli is not None:
            for d in self._milli:
                self.ctx.free(d)
            self._milli = None
        if self._milli32 is not None:
            for d in self._milli32:
                if d:
                    self.ctx.free(d)
            self._milli32 = None
        if self.segs:
            L.abw_segments_destroy(self.segs)
            self.segs = None
        if self.seqset:
            L.abw_seqset_destroy(self.seqset)
            self.seqset = None


class ReadSample:
    """One sample's read records for build_features: either abw_read records (READ_DTYPE, the device applies the filter of abawaca-build.cpp:546-550),
    compact abw_read8 records of the reads that passed it on the host (compact_reads), or the same reads coordinate-sorted in about 2 bytes each
    (sorted_reads: uint16 deltas in `recs`, plus `runs` and `exc`), as host arrays or as device pointers (d_recs, d_runs, d_exc with nruns, nexc)."""

    def __init__(self, fmt, n, recs=None, length=0, len16=None, d_recs=None, d_len16=None, runs=None, exc=None, d_runs=None, d_exc=None, nruns=0, nexc=0):
        self.fmt, self.n, self.recs, self.length, self.len16, self.d_recs, self.d_len16 = fmt, int(n), recs, int(length), len16, d_recs, d_len16
        self.runs, self.exc, self.d_runs, self.d_exc = runs, exc, d_runs, d_exc
        self.nruns = int(runs.size) if runs is not None else int(nruns)
        self.nexc = int(exc.size) if exc is not None else int(nexc)

    @property
    def nbytes(self):
        per_read = {capi.READS_FULL: 16, capi.READS_COMPACT: 8, capi.READS_SORTED: 2}[self.fmt]
        return self.n * per_read + (2 * self.n if (self.len16 is not None or self.d_len16) else 0) + 8 * self.nruns + 4 * self.nexc


def _host_filter(r, nscaf, max_snps):
    """the read filter of abawaca-build.cpp:546-550 (mapped, not a secondary alignment, at most max_snps mismatches, scaffold known), file order kept"""
    flag, nsnps = r["flag_nsnps"] & 0xFFFF, r["flag_nsnps"] >> 16
    return r[((flag & 0x104) == 0) & (nsnps <= max_snps) & (r["scaf"] < nscaf)]


def _lengths(lens):
    """(one length for the sample, None) when all reads are that long, else (0, uint16 per-read lengths)"""
    if lens.size == 0 or bool((lens == lens[0]).all()):
        return (int(lens[0]) if lens.size else 0), None
    if int(lens.max()) > 65535:
        raise ValueError("reads longer than 65535 bases need the full record format")
    return 0, lens.astype(np.uint16)


def compact_reads(r, nscaf, max_snps=15) -> ReadSample:
    """What a host-side SAM parser hands over when it applies the read filter itself (abawaca-build.cpp:546-550: mapped, not a secondary alignment,
    at most max_snps mismatches, scaffold known; SURVEY.md section 8b(4)): 8-byte records in SAM order, one length for the sample or uint16 lengths."""
    rr = _host_filter(r, nscaf, max_snps)
    out = np.empty(rr.size, dtype=capi.READ8_DTYPE)
    out["scaf"], out["pos0"] = rr["scaf"], rr["pos0"]
    length, len16 = _lengths(rr["len"])
    return ReadSample(capi.READS_COMPACT, out.size, out, length, len16)


def sorted_reads(r, nscaf, max_snps=15) -> ReadSample:
    """The reads of compact_reads, in the same order, in the ABW_READS_SORTED format (include/abawaca_b200.h): runs of consecutive reads on one
    scaffold, a uint16 position delta per read (0xFFFF: the position is the next entry of `exc`).  About 2 bytes per read when the SAM file is
    coordinate sorted; any order is encoded losslessly."""
    rr = _host_filter(r, nscaf, max_snps)
    n = rr.size
    scaf = rr["scaf"].astype(np.uint32)
    pos = rr["pos0"].astype(np.int64)
    starts = np.flatnonzero(np.concatenate(([n > 0], scaf[1:] != scaf[:-1])))
    runs = np.empty(starts.size, dtype=capi.READ_RUN_DTYPE)
    runs["scaf"] = scaf[starts]
    runs["count"] = np.diff(np.append(starts, n))
    prev = np.empty(n, dtype=np.int64)
    prev[1:] = pos[:-1]
    prev[starts] = 0
    diff = pos - prev
    esc = (diff < 0) | (diff >= 0xFFFF)
    delta = np.where(esc, 0xFFFF, diff).astype(np.uint16)
    length, len16 = _lengths(rr["len"])
    return ReadSample(capi.READS_SORTED, n, delta, length, len16, runs=runs, exc=pos[esc].astype(np.uint32))


def build_features(ctx: capi.Context, seq, offsets, reads, this_sample=0, params=None, kind=capi.FEAT_TRUNC3, skip_A=True,
                   seq_on_device=False, reads_on_device=False, nreads=None, timings=None, overlap_h2d=False, seqset=None, per_sample_calls=False) -> FeatureBuild:
    """seq: uint8 ASCII (numpy array, or a device pointer int when seq_on_device), or a PackedAssembly (offsets is then ignored and may be None);
    offsets: uint64 [nscaf+1];
    reads: per sample a structured array (capi.READ_DTYPE), a ReadSample, or a device pointer of abw_read records (reads_on_device, with nreads).
    All samples go through ONE abw_coverage_batch call (per_sample_calls=True: one abw_coverage call per sample, full records only)."""
    L = ctx.lib
    p = params or capi.default_params()
    packed = isinstance(seq, PackedAssembly)
    if packed:
        offsets = None
        nscaf = seq.nscaf
    else:
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        nscaf = offsets.size - 1
    t_last = [time.perf_counter()]

    def lap(name):
        if timings is not None:
            ctx.synchronize()
            now = time.perf_counter()
            timings[name] = timings.get(name, 0.0) + 1000.0 * (now - t_last[0])
            t_last[0] = now
    samples = []
    for j, r in enumerate(reads):
        if isinstance(r, ReadSample):
            samples.append(r)
        elif reads_on_device:
            samples.append(ReadSample(capi.READS_FULL, nreads[j], d_recs=r))
        else:
            r = np.ascontiguousarray(r)
            samples.append(ReadSample(capi.READS_FULL, r.size, r))
    staged = []
    tickets = [0] * len(samples)
    t_seq = 0
    d_2bit = None
    if packed and seqset is None:
        # codes and runs behind one ticket: copies of one stream complete in order, so the ticket of the codes covers the runs
        d_codes = ctx.alloc(max(seq.codes.nbytes, 16))
        d_runs = ctx.alloc(max(seq.runs.nbytes, 16))
        staged += [d_codes, d_runs]
        for a, d in ((seq.runs, d_runs), (seq.codes, d_codes)):
            if a.size == 0:
                continue
            if overlap_h2d:
                t_seq = ctx.h2d_async(d, a)
            else:
                ctx.to_device(d, a)
        d_2bit = (d_codes, d_runs)
    elif not seq_on_device and seqset is None and overlap_h2d:
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        d_seq = ctx.alloc(seq.nbytes + 64)
        staged.append(d_seq)
        t_seq = ctx.h2d_async(d_seq, seq)                  # enqueue every host->device copy up front on the copy stream (inputs should be pinned)
        seq, seq_on_device = d_seq, True
    dev = []                                               # (records, len16, runs, exc) device pointers per sample
    for j, sm in enumerate(samples):
        if sm.d_recs is not None:
            dev.append((sm.d_recs, sm.d_len16, sm.d_runs, sm.d_exc))
            continue
        arrays = [np.ascontiguousarray(a) if a is not None else None for a in (sm.recs, sm.len16, sm.runs, sm.exc)]
        ptrs = []
        for a in arrays:
            d = None
            if a is not None:
                d = ctx.alloc(max(a.nbytes, 16))
                staged.append(d)
            ptrs.append(d)
        # records last: copies of one stream complete in order, so the ticket of the records covers the sample's other arrays too
        for a, d in list(zip(arrays, ptrs))[1:] + [(arrays[0], ptrs[0])]:
            if a is None or a.size == 0:
                continue
            if overlap_h2d:
                tickets[j] = ctx.h2d_async(d, a)
            else:
                ctx.to_device(d, a)
        dev.append(tuple(ptrs))
    if t_seq and not packed:
        ctx.wait_h2d(t_seq)
    if seqset is not None:
        pass                                               # packed elsewhere (fasta_to_seqset); offsets only carry the scaffold count
    elif packed:
        seqset = pack_2bit(ctx, seq, d_2bit[0], d_2bit[1], t_seq)      # waits for the ticket on the device, not on the host
    elif seq_on_device:
        seqset = C.c_void_p()
        ctx.check(L.abw_pack_sequences(ctx.h, C.c_void_p(seq), 1, capi._p(offsets), nscaf, C.byref(seqset)))
    else:
        seqset = C.c_void_p()
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        ctx.check(L.abw_pack_sequences(ctx.h, capi._p(seq), 0, capi._p(offsets), nscaf, C.byref(seqset)))
    lap("pack_ms")
    segs = C.c_void_p()
    ctx.check(L.abw_segment(ctx.h, seqset, p.window_size, C.byref(segs)))
    lap("segment_ms")
    nseg = int(L.abw_segments_count(segs))
    nk = capi.NKMER - (1 if skip_A else 0)
    ncols = nk + len(samples)
    d_rows = ctx.alloc(max(nseg * ncols, 1) * 8)
    d_nbps = ctx.alloc(max(nscaf, 1) * 8)
    ctx.memset(d_nbps, 0, max(nscaf, 1) * 8)
    ctx.check(L.abw_kmer_features(ctx.h, seqset, segs, kind, 1 if skip_A else 0, C.c_void_p(d_rows), ncols, 0))
    lap("kmer_ms")
    if per_sample_calls:
        for j, sm in enumerate(samples):
            assert sm.fmt == capi.READS_FULL
            ctx.wait_h2d(tickets[j])
            nb = C.c_void_p(d_nbps) if j == this_sample else None
            ctx.check(L.abw_coverage(ctx.h, segs, C.c_void_p(dev[j][0]), sm.n, 1, p.max_snps, kind, C.c_void_p(d_rows), ncols, nk + j, nb))
    elif samples:
        arr = (capi.Sample * len(samples))()
        for j, sm in enumerate(samples):
            arr[j].reads, arr[j].nreads, arr[j].format, arr[j].len, arr[j].len16, arr[j].h2d_ticket = dev[j][0], sm.n, sm.fmt, sm.length, dev[j][1], tickets[j]
            if sm.fmt == capi.READS_SORTED:
                arr[j].runs, arr[j].nruns, arr[j].exc, arr[j].nexc = dev[j][2], sm.nruns, dev[j][3], sm.nexc
        ctx.check(L.abw_coverage_batch(ctx.h, segs, arr, len(samples), p.max_snps, kind, C.c_void_p(d_rows), ncols, nk,
                                       this_sample if this_sample is not None else -1, C.c_void_p(d_nbps)))
    ctx.synchronize()
    for d in staged:
        ctx.free(d)
    lap("coverage_ms")
    return FeatureBuild(ctx, seqset, segs, d_rows, nseg, ncols, nscaf, d_nbps, nk)


def search_problem_from_counts(counts):
    """Same as search_problem_from_features, from the number of windows of every scaffold (diff of seg_first)"""
    counts = np.asarray(counts, dtype=np.int64)
    keep_scaf = counts >= 2
    kept = np.nonzero(keep_scaf)[0]
    T = counts[kept].astype(np.uint32)
    keep_rows = np.repeat(keep_scaf, counts)
    dp2scaf = np.repeat(np.arange(kept.size, dtype=np.uint32), T)
    return keep_rows, dp2scaf, T, kept


def search_rows_from_counts(counts):
    """The same problem in the form abw_search_create derives the rest from: (row_of_dp or None, T, kept_scaffolds or None, N).
    Scaffolds with fewer than two windows are dropped (quirk Q1); row_of_dp lists the matrix rows that remain (None: all of them) and
    dp2scaf is left to the library (datapoints of a scaffold are consecutive)."""
    counts = np.asarray(counts, dtype=np.int64)
    drop = counts < 2
    if not drop.any():
        return None, counts.astype(np.uint32), None, int(counts.sum())
    kept = np.flatnonzero(~drop)
    end = np.cumsum(counts)
    mask = np.ones(int(end[-1]), dtype=bool)
    mask[(end - counts)[counts == 1]] = False              # the single row of every dropped scaffold
    row_of_dp = np.flatnonzero(mask).view(np.uint64)       # int64 >= 0: the same bits
    return row_of_dp, counts[kept].astype(np.uint32), kept, int(row_of_dp.size)


def search_problem_from_features(seg_scaf, nscaf):
    """ScafDpData.cpp:91-99: drop scaffolds with exactly one datapoint (quirk Q1), renumber the rest in order.

    Returns (keep_rows, dp2scaf, T, kept_scaffolds)."""
    seg_scaf = np.asarray(seg_scaf)
    counts = np.bincount(seg_scaf, minlength=nscaf)
    keep_scaf = counts != 1
    keep_scaf &= counts > 0
    new_id = np.cumsum(keep_scaf) - 1
    keep_rows = keep_scaf[seg_scaf]
    dp2scaf = new_id[seg_scaf[keep_rows]].astype(np.uint32)
    T = counts[keep_scaf].astype(np.uint32)
    return keep_rows, dp2scaf, T, np.nonzero(keep_scaf)[0]


class SearchResult:
    def __init__(self, recs, dp2cluster, scaf2cluster, profile):
        self.recs, self.dp2cluster, self.scaf2cluster, self.profile = recs, dp2cluster, scaf2cluster, profile


def search(ctx: capi.Context, values, dp2scaf, T, length, scgmask, params=None, strategy=capi.SENS_SPEC, layout=capi.LAYOUT_COLMAJOR,
           values_on_device=False, N=None, D=None, ld=None, want_bins=True, row_of_dp=None, nrows=None, timings=None,
           collectives=None, dim_offset=0, D_total=None, scaf_gc=None, scaf_cvg=None, buffers=None, dim_stride=1) -> SearchResult:
    """values: numpy [D][nrows] (column major) or [nrows][D] (row major), or a device pointer with nrows, D, ld given.
    row_of_dp (uint64 [N], optional): the matrix row of every datapoint; default: N = nrows, datapoint i = row i."""
    L = ctx.lib
    p = params or capi.default_params()
    if not values_on_device:
        values = np.ascontiguousarray(values, dtype=np.float64)
        if layout == capi.LAYOUT_COLMAJOR:
            D, nrows = values.shape
            ld = nrows
        else:
            nrows, D = values.shape
            ld = D
        vptr = capi._p(values)
    else:
        vptr = C.c_void_p(values)
        if nrows is None:
            nrows = N
    if row_of_dp is not None:
        row_of_dp = np.ascontiguousarray(row_of_dp, dtype=np.uint64)
        N = row_of_dp.size
    else:
        N = nrows
    if dp2scaf is not None:                            # None: the matrix holds all T datapoints of every scaffold, in scaffold order
        dp2scaf = np.ascontiguousarray(dp2scaf, dtype=np.uint32)
    T = np.ascontiguousarray(T, dtype=np.uint32)
    length = np.ascontiguousarray(length, dtype=np.uint64)
    scgmask = np.ascontiguousarray(scgmask, dtype=np.uint64)
    if scgmask.ndim == 1:
        scgmask = scgmask.reshape(-1, 1)
    S, W = T.size, scgmask.shape[1]
    h = C.c_void_p()
    t0 = time.perf_counter()
    ctx.check(L.abw_search_create(ctx.h, vptr, 1 if values_on_device else 0, layout, ld, nrows, capi._p(row_of_dp), N, D, capi._p(dp2scaf), S, capi._p(T), capi._p(length),
                                  capi._p(scgmask), W, C.byref(p), strategy, C.byref(h)))
    return _run_search(ctx, h, N, S, D, p, t0, want_bins, timings, collectives, dim_offset, D_total, scaf_gc, scaf_cvg, buffers, dim_stride)


def search_features(ctx: capi.Context, fb: "FeatureBuild", length, scgmask, params=None, strategy=capi.SENS_SPEC, want_bins=True, timings=None, buffers=None):
    """The split search straight from a feature build that is still on the device (abw_search_create_from_features): windows per scaffold, the scaffolds
    ScafDpData would drop and the row index are derived on the device.  length / scgmask: per scaffold of the ASSEMBLY.
    Returns (SearchResult, kept) -- kept[i] = assembly index of scaffold i of the result."""
    L = ctx.lib
    p = params or capi.default_params()
    length = np.ascontiguousarray(length, dtype=np.uint64)
    scgmask = np.ascontiguousarray(scgmask, dtype=np.uint64)
    if scgmask.ndim == 1:
        scgmask = scgmask.reshape(-1, 1)
    W = scgmask.shape[1]
    kept = buffers.get("kept") if buffers is not None else None
    if kept is None or kept.size < fb.nscaf:
        kept = np.zeros(fb.nscaf, dtype=np.uint32)
        if buffers is not None:
            buffers["kept"] = kept
    S, N = C.c_uint32(), C.c_uint64()
    h = C.c_void_p()
    t0 = time.perf_counter()
    ctx.check(L.abw_search_create_from_features(ctx.h, fb.segs, C.c_void_p(fb.d_rows), fb.ncols, fb.ncols, capi._p(length), capi._p(scgmask), W, C.byref(p), strategy,
                                                C.byref(S), C.byref(N), capi._p(kept), C.byref(h)))
    res = _run_search(ctx, h, int(N.value), int(S.value), fb.ncols, p, t0, want_bins, timings, None, 0, None, None, None, buffers)
    return res, kept[:S.value]


def cluster_scg(ctx: capi.Context, scgmask, scaf_lists):
    """ClusterQuality::scg of every scaffold list in scaf_lists through abw_cluster_scg: [(unique SCG names, average copies per name)].
    scgmask: uint64 [S][W] SCG masks of the scaffolds.  abw_cluster_scg reads the masks of a search, so every call creates (and destroys) a
    search of S scaffolds of two equal datapoints each that holds them and is never run: a device sort of 2 S values per call, meant for tests
    and tools that hold the masks on the host, not for tallies inside a search loop."""
    L = ctx.lib
    scgmask = np.ascontiguousarray(scgmask, dtype=np.uint64)
    if scgmask.ndim == 1:
        scgmask = scgmask.reshape(-1, 1)
    S, W = scgmask.shape
    N = 2 * S
    T = np.full(S, 2, dtype=np.uint32)
    values = np.zeros((1, N), dtype=np.float64)
    length = np.zeros(S, dtype=np.uint64)
    p = capi.default_params()
    h = C.c_void_p()
    ctx.check(L.abw_search_create(ctx.h, capi._p(values), 0, capi.LAYOUT_COLMAJOR, N, N, None, N, 1, None, S, capi._p(T), capi._p(length), capi._p(scgmask), W,
                                  C.byref(p), capi.SENS_SPEC, C.byref(h)))
    try:
        out = []
        for scafs in scaf_lists:
            scafs = np.ascontiguousarray(scafs, dtype=np.uint32)
            u, avg = C.c_uint32(), C.c_double()
            ctx.check(L.abw_cluster_scg(ctx.h, h, capi._p(scafs), scafs.size, C.byref(u), C.byref(avg)))
            out.append((u.value, avg.value))
        return out
    finally:
        L.abw_search_destroy(h)


def _run_search(ctx, h, N, S, D, p, t0, want_bins, timings, collectives, dim_offset, D_total, scaf_gc, scaf_cvg, buffers, dim_stride=1):
    L = ctx.lib
    t1 = time.perf_counter()
    try:
        if scaf_gc is not None:
            gc_a, cv_a = np.ascontiguousarray(scaf_gc, dtype=np.float64), np.ascontiguousarray(scaf_cvg, dtype=np.float64)
            ctx.check(L.abw_search_set_scaffold_stats(ctx.h, h, capi._p(gc_a), capi._p(cv_a)))
        cap = int(max(64, 2 * (N // max(p.cluster_ndps_threshold, 1)) + 64))
        n = C.c_uint32()
        if buffers is not None:
            # result buffers kept by the caller across calls (no fresh pages to fault in on every pass)
            if buffers.get("cap", 0) < cap or buffers.get("N", 0) < N or buffers.get("S", 0) < S:
                buffers.update(cap=cap, N=N, S=S, recs=(capi.ClusterRec * cap)(), dp2c=np.zeros(N, dtype=np.uint32), s2c=np.zeros(S, dtype=np.uint32))
            recs, cap = buffers["recs"], buffers["cap"]
            dp2c = buffers["dp2c"][:N] if want_bins else None
            s2c = buffers["s2c"][:S] if want_bins else None
        else:
            recs = (capi.ClusterRec * cap)()
            dp2c = np.zeros(N, dtype=np.uint32) if want_bins else None
            s2c = np.zeros(S, dtype=np.uint32) if want_bins else None
        if collectives is None:
            ctx.check(L.abw_search_run(ctx.h, h, recs, cap, C.byref(n), capi._p(dp2c), capi._p(s2c)))
        else:
            # dimension-sharded search: `values` holds dimensions [dim_offset, dim_offset + D) of D_total on this rank
            ctx.check(L.abw_search_set_shard_strided(h, dim_offset, dim_stride, D_total if D_total is not None else D))
            ctx.check(L.abw_search_run_sharded(ctx.h, h, C.byref(collectives.struct), recs, cap, C.byref(n), capi._p(dp2c), capi._p(s2c)))
        if timings is not None:
            timings["search_create_ms"] = timings.get("search_create_ms", 0.0) + 1000.0 * (t1 - t0)
            timings["search_run_ms"] = timings.get("search_run_ms", 0.0) + 1000.0 * (time.perf_counter() - t1)
        prof = capi.SearchProfile()
        L.abw_search_get_profile(h, C.byref(prof))
        return SearchResult([recs[i] for i in range(min(n.value, cap))], dp2c, s2c, prof)
    finally:
        L.abw_search_destroy(h)
