"""The assembly in 2 bits per base (abw_pack_2bit, pipeline.packed_assembly) and UCSC .2bit files (abw_twobit_*, hostio.write_twobit).

On the CPU: a numpy restatement of the decode rules of include/abawaca_b200.h takes packed_assembly's output back to the classification of the
ASCII (code, valid bit, N bit per base); a lower-case 'n' is refused; a test-local .2bit writer and reader round-trip in both versions and byte
orders, and agree with hostio.write_twobit.
On the GPU: abw_pack_2bit against abw_pack_sequences on the same assemblies (counts, windows, k-mer rows in both value kinds, coverage rows),
with scaffolds at every byte offset mod 16; malformed runs; staging behind a ticket; abw_twobit_* against the test-local reader; the feature
build from a PackedAssembly against the ASCII path; and the command lines on .2bit files against the same assemblies as FASTA."""
import gzip
import json
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

from golden_util import GOLDEN, load_set

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "abawaca_b200", "bin")
INTERNAL = np.array([3, 1, 0, 2], dtype=np.uint8)        # UCSC code (T C A G) -> code of the packed arrays (A=0 C=1 G=2 T=3)


# ---------------------------------------------------------------------------------------------------------------- restatements and inputs
def ref_decode(pa):
    """per scaffold (code, valid, N) arrays from a PackedAssembly by the rules of include/abawaca_b200.h, run by run"""
    out = []
    for s in range(pa.nscaf):
        L, b = int(pa.lengths[s]), int(pa.byte_off[s])
        i = np.arange(L)
        code = INTERNAL[(pa.codes[b + (i >> 2)] >> (6 - 2 * (i & 3))) & 3] if L else np.zeros(0, np.uint8)
        out.append([code.astype(np.uint8), np.ones(L, bool), np.zeros(L, bool)])
    for scaf, start, ln, kind in pa.runs.tolist():
        if scaf >= pa.nscaf or start >= int(pa.lengths[scaf]) or ln == 0:
            continue
        code, valid, nb = out[scaf]
        sl = slice(start, min(start + ln, int(pa.lengths[scaf])))
        code[sl] = 0
        valid[sl] = False
        if kind == 0:
            nb[sl] = True
    return out


def classify_ascii(seq, offsets):
    """what abw_pack_sequences makes of every character: (code, valid, N) per scaffold"""
    out = []
    for s in range(offsets.size - 1):
        a = seq[int(offsets[s]):int(offsets[s + 1])]
        u = a & 0xDF
        code = np.zeros(a.size, np.uint8)
        for c, v in zip(b"ACGT", range(4)):
            code[u == c] = v
        valid = np.isin(u, list(b"ACGT"))
        out.append([code, valid, u == ord("N")])
    return out


def ascii_of(decoded):
    """ASCII that abw_pack_sequences classifies as `decoded` (OTHER positions become 'R')"""
    seqs = []
    for code, valid, nb in decoded:
        a = np.frombuffer(b"ACGT", np.uint8)[code].copy()
        a[~valid] = ord("R")
        a[nb] = ord("N")
        seqs.append(a)
    return seqs


LENGTHS = [0, 1, 3, 4, 5, 15, 16, 17, 31, 32, 33, 127, 128, 129, 4000, 4001]


def random_assembly(seed, lengths=LENGTHS, iupac=True, lower=True):
    """ASCII scaffolds with upper and lower case, IUPAC codes, and N runs at the first and last base and across 16- and 32-base words"""
    rng = np.random.default_rng(seed)
    seqs = []
    for L in lengths:
        a = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)].copy()
        if L:
            for _ in range(rng.integers(0, 4)):
                st = int(rng.integers(0, L))
                a[st:st + int(rng.integers(1, 40))] = ord("N")
            if rng.random() < 0.5:
                a[0] = ord("N")
            if rng.random() < 0.5:
                a[-1] = ord("N")
            for w in (16, 32):
                if L > w + 2:
                    a[w - 2:w + 2] = ord("N")
            if iupac:
                pos = rng.integers(0, L, max(1, L // 50))
                a[pos] = np.frombuffer(b"RYKMSWBDHV-.", np.uint8)[rng.integers(0, 12, pos.size)]
            if lower:
                low = (rng.random(L) < 0.3) & (a != ord("N"))
                a[low] |= 0x20
        seqs.append(a)
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([s.size for s in seqs])
    return np.concatenate(seqs) if seqs else np.zeros(0, np.uint8), offsets


def relocate(pa, seed=0):
    """the same PackedAssembly with scaffold s starting at a byte offset = s mod 16, with junk bytes between scaffolds"""
    from abawaca_b200 import pipeline
    rng = np.random.default_rng(seed)
    parts, off, pos = [], [], 0
    for s in range(pa.nscaf):
        nb = (int(pa.lengths[s]) + 3) // 4
        gap = (s - pos) % 16 + 16
        parts.append(rng.integers(0, 256, gap).astype(np.uint8))
        pos += gap
        off.append(pos)
        b = int(pa.byte_off[s])
        parts.append(pa.codes[b:b + nb])
        pos += nb
    parts.append(rng.integers(0, 256, 5).astype(np.uint8))
    return pipeline.PackedAssembly(np.concatenate(parts), np.array(off, dtype=np.uint64), pa.lengths.copy(), pa.runs.copy())


# ---------------------------------------------------------------------------------------------------------------- test-local .2bit writer / reader
def tl_write(names, seqs, version=0, big_endian=False):
    e = ">" if big_endian else "<"
    recs = []
    for s in seqs:
        s = bytes(s)
        nblk, mblk = [], []
        for i, ch in enumerate(s):
            isn = chr(ch).upper() not in "ACGT"
            islow = chr(ch).islower()
            for blk, flag in ((nblk, isn), (mblk, islow)):
                if flag:
                    if blk and blk[-1][0] + blk[-1][1] == i:
                        blk[-1][1] += 1
                    else:
                        blk.append([i, 1])
        dna = bytearray()
        for i in range(0, len(s), 4):
            byte = 0
            for j in range(4):
                ch = chr(s[i + j]).upper() if i + j < len(s) else "T"
                byte = (byte << 2) | ("TCAG".index(ch) if ch in "TCAG" else 0)
            dna.append(byte)
        r = struct.pack(e + "II", len(s), len(nblk)) + b"".join(struct.pack(e + "I", b[0]) for b in nblk) + b"".join(struct.pack(e + "I", b[1]) for b in nblk)
        r += struct.pack(e + "I", len(mblk)) + b"".join(struct.pack(e + "I", b[0]) for b in mblk) + b"".join(struct.pack(e + "I", b[1]) for b in mblk)
        recs.append(r + struct.pack(e + "I", 0) + bytes(dna))
    off = 16 + sum(1 + len(n) + (8 if version else 4) for n in names)
    out = struct.pack(e + "IIII", 0x1A412743, version, len(names), 0)
    for n, r in zip(names, recs):
        out += bytes([len(n)]) + n.encode() + struct.pack(e + ("Q" if version else "I"), off)
        off += len(r)
    return out + b"".join(recs)


def tl_read(data):
    """[(name, twoBitToFa sequence)]"""
    e = "<" if struct.unpack("<I", data[:4])[0] == 0x1A412743 else ">"
    _, version, count, _ = struct.unpack(e + "IIII", data[:16])
    at, out = 16, []
    for _ in range(count):
        n = data[at]
        name = data[at + 1:at + 1 + n].decode()
        at += 1 + n
        off = struct.unpack(e + ("Q" if version else "I"), data[at:at + (8 if version else 4)])[0]
        at += 8 if version else 4
        L, nn = struct.unpack(e + "II", data[off:off + 8])
        p = off + 8
        ns = struct.unpack(e + "%dI" % nn, data[p:p + 4 * nn]); p += 4 * nn
        nz = struct.unpack(e + "%dI" % nn, data[p:p + 4 * nn]); p += 4 * nn
        nm = struct.unpack(e + "I", data[p:p + 4])[0]; p += 4
        ms = struct.unpack(e + "%dI" % nm, data[p:p + 4 * nm]); p += 4 * nm
        mz = struct.unpack(e + "%dI" % nm, data[p:p + 4 * nm]); p += 4 * nm
        p += 4
        seq = bytearray("TCAG"[(data[p + i // 4] >> (6 - 2 * (i % 4))) & 3].encode()[0] for i in range(L))
        for st, sz in zip(ns, nz):
            seq[st:st + sz] = b"N" * sz
        for st, sz in zip(ms, mz):
            seq[st:st + sz] = seq[st:st + sz].lower()
        out.append((name, bytes(seq)))
    return out


def twobit_view(seq_bytes):
    """what twoBitToFa prints for a FASTA sequence that went through faToTwoBit: every non-ACGT character N, case kept"""
    return bytes((c if chr(c).upper() in "ACGT" else (ord("n") if chr(c).islower() else ord("N"))) for c in seq_bytes)


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_encoder_round_trips_to_the_ascii_classification(seed):
    from abawaca_b200 import pipeline
    seq, offsets = random_assembly(seed)
    pa = pipeline.packed_assembly(seq, offsets)
    assert pa.codes.nbytes == sum((int(L) + 3) // 4 for L in np.diff(offsets.astype(np.int64)))
    for got, want in zip(ref_decode(pa), classify_ascii(seq, offsets)):
        for g, w in zip(got, want):
            assert np.array_equal(g, w)
    # runs are maximal: no two runs of one kind touch inside a scaffold
    r = pa.runs
    touch = (r["scaf"][1:] == r["scaf"][:-1]) & (r["start"][:-1] + r["len"][:-1] == r["start"][1:]) & (r["kind"][1:] == r["kind"][:-1])
    assert not touch.any()


def test_encoder_keeps_iupac_codes_of_the_golden_set():
    from abawaca_b200 import pipeline
    kat = json.loads(gzip.open(os.path.join(GOLDEN, "kat_features.json.gz"), "rb").read())
    seqs = [s.encode() for _, s in kat["seqs"]]
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([len(s) for s in seqs])
    seq = np.frombuffer(b"".join(seqs), np.uint8)
    pa = pipeline.packed_assembly(seq, offsets)
    assert (pa.runs["kind"] == 1).any()
    for got, want in zip(ref_decode(pa), classify_ascii(seq, offsets)):
        for g, w in zip(got, want):
            assert np.array_equal(g, w)


def test_encoder_refuses_lower_case_n():
    from abawaca_b200 import pipeline
    seq = np.frombuffer(b"ACGTACGTnACGT", np.uint8)
    with pytest.raises(ValueError, match="lower-case 'n'"):
        pipeline.packed_assembly(seq, np.array([0, seq.size], dtype=np.uint64))


@pytest.mark.parametrize("version", [0, 1])
@pytest.mark.parametrize("big_endian", [False, True])
def test_twobit_writer_and_reader_round_trip(tmp_path, version, big_endian):
    from abawaca_b200 import hostio
    assert tl_write(["x"], [b"ACGT"])[-1] == 0x9C                   # A=10 C=01 G=11 T=00, first base in the high bits
    assert tl_read(tl_write(["x"], [b"ACGT"])) == [("x", b"ACGT")]
    seq, offsets = random_assembly(5)
    seqs = [bytes(seq[int(offsets[i]):int(offsets[i + 1])]) for i in range(offsets.size - 1)]
    names = ["scaf_%d" % i for i in range(len(seqs))]
    data = tl_write(names, seqs, version, big_endian)
    assert tl_read(data) == [(n, twobit_view(s)) for n, s in zip(names, seqs)]
    p = str(tmp_path / "a.2bit")
    hostio.write_twobit(p, names, seqs, version=version, big_endian=big_endian)
    assert open(p, "rb").read() == data


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def random_reads(lengths, seed, n=4000):
    from abawaca_b200 import capi
    rng = np.random.default_rng(seed)
    lengths = np.asarray(lengths, dtype=np.int64)
    ok = np.flatnonzero(lengths > 0)
    r = np.zeros(n, dtype=capi.READ_DTYPE)
    r["scaf"] = ok[rng.integers(0, ok.size, n)]
    r["pos0"] = (rng.random(n) * lengths[r["scaf"]]).astype(np.uint32)
    r["len"] = rng.integers(50, 150, n)
    r["flag_nsnps"] = rng.integers(0, 3, n) << 16
    return r


def features_of(ctx, make_seqset, nscaf, reads, window, kind):
    """stats, window table and rows of a seqset made by make_seqset() (destroyed with the build)"""
    from abawaca_b200 import capi, pipeline
    p = capi.default_params()
    p.window_size = window
    fb = pipeline.build_features(ctx, None, np.zeros(nscaf + 1, dtype=np.uint64), reads, seqset=make_seqset(), params=p, kind=kind)
    nN = np.zeros(nscaf, dtype=np.uint64)
    nGC = np.zeros(nscaf, dtype=np.uint64)
    ctx.check(ctx.lib.abw_seqset_stats(ctx.h, fb.seqset, capi._p(nN), capi._p(nGC)))
    out = dict(nN=nN, nGC=nGC, rows=fb.rows_host().copy(), **fb.segments_host())
    fb.close()
    return out


def pack_ascii(ctx, seq, offsets):
    import ctypes as C
    from abawaca_b200 import capi
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    ss = C.c_void_p()
    ctx.check(ctx.lib.abw_pack_sequences(ctx.h, capi._p(seq) if seq.size else None, 0, capi._p(offsets), offsets.size - 1, C.byref(ss)))
    return ss


def pack_2bit_host(ctx, pa, ticket_arrays=False):
    """abw_pack_2bit with codes and runs copied to the device first (or staged behind one abw_h2d_async ticket); the buffers are freed once the
    context has drained"""
    from abawaca_b200 import pipeline
    d_codes = ctx.alloc(max(pa.codes.nbytes, 16))
    d_runs = ctx.alloc(max(pa.runs.nbytes, 16))
    t = 0
    for a, d in ((pa.runs, d_runs), (pa.codes, d_codes)):
        if a.size:
            if ticket_arrays:
                t = ctx.h2d_async(d, a)
            else:
                ctx.to_device(d, a)
    ss = pipeline.pack_2bit(ctx, pa, d_codes, d_runs, t)
    ctx.synchronize()
    ctx.free(d_codes)
    ctx.free(d_runs)
    return ss


def assert_same_features(ctx, seq, offsets, pa, window, kinds=(0, 1), seed=0, staged=False):
    nscaf = offsets.size - 1
    reads = [random_reads(np.diff(offsets.astype(np.int64)), seed)] if nscaf else []
    for kind in kinds:
        a = features_of(ctx, lambda: pack_ascii(ctx, seq, offsets), nscaf, reads, window, kind)
        b = features_of(ctx, lambda: pack_2bit_host(ctx, pa, staged), nscaf, reads, window, kind)
        for k in a:
            assert np.array_equal(a[k], b[k]), k


@gpu
@pytest.mark.parametrize("window", [50, 2000])
@pytest.mark.parametrize("seed", [11, 12])
def test_pack_2bit_matches_pack_sequences(ctx, seed, window):
    from abawaca_b200 import pipeline
    seq, offsets = random_assembly(seed, LENGTHS + [0, 2, 600, 9000] + [int(x) for x in np.random.default_rng(seed).integers(1, 3000, 20)])
    # one all-N scaffold: every character becomes a window
    seq = np.concatenate((seq, np.frombuffer(b"N" * 300, np.uint8)))
    offsets = np.append(offsets, offsets[-1] + 300).astype(np.uint64)
    pa = pipeline.packed_assembly(seq, offsets)
    assert_same_features(ctx, seq, offsets, pa, window, seed=seed)
    ra = relocate(pa, seed)
    assert sorted(set((ra.byte_off % 16).tolist())) == list(range(16))
    assert_same_features(ctx, seq, offsets, ra, window, seed=seed)


@gpu
def test_malformed_runs_follow_the_header_rules(ctx):
    from abawaca_b200 import capi, pipeline
    seq, offsets = random_assembly(21, [100, 37, 64, 300, 5])
    pa = pipeline.packed_assembly(seq, offsets)
    extra = np.array([(99, 0, 10, 0),          # scaffold out of range: skipped
                      (1, 37, 5, 0),           # start at the length: skipped
                      (1, 40, 5, 1),           # start past the length: skipped
                      (0, 90, 1000, 0),        # reaches past the end: clipped
                      (3, 10, 50, 1), (3, 30, 50, 0), (3, 60, 10, 1),     # N and OTHER overlapping, in both orders
                      (2, 20, 20, 7),          # unknown kind: OTHER
                      (2, 25, 5, 0),           # N inside it
                      (4, 0, 0, 0),            # empty
                      (4, 4, 0xFFFFFFFF, 1)],  # length near 2^32: clipped
                     dtype=capi.BASE_RUN_DTYPE)
    rng = np.random.default_rng(3)
    runs = np.concatenate((pa.runs, extra))[rng.permutation(pa.runs.size + extra.size)]
    bad = pipeline.PackedAssembly(pa.codes, pa.byte_off, pa.lengths, runs)
    want = ascii_of(ref_decode(bad))
    wseq = np.concatenate(want)
    assert_same_features(ctx, wseq, offsets, bad, 20)
    assert_same_features(ctx, wseq, offsets, relocate(bad, 4), 20)


@gpu
def test_staged_behind_a_ticket(ctx):
    import torch
    from abawaca_b200 import pipeline
    seq, offsets = random_assembly(31, [int(x) for x in np.random.default_rng(31).integers(1, 20000, 300)])
    pa = pipeline.packed_assembly(seq, offsets)
    pinned = []
    for name in ("codes", "runs"):
        a = getattr(pa, name)
        t = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
        t.numpy()[:] = a.view(np.uint8).reshape(-1)
        pinned.append(t)
        setattr(pa, name, t.numpy().view(a.dtype))
    launches = ctx.launches
    assert_same_features(ctx, seq, offsets, pa, 2000, staged=True)
    assert ctx.launches > launches
    # through build_features: codes and runs behind one ticket, the pack waits for it on the device
    reads = [random_reads(np.diff(offsets.astype(np.int64)), 5)]
    a = pipeline.build_features(ctx, seq, offsets, reads, overlap_h2d=True)
    b = pipeline.build_features(ctx, pa, None, reads, overlap_h2d=True)
    assert np.array_equal(a.rows_host(), b.rows_host())
    a.close(); b.close()


def scan(ctx, data):
    import ctypes as C
    from abawaca_b200 import capi
    arr = np.frombuffer(data, np.uint8)
    t = C.c_void_p()
    rc = ctx.lib.abw_twobit_scan(ctx.h, capi._p(arr) if arr.size else None, arr.size, C.byref(t))
    return rc, t


@gpu
@pytest.mark.parametrize("version,big_endian", [(0, False), (1, False), (0, True), (1, True)])
def test_twobit_entry_points_match_the_local_reader(ctx, version, big_endian):
    from abawaca_b200 import capi
    seq, offsets = random_assembly(41)
    seqs = [bytes(seq[int(offsets[i]):int(offsets[i + 1])]).replace(b"n", b"N") for i in range(offsets.size - 1)]
    names = ["s%02d" % i for i in range(len(seqs))]
    data = tl_write(names, seqs, version, big_endian)
    rc, t = scan(ctx, data)
    assert rc == 0
    try:
        n = int(ctx.lib.abw_twobit_count(t))
        assert n == len(seqs)
        no, nl, sl = np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint64)
        ctx.check(ctx.lib.abw_twobit_get(ctx.h, t, capi._p(no), capi._p(nl), capi._p(sl)))
        arr = np.frombuffer(data, np.uint8)
        for i, (name, s) in enumerate(tl_read(data)):
            assert data[int(no[i]):int(no[i]) + int(nl[i])].decode() == name and int(sl[i]) == len(s)
            out = np.zeros(max(len(s), 1), np.uint8)
            ctx.check(ctx.lib.abw_twobit_decode(ctx.h, t, i, capi._p(arr), capi._p(out)))
            assert out[:len(s)].tobytes() == s
    finally:
        ctx.lib.abw_twobit_destroy(t)


@gpu
def test_twobit_scan_rejects_malformed_files(ctx):
    good = tl_write(["a", "b"], [b"ACGTNNAC", b"acgtACGT"])
    assert scan(ctx, good)[0] == 0
    ctx.lib.abw_twobit_destroy(scan(ctx, good)[1])
    cases = {"truncated header": good[:10], "truncated record": good[:-1], "bad signature": b"\0" * 4 + good[4:],
             "version 2": good[:4] + struct.pack("<I", 2) + good[8:], "empty name": tl_write([""], [b"ACGT"]),
             "offset outside": good[:18] + struct.pack("<I", 1 << 30) + good[22:]}
    # N blocks: outside the sequence, unsorted, overlapping
    def with_blocks(starts, sizes, L=20):
        rec = struct.pack("<II", L, len(starts)) + struct.pack("<%dI" % len(starts), *starts) + struct.pack("<%dI" % len(sizes), *sizes)
        rec += struct.pack("<II", 0, 0) + b"\0" * ((L + 3) // 4)
        return struct.pack("<IIII", 0x1A412743, 0, 1, 0) + b"\x01x" + struct.pack("<I", 22) + rec
    assert scan(ctx, with_blocks([2, 8], [3, 4]))[0] == 0
    cases.update({"block outside": with_blocks([18], [5]), "unsorted": with_blocks([8, 2], [1, 1]), "overlapping": with_blocks([2, 4], [3, 1])})
    for what, data in cases.items():
        rc, t = scan(ctx, data)
        assert rc == 2, what


@gpu
def test_twobit_pack_refuses_n_under_a_mask_block(ctx):
    import ctypes as C
    from abawaca_b200 import capi
    data = tl_write(["a", "b"], [b"ACGTACGT", b"ACGTnACGT"])     # 'n': an N block inside a mask block
    rc, t = scan(ctx, data)
    assert rc == 0
    arr = np.frombuffer(data, np.uint8)
    d = ctx.alloc(arr.size)
    ctx.to_device(d, arr)
    try:
        ss = C.c_void_p()
        order = np.array([0], np.uint32)
        assert ctx.lib.abw_twobit_pack(ctx.h, t, C.c_void_p(d), 0, capi._p(order), 1, C.byref(ss)) == 0      # record "a" alone is fine
        ctx.lib.abw_seqset_destroy(ss)
        order = np.array([0, 1], np.uint32)
        assert ctx.lib.abw_twobit_pack(ctx.h, t, C.c_void_p(d), 0, capi._p(order), 2, C.byref(ss)) == 3
        assert "Illegal_DNAString" in ctx.lib.abw_last_error(ctx.h).decode()
    finally:
        ctx.free(d)
        ctx.lib.abw_twobit_destroy(t)


def _kat():
    kat = json.loads(gzip.open(os.path.join(GOLDEN, "kat_features.json.gz"), "rb").read())
    from abawaca_b200 import capi
    seqs = sorted(kat["seqs"], key=lambda x: x[0].encode())
    idx = {n: i for i, (n, _) in enumerate(seqs)}
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([len(s) for _, s in seqs])
    seq = np.frombuffer("".join(s for _, s in seqs).encode(), dtype=np.uint8)
    reads = []
    for rr in kat["reads"]:
        rec = np.zeros(len(rr), dtype=capi.READ_DTYPE)
        for i, (rname, pos1, ln, flag, nsnps) in enumerate(rr):
            rec[i] = (idx.get(rname, 0xFFFFFFFF), (pos1 - 1) & 0xFFFFFFFF, ln, (flag & 0xFFFF) | (nsnps << 16))
        reads.append(rec)
    return seq, offsets, reads


@gpu
@pytest.mark.parametrize("which", ["kat_features", "tiny_noisy", "synth"])
def test_build_features_from_a_packed_assembly(ctx, which):
    from abawaca_b200 import pipeline, synth
    if which == "kat_features":
        seq, offsets, reads = _kat()
    elif which == "tiny_noisy":
        mg = load_set("tiny_noisy")["mg"]
        seq, offsets, reads = mg.seq, mg.offsets, mg.reads
    else:
        mg = synth.make_metagenome(400, 3, 4, 777, shuffle_reads=True)
        seq, offsets, reads = mg.seq, mg.offsets, mg.reads
    pa = pipeline.packed_assembly(seq, offsets)
    for overlap in (False, True):
        a = pipeline.build_features(ctx, seq, offsets, reads, this_sample=0, overlap_h2d=overlap)
        b = pipeline.build_features(ctx, pa, None, reads, this_sample=0, overlap_h2d=overlap)
        assert np.array_equal(a.rows_host(), b.rows_host())
        assert pipeline.format_lrn_rows(ctx, a.d_rows, a.ncols, a.ncols, nlines=a.nseg) == pipeline.format_lrn_rows(ctx, b.d_rows, b.ncols, b.ncols, nlines=b.nseg)
        lengths = np.diff(np.asarray(offsets, dtype=np.int64))
        sa, sb = a.scaffold_stats_host(lengths), b.scaffold_stats_host(lengths)
        assert all(np.array_equal(sa[k], sb[k]) for k in sa)
        a.close(); b.close()


# ---------------------------------------------------------------------------------------------------------------- command lines
def _run_cli(wd, assembly, sams, paths):
    build, out = os.path.join(wd, "build"), os.path.join(wd, "out")
    for d in (build, out):
        shutil.rmtree(d, ignore_errors=True)
    r1 = subprocess.run([os.path.join(BIN, "abawaca-build"), "-f", assembly, "-o", build, "-s", sams, "-c", paths["sams"][0]], capture_output=True, text=True)
    if r1.returncode != 0:
        return r1, None
    env = dict(os.environ, ABW_SCG_LIST=paths["scg_list"])
    r2 = subprocess.run([os.path.join(BIN, "abawaca"), "-u", build, "-o", out, "-c", paths["gene2scg"], "-p", "8"], capture_output=True, text=True, env=env)
    assert r2.returncode == 0, r2.stderr[-2000:]
    files = {}
    for base in (build, out):
        for dp, _, fs in os.walk(base):
            for f in fs:
                if f != "log":
                    p = os.path.join(dp, f)
                    files[os.path.relpath(p, wd)] = open(p, "rb").read()
    return r1, files


@gpu
@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
def test_command_lines_on_twobit_files(tmp_path, name):
    from abawaca_b200 import hostio, synth
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "abawaca_b200", "host")], check=True)
    wd = str(tmp_path)
    paths = synth.write_reference_inputs(load_set(name)["mg"], wd)
    names, seqs = hostio.read_fasta(paths["fasta"])
    seqs = [twobit_view(s) for s in seqs]                      # IUPAC codes to N in both arms
    os.makedirs(os.path.join(wd, "fa")); os.makedirs(os.path.join(wd, "tb")); os.makedirs(os.path.join(wd, "be"))
    fa, tb, be = os.path.join(wd, "fa", "assembly"), os.path.join(wd, "tb", "assembly"), os.path.join(wd, "be", "assembly")
    with open(fa, "w") as f:
        for n, s in zip(names, seqs):
            f.write(">%s\n%s\n" % (n, s.decode()))
    hostio.write_twobit(tb, names, seqs)
    hostio.write_twobit(be, names, seqs, version=1, big_endian=True)
    sams = os.path.join(wd, "sample*.sam")
    _, want = _run_cli(wd, fa, sams, paths)
    for path in (tb, be):
        r, got = _run_cli(wd, path, sams, paths)
        assert r.returncode == 0, r.stderr[-2000:]
        assert sorted(got) == sorted(want)
        for k in want:
            if k.endswith("data.txt"):
                a = [l for l in want[k].decode().splitlines() if not l.startswith("Assembly\t")]
                b = [l for l in got[k].decode().splitlines() if not l.startswith("Assembly\t")]
                assert a == b and ("Assembly\t" + path) in got[k].decode()
            else:
                assert got[k] == want[k], k
    assert any(k.startswith(os.path.join("out", "final-clusters")) for k in want)
    # a lower-case 'n' fails as its FASTA does
    seqs[0] = seqs[0][:10] + b"n" + seqs[0][11:]
    with open(fa, "w") as f:
        for n, s in zip(names, seqs):
            f.write(">%s\n%s\n" % (n, s.decode()))
    hostio.write_twobit(tb, names, seqs)
    r_fa, _ = _run_cli(wd, fa, sams, paths)
    r_tb, _ = _run_cli(wd, tb, sams, paths)
    assert r_fa.returncode != 0 and r_tb.returncode == r_fa.returncode
    assert "Fatal error, attempted to initialize DNAString with illegal string" in r_tb.stderr
