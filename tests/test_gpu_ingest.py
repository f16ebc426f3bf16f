"""GPU tests of the SAM ingest (abw_parse_sam): the records must equal what the reference's line parser produces.

The checker is a plain-Python restatement of SAMReader::next_mapping (ReadMappingReader.cpp:80-116), ReadMapping::ReadMapping(const char*)
(ReadMapping.cpp:23-72) and the SNP count of ReadMapping::determine_snps (:78-185); it is pinned by the golden sets: the SAM text written for
them is the text the unmodified reference read when tests/golden/make_golden.py produced the committed .lrn files, and the coverage columns
computed from the parsed records must reproduce those files (test below)."""
import os

import numpy as np
import pytest

from golden_util import load_set, parse_lrn_text

pytestmark = pytest.mark.gpu


def ref_parse_sam(text, index):
    """(scaf, pos0, len, flag | nsnps << 16) per record line, as the reference sees the file"""
    out = []
    for line in text.split("\n"):
        line = line.rstrip("\r\n")
        if line == "" or line[0] == "@":
            continue
        fs = line.split("\t")
        assert len(fs) >= 11
        flag = _atoi(fs[1])
        scaf = index.get(fs[2], 0xFFFFFFFF)
        pos0 = (_atoi(fs[3]) - 1) & 0xFFFFFFFF
        md = ""
        for f in fs[11:]:
            k = f.find("MD:Z:")
            if k >= 0:
                e = f.find(" ", k)
                md = f[k:] if e < 0 else f[k:e]
                break
        nsnps = 0
        if md:
            i = 5
            while i < len(md) and md[i].isdigit():
                i += 1
            while i < len(md):
                if md[i] == "^":
                    i += 1
                    while i < len(md) and not md[i].isdigit():
                        nsnps += 1
                        i += 1
                else:
                    assert "A" <= md[i] <= "Z"
                    nsnps += 1
                    i += 1
                assert i < len(md) and md[i].isdigit()
                while i < len(md) and md[i].isdigit():
                    i += 1
            nsnps += fs[5].count("I")
        out.append((scaf, pos0, len(fs[9]), (flag & 0xFFFF) | (min(nsnps, 0xFFFF) << 16)))
    return out


def _atoi(s):
    s = s.lstrip(" \t\n\v\f\r")
    sign = 1
    if s[:1] in ("+", "-"):
        sign = -1 if s[0] == "-" else 1
        s = s[1:]
    v = 0
    for c in s:
        if not c.isdigit():
            break
        v = v * 10 + ord(c) - 48
    return sign * v


@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


EDGE = "\n".join([
    "@HD\tVN:1.0\tSO:unsorted",
    "@SQ\tSN:s1\tLN:5000",
    "r1\t0\ts1\t1\t42\t100M\t*\t0\t0\t" + "A" * 100 + "\t" + "I" * 100 + "\tMD:Z:100",
    "r2\t16\ts2\t2151\t42\t50M2I48M\t=\t100\t-300\t" + "C" * 100 + "\t" + "I" * 100 + "\tXA:i:0\tMD:Z:5A46^AC10T35\tNM:i:6",          # 2 mismatches + 2 deleted + 1 insertion
    "r3\t256\ts1\t10\t0\t100M\t*\t0\t0\t" + "G" * 100 + "\t" + "I" * 100 + "\tMD:Z:100",                                        # secondary
    "r4\t4\t*\t0\t0\t*\t*\t0\t0\t" + "T" * 100 + "\t" + "I" * 100 + "\tXM:i:0",                                                  # unmapped, no MD
    "r5\t0\tnot_a_scaffold\t7\t42\t100M\t*\t0\t0\t" + "A" * 100 + "\t" + "I" * 100 + "\tMD:Z:100",                               # unknown reference name
    "r6\t0\ts10\t 12\t42\t30M\t*\t0\t0\t" + "ACGTNRYacgt" * 2 + "AC" + "GT" * 3 + "\t" + "I" * 30 + "\tZZ:Z:x MD:Z:3C2G0T21 tail\tMD:Z:30",  # MD inside a field, up to the space; first match wins
    "",
    "r7\t1024\ts1\t4901\t42\t100M\t*\t0\t0\t" + "A" * 100 + "\t" + "I" * 100 + "\tMD:Z:0" + "C0" * 15 + "C84\r",                 # 16 mismatches, CR before the newline
    "r8\t0\ts2\t+33\t42\t10M\t*\t0\t0\tACGTACGTAC\tIIIIIIIIII",                                                                  # exactly 11 fields, no trailing newline
])


def test_edge_lines(ctx):
    from abawaca_b200 import pipeline
    names = ["s1", "s10", "s2"]
    index = {n: i for i, n in enumerate(names)}
    sp = pipeline.SamParser(ctx, names)
    try:
        for text in (EDGE, EDGE + "\n", EDGE.replace("\n", "\r\n"), "@only\theader\n", "", "\n\n"):
            got = sp.parse_to_host(text.encode())
            exp = ref_parse_sam(text, index)
            assert [tuple(int(x) for x in r) for r in got.tolist()] == exp
        exp = ref_parse_sam(EDGE, index)
        assert exp[1] == (2, 2150, 100, 16 | (5 << 16)) and exp[5][3] >> 16 == 3 and exp[6][3] >> 16 == 16 and exp[3][0] == 0xFFFFFFFF
    finally:
        sp.close()


def test_errors_like_the_reference(ctx):
    from abawaca_b200 import capi, pipeline
    sp = pipeline.SamParser(ctx, ["s1"])
    try:
        with pytest.raises(capi.AbwError, match="Illegal_DNAString"):
            sp.parse_to_host(b"r\t0\ts1\t1\t42\t4M\t*\t0\t0\tACnT\tIIII\n")
        with pytest.raises(capi.AbwError, match="fewer than 11"):
            sp.parse_to_host(b"r\t0\ts1\t1\t42\t4M\t*\t0\t0\tACGT\n")
        with pytest.raises(capi.AbwError, match="MD:Z"):
            sp.parse_to_host(b"r\t0\ts1\t1\t42\t4M\t*\t0\t0\tACGT\tIIII\tMD:Z:2a1\n")
        for blank in (b" ", b"  \t ", b" \r"):          # chomp strips only '\r' and '\n': a line of blanks is a record, as the reference reads it
            with pytest.raises(capi.AbwError, match="fewer than 11"):
                sp.parse_to_host(b"r\t0\ts1\t1\t42\t4M\t*\t0\t0\tACGT\tIIII\n" + blank + b"\n")
    finally:
        sp.close()


@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
def test_sam_text_of_the_golden_sets(ctx, tmp_path, name):
    """parse the SAM files the reference read -> same records as the generator's, and the coverage columns of the committed .lrn"""
    from abawaca_b200 import capi, pipeline, synth
    g = load_set(name)
    mg = g["mg"]
    paths = synth.write_reference_inputs(mg, str(tmp_path))
    index = {n: i for i, n in enumerate(mg.names)}
    sp = pipeline.SamParser(ctx, mg.names)
    try:
        parsed = []
        for j, path in enumerate(paths["sams"]):
            text = open(path, "rb").read()
            got = sp.parse_to_host(text)
            assert [tuple(int(x) for x in r) for r in got.tolist()] == ref_parse_sam(text.decode(), index)
            # against the generator: identical for every record that is not unmapped (those carry RNAME '*' and POS 0 in the file)
            src = mg.reads[j]
            mapped = (src["flag_nsnps"] & 0x4) == 0
            assert got.size == src.size and np.array_equal(got[mapped], src[mapped]) and np.array_equal(got["flag_nsnps"], src["flag_nsnps"])
            parsed.append(got)
        fb = pipeline.build_features(ctx, mg.seq, mg.offsets, parsed, this_sample=0)
        heads, vals = parse_lrn_text(g["lrn_text"])
        assert np.array_equal(fb.rows_host(), vals)
        fb.close()
    finally:
        sp.close()


def test_chunked_parsing_of_a_larger_file(ctx, tmp_path):
    """chunks cut at line boundaries, records appended on the device, one abw_coverage call per sample"""
    from abawaca_b200 import capi, pipeline, synth
    mg = synth.make_metagenome(300, 1, 3, 4243, shuffle_reads=True)
    paths = synth.write_reference_inputs(mg, str(tmp_path))
    text = open(paths["sams"][0], "rb").read()
    sp = pipeline.SamParser(ctx, mg.names)
    try:
        cap = mg.reads[0].size + 16
        d = ctx.alloc(cap * 16)
        n = 0
        pos = 0
        chunk = 1 << 20
        while pos < len(text):
            end = min(len(text), pos + chunk)
            if end < len(text):
                end = text.rfind(b"\n", pos, end) + 1
            n += sp.parse(text[pos:end], d + 16 * n, cap - n)
            pos = end
        got = np.zeros(n, dtype=capi.READ_DTYPE)
        ctx.to_host(got, d)
        ctx.free(d)
        src = mg.reads[0]
        mapped = (src["flag_nsnps"] & 0x4) == 0
        assert n == src.size and np.array_equal(got[mapped], src[mapped])
    finally:
        sp.close()


# ---------------------------------------------------------------------------------------------------
# FASTA ingest (abw_fasta_scan / abw_fasta_pack)
# ---------------------------------------------------------------------------------------------------
def ref_read_fasta(text):
    """[(id, sequence)] as SeqIORead_fasta<S>::next_seq (SeqIORead_fasta.h:51-103) with getline(true) (SeqIORead.h:85-121) reads the file"""
    ws = " \t\n\v\f\r"
    out = []
    for line in text.split("\n"):
        t = line.strip(ws)
        if t == "":
            continue
        if t[0] == ">":
            i = 1
            while i < len(t) and t[i] not in ws:
                i += 1
            assert i > 1
            out.append([t[1:i], ""])
        else:
            assert out
            out[-1][1] += t
    return [(a, b) for a, b in out]


FASTA_EDGE = "\n".join([
    "", "   ",
    ">s2 some description here",
    "ACGTACGTAC  ",
    "  acgtNNNNacgt",
    "",
    ">s1\tdesc",
    "AC GT\tAC",                    # interior white space is part of the sequence
    "RYKM" * 10 + "\r",
    "> s0",                          # never reached in the good file: see the error test
])


def _pack_and_compare(ctx, text):
    from abawaca_b200 import pipeline
    recs = ref_read_fasta(text)
    first = {}
    for i, (name, _) in enumerate(recs):
        first.setdefault(name.encode(), i)
    names = sorted(first)
    seqs = [recs[first[k]][1] for k in names]
    ss, got_names, lens = pipeline.fasta_to_seqset(ctx, text.encode())
    assert got_names == [k.decode() for k in names]
    assert lens.tolist() == [len(s) for s in seqs]
    # the same windows, k-mer rows and per-scaffold statistics as packing the host-parsed sequences
    seq = np.frombuffer("".join(seqs).encode(), dtype=np.uint8)
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([len(s) for s in seqs])
    a = pipeline.build_features(ctx, None, offsets, [], seqset=ss)
    b = pipeline.build_features(ctx, seq, offsets, [])
    assert np.array_equal(a.rows_host(), b.rows_host())
    sa, sb = a.segments_host(), b.segments_host()
    assert all(np.array_equal(sa[k], sb[k]) for k in sa)
    lengths = np.diff(offsets.astype(np.int64))
    ta, tb = a.scaffold_stats_host(lengths), b.scaffold_stats_host(lengths)
    assert np.array_equal(ta["gc"], tb["gc"]) and np.array_equal(ta["Ns"], tb["Ns"])
    a.close(); b.close()


def test_fasta_edge_cases(ctx):
    from abawaca_b200 import capi, pipeline
    good = FASTA_EDGE.rsplit("\n", 1)[0]
    for text in (good, good + "\n", good.replace("\n", "\r\n"), ">a\nACGT" * 1 + "\n>a\nTTTT\n>b\n" + "ACGT" * 700 + "\n"):
        _pack_and_compare(ctx, text)
    with pytest.raises(capi.AbwError, match="header line"):
        pipeline.fasta_to_seqset(ctx, FASTA_EDGE.encode())            # '>' followed by white space
    with pytest.raises(capi.AbwError, match="header line"):
        pipeline.fasta_to_seqset(ctx, b"ACGT\n>a\nACGT\n")              # sequence text before the first header


@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
def test_fasta_text_of_the_golden_sets(ctx, tmp_path, name):
    """the FASTA file the reference read -> the committed .lrn / .info (k-mer columns, GC, N counts) through the device-side reader"""
    from abawaca_b200 import pipeline, synth
    g = load_set(name)
    mg = g["mg"]
    paths = synth.write_reference_inputs(mg, str(tmp_path))
    text = open(paths["fasta"], "rb").read()
    ss, names, lens = pipeline.fasta_to_seqset(ctx, text)
    assert names == mg.names and np.array_equal(lens.astype(np.int64), np.diff(mg.offsets.astype(np.int64)))
    fb = pipeline.build_features(ctx, None, mg.offsets, mg.reads, this_sample=0, seqset=ss)
    heads, vals = parse_lrn_text(g["lrn_text"])
    assert np.array_equal(fb.rows_host(), vals)
    st = fb.scaffold_stats_host(np.diff(mg.offsets.astype(np.int64)))
    info = [l.split("\t") for l in g["info_text"].splitlines()]
    assert ["%.3f" % v for v in st["gc"]] == [x[3] for x in info] and [int(x[4]) for x in info] == st["Ns"].tolist()
    fb.close()


# ---------------------------------------------------------------------------------------------------
# .lrn data lines (abw_parse_lrn)
# ---------------------------------------------------------------------------------------------------
def test_lrn_values_equal_atof(ctx):
    """every value must be the double the C library's strtod gives (atof, ClusterData.cpp:159): device fast path and host fallback"""
    from abawaca_b200 import capi, pipeline
    rng = np.random.default_rng(5)
    special = ["0", "-0", "0.000", "1", "-1.5", "0.001", "123456789.123", "1e5", "1E-5", "2.5e+3", ".5", "5.", "+7.25", "9007199254740991", "9007199254740993",
               "0.1234567890123456789", "1e22", "1e23", "1e-22", "1e-23", "1e400", "-1e-400", "inf", "-inf", "nan", "0x1p-3", "12abc", "abc", "", " 3.5", "4.25e", "1.7976931348623157e308",
               "4.9e-324", "0.30000000000000004", "179769313486231570000000000000000000000", "-2147483.648", "65.432"]
    D = 7
    rows = []
    vals = special + ["%.3f" % x for x in rng.uniform(0, 70, 400)] + [repr(float(x)) for x in rng.normal(0, 1e3, 200)] + ["%.17g" % x for x in rng.uniform(-1, 1, 100)]
    while len(vals) % D:
        vals.append("0.5")
    for i in range(0, len(vals), D):
        rows.append(vals[i:i + D])
    text = "% a comment line\n\n" + "".join("%d\t%s\n" % (10 * r + 3, "\t".join(row)) for r, row in enumerate(rows)) + "%\n"
    keys, d_vals, n = pipeline.parse_lrn_rows(ctx, text.encode(), D)
    got = np.zeros((n, D), dtype=np.float64)
    ctx.to_host(got, d_vals)
    ctx.free(d_vals)
    assert n == len(rows) and keys.tolist() == [10 * r + 3 for r in range(len(rows))]
    import ctypes
    libc = ctypes.CDLL(None)
    libc.atof.restype = ctypes.c_double
    exp = np.array([[libc.atof(v.encode()) for v in row] for row in rows])
    assert np.array_equal(got.view(np.uint64), exp.view(np.uint64)), [(v, g, e) for v, g, e in zip(sum(rows, []), got.ravel(), exp.ravel()) if np.float64(g).view(np.uint64) != np.float64(e).view(np.uint64)][:10]
    # a data line ends at its last non-blank character: CRLF, trailing blanks and tabs, lines of blanks (skipped), no final newline
    body = ["%d\t%s" % (10 * r + 3, "\t".join(row)) for r, row in enumerate(rows)]
    for text in ("\r\n".join(body) + "\r\n", " \t\n".join(body) + "\t ", "\n \t  \n".join(body) + "\n \n", "\n".join(body)):
        keys2, d_vals2, n2 = pipeline.parse_lrn_rows(ctx, text.encode(), D)
        got2 = np.zeros((n2, D), dtype=np.float64)
        ctx.to_host(got2, d_vals2)
        ctx.free(d_vals2)
        assert n2 == len(rows) and keys2.tolist() == keys.tolist() and np.array_equal(got2.view(np.uint64), got.view(np.uint64))
    with pytest.raises(capi.AbwError, match="number of tab-separated fields"):
        pipeline.parse_lrn_rows(ctx, b"1\t0.5\t0.25\n2\t0.5\n", 2)


@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
def test_lrn_text_of_the_golden_sets(ctx, name):
    """the .lrn file written by the unmodified reference abawaca-build -> the matrix, handed to the split search without leaving the device"""
    from abawaca_b200 import capi, pipeline
    from golden_util import search_problem
    g = load_set(name)
    lines = g["lrn_text"].split("\n")
    heads, vals = parse_lrn_text(g["lrn_text"])
    D = vals.shape[1]
    body = "\n".join(lines[4:]).encode()
    keys, d_vals, n = pipeline.parse_lrn_rows(ctx, body, D)
    got = np.zeros((n, D), dtype=np.float64)
    ctx.to_host(got, d_vals)
    assert n == vals.shape[0] and np.array_equal(got, vals) and keys.tolist() == list(range(1, n + 1))
    prob = search_problem(name)
    ref = pipeline.search(ctx, prob["values"], prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"])
    if prob["values"].shape[1] == n:                     # (rows of scaffolds with a single window would need row_of_dp: none in these sets)
        res = pipeline.search(ctx, d_vals, prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"], layout=capi.LAYOUT_ROWMAJOR, values_on_device=True, nrows=n, D=D, ld=D)
        assert res.scaf2cluster.tolist() == ref.scaf2cluster.tolist() and [(r.id, r.split, r.best.dim, r.best.value) for r in res.recs] == [(r.id, r.split, r.best.dim, r.best.value) for r in ref.recs]
    ctx.free(d_vals)


# ---------------------------------------------------------------------------------------------------
# Text already on the device (text_on_device = 1), at aligned and unaligned addresses, with newlines on the 4 KB tiles of the line index
# ---------------------------------------------------------------------------------------------------
TILE = 4096


def tile_edge_texts(make, minlen):
    """texts of lines make(i, length) with newlines at the last byte of a tile, at the first byte of the next (alone, and after an empty line),
    and texts of exactly one tile with and without a final newline; every other line is at least minlen bytes long"""
    out = []
    for marks, end in (([TILE - 1], 3 * TILE + 77), ([TILE], 2 * TILE + 1000), ([2 * TILE - 1, 2 * TILE], 3 * TILE), ([TILE - 1], TILE), ([], TILE)):
        cuts = sorted(marks + [p for p in range(120, end, 120) if all(abs(p - m) > minlen for m in marks + [end])])
        lines, prev = [], -1
        for i, c in enumerate(cuts):
            lines.append(make(i, c - prev - 1) + "\n")
            prev = c
        lines.append(make(len(cuts), end - prev - 1))
        text = "".join(lines).encode()
        assert len(text) == end and all(text[m] == 10 for m in marks)
        out.append(text)
    return out


def _pad(head, n, tail="", fill="x"):
    assert n == 0 or len(head) + len(tail) <= n
    return head + fill * (n - len(head) - len(tail)) + tail if n else ""


def sam_line(i, n):
    if i % 11 == 3:
        return _pad("@CO\t", n)
    return _pad("r%d\t%d\ts%d\t%d\t42\t4M\t*\t0\t0\tACGT\tIIII\tMD:Z:%dA%d\tXP:Z:" % (i, 16 * (i % 2), i % 3, i + 1, i % 3, 3 - i % 3), n)


def fasta_line(i, n):
    if i % 6 == 0:
        return _pad(">c%d " % i, n)
    return ("ACGTTGCANC" * (n // 10 + 2))[i % 10:i % 10 + n]


def lrn_line(i, n):
    if i % 13 == 5:
        return _pad("%", n)
    v = "1e30" if i % 7 == 3 else "%d.25" % i              # 1e30 is converted by the host, which reads it from the device text
    return _pad("%d\t" % (i + 1), n, v + "\t0.5", fill="0")


def _device_text(ctx, text, off):
    """device buffer holding text at byte offset off -> (buffer, text pointer)"""
    buf = np.zeros(len(text) + 32, dtype=np.uint8)
    buf[off:off + len(text)] = np.frombuffer(text, dtype=np.uint8)
    d = ctx.alloc(buf.size)
    ctx.to_device(d, buf)
    return d, d + off


def _sam_records(ctx, sp, text, ptr):
    import ctypes as C
    from abawaca_b200 import capi
    cap = text.count(b"\n") + 1
    d = ctx.alloc(cap * 16)
    n = C.c_uint64()
    try:
        ctx.check(ctx.lib.abw_parse_sam(ctx.h, sp.h, C.c_void_p(ptr), len(text), 1, C.c_void_p(d), cap, C.byref(n)))
        out = np.zeros(n.value, dtype=capi.READ_DTYPE)
        ctx.to_host(out, d)
        return out
    finally:
        ctx.free(d)


def _fasta_records(ctx, text, ptr):
    """ids, lengths, N and GC counts and 50-base k-mer rows of all records, through abw_fasta_scan of the host text (ptr None) or of device text"""
    import ctypes as C
    from abawaca_b200 import capi, pipeline
    L = ctx.lib
    arr = np.frombuffer(text, dtype=np.uint8)
    f = C.c_void_p()
    ctx.check(L.abw_fasta_scan(ctx.h, capi._p(arr) if ptr is None else C.c_void_p(ptr), len(text), 0 if ptr is None else 1, C.byref(f)))
    try:
        n = int(L.abw_fasta_count(f))
        id_off, id_len, seq_len = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint64)
        ctx.check(L.abw_fasta_get(ctx.h, f, capi._p(id_off), capi._p(id_len), capi._p(seq_len)))
        order = np.arange(n, dtype=np.uint32)
        ss = C.c_void_p()
        ctx.check(L.abw_fasta_pack(ctx.h, f, capi._p(order), n, C.byref(ss)))
    finally:
        L.abw_fasta_destroy(f)
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(seq_len)
    p = capi.default_params()
    p.window_size = 50
    fb = pipeline.build_features(ctx, None, offsets, [], seqset=ss, params=p)
    nN, nGC = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint64)
    ctx.check(L.abw_seqset_stats(ctx.h, fb.seqset, capi._p(nN), capi._p(nGC)))
    out = [id_off.tolist(), id_len.tolist(), seq_len.tolist(), nN.tolist(), nGC.tolist(), fb.rows_host().tobytes()]
    fb.close()
    return out


def _lrn_rows(ctx, text, ptr, D):
    import ctypes as C
    cap = text.count(b"\n") + 1
    d_keys, d_vals = ctx.alloc(cap * 8), ctx.alloc(cap * D * 8)
    n = C.c_uint64()
    try:
        ctx.check(ctx.lib.abw_parse_lrn(ctx.h, C.c_void_p(ptr), len(text), 1, D, C.c_void_p(d_keys), C.c_void_p(d_vals), cap, C.byref(n)))
        keys, vals = np.zeros(n.value, dtype=np.uint64), np.zeros((n.value, D), dtype=np.float64)
        ctx.to_host(keys, d_keys)
        ctx.to_host(vals, d_vals)
        return keys, vals
    finally:
        ctx.free(d_keys); ctx.free(d_vals)


@pytest.mark.parametrize("fmt", ["sam", "fasta", "lrn"])
def test_text_on_the_device(ctx, fmt):
    """each parser returns for text on the device, at byte offsets 0, 1 and 15 of a buffer, exactly what it returns for the same text on the host;
    the texts put newlines on the last byte of a 4 KB tile and the first byte of the next, and are one tile long"""
    from abawaca_b200 import pipeline
    names = ["s0", "s1", "s2"]
    sp = pipeline.SamParser(ctx, names)
    try:
        for text in tile_edge_texts({"sam": sam_line, "fasta": fasta_line, "lrn": lrn_line}[fmt], 64):
            if fmt == "sam":
                want = sp.parse_to_host(text)
                assert [tuple(int(x) for x in r) for r in want.tolist()] == ref_parse_sam(text.decode(), {n: i for i, n in enumerate(names)})
            elif fmt == "fasta":
                want = _fasta_records(ctx, text, None)
                assert [bytes(text[a:a + l]).decode() for a, l in zip(want[0], want[1])] == [r[0] for r in ref_read_fasta(text.decode())]
            else:
                keys, d_vals, n = pipeline.parse_lrn_rows(ctx, text, 2)
                vals = np.zeros((n, 2), dtype=np.float64)
                ctx.to_host(vals, d_vals)
                ctx.free(d_vals)
                assert n > 10 and 1e30 in vals[:, 0]
            for off in (0, 1, 15):
                d, ptr = _device_text(ctx, text, off)
                try:
                    if fmt == "sam":
                        assert _sam_records(ctx, sp, text, ptr).tobytes() == want.tobytes()
                    elif fmt == "fasta":
                        assert _fasta_records(ctx, text, ptr) == want
                    else:
                        k2, v2 = _lrn_rows(ctx, text, ptr, 2)
                        assert np.array_equal(k2, keys) and np.array_equal(v2.view(np.uint64), vals.view(np.uint64))
                finally:
                    ctx.free(d)
    finally:
        sp.close()
