"""FASTA text of chosen records made on the device (abw_fasta_format, abw_twobit_format), per-record base counts without packing
(abw_fasta_base_counts, abw_twobit_base_counts), and abawaca writing final-clusters/<id>.fasta through them.

On the CPU: the test-local restatement of the rules of include/abawaca_b200.h (records as SeqIORead_fasta reads them, text as abawaca writes it)
against hand-written expectations.
On the GPU: both formats against the restatement byte for byte over texts with every line quirk, text on the host and at device offsets, output at
every address mod 16; windows of every size; the counts against numpy and abw_seqset_stats; the command line on FASTA, reformatted FASTA and .2bit
assemblies against the golden bins."""
import ctypes as C
import hashlib
import os
import shutil
import subprocess

import numpy as np
import pytest

from golden_util import load_set

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "abawaca_b200", "bin")
WS = b" \t\n\v\f\r"                                        # C isspace
UPPER = bytes(c - 32 if 0x61 <= c <= 0x7A else c for c in range(256))


# ---------------------------------------------------------------------------------------------------------------- restatement
def ref_records(text):
    """[(id, desc, seq)] in file order: lines trimmed of white space on both ends, blank lines skipped, '>' opens a record whose id runs to the
    first white space and whose description is the rest after the white space that follows; other lines are appended to the open record"""
    recs = []
    for line in text.split(b"\n"):
        t = line.strip(WS)
        if not t:
            continue
        if t[:1] == b">":
            rest = t[1:]
            i = next((k for k, c in enumerate(rest) if c in WS), len(rest))
            recs.append([rest[:i], rest[i:].lstrip(WS), []])
        else:
            recs[-1][2].append(t)
    return [(i, d, b"".join(s)) for i, d, s in recs]


def ref_text(recs, order):
    """what abawaca writes for the records `order` of recs: header "><id> <desc>", sequence upper-cased (a-z only) in floor(L/60) + 1 lines of 60"""
    out = []
    for r in order:
        rid, desc, seq = recs[r]
        out.append(b">" + rid + b" " + desc + b"\n")
        up = seq.translate(UPPER)
        out.extend(up[j:j + 60] + b"\n" for j in range(0, len(up) + 1, 60))
    return b"".join(out)


def ref_counts(recs):
    up = [np.frombuffer(s.translate(UPPER), np.uint8) for _, _, s in recs]
    return (np.array([int((u == ord("N")).sum()) for u in up], np.uint64),
            np.array([int(((u == ord("C")) | (u == ord("G"))).sum()) for u in up], np.uint64))


def test_restatement_on_hand_written_text():
    text = b"  >a  x \t y\t \r\nac gt\r\n\n\t>b\nNNNN\n>a\n" + b"n" * 60 + b"\n>c desc"
    recs = ref_records(text)
    assert recs == [(b"a", b"x \t y", b"ac gt"), (b"b", b"", b"NNNN"), (b"a", b"", b"n" * 60), (b"c", b"desc", b"")]
    assert ref_text(recs, [0, 2, 3, 0]) == (b">a x \t y\nAC GT\n" + b">a \n" + b"N" * 60 + b"\n\n" + b">c desc\n\n" + b">a x \t y\nAC GT\n")
    assert ref_text([(b"s", b"", bytes(range(0x5B, 0x80)) * 2)], [0]).count(b"\n") == 3
    assert ref_text([(b"s", b"", b"\xe9a{z`")], [0]) == b">s \n\xe9A{Z`\n"
    n, gc = ref_counts(recs)
    assert n.tolist() == [0, 4, 60, 0] and gc.tolist() == [2, 0, 0, 0]


# ---------------------------------------------------------------------------------------------------------------- inputs
LENGTHS = [0, 1, 59, 60, 61, 119, 120, 121, 200000]
ALPHABET = np.frombuffer(b"ACGTACGTACGTacgtacgtNnRYKMSWBDHVrykm-.*" + bytes([0x80, 0xC3, 0xE9, 0xFF]), np.uint8)


def quirky_fasta(seed, lengths=LENGTHS):
    """FASTA text whose records have the given sequence lengths (and a few repeated ids), with input line widths 1, 59, 60, 61, 80 and single lines,
    LF and CRLF, blank lines, leading and trailing blanks and tabs, interior blanks and tabs, every kind of description, no final newline"""
    rng = np.random.default_rng(seed)
    out = []
    for k, L in enumerate(lengths):
        seq = ALPHABET[rng.integers(0, ALPHABET.size, L)].tobytes()
        if L > 10 and k % 2:
            seq = seq[:3] + b" \t " + seq[3:-4] + b"\t" + seq[-4:]          # interior white space stays in the sequence
        rid = b"r%d" % (k % 7 if k >= 7 else k)                              # ids r0 .. r6 repeat
        desc = [b"", b" some words", b" \t  spaced\tout  ", b"\tx\t\t", b"  trailing \t "][k % 5]
        eol = b"\r\n" if k % 3 == 1 else b"\n"
        lead = [b"", b" ", b"\t", b" \t"][k % 4]
        out.append(lead + b">" + rid + desc + eol)
        if k % 4 == 2:
            out.append(b"\n" + b" \t" + eol)
        width = [1, 59, 60, 61, 80, 0][k % 6] if L < 100000 else [80, 61][k % 2]
        chunks = [seq] if width == 0 else [seq[j:j + width] for j in range(0, len(seq), width)]
        for j, c in enumerate(chunks):
            pad = b" " if j % 5 == 4 else b""
            out.append(pad + c + (b"\t " if j % 7 == 3 else b"") + eol)
    text = b"".join(out)
    return text.rstrip(b"\r\n")                                              # no final newline


def window_cases():
    text = quirky_fasta(3, [0, 1, 59, 60, 61, 119, 120, 121, 7, 300])
    recs = ref_records(text)
    order = [9, 0, 3, 3, 8, 1, 2, 7, 5, 4, 6, 9]
    return text, recs, order


# ---------------------------------------------------------------------------------------------------------------- device helpers
@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def windows(asm, ctx, recs, cap, d_base, off, byte0=0):
    """concatenated windows of `cap` bytes from byte0, written at d_base + off -> (text, total)"""
    recs = np.ascontiguousarray(recs, np.uint32)
    out, total = [], None
    while True:
        total, n = asm.format_window(recs, byte0, d_base + off, cap)
        if n:
            buf = np.empty(n, np.uint8)
            ctx.to_host(buf, d_base + off)
            out.append(buf.tobytes())
        byte0 += n
        if byte0 >= total:
            return b"".join(out), total


@gpu
@pytest.mark.parametrize("text_at", ["host", 0, 1, 15])
def test_fasta_format_matches_the_restatement(ctx, text_at):
    from abawaca_b200 import pipeline
    text = quirky_fasta(11)
    recs = ref_records(text)
    assert len(recs) == len(LENGTHS) and all(len(r[2]) >= L for r, L in zip(recs, LENGTHS))
    d_src = None
    if text_at != "host":
        d_src = ctx.alloc(len(text) + 32)
        ctx.to_device(d_src + text_at, np.frombuffer(text, np.uint8))
    asm = pipeline.AssemblyFile(ctx, text, None if d_src is None else d_src + text_at)
    try:
        ids, lens = asm.records()
        assert ids == [r[0] for r in recs] and lens.tolist() == [len(r[2]) for r in recs]
        rng = np.random.default_rng(5)
        orders = [list(range(len(recs))), rng.permutation(len(recs)).tolist() + [8, 0, 0, 3], [8], []]
        for order in orders:
            assert pipeline.format_fasta(ctx, asm, order) == ref_text(recs, order)
        # output at every address mod 16 of interest
        d_out = ctx.alloc(len(ref_text(recs, orders[1])) + 64)
        try:
            for off in (0, 1, 3, 15):
                got, total = windows(asm, ctx, orders[1], 1 << 20, d_out, off)
                assert got == ref_text(recs, orders[1]) and total == len(got)
        finally:
            ctx.free(d_out)
    finally:
        asm.close()
        if d_src is not None:
            ctx.free(d_src)


def twobit_inputs(seed):
    """sequences with N runs, masked (lower-case) stretches, 'n' (an N block under a mask block) and lengths around multiples of 4 and 60"""
    rng = np.random.default_rng(seed)
    lens = [0, 1, 3, 4, 5, 59, 60, 61, 63, 64, 65, 119, 120, 121, 240, 1001, 4001]
    seqs = []
    for L in lens:
        a = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)].copy()
        if L > 8:
            st = int(rng.integers(0, L - 4)); a[st:st + int(rng.integers(1, 40))] = ord("N")
            st = int(rng.integers(0, L - 4)); a[st:st + int(rng.integers(1, 60))] |= 0x20
            a[int(rng.integers(0, L))] = ord("n")
            a[0] = ord("N") if L % 2 else a[0]
        seqs.append(a.tobytes())
    return ["t%02d" % i for i in range(len(seqs))], seqs


@gpu
@pytest.mark.parametrize("version,big_endian", [(0, False), (1, True)])
def test_twobit_format_matches_the_decoded_records(ctx, tmp_path, version, big_endian):
    from abawaca_b200 import capi, hostio, pipeline
    names, seqs = twobit_inputs(21 + version)
    path = str(tmp_path / "a.2bit")
    hostio.write_twobit(path, names, seqs, version=version, big_endian=big_endian)
    data = open(path, "rb").read()
    asm = pipeline.AssemblyFile(ctx, data)
    try:
        assert asm.twobit and asm.count == len(seqs)
        arr = np.frombuffer(data, np.uint8)
        recs = []
        for i, n in enumerate(names):
            out = np.zeros(max(len(seqs[i]), 1), np.uint8)
            ctx.check(ctx.lib.abw_twobit_decode(ctx.h, asm.h, i, capi._p(arr), capi._p(out)))
            recs.append((n.encode(), b"", out[:len(seqs[i])].tobytes()))
        assert any(r[2] != r[2].upper() for r in recs)                           # mask blocks: the decode has lower case to upper-case
        order = list(range(len(recs))) + [16, 2, 2, 0]
        assert pipeline.format_fasta(ctx, asm, order) == ref_text(recs, order)
        d_out = ctx.alloc(len(ref_text(recs, order)) + 64)
        try:
            for off in (1, 15):
                assert windows(asm, ctx, order, 4096, d_out, off)[0] == ref_text(recs, order)
        finally:
            ctx.free(d_out)
        n, gc = pipeline.base_counts(ctx, asm)
        wn, wgc = ref_counts(recs)
        assert n.tolist() == wn.tolist() and gc.tolist() == wgc.tolist()
    finally:
        asm.close()


@gpu
def test_windows_of_every_size(ctx):
    from abawaca_b200 import pipeline
    text, recs, order = window_cases()
    want = ref_text(recs, order)
    asm = pipeline.AssemblyFile(ctx, text)
    d_out = ctx.alloc(len(want) + 64)
    try:
        for cap in (1, 7, 60, 61, 4096, len(want) - 1, len(want), len(want) + 5):
            got, total = windows(asm, ctx, order, cap, d_out, 3)
            assert total == len(want) and got == want, cap
        # from byte0 >= total nothing is written
        ctx.memset(d_out, 0x5A, len(want) + 64)
        for byte0 in (len(want), len(want) + 1):
            total, n = asm.format_window(np.array(order, np.uint32), byte0, d_out, 64)
            assert (total, n) == (len(want), 0)
        buf = np.empty(len(want) + 64, np.uint8)
        ctx.to_host(buf, d_out)
        assert (buf == 0x5A).all()
        assert asm.format_window(np.zeros(0, np.uint32), 0, d_out, 64) == (0, 0)
        total, n = C.c_uint64(), C.c_uint64()
        bad = np.array([0, len(recs)], np.uint32)
        assert ctx.lib.abw_fasta_format(ctx.h, asm.h, bad.ctypes.data_as(C.c_void_p), 2, 0, C.c_void_p(d_out), 64, C.byref(total), C.byref(n)) == 2
    finally:
        ctx.free(d_out)
        asm.close()


@gpu
def test_output_larger_than_one_window(ctx):
    """an assembly whose text exceeds 64 MB, written in 64 MB windows"""
    from abawaca_b200 import pipeline
    rng = np.random.default_rng(9)
    L, nrec = 100003, 700
    body = np.frombuffer(b"ACGTacgtN", np.uint8)[rng.integers(0, 9, L * nrec)]
    parts, recs = [], []
    for r in range(nrec):
        s = body[r * L:(r + 1) * L].tobytes()
        recs.append((b"big%d" % r, b"d", s))
        parts.append(b">big%d d\n" % r + b"\n".join(s[j:j + 80] for j in range(0, L, 80)) + b"\n")
    text = b"".join(parts)
    order = list(range(nrec))
    want = ref_text(recs, order)
    assert len(want) > 64 << 20
    asm = pipeline.AssemblyFile(ctx, text)
    try:
        got = pipeline.format_fasta(ctx, asm, order, cap=64 << 20)
        assert len(got) == len(want) and hashlib.sha256(got).hexdigest() == hashlib.sha256(want).hexdigest()
    finally:
        asm.close()


@gpu
def test_base_counts(ctx, tmp_path):
    from abawaca_b200 import capi, hostio, pipeline
    text = quirky_fasta(17)
    recs = ref_records(text)
    asm = pipeline.AssemblyFile(ctx, text)
    try:
        n, gc = pipeline.base_counts(ctx, asm)
        wn, wgc = ref_counts(recs)
        assert n.tolist() == wn.tolist() and gc.tolist() == wgc.tolist()
    finally:
        asm.close()
    # on records abw_*_pack accepts (no lower-case 'n') the counts are abw_seqset_stats'
    text = text.replace(b"n", b"N")
    recs = ref_records(text)
    names, seqs = [r[0].decode() for r in recs], [r[2] for r in recs]
    path = str(tmp_path / "a.2bit")
    hostio.write_twobit(path, names, [s.upper() for s in seqs])                # no mask blocks: an IUPAC code under one is an 'n' to the pack
    for data in (text, open(path, "rb").read()):
        asm = pipeline.AssemblyFile(ctx, data)
        try:
            n, gc = pipeline.base_counts(ctx, asm)
            ss, snames, _ = (pipeline.twobit_to_seqset if asm.twobit else pipeline.fasta_to_seqset)(ctx, data)
            try:
                sn, sgc = np.zeros(len(snames), np.uint64), np.zeros(len(snames), np.uint64)
                ctx.check(ctx.lib.abw_seqset_stats(ctx.h, ss, capi._p(sn), capi._p(sgc)))
            finally:
                ctx.lib.abw_seqset_destroy(ss)
            first = {}
            for i, nm in enumerate(names):
                first.setdefault(nm, i)
            idx = [first[s] for s in snames]
            assert n[idx].tolist() == sn.tolist() and gc[idx].tolist() == sgc.tolist()
        finally:
            asm.close()


# ---------------------------------------------------------------------------------------------------------------- command line
def _reformat(names, seqs, rng):
    """the same assembly with line widths 50, 61, 80 and 7, CRLF for every other record, mixed-case ACGT, descriptions, and for three ids an
    earlier decoy record (the last record of a name is the one abawaca takes)"""
    out = []
    for k, n in enumerate(names[:3]):
        out.append(b">%s decoy\nACGTTTGCA\n" % n.encode())
    for k, (n, s) in enumerate(zip(names, seqs)):
        a = np.frombuffer(s, np.uint8).copy()
        low = (rng.random(a.size) < 0.3) & np.isin(a, list(b"ACGT"))
        a[low] |= 0x20
        s = a.tobytes()
        eol = b"\r\n" if k % 2 else b"\n"
        w = [50, 61, 80, 7][k % 4]
        out.append(b">" + n.encode() + [b"", b" x y", b"\t desc\t "][k % 3] + eol)
        out.extend(s[j:j + w] + eol for j in range(0, len(s), w))
    return b"".join(out)


def _abawaca(build, out, fasta, paths):
    shutil.rmtree(out, ignore_errors=True)
    env = dict(os.environ, ABW_SCG_LIST=paths["scg_list"])
    cmd = [os.path.join(BIN, "abawaca"), "-u", build]
    if fasta:
        cmd += ["-f", fasta]                                     # after -u: a later -u would override it from data.txt
    return subprocess.run(cmd + ["-o", out, "-c", paths["gene2scg"], "-p", "8"], capture_output=True, text=True, env=env)


@gpu
@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
def test_command_line_bins(tmp_path, name):
    from abawaca_b200 import hostio, synth
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "abawaca_b200", "host")], check=True)
    g = load_set(name)
    wd = str(tmp_path)
    paths = synth.write_reference_inputs(g["mg"], wd)
    build = os.path.join(wd, "build")
    r = subprocess.run([os.path.join(BIN, "abawaca-build"), "-f", paths["fasta"], "-o", build, "-s", os.path.join(wd, "sample*.sam"), "-c", paths["sams"][0]],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    names, seqs = hostio.read_fasta(paths["fasta"])
    refmt = os.path.join(wd, "reformatted.fa")
    with open(refmt, "wb") as f:
        f.write(_reformat(names, seqs, np.random.default_rng(4)))
    tb = os.path.join(wd, "assembly.2bit")
    hostio.write_twobit(tb, names, seqs)
    for fasta in (None, refmt, tb):
        out = os.path.join(wd, "out")
        r = _abawaca(build, out, fasta, paths)
        assert r.returncode == 0, r.stderr[-2000:]
        assert open(os.path.join(out, "scaf2cluster.txt")).read() == g["meta"]["scaf2cluster"]
        assert open(os.path.join(out, "summary.txt")).read() == g["meta"]["summary"]
        if fasta == tb:
            recs = [(n.encode(), b"", s) for n, s in zip(names, seqs)]
        else:
            recs = ref_records(open(fasta or paths["fasta"], "rb").read())
        last = {rid: i for i, (rid, _, _) in enumerate(recs)}
        bins = {}
        for line in g["meta"]["scaf2cluster"].splitlines():
            scaf, cid = line.split("\t")
            bins.setdefault(int(cid), []).append(last[scaf.encode()])
        files = os.listdir(os.path.join(out, "final-clusters"))
        assert set("%d.fasta" % c for c in bins if c) <= set(files)
        for f in files:
            got = open(os.path.join(out, "final-clusters", f), "rb").read()
            assert got == ref_text(recs, bins.get(int(f.split(".")[0]), [])), (fasta, f)
    # a scaffold missing from the -f assembly is still an error, with the same message
    missing = sorted(l.split("\t")[0] for l in g["meta"]["scaf2cluster"].splitlines())[0]
    short = os.path.join(wd, "short.fa")
    with open(short, "w") as f:
        for n, s in zip(names, seqs):
            if n != missing:
                f.write(">%s\n%s\n" % (n, s.decode()))
    r = _abawaca(build, os.path.join(wd, "out"), short, paths)
    assert r.returncode != 0
    assert "scaffold %s is not in %s" % (missing, short) in r.stderr
