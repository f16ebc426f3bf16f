"""GPU tests of the .lrn writer on the device (abw_format_lrn): every value must be byte-identical to what the C library's printf writes.

The reference text comes from libc snprintf through ctypes, not from Python's % operator (which prints a NaN with its sign bit set as "nan",
where glibc writes "-nan")."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from golden_util import load_set, search_problem

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "abawaca_b200", "bin")

_libc = ctypes.CDLL(None)
_FMT = {0: b"%.3lf", 1: b"%lf"}


def c_fmt(x, fmt):
    b = ctypes.create_string_buffer(512)
    _libc.snprintf(b, 512, _FMT[fmt], ctypes.c_double(float(x)))
    return b.value


def ref_lines(M, rows, fmt, col0=0, ncols=None):
    ncols = M.shape[1] - col0 if ncols is None else ncols
    return b"".join(b"%d\t" % (r + 1) + b"\t".join(c_fmt(x, fmt) for x in M[r, col0:col0 + ncols]) + b"\n" if ncols else b"%d\n" % (r + 1) for r in rows)


@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def _upload(ctx, M):
    M = np.ascontiguousarray(M, dtype=np.float64)
    d = ctx.alloc(max(M.nbytes, 8))
    if M.size:
        ctx.to_device(d, M)
    return d


def _values_vs_libc(ctx, vals, fmt, D=97):
    from abawaca_b200 import pipeline
    vals = np.asarray(vals, dtype=np.float64)
    pad = (-vals.size) % D
    M = np.concatenate([vals, np.zeros(pad)]).reshape(-1, D)
    d = _upload(ctx, M)
    try:
        got = pipeline.format_lrn_rows(ctx, d, D, D, nlines=M.shape[0], fmt=fmt)
    finally:
        ctx.free(d)
    exp = ref_lines(M, range(M.shape[0]), fmt)
    if got != exp:
        gl, el = got.split(b"\n"), exp.split(b"\n")
        bad = [(i, a, b) for i, (a, b) in enumerate(zip(gl, el)) if a != b][:1]
        if bad:
            i, a, b = bad[0]
            diffs = [(M[i, j], x, y) for j, (x, y) in enumerate(zip(a.split(b"\t")[1:], b.split(b"\t")[1:])) if x != y][:5]
            pytest.fail(f"line {i}: {diffs}")
        pytest.fail(f"{len(gl)} lines against {len(el)}")


def _special_values():
    u = np.uint64
    bits = lambda b: np.array([b], dtype=u).view(np.float64)[0]     # noqa: E731
    v = [0.0, -0.0, 0.0625, -0.0625, 1 / 128, -1 / 128, 0.0005, 0.0015, 0.0025, 5e-7, 1.5e-6, 2.5e-6, -1e-9, 1e-300, -1e-300, 5e-324, -5e-324,
         2.2250738585072014e-308, 2.225073858507201e-308, 1.7976931348623157e308, -1.7976931348623157e308, 1e20, -1e20, 1e22, 1e300,
         np.inf, -np.inf, np.nan, bits(0xFFF8000000000000), bits(0x7FF0000000000001), bits(0xFFF0000000000001), 0.1, 0.2, 0.3, 1 / 3, 2 / 3, 999.9995, 999.9994999]
    for edge in (2.0 ** 53, 2.0 ** 63, 2.0 ** 64, 1e13, 2.0 ** 64 / 1e3, 2.0 ** 64 / 1e6, 1e16):
        for k in range(-3, 4):
            x = np.float64(edge)
            for _ in range(abs(k)):
                x = np.nextafter(x, np.inf if k > 0 else -np.inf)
            v += [float(x), -float(x), float(x) + 0.5, float(x) - 0.25]
    return v


@pytest.mark.parametrize("fmt", [0, 1])
def test_values_equal_libc(ctx, fmt):
    rng = np.random.default_rng(11 + fmt)
    vals = [np.arange(0, 10 ** 6 + 1) / 1000.0, rng.integers(0, 2 ** 31, 200000) / 1000.0, -(rng.integers(0, 2 ** 31, 20000) / 1000.0)]
    vals.append(rng.integers(0, 2 ** 64, 200000, dtype=np.uint64).view(np.float64))                  # random bit patterns: every exponent, both signs
    vals.append(rng.uniform(-1, 1, 100000) * np.exp2(rng.integers(-90, 80, 100000)))
    j = np.arange(0, 20000)
    vals.append((2 * j + 1) / 16.0 if fmt == 0 else (2 * j + 1) / 128.0)                               # exact ties of the last printed digit
    vals.append(-(2 * j + 1) / 16.0 if fmt == 0 else -(2 * j + 1) / 128.0)
    vals.append(np.array(_special_values()))
    _values_vs_libc(ctx, np.concatenate(vals), fmt)


def test_shapes(ctx):
    from abawaca_b200 import capi, pipeline
    rng = np.random.default_rng(3)
    M = rng.integers(0, 100000, (700, 300)) / 1000.0
    M[5, 7], M[9, 299], M[600, 0] = np.nan, 1e300, -np.inf
    d = _upload(ctx, M)
    try:
        full = pipeline.format_lrn_rows(ctx, d, 300, 300, nlines=700, fmt=capi.TEXT_LF)
        assert full == ref_lines(M, range(700), 1)                                                         # D = 300, rows == NULL
        rows = rng.permutation(700)[:400].astype(np.uint64)
        rows.sort()
        assert pipeline.format_lrn_rows(ctx, d, 300, 300, rows=rows, fmt=capi.TEXT_LF) == ref_lines(M, rows, 1)      # host row list
        d_rows = ctx.alloc(rows.nbytes)
        ctx.to_device(d_rows, rows)
        try:
            assert pipeline.format_lrn_rows(ctx, d, 300, 300, rows=d_rows, nlines=rows.size, rows_on_device=True, fmt=capi.TEXT_LF) == ref_lines(M, rows, 1)
        finally:
            ctx.free(d_rows)
        for col0, ncols in ((17, 40), (299, 1), (0, 1), (5, 0), (100, 200)):                             # column sub-ranges
            assert pipeline.format_lrn_rows(ctx, d, 300, ncols, col0=col0, rows=rows[:50], fmt=capi.TEXT_3LF) == ref_lines(M, rows[:50], 0, col0, ncols)
        assert pipeline.format_lrn_rows(ctx, d, 300, 300, nlines=0) == b""
        # a capacity that forces hundreds of pieces: their concatenation is the text of one call
        line_max = max(len(l) for l in full.split(b"\n")) + 1
        pieces = pipeline.format_lrn_rows(ctx, d, 300, 300, nlines=700, fmt=capi.TEXT_LF, cap=line_max + 13)
        assert pieces == full
        # a capacity below the size of the first line: ABW_ERR_ARG and the size needed
        d_text = ctx.alloc(4096)
        done, nbytes = ctypes.c_uint64(), ctypes.c_uint64()
        rc = ctx.lib.abw_format_lrn(ctx.h, ctypes.c_void_p(d), 300, 0, 300, None, 0, 0, 700, capi.TEXT_LF, ctypes.c_void_p(d_text), 100, ctypes.byref(done), ctypes.byref(nbytes))
        ctx.free(d_text)
        assert rc == 2 and done.value == 0 and nbytes.value == len(full.split(b"\n")[0]) + 1
    finally:
        ctx.free(d)


def test_round_trip_through_parse(ctx):
    """abw_parse_lrn(abw_format_lrn(M, "%.3lf")) == M bit for bit for matrices of thousandths"""
    from abawaca_b200 import pipeline
    rng = np.random.default_rng(8)
    M = rng.integers(0, 2 ** 31, (5000, 189)) / 1000.0
    M[:, :179] = rng.integers(0, 1001, (5000, 179)) / 1000.0
    d = _upload(ctx, M)
    try:
        text = pipeline.format_lrn_rows(ctx, d, 189, 189, nlines=5000, cap=1 << 20)
    finally:
        ctx.free(d)
    keys, d_vals, n = pipeline.parse_lrn_rows(ctx, text, 189)
    got = np.zeros((n, 189), dtype=np.float64)
    ctx.to_host(got, d_vals)
    ctx.free(d_vals)
    assert n == 5000 and keys.tolist() == list(range(1, 5001))
    assert np.array_equal(got.view(np.uint64), M.view(np.uint64))


def _norm_lrn(text):
    lines = text.split("\n")
    lines[3] = "\t".join(os.path.basename(x) for x in lines[3].split("\t"))
    return "\n".join(lines)


def test_command_lines_on_cfg1(tmp_path, ctx):
    """both command lines on the reference's configs[0] output: the files the reference wrote byte for byte, and every clusters/<id>.lrn holds the
    datapoints of cluster id in ascending order, each value printed as libc's "%lf" of the input value"""
    from abawaca_b200 import pipeline, synth
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "abawaca_b200", "host")], check=True)
    g = load_set("cfg1")
    wd = str(tmp_path)
    paths = synth.write_reference_inputs(g["mg"], wd)
    build = os.path.join(wd, "build")
    r = subprocess.run([os.path.join(BIN, "abawaca-build"), "-f", paths["fasta"], "-o", build, "-s", os.path.join(wd, "sample*.sam"), "-c", paths["sams"][0]],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert _norm_lrn(open(os.path.join(build, "abawaca.lrn")).read()) == _norm_lrn(g["lrn_text"])
    assert open(os.path.join(build, "abawaca.names")).read() == g["names_text"]
    assert open(os.path.join(build, "abawaca.info")).read() == g["info_text"]
    out = os.path.join(wd, "out")
    env = dict(os.environ, ABW_SCG_LIST=paths["scg_list"])
    r = subprocess.run([os.path.join(BIN, "abawaca"), "-u", build, "-o", out, "-c", paths["gene2scg"], "-p", "8"], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    meta = g["meta"]
    assert open(os.path.join(out, "scaf2cluster.txt")).read() == meta["scaf2cluster"]
    assert open(os.path.join(out, "summary.txt")).read() == meta["summary"]

    prob = search_problem("cfg1")
    vals = prob["values"]                                      # [D][N], datapoints in the order of their ids
    res = pipeline.search(ctx, vals, prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"])
    parent = {rec.id: rec.parent for rec in res.recs}
    dp2c = [int(l.split("\t")[1]) for l in open(os.path.join(out, "dp2cluster.txt")).read().splitlines()[1:]]
    members = {}
    for dp, c in enumerate(dp2c):
        while c:
            members.setdefault(c, []).append(dp)
            c = parent[c]
    children = [c for rec in res.recs if rec.split for c in (rec.child1, rec.child2)]
    assert len(children) == 2 * len(meta["best_separation_log"])
    for cid in children:
        lines = open(os.path.join(out, "clusters", f"{cid}.lrn"), "rb").read().split(b"\n")
        assert lines[0] == b"%% %d" % len(members[cid]) and lines[-1] == b""
        body = lines[4:-1]
        assert [int(l.split(b"\t", 1)[0]) - 1 for l in body] == members[cid]
        for l in body:
            f = l.split(b"\t")
            dp = int(f[0]) - 1
            assert f[1:] == [c_fmt(x, 1) for x in vals[:, dp]], (cid, dp)


def _format_at(ctx, d, ld, nlines, fmt, d_text, cap):
    """one abw_format_lrn call into d_text (any byte address); returns (status, lines done, bytes)"""
    done, nbytes = ctypes.c_uint64(), ctypes.c_uint64()
    rc = ctx.lib.abw_format_lrn(ctx.h, ctypes.c_void_p(d), ld, 0, ld, None, 0, 0, nlines, fmt, ctypes.c_void_p(d_text), cap, ctypes.byref(done), ctypes.byref(nbytes))
    return rc, done.value, nbytes.value


@pytest.mark.parametrize("fmt", [0, 1])
def test_long_values_and_unaligned_text(ctx, fmt):
    """rows whose 32 consecutive values are printed by the host and do not fit the 4 KB staging buffer (written straight to the output), and
    text buffers that start at every address mod 16: the bytes equal libc's and nothing outside [d_text, d_text + nbytes) is touched"""
    rng = np.random.default_rng(21 + fmt)
    D = 70
    M = rng.integers(0, 10 ** 6, (40, D)) / 1000.0
    M[3, 0:40] = 1.7976931348623157e308
    M[4, 5:37] = -1.7976931348623157e308
    M[4, 37:70] = 1e300
    M[17, 1:33] = np.where(np.arange(32) % 2, 1.7976931348623157e308, 1e-5)
    M[30:, :] = rng.integers(0, 2 ** 64, (10, D), dtype=np.uint64).view(np.float64)
    exp = ref_lines(M, range(40), fmt)
    assert max(len(l) for l in exp.split(b"\n")) > 32 * 300
    d = _upload(ctx, M)
    cap = len(exp)
    d_text = ctx.alloc(cap + 64)
    try:
        for k in range(16):
            ctx.memset(d_text, 0xAB, cap + 64)
            rc, done, nbytes = _format_at(ctx, d, D, 40, fmt, d_text + k, cap)
            assert (rc, done, nbytes) == (0, 40, len(exp)), k
            got = np.empty(cap + 64, dtype=np.uint8)
            ctx.to_host(got, d_text)
            assert got[k:k + nbytes].tobytes() == exp, k
            assert (got[:k] == 0xAB).all() and (got[k + nbytes:] == 0xAB).all(), k
    finally:
        ctx.free(d_text)
        ctx.free(d)


def test_gather_rows(ctx):
    """abw_gather_rows: rows picked from a host or device list, the first ncols values of each, into a matrix of another stride"""
    rng = np.random.default_rng(4)
    src = rng.standard_normal((500, 37))
    rows = rng.integers(0, 500, 800).astype(np.uint64)
    d_src = _upload(ctx, src)
    d_dst = ctx.alloc(800 * 40 * 8)
    d_rows = ctx.alloc(rows.nbytes)
    ctx.to_device(d_rows, rows)
    try:
        for on_device in (0, 1):
            ctx.memset(d_dst, 0, 800 * 40 * 8)
            r = ctypes.c_void_p(d_rows) if on_device else rows.ctypes.data_as(ctypes.c_void_p)
            ctx.check(ctx.lib.abw_gather_rows(ctx.h, ctypes.c_void_p(d_src), 37, r, on_device, 800, 33, ctypes.c_void_p(d_dst), 40))
            got = np.empty((800, 40))
            ctx.to_host(got, d_dst)
            assert np.array_equal(got[:, :33], src[rows.astype(np.int64), :33]) and not got[:, 33:].any()
    finally:
        ctx.free(d_rows)
        ctx.free(d_dst)
        ctx.free(d_src)


def test_helper_requires_nlines(ctx):
    from abawaca_b200 import pipeline
    with pytest.raises(ValueError, match="nlines"):
        pipeline.format_lrn_rows(ctx, 0, 10, 10)
