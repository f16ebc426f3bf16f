"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C ABI, against
 (a) the committed golden vectors produced by the unmodified reference, and
 (b) the flat-array oracle on seeded random inputs (edge cases: heavy ties, partial scaffolds, SCG filters)."""
import gzip
import json
import os

import numpy as np
import pytest

from golden_util import GOLDEN, load_set, parse_lrn_text, parse_ref_search, search_problem, compare_cluster_records, _random_problem, \
    assert_search_matches_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def _kat_arrays():
    kat = json.loads(gzip.open(os.path.join(GOLDEN, "kat_features.json.gz"), "rb").read())
    from abawaca_b200 import capi
    seqs = sorted(kat["seqs"], key=lambda x: x[0].encode())
    names = [n for n, _ in seqs]
    idx = {n: i for i, n in enumerate(names)}
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([len(s) for _, s in seqs])
    seq = np.frombuffer("".join(s for _, s in seqs).encode(), dtype=np.uint8)
    reads = []
    for rr in kat["reads"]:
        rec = np.zeros(len(rr), dtype=capi.READ_DTYPE)
        for i, (rname, pos1, ln, flag, nsnps) in enumerate(rr):
            rec[i] = (idx.get(rname, 0xFFFFFFFF), (pos1 - 1) & 0xFFFFFFFF, ln, (flag & 0xFFFF) | (nsnps << 16))
        reads.append(rec)
    return kat, names, seq, offsets, reads


def test_kat_features_bit_exact(ctx):
    from abawaca_b200 import capi, pipeline
    kat, names, seq, offsets, reads = _kat_arrays()
    fb = pipeline.build_features(ctx, seq, offsets, reads, this_sample=0)
    heads, vals = parse_lrn_text(kat["lrn"])
    rows = fb.rows_host()
    assert rows.shape == vals.shape
    assert np.array_equal(rows, vals)
    sg = fb.segments_host()
    recs = [l.split("\t") for l in kat["names"].splitlines()[1:]]
    per = {}
    for i, r in enumerate(recs):
        s = int(sg["seg_scaf"][i]); per[s] = per.get(s, 0) + 1
        ln = int(sg["seg_end"][i] - sg["seg_start"][i] + 1)
        assert r[2] == f"{names[s]}:({int(sg['seg_start'][i])}, {int(sg['seg_end'][i])}), {int(sg['seg_nonN'][i])}/{ln} non-Ns bps"
    st = fb.scaffold_stats_host(np.diff(offsets.astype(np.int64)))
    for i, l in enumerate(kat["info"].splitlines()):
        nm, ln, cvg, gc, Ns = l.split("\t")
        assert ("%.3f" % st["cvg"][i], "%.3f" % st["gc"][i], int(st["Ns"][i])) == (cvg, gc, int(Ns))
    fb.close()
    # un-truncated doubles
    fb = pipeline.build_features(ctx, seq, offsets, reads, this_sample=0, kind=capi.FEAT_RAW, skip_A=False)
    raw = np.array([[float(x) for x in l.split("\t")[3:]] for l in kat["raw"].splitlines() if l.startswith("SEG")])
    assert np.array_equal(fb.rows_host(), raw)
    fb.close()


def test_lowercase_n_is_rejected_like_the_reference(ctx):
    from abawaca_b200 import capi, pipeline
    seq = np.frombuffer(b"ACGT" * 600 + b"n" + b"ACGT" * 10, dtype=np.uint8)
    with pytest.raises(capi.AbwError, match="Illegal_DNAString"):
        pipeline.build_features(ctx, seq, np.array([0, seq.size], dtype=np.uint64), [])


@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
def test_features_match_reference_files(ctx, name):
    from abawaca_b200 import capi, pipeline
    g = load_set(name)
    mg = g["mg"]
    fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=0)
    heads, vals = parse_lrn_text(g["lrn_text"])
    assert np.array_equal(fb.rows_host(), vals)
    st = fb.scaffold_stats_host(np.diff(mg.offsets.astype(np.int64)))
    info = [l.split("\t") for l in g["info_text"].splitlines()]
    assert ["%.3f" % v for v in st["cvg"]] == [x[2] for x in info]
    assert ["%.3f" % v for v in st["gc"]] == [x[3] for x in info]
    assert [int(x[4]) for x in info] == st["Ns"].tolist()
    fb.close()
    fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=0, kind=capi.FEAT_RAW, skip_A=False)
    assert np.array_equal(fb.rows_host()[:, 180:], g["rawcov"])
    fb.close()


@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
@pytest.mark.parametrize("strategy", [0, 1])
def test_search_matches_reference(ctx, name, strategy):
    from abawaca_b200 import capi, pipeline
    g = load_set(name)
    prob = search_problem(name)
    ref_clusters, ref_bins = parse_ref_search(g["meta"]["ref_search"]["sensspec" if strategy == 0 else "splitscafs"])
    # full fidelity: also the best separation the reference logs for terminal clusters
    p = capi.default_params()
    p.min_reported_score = 0.0
    res = pipeline.search(ctx, prob["values"], prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"], params=p, strategy=strategy)
    assert compare_cluster_records(ref_clusters, res.recs, strategy) == []
    assert [b for _, b in ref_bins] == res.scaf2cluster.tolist()
    # default parameters: identical splits and bins
    res = pipeline.search(ctx, prob["values"], prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"], strategy=strategy)
    assert compare_cluster_records(ref_clusters, res.recs, strategy, check_illegal_best=(strategy == 1)) == []
    assert [b for _, b in ref_bins] == res.scaf2cluster.tolist()
    # row-major input (the .lrn layout) gives the same answer
    res2 = pipeline.search(ctx, np.ascontiguousarray(prob["values"].T), prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"], strategy=strategy,
                           layout=capi.LAYOUT_ROWMAJOR)
    assert res2.scaf2cluster.tolist() == res.scaf2cluster.tolist() and res2.dp2cluster.tolist() == res.dp2cluster.tolist()


@pytest.mark.parametrize("seed,partial,scg,strategy", [(1, False, True, 0), (2, True, True, 0), (3, False, False, 0), (4, True, True, 1), (5, False, True, 1),
                                                     (6, False, True, 0), (7, True, False, 0)])
def test_search_matches_oracle_on_random_problems(ctx, oracle, seed, partial, scg, strategy):
    from abawaca_b200 import capi, pipeline
    rng = np.random.default_rng(seed)
    S = int(rng.integers(150, 500))
    D = int(rng.integers(3, 12))
    vals, dp2scaf, T, length, mask = _random_problem(rng, S, D, partial=partial, scg=scg, nclus=int(rng.integers(2, 5)))
    O = oracle.Search(vals, dp2scaf, T, length, mask)
    orecs, odp, osc = O.run(strategy=strategy)
    p = capi.default_params()
    p.min_reported_score = 0.0
    res = pipeline.search(ctx, vals, dp2scaf, T, length, mask, params=p, strategy=strategy)
    assert_search_matches_oracle(orecs, odp, osc, res)


def test_small_and_degenerate_searches(ctx, oracle):
    from abawaca_b200 import pipeline
    rng = np.random.default_rng(11)
    # fewer than 2 x 100 datapoints: never splits; constant columns: no boundary at all
    for S, D, const in ((20, 2, False), (300, 3, True)):
        vals, dp2scaf, T, length, mask = _random_problem(rng, S, D)
        if const:
            vals[:] = 0.25
        O = oracle.Search(vals, dp2scaf, T, length, mask)
        orecs, odp, osc = O.run()
        res = pipeline.search(ctx, vals, dp2scaf, T, length, mask)
        assert len(res.recs) == len(orecs) == 1 and res.recs[0].split == 0
        assert res.scaf2cluster.tolist() == osc.tolist() and res.dp2cluster.tolist() == odp.tolist()


def test_features_match_oracle_on_a_larger_random_assembly(ctx, oracle):
    """size-independent check at a size the oracle still finishes quickly: 3000 scaffolds, shuffled reads"""
    from abawaca_b200 import pipeline, synth
    mg = synth.make_metagenome(3000, 2, 6, 991, shuffle_reads=True, n_run_frac=0.05)
    f = oracle.build_features(mg.seq, mg.offsets, mg.reads, this_sample=1)
    fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=1)
    assert np.array_equal(fb.rows_host(), f["rows"])
    sg = fb.segments_host()
    assert np.array_equal(sg["seg_start"], f["seg_start"]) and np.array_equal(sg["seg_end"], f["seg_end"]) and np.array_equal(sg["seg_scaf"], f["seg_scaf"])
    st = fb.scaffold_stats_host(np.diff(mg.offsets.astype(np.int64)))
    assert np.array_equal(st["cvg"], f["info_cvg"]) and np.array_equal(st["gc"], f["info_gc"]) and np.array_equal(st["Ns"], f["info_Ns"])
    fb.close()


def test_row_index_skips_dropped_rows(ctx):
    """abawaca-build writes rows for scaffolds with a single window; ScafDpData drops them (quirk Q1): row_of_dp does the same without a copy."""
    from abawaca_b200 import capi, pipeline
    prob = search_problem("tiny_clean")
    vals = prob["values"]                                   # [D][N]
    D, N = vals.shape
    rng = np.random.default_rng(3)
    nrows = N + 37
    pos = np.sort(rng.choice(nrows, size=N, replace=False)).astype(np.uint64)
    big = rng.normal(size=(nrows, D))
    big[pos] = vals.T
    ref = pipeline.search(ctx, vals, prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"])
    for layout, mat in ((capi.LAYOUT_ROWMAJOR, big), (capi.LAYOUT_COLMAJOR, np.ascontiguousarray(big.T))):
        res = pipeline.search(ctx, mat, prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"], layout=layout, row_of_dp=pos)
        assert res.scaf2cluster.tolist() == ref.scaf2cluster.tolist() and res.dp2cluster.tolist() == ref.dp2cluster.tolist()
        assert [(r.id, r.split, r.best.dim, r.best.value) for r in res.recs] == [(r.id, r.split, r.best.dim, r.best.value) for r in ref.recs]


def test_search_without_dp2scaf(ctx):
    """dp2scaf may be omitted when the matrix holds all T datapoints of every scaffold (the reference's own flow): the device derives it from T"""
    from abawaca_b200 import pipeline
    prob = search_problem("tiny_clean")
    assert np.array_equal(np.bincount(prob["dp2scaf"]), prob["T"])
    ref = pipeline.search(ctx, prob["values"], prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"])
    res = pipeline.search(ctx, prob["values"], None, prob["T"], prob["len"], prob["scgmask"])
    assert res.scaf2cluster.tolist() == ref.scaf2cluster.tolist() and res.dp2cluster.tolist() == ref.dp2cluster.tolist()
    assert [(r.id, r.split, r.best.dim, r.best.value) for r in res.recs] == [(r.id, r.split, r.best.dim, r.best.value) for r in ref.recs]
    from abawaca_b200 import capi
    with pytest.raises(capi.AbwError, match="sum\\(T\\)"):
        pipeline.search(ctx, prob["values"][:, :-1], None, prob["T"], prob["len"], prob["scgmask"])


def test_terminal_bin_statistics(ctx):
    """ClusterQuality::gc / cvg of the terminal bins (ClusterQuality.cpp:6-27,51-75): length-weighted mean and standard deviation over the assigned
    scaffolds in scaffold order, the same fp64 operations in the same order (python floats are IEEE doubles, evaluated left to right)"""
    import math
    from abawaca_b200 import pipeline
    prob = search_problem("tiny_noisy")
    rng = np.random.default_rng(17)
    S = prob["T"].size
    gc = np.trunc(1000 * rng.uniform(0.25, 0.75, S)) / 1000
    cvg = np.trunc(1000 * rng.uniform(0.0, 40.0, S)) / 1000
    res = pipeline.search(ctx, prob["values"], prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"], scaf_gc=gc, scaf_cvg=cvg)
    nterm = 0
    for r in res.recs:
        if r.split:
            continue
        nterm += 1
        scafs = np.nonzero(res.scaf2cluster == r.id)[0]          # assigned scaffolds of the bin, ascending id
        for x, got_mean, got_sd in ((gc, r.gc_avg, r.gc_sd), (cvg, r.cvg_avg, r.cvg_sd)):
            if scafs.size == 0:
                assert (got_mean, got_sd) == (-1.0, -1.0)
                continue
            mean, total = 0.0, 0
            for s in scafs:
                mean += float(int(prob["len"][s])) * float(x[s])
                total += int(prob["len"][s])
            mean /= float(total)
            sd = 0.0
            for s in scafs:
                sd += float(int(prob["len"][s])) * (float(x[s]) - mean) * (float(x[s]) - mean)
            sd = math.sqrt(sd / float(total - 1))
            assert (got_mean, got_sd) == (mean, sd)
    assert nterm >= 2


def test_coverage_when_the_order_of_the_reads_decides_the_third_decimal(ctx, oracle):
    """Round window lengths: for many windows 1000 * sum(overlaps) / length is an integer, which is where abw_coverage cannot take the value
    from the integer sum (DESIGN.md section 4) and falls back to the in-order accumulation; plus a read over more than 255 windows."""
    from abawaca_b200 import capi, pipeline
    from golden_util import coverage_edge_workload
    seq, offsets, reads = coverage_edge_workload()
    f = oracle.build_features(seq, offsets, reads, this_sample=1, want_raw=True)
    fb = pipeline.build_features(ctx, seq, offsets, reads, this_sample=1)
    rows = fb.rows_host()
    assert np.array_equal(rows, f["rows"])
    st = fb.scaffold_stats_host(np.diff(offsets.astype(np.int64)))
    assert np.array_equal(st["cvg"], f["info_cvg"])
    fb.close()
    fb = pipeline.build_features(ctx, seq, offsets, reads, this_sample=1, kind=capi.FEAT_RAW, skip_A=False)
    assert np.array_equal(fb.rows_host(), f["raw"])
    fb.close()
    # without the all-N scaffold no read covers more than 255 windows: the integer-sum path with its in-order remainder
    keep = offsets.size - 2
    reads2 = [r[r["scaf"] < keep] for r in reads]
    f2 = oracle.build_features(seq[:int(offsets[keep])], offsets[:keep + 1], reads2, this_sample=0)
    fb = pipeline.build_features(ctx, seq[:int(offsets[keep])], offsets[:keep + 1], reads2, this_sample=0)
    assert np.array_equal(fb.rows_host(), f2["rows"])
    fb.close()


def test_coverage_order_windows_match_reference_files(ctx):
    """tests/golden/kat_coverage_order.json.gz: the unmodified reference on windows of round lengths, where the order of the reads decides the
    third decimal of the coverage (the same fixture pins the oracle in tests/test_oracle_vs_reference.py)."""
    import hashlib
    from abawaca_b200 import capi, pipeline
    from golden_util import coverage_edge_workload
    fix = json.loads(gzip.open(os.path.join(GOLDEN, "kat_coverage_order.json.gz"), "rb").read())
    seq, offsets, reads = coverage_edge_workload(**fix["args"])
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()   # noqa: E731
    assert fix["digests"] == dict(seq=sha(seq), offsets=sha(offsets), reads=[sha(r) for r in reads])
    heads, vals = parse_lrn_text(fix["lrn"])
    fb = pipeline.build_features(ctx, seq, offsets, reads, this_sample=0)
    assert np.array_equal(fb.rows_host(), vals)
    st = fb.scaffold_stats_host(np.diff(offsets.astype(np.int64)))
    for i, l in enumerate(fix["info"].splitlines()):
        assert "%.3f" % st["cvg"][i] == l.split("\t")[2]
    fb.close()
    fb = pipeline.build_features(ctx, seq, offsets, reads, this_sample=0, kind=capi.FEAT_RAW, skip_A=False)
    assert np.array_equal(fb.rows_host()[:, 180:], np.array(fix["rawcov"], dtype=np.float64))
    fb.close()


def test_cfg1_matches_reference_files(ctx):
    """BASELINE.json configs[0] (2 000 scaffolds, 3 samples, 8 genomes), the one configuration the unmodified reference runs in full: its .lrn,
    .info, un-truncated coverage, every evaluated cluster of the live strategy and the bins of the real `abawaca` binary (tests/golden/cfg1.*)."""
    from abawaca_b200 import capi, pipeline
    g = load_set("cfg1")
    mg = g["mg"]
    fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=0)
    heads, vals = parse_lrn_text(g["lrn_text"])
    assert np.array_equal(fb.rows_host(), vals)
    st = fb.scaffold_stats_host(np.diff(mg.offsets.astype(np.int64)))
    info = [l.split("\t") for l in g["info_text"].splitlines()]
    assert ["%.3f" % v for v in st["cvg"]] == [x[2] for x in info]
    assert ["%.3f" % v for v in st["gc"]] == [x[3] for x in info]
    assert [int(x[4]) for x in info] == st["Ns"].tolist()
    fb.close()
    fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=0, kind=capi.FEAT_RAW, skip_A=False)
    assert np.array_equal(fb.rows_host()[:, 180:], g["rawcov"])
    fb.close()
    prob = search_problem("cfg1")
    ref_clusters, ref_bins = parse_ref_search(g["meta"]["ref_search"]["sensspec"])
    res = pipeline.search(ctx, prob["values"], prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"])
    assert compare_cluster_records(ref_clusters, res.recs, 0, check_illegal_best=False) == []
    assert [b for _, b in ref_bins] == res.scaf2cluster.tolist()
    lines = [l.split("\t") for l in g["meta"]["scaf2cluster"].splitlines()]      # the real binary's scaf2cluster.txt (abawaca.cpp:205-210)
    assert [int(x[1]) for x in lines] == res.scaf2cluster.tolist()
    assert len(set(res.scaf2cluster.tolist()) - {0}) == 8


def test_search_from_features_equals_the_explicit_problem(ctx):
    """abw_search_create_from_features derives T, the dropped scaffolds (a single window, ScafDpData.cpp:92-93) and the row index on the device: same records
    and bins as abw_search_create on the problem the host derives from the window table."""
    from abawaca_b200 import capi, pipeline, synth
    for min_len, seed in ((1500, 31), (4000, 32)):          # with and without dropped scaffolds
        mg = synth.make_metagenome(1500, 3, 4, seed, min_len=min_len, mean_extra=3000)
        fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=0)
        counts = np.diff(fb.seg_first_host().astype(np.int64))
        assert ((counts < 2).any()) == (min_len == 1500)
        keep, dp2scaf, T, kept = pipeline.search_problem_from_counts(counts)
        length = np.diff(mg.offsets.astype(np.int64)).astype(np.uint64)
        mask = mg.scg_masks()
        p = capi.default_params()
        p.min_reported_score = 0.0
        a = pipeline.search(ctx, fb.d_rows, dp2scaf, T, length[kept], mask[kept], params=p, layout=capi.LAYOUT_ROWMAJOR, values_on_device=True, nrows=fb.nseg,
                            D=fb.ncols, ld=fb.ncols, row_of_dp=None if keep.all() else np.nonzero(keep)[0].astype(np.uint64))
        b, kept_b = pipeline.search_features(ctx, fb, length, mask, params=p)
        fb.close()
        assert kept_b.tolist() == kept.tolist()
        key = lambda r: (r.id, r.parent, r.ndps, r.nscafs, r.split, r.best.found, r.best.dim, r.best.value, r.best.a, r.best.b, r.child1, r.child2,   # noqa: E731
                         r.child1_ndps, r.child2_ndps, r.child1_nscafs, r.child2_nscafs, r.child1_raw, r.child2_raw, r.total_size, r.scg_unique, r.scg_avg)
        assert [key(r) for r in a.recs] == [key(r) for r in b.recs] and len(a.recs) > 1
        assert a.scaf2cluster.tolist() == b.scaf2cluster.tolist() and a.dp2cluster.tolist() == b.dp2cluster.tolist()


def test_matrix_of_integer_thousandths_gives_the_same_search(ctx):
    """ABW_LAYOUT_ROWMAJOR_MILLI32: the matrix as uint32 thousandths (abw_rows_to_milli) -- what the ranks of a dimension-sharded search exchange -- gives
    the records of the search on the doubles, separating values included (value = k / 1000.0, the double abawaca-build prints, abawaca-build.cpp:603)."""
    from abawaca_b200 import capi, pipeline, synth
    for min_len, seed in ((1500, 41), (4000, 42)):          # with and without a row index
        mg = synth.make_metagenome(1200, 3, 4, seed, min_len=min_len, mean_extra=3000)
        fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=0)
        counts = np.diff(fb.seg_first_host().astype(np.int64))
        keep, dp2scaf, T, kept = pipeline.search_problem_from_counts(counts)
        length = np.diff(mg.offsets.astype(np.int64)).astype(np.uint64)[kept]
        mask = mg.scg_masks()[kept]
        p = capi.default_params()
        p.min_reported_score = 0.0
        rod = None if keep.all() else np.nonzero(keep)[0].astype(np.uint64)
        a = pipeline.search(ctx, fb.d_rows, dp2scaf, T, length, mask, params=p, layout=capi.LAYOUT_ROWMAJOR, values_on_device=True, nrows=fb.nseg,
                            D=fb.ncols, ld=fb.ncols, row_of_dp=rod)
        d32 = fb.rows_milli32_device()
        assert fb.milli_inexact() == 0
        b = pipeline.search(ctx, d32, dp2scaf, T, length, mask, params=p, layout=capi.LAYOUT_ROWMAJOR_MILLI32, values_on_device=True, nrows=fb.nseg,
                            D=fb.ncols, ld=fb.ncols, row_of_dp=rod)
        # a block of columns with a stride, as a rank of the sharded search holds them
        c = pipeline.search(ctx, d32 + 4 * 5, dp2scaf, T, length, mask, params=p, layout=capi.LAYOUT_ROWMAJOR_MILLI32, values_on_device=True, nrows=fb.nseg,
                            D=40, ld=fb.ncols, row_of_dp=rod)
        c_ref = pipeline.search(ctx, fb.d_rows + 8 * 5, dp2scaf, T, length, mask, params=p, layout=capi.LAYOUT_ROWMAJOR, values_on_device=True, nrows=fb.nseg,
                                D=40, ld=fb.ncols, row_of_dp=rod)
        fb.close()
        key = lambda r: (r.id, r.parent, r.ndps, r.nscafs, r.split, r.best.found, r.best.dim, r.best.value, r.best.a, r.best.b, r.child1, r.child2,   # noqa: E731
                         r.child1_ndps, r.child2_ndps, r.child1_nscafs, r.child2_nscafs, r.child1_raw, r.child2_raw, r.total_size, r.scg_unique, r.scg_avg)
        assert [key(r) for r in a.recs] == [key(r) for r in b.recs] and len(a.recs) > 1
        assert a.scaf2cluster.tolist() == b.scaf2cluster.tolist() and a.dp2cluster.tolist() == b.dp2cluster.tolist()
        assert [key(r) for r in c.recs] == [key(r) for r in c_ref.recs]
    with pytest.raises(Exception):                          # a host matrix of integers is refused, not misread
        pipeline.search(ctx, np.zeros((4, 2)), np.array([0, 0, 1, 1]), np.array([2, 2]), np.array([10, 10]), np.zeros((2, 1)), layout=capi.LAYOUT_ROWMAJOR_MILLI32)
