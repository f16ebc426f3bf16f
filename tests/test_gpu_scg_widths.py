"""Single-copy-gene (SCG) masks of every width the library takes, against the oracle.

A scaffold's SCG set is a mask of W 64-bit words, W = ceil(G / 64) for G names, up to W = 8 (512 names).  Every kernel that reads the masks loops over
the words: the SCG pass table of the sens/spec sweep (k_pass_table), the masks of the scaffolds that can never flip (k_tab_scaffolds, k_scaf_sides),
the tallies of the terminal bins (k_finalize_terminal), the mask copy of abw_search_create_from_features and abw_cluster_scg (k_scg_tally).  The
problems here put names on both sides of every word boundary, on dense scaffolds and as contamination across cluster centres, and every result is
compared bit for bit with the oracle, which handles any W."""
import os
import subprocess

import numpy as np
import pytest

from golden_util import _random_problem, assert_search_matches_oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "abawaca_b200", "bin")

PT_WARPS = 8           # warps of k_pass_table: the K + 1 entries of a pass table are cut into 8 chunks of a multiple of 32 entries


@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def _params():
    from abawaca_b200 import capi
    p = capi.default_params()
    p.min_reported_score = 0.0
    return p


def _or(masks, W):
    return np.bitwise_or.reduce(masks, axis=0) if len(masks) else np.zeros(W, dtype=np.uint64)


def _pop(masks):
    return np.bitwise_count(masks).sum(axis=-1, dtype=np.int64)


def scg_test(vals, dp2scaf, T, length, mask, overlap=0.2, min_size=500000, min_dps=100):
    """The SCG test of ClusterQuality::is_split_better (ClusterQuality.cpp:96-136) at every candidate of the sens/spec sweep of one cluster, restated in
    numpy.  vals [D][n] / dp2scaf [n]: the datapoints of the cluster; T: the scaffolds' datapoints in the whole problem.

    Side 1 of the candidate after the datapoints with value <= v holds the scaffolds with more than T/2 of their datapoints among them; only
    candidates with at least min_dps datapoints on each side are scored.  Returns, over every dimension, per candidate: the SCG names of side 1 (g1),
    of side 2 (g2), of both (g12), the two side lengths and whether the test accepts."""
    S, N = T.size, dp2scaf.size
    W = mask.shape[1]
    n = np.bincount(dp2scaf, minlength=S)
    flip_rank = T.astype(np.int64) // 2                    # 0-based rank of the datapoint that flips the scaffold
    flippable = n > flip_rank
    carrier = mask.any(axis=1)
    never = _or(mask[carrier & ~flippable], W)             # SCG names on scaffolds that stay on side 2
    out = {k: [] for k in ("g1", "g2", "g12", "size1", "size2")}
    for col in vals:
        order = np.lexsort((np.arange(N), col))
        scaf = dp2scaf[order]
        by_scaf = np.argsort(scaf, kind="stable")          # positions in sweep order, grouped by scaffold
        first = np.concatenate(([0], np.cumsum(n)[:-1]))
        flip_pos = np.full(S, N, dtype=np.int64)
        flip_pos[flippable] = by_scaf[first[flippable] + flip_rank[flippable]]
        sv = col[order]
        ends = np.concatenate((np.flatnonzero(sv[1:] != sv[:-1]) + 1, [N]))
        ends = ends[(ends >= min_dps) & (N - ends >= min_dps)]
        ev = np.flatnonzero(carrier & flippable)
        ev = ev[np.argsort(flip_pos[ev], kind="stable")]
        m = mask[ev]
        pre = np.vstack((np.zeros((1, W), dtype=np.uint64), np.bitwise_or.accumulate(m, axis=0))) if ev.size else np.zeros((1, W), dtype=np.uint64)
        suf = np.vstack((np.bitwise_or.accumulate(m[::-1], axis=0)[::-1], np.zeros((1, W), dtype=np.uint64))) if ev.size else np.zeros((1, W), dtype=np.uint64)
        k = np.searchsorted(flip_pos[ev], ends, side="left")
        side1, side2 = pre[k], suf[k] | never
        out["g1"].append(_pop(side1))
        out["g2"].append(_pop(side2))
        out["g12"].append(_pop(side1 & side2))
        fl = np.sort(flip_pos[flippable])
        cum = np.concatenate(([0], np.cumsum(length[flippable][np.argsort(flip_pos[flippable], kind="stable")].astype(np.int64))))
        s1 = cum[np.searchsorted(fl, ends, side="left")]
        out["size1"].append(s1)
        out["size2"].append(int(length.sum(dtype=np.int64)) - s1)
    r = {k: np.concatenate(v) for k, v in out.items()}
    g1, g2, g12 = r["g1"], r["g2"], r["g12"]
    by_size = (g1 == 0) | (g2 == 0)
    ratio = g12 / np.maximum(np.minimum(g1, g2), 1)
    r["by_size"] = by_size
    r["ratio"] = np.where(by_size, np.nan, ratio)
    r["ok"] = np.where(by_size, (r["size1"] >= min_size) & (r["size2"] >= min_size), ratio >= overlap)
    return r


def scg_test_in_clusters(prob, dp2cluster, ids):
    """scg_test over the root (id 1) and the clusters `ids` of a finished search (terminal ones: dp2cluster holds their datapoints), concatenated."""
    vals, dp2scaf, T, length, mask = prob
    parts = []
    for c in ids:
        dps = np.arange(dp2scaf.size) if c == 1 else np.flatnonzero(dp2cluster == c)
        sc, inv = np.unique(dp2scaf[dps], return_inverse=True)
        parts.append(scg_test(vals[:, dps], inv.astype(np.uint32), T[sc], length[sc], mask[sc]))
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


def _run_both(ctx, oracle, prob, strategy):
    from abawaca_b200 import pipeline
    vals, dp2scaf, T, length, mask = prob
    orecs, odp, osc = oracle.Search(vals, dp2scaf, T, length, mask).run(strategy=strategy)
    res = pipeline.search(ctx, vals, dp2scaf, T, length, mask, params=_params(), strategy=strategy)
    assert_search_matches_oracle(orecs, odp, osc, res)
    return orecs, res


def width_problem(G, seed, partial=False, S=1500, D=4):
    """Five centres, each name on one scaffold of a centre; contamination puts about one more copy of a name in every centre, so that splits inside a
    centre see overlaps on both sides of scg_overlap_threshold."""
    rng = np.random.default_rng(seed)
    return _random_problem(rng, S, D, partial=partial, ties=False, nclus=5, G=G, contamination=0.001, dense=6)


def _assert_highest_name_used(mask, G):
    W = mask.shape[1]
    assert W == (G + 63) // 64
    assert ((mask[:, W - 1] >> np.uint64((G - 1) % 64)) & np.uint64(1)).any()


WIDTH_CASES = [(G, 0, False) for G in (1, 63, 64, 65, 128, 129, 200, 448, 511, 512)] + \
              [(G, 1, False) for G in (64, 129, 512)] + [(G, 0, True) for G in (65, 200, 511)]


@pytest.mark.parametrize("G,strategy,partial", WIDTH_CASES)
def test_search_at_every_mask_width_matches_oracle(ctx, oracle, G, strategy, partial):
    prob = width_problem(G, 1000 + G + 7 * strategy + 29 * partial, partial=partial)
    vals, dp2scaf, T, length, mask = prob
    _assert_highest_name_used(mask, G)
    if partial:
        n = np.bincount(dp2scaf, minlength=T.size)
        assert (mask.any(axis=1) & (n < T // 2 + 1)).any()
    orecs, res = _run_both(ctx, oracle, prob, strategy)
    assert sum(r.split for r in orecs) >= 1
    if strategy == 0:
        r = scg_test_in_clusters(prob, res.dp2cluster, [1] + [o.id for o in orecs if not o.split])
        assert r["ok"].any() and not r["ok"].all()


def chunk_problem(K, G, seed, len_hi=400000):
    """S scaffolds of which exactly K carry SCG names and can all flip (n = T): the root's pass table has K + 1 entries."""
    rng = np.random.default_rng(seed)
    S = max(600, K + K // 5)
    return _random_problem(rng, S, 3, ties=False, nclus=5, G=G, carriers=K, contamination=0.001, dense=min(4, K), len_hi=len_hi)


CHUNK_CASES = [(K, G) for K in (31, 32, 255, 256, 257, 511, 512, 5000) for G in (60, 170)]


@pytest.mark.parametrize("K,G", CHUNK_CASES)
def test_pass_table_chunk_edges_match_oracle(ctx, oracle, K, G):
    prob = chunk_problem(K, G, 2000 + K + G)
    vals, dp2scaf, T, length, mask = prob
    n = np.bincount(dp2scaf, minlength=T.size)
    assert np.count_nonzero(mask.any(axis=1) & (n >= T // 2 + 1)) == K
    _assert_highest_name_used(mask, G)
    ech = (-(-(K + 1) // PT_WARPS) + 31) // 32 * 32     # entries per warp of k_pass_table
    if K >= 5000:
        assert ech >= 4 * 32                             # every warp walks several 32-entry blocks
    orecs, res = _run_both(ctx, oracle, prob, 0)
    r = scg_test_in_clusters(prob, res.dp2cluster, [1] + [o.id for o in orecs if not o.split])
    assert r["ok"].any() and not r["ok"].all()


def test_pass_table_size_rule_and_exact_threshold(ctx, oracle):
    """Candidates where one side has no SCG name (the decision falls to scg_min_size, side lengths on both sides of 500000) and candidates whose
    overlap g12 / min(g1, g2) is exactly the threshold 0.2 (accepted: the test is `< 0.2` rejects)."""
    prob = chunk_problem(31, 60, 81, len_hi=60000)
    orecs, res = _run_both(ctx, oracle, prob, 0)
    r = scg_test_in_clusters(prob, res.dp2cluster, [1] + [o.id for o in orecs if not o.split])
    sz = r["by_size"]
    assert (sz & r["ok"]).any() and (sz & ~r["ok"]).any()
    assert (r["size1"][sz] >= 500000).any() and (r["size1"][sz] < 500000).any()
    assert (r["ratio"] == 0.2).any()


def never_flip_problem(seed):
    """Names 64..127 only on the scaffolds that can never flip (n < T/2 + 1), names 0..63 on at most four scaffolds that can.  The scaffolds that can
    never flip all go to the first child of a split, where k_scaf_sides gathers their names; there the second word decides the SCG test of every
    candidate after the last flippable carrier has flipped (no name of side 2 without it)."""
    rng = np.random.default_rng(seed)
    vals, dp2scaf, T, length, mask = _random_problem(rng, 1500, 4, partial=True, ties=False, nclus=5, G=128, carriers=4)
    nf = np.bincount(dp2scaf, minlength=T.size) < T // 2 + 1
    mask[~nf, 1] = 0
    mask[nf, 0] = 0
    mask[nf, 1] = rng.integers(0, 2 ** 64, int(nf.sum()), dtype=np.uint64) & rng.integers(0, 2 ** 64, int(nf.sum()), dtype=np.uint64)
    return (vals, dp2scaf, T, length, mask), nf


@pytest.mark.parametrize("seed", [6001, 6003, 6007])
def test_names_of_scaffolds_that_never_flip_in_child_clusters(ctx, oracle, seed):
    prob, nf = never_flip_problem(seed)
    orecs, res = _run_both(ctx, oracle, prob, 0)
    term = [o.id for o in orecs if not o.split and o.id != 1]
    assert term
    cut = prob[4].copy()
    cut[nf, 1] = 0
    r = scg_test_in_clusters(prob, res.dp2cluster, term)
    rc = scg_test_in_clusters(prob[:4] + (cut,), res.dp2cluster, term)
    assert (r["ok"] != rc["ok"]).any()                   # the second word of those masks changes the verdict of some candidate of a child


def test_no_scg_database_equals_all_zero_masks(ctx):
    """W = 0 (no gene2scg) gives the records of W = 1 with all-zero masks."""
    from abawaca_b200 import pipeline
    vals, dp2scaf, T, length, _ = width_problem(64, 5)
    S = T.size
    a = pipeline.search(ctx, vals, dp2scaf, T, length, np.zeros((S, 0), dtype=np.uint64), params=_params())
    b = pipeline.search(ctx, vals, dp2scaf, T, length, np.zeros((S, 1), dtype=np.uint64), params=_params())
    key = lambda r: (r.id, r.parent, r.ndps, r.nscafs, r.split, r.best.found, r.best.dim, r.best.value, r.best.a, r.best.b, r.child1, r.child2,   # noqa: E731
                     r.child1_ndps, r.child2_ndps, r.child1_nscafs, r.child2_nscafs, r.child1_raw, r.child2_raw, r.total_size, r.scg_unique, r.scg_avg)
    assert [key(r) for r in a.recs] == [key(r) for r in b.recs] and len(a.recs) > 1
    assert a.scaf2cluster.tolist() == b.scaf2cluster.tolist() and a.dp2cluster.tolist() == b.dp2cluster.tolist()
    assert pipeline.cluster_scg(ctx, np.zeros((S, 0), dtype=np.uint64), [np.arange(S)]) == [(0, 0.0)]


def test_search_from_features_with_three_word_masks(ctx):
    """abw_search_create_from_features copies the masks of the scaffolds it keeps to their new index: the same records and bins as abw_search_create on
    the problem the host derives, with 150 SCG names (W = 3) and scaffolds of a single window dropped."""
    from abawaca_b200 import capi, pipeline, synth
    mg = synth.make_metagenome(1500, 3, 4, 51, min_len=1500, mean_extra=3000, n_scg=150)
    fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=0)
    counts = np.diff(fb.seg_first_host().astype(np.int64))
    keep, dp2scaf, T, kept = pipeline.search_problem_from_counts(counts)
    length = np.diff(mg.offsets.astype(np.int64)).astype(np.uint64)
    mask = mg.scg_masks()
    assert mask.shape[1] == 3 and mask[kept, 2].any()
    dropped = np.setdiff1d(np.arange(mg.nscaf), kept)
    assert dropped.size and mask[dropped].any()          # the kept masks move to new indices
    a = pipeline.search(ctx, fb.d_rows, dp2scaf, T, length[kept], mask[kept], params=_params(), layout=capi.LAYOUT_ROWMAJOR, values_on_device=True,
                        nrows=fb.nseg, D=fb.ncols, ld=fb.ncols, row_of_dp=np.nonzero(keep)[0].astype(np.uint64))
    b, kept_b = pipeline.search_features(ctx, fb, length, mask, params=_params())
    fb.close()
    assert kept_b.tolist() == kept.tolist()
    key = lambda r: (r.id, r.parent, r.ndps, r.nscafs, r.split, r.best.found, r.best.dim, r.best.value, r.best.a, r.best.b, r.child1, r.child2,   # noqa: E731
                     r.child1_ndps, r.child2_ndps, r.child1_nscafs, r.child2_nscafs, r.child1_raw, r.child2_raw, r.total_size, r.scg_unique, r.scg_avg)
    assert [key(r) for r in a.recs] == [key(r) for r in b.recs] and len(a.recs) > 1
    assert a.scaf2cluster.tolist() == b.scaf2cluster.tolist() and a.dp2cluster.tolist() == b.dp2cluster.tolist()
    assert mask[kept][a.scaf2cluster != 0, 2].any()      # the bins' tallies see the third word


def _expected_scg(mask, scafs):
    s = np.unique(np.asarray(scafs, dtype=np.int64))
    u = int(_pop(_or(mask[s], mask.shape[1])))
    copies = int(_pop(mask[s]).sum())
    return u, (0.0 if copies == 0 else copies / u)


@pytest.mark.parametrize("G", [1, 63, 64, 65, 128, 129, 200, 448, 511, 512])
def test_cluster_scg_matches_oracle(ctx, oracle, G):
    """abw_cluster_scg on the empty list, one scaffold, random lists with repeated scaffolds and lists of more than 128 x 1024 scaffolds (the kernel's grid
    is capped at 1024 CTAs of 128 threads)."""
    from abawaca_b200 import pipeline
    rng = np.random.default_rng(3000 + G)
    S = 140000
    W = (G + 63) // 64
    r = lambda: rng.integers(0, 2 ** 64, (S, W), dtype=np.uint64)   # noqa: E731
    mask = r() & r() & r()                               # one name in eight
    if G % 64:
        mask[:, W - 1] &= np.uint64((1 << (G % 64)) - 1)
    mask[rng.random(S) < 0.6] = 0
    mask[rng.choice(S, 20, replace=False)] = ~np.uint64(0)
    if G % 64:
        mask[:, W - 1] &= np.uint64((1 << (G % 64)) - 1)
    sub = rng.choice(S, 3000, replace=False)
    lists = [np.zeros(0, dtype=np.uint32), np.array([int(np.flatnonzero(mask.any(axis=1))[0])]), rng.permutation(S),
             sub, np.concatenate((sub, sub[:1000], sub[:10])), rng.integers(0, S, 200000), rng.integers(0, 50, 1000)]
    got = pipeline.cluster_scg(ctx, mask, lists)
    O = oracle.Search(np.zeros((1, 2 * S)), np.repeat(np.arange(S, dtype=np.uint32), 2), np.full(S, 2, dtype=np.uint32), np.zeros(S, dtype=np.uint64), mask)
    for scafs, g in zip(lists, got):
        assert g == O.cluster_scg(scafs) == _expected_scg(mask, scafs)
    assert got[0] == (0, 0.0)
    assert got[2][0] == G                                # every name occurs
    assert got[3] == got[4]                              # a scaffold listed twice counts once


def test_cluster_scg_rejects_an_index_past_the_scaffolds(ctx):
    from abawaca_b200 import capi, pipeline
    mask = np.ones((10, 2), dtype=np.uint64)
    assert pipeline.cluster_scg(ctx, mask, [np.arange(10)]) == [(2, 10.0)]
    with pytest.raises(capi.AbwError, match="^status 2:"):
        pipeline.cluster_scg(ctx, mask, [np.array([3, 10])])


def test_cluster_scg_of_the_terminal_bins_gives_their_records(ctx, oracle):
    """abw_cluster_scg over the assigned scaffolds of every terminal bin of a search gives the scg_unique / scg_avg that k_finalize_terminal wrote
    into the bin's record.  The tallies are taken on a second search of the same masks (pipeline.cluster_scg), not on the handle that ran."""
    from abawaca_b200 import pipeline
    prob = width_problem(200, 1207)
    orecs, res = _run_both(ctx, oracle, prob, 0)
    term = [r for r in res.recs if not r.split]
    assert len(term) > 1
    got = pipeline.cluster_scg(ctx, prob[4], [np.flatnonzero(res.scaf2cluster == r.id) for r in term])
    assert got == [(r.scg_unique, r.scg_avg) for r in term]


def test_command_lines_with_three_word_masks(tmp_path, oracle):
    """abawaca-build and abawaca -c <gene2scg> on a set with 150 SCG names (W = 3): scaf2cluster.txt holds the oracle's bins of the problem read back from
    the build's own files, and the #SCG / Avg columns of summary.txt its terminal records."""
    from abawaca_b200 import hostio, synth
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "abawaca_b200", "host")], check=True)
    mg = synth.make_metagenome(500, 3, 4, 4321, n_scg=150, shuffle_reads=True)
    wd = str(tmp_path)
    paths = synth.write_reference_inputs(mg, wd)
    build = os.path.join(wd, "build")
    r = subprocess.run([os.path.join(BIN, "abawaca-build"), "-f", paths["fasta"], "-o", build, "-s", os.path.join(wd, "sample*.sam"), "-c", paths["sams"][0]],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    out = os.path.join(wd, "out")
    env = dict(os.environ, ABW_SCG_LIST=paths["scg_list"])
    r = subprocess.run([os.path.join(BIN, "abawaca"), "-u", build, "-o", out, "-c", paths["gene2scg"], "-p", "8"], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    prob = hostio.load_search_problem(os.path.join(build, "abawaca.names"), os.path.join(build, "abawaca.lrn"), paths["fasta"], paths["gene2scg"])
    assert prob["scgmask"].shape[1] == 3
    orecs, _, osc = oracle.Search(prob["values"], prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"]).run()
    assert open(os.path.join(out, "scaf2cluster.txt")).read() == "".join(f"{n}\t{c}\n" for n, c in zip(prob["scaf_names"], osc.tolist()))
    rows = [l.split("\t") for l in open(os.path.join(out, "summary.txt")).read().splitlines()[1:]]
    term = [o for o in orecs if not o.split]
    assert len(term) > 1 and max(o.scg_unique for o in term) > 128
    assert [(int(x[0]), x[8], x[9]) for x in rows] == [(o.id, "%g" % o.scg_unique, "%g" % (int(100 * o.scg_avg) / 100.0)) for o in term]
