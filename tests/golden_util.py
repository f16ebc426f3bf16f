"""Helpers shared by the CPU (oracle) and GPU parity tests: load the committed golden fixtures."""
import gzip
import hashlib
import io
import json
import os
import functools

import numpy as np

from abawaca_b200 import synth, hostio

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@functools.lru_cache(maxsize=None)
def load_set(name):
    """Regenerate the synthetic inputs of a golden set from its seed and load the reference outputs."""
    meta = json.load(open(os.path.join(GOLDEN, f"{name}.json")))
    mg = synth.make_metagenome(**meta["args"])
    dg = meta["digests"]
    assert _sha(mg.seq) == dg["seq"], "synthetic generator drifted from the committed fixture (sequence)"
    assert [_sha(r) for r in mg.reads] == dg["reads"], "synthetic generator drifted from the committed fixture (reads)"
    assert hashlib.sha256("\n".join(mg.names).encode()).hexdigest() == dg["names"]
    lrn_text = gzip.open(os.path.join(GOLDEN, f"{name}.lrn.gz"), "rt").read()
    names_text = gzip.open(os.path.join(GOLDEN, f"{name}.names.gz"), "rt").read()
    info_text = gzip.open(os.path.join(GOLDEN, f"{name}.info.gz"), "rt").read()
    rawcov = np.load(os.path.join(GOLDEN, f"{name}.rawcov.npy"))
    return dict(meta=meta, mg=mg, lrn_text=lrn_text, names_text=names_text, info_text=info_text, rawcov=rawcov)


def parse_lrn_text(text):
    lines = text.splitlines()
    ndps = int(lines[0].split()[1])
    heads = lines[3].split("\t")[1:]
    vals = np.array([[float(x) for x in l.split("\t")[1:]] for l in lines[4:4 + ndps]], dtype=np.float64)
    return heads, vals


def parse_ref_search(text):
    """Parse a ref_search dump (oracle/ref_search_harness.cpp) into cluster records and scaffold bins."""
    clusters, bins = [], []
    for line in text.splitlines():
        f = line.split("\t")
        if f[0] == "C":
            c = dict(id=int(f[1]), ndps=int(f[2]), nscafs=int(f[3]), split=int(f[4]), dim=int(f[5]), value=float(f[6]), a=float(f[7]), b=float(f[8]))
            if c["split"]:
                c.update(child1=int(f[9]), child1_ndps=int(f[10]), child1_nscafs=int(f[11]), child1_raw=int(f[12]),
                         child2=int(f[13]), child2_ndps=int(f[14]), child2_nscafs=int(f[15]), child2_raw=int(f[16]))
            else:
                c.update(total_size=int(f[10]), scg_unique=float(f[11]), scg_avg=float(f[12]))
            clusters.append(c)
        elif f[0] == "S":
            bins.append((f[1], int(f[2])))
    return clusters, bins


@functools.lru_cache(maxsize=None)
def search_problem(name):
    """Flat search arrays built from the golden .names/.lrn exactly as ScafDpData/ClusterData/SCGdb would."""
    g = load_set(name)
    mg = g["mg"]
    import tempfile
    with tempfile.TemporaryDirectory() as wd:
        p_names = os.path.join(wd, "n"); open(p_names, "w").write(g["names_text"])
        p_lrn = os.path.join(wd, "l"); open(p_lrn, "w").write(g["lrn_text"])
        p_fa = os.path.join(wd, "f")
        with open(p_fa, "w") as f:
            for i, nm in enumerate(mg.names):
                f.write(f">{nm}\n{mg.scaffold(i).tobytes().decode()}\n")
        p_scg = os.path.join(wd, "g")
        with open(p_scg, "w") as f:
            for gene, scg in mg.gene2scg:
                f.write(f"{gene}\t{scg}\n")
        return hostio.load_search_problem(p_names, p_lrn, p_fa, p_scg)


def compare_cluster_records(ref_clusters, recs, strategy, check_illegal_best=True):
    """recs: objects with the abwo_cluster_rec / abw_cluster_rec fields. Returns a list of mismatch strings."""
    bad = []
    if len(ref_clusters) != len(recs):
        bad.append(f"number of evaluated clusters {len(recs)} != reference {len(ref_clusters)}")
    for r, o in zip(ref_clusters, recs):
        odim = o.best.dim if o.best.found else -1
        ok = r["id"] == o.id and r["ndps"] == o.ndps and r["nscafs"] == o.nscafs and r["split"] == o.split
        if r["split"] or check_illegal_best:
            ok = ok and r["dim"] == odim and r["value"] == o.best.value and r["a"] == o.best.a and (strategy == 1 or r["b"] == o.best.b)
        if r["split"]:
            ok = ok and (r["child1"], r["child1_ndps"], r["child1_nscafs"], r["child1_raw"]) == (o.child1, o.child1_ndps, o.child1_nscafs, o.child1_raw)
            ok = ok and (r["child2"], r["child2_ndps"], r["child2_nscafs"], r["child2_raw"]) == (o.child2, o.child2_ndps, o.child2_nscafs, o.child2_raw)
        else:
            ok = ok and r["total_size"] == o.total_size and r["scg_unique"] == o.scg_unique and r["scg_avg"] == o.scg_avg
        if not ok:
            bad.append(f"cluster {r['id']}: reference {r} != ({o.id},{o.ndps},{o.nscafs},{o.split},{odim},{o.best.value},{o.best.a},{o.best.b})")
    return bad


def coverage_edge_workload(seed=7, nscaf=160, nsamples=3, depth=40, cover_all_n=False):
    """Scaffolds whose windows have round lengths (2000, 2500, 2048, 3125 ...), so that 1000 * (sum of overlaps) / length is an integer for a
    large share of the windows -- the case in which the order of the reads decides the third decimal (quirk Q5) -- plus an all-N scaffold (one
    window per character, a read over more than 255 windows), N runs, reads hanging over window and scaffold ends, shuffled read order.
    cover_all_n: see below (needed when the unmodified reference is to print the rows).
    Returns (seq, offsets, reads) in the layout of abw_pack_sequences / abw_coverage."""
    read_dtype = np.dtype([("scaf", "<u4"), ("pos0", "<u4"), ("len", "<u4"), ("flag_nsnps", "<u4")])   # abw_read
    rng = np.random.default_rng(seed)
    lens = [int(rng.choice([4000, 5000, 4096, 6000, 6250, 8000, 7500, 10000, 12000, 4001, 9999])) for _ in range(nscaf)]
    seqs = []
    for i, n in enumerate(lens):
        s = rng.integers(0, 4, n).astype(np.uint8)
        a = np.frombuffer(b"ACGT", dtype=np.uint8)[s].copy()
        if i % 17 == 3:                                     # a run of N inside the scaffold
            p = int(rng.integers(100, n - 400)); a[p:p + int(rng.integers(10, 300))] = ord("N")
        seqs.append(a)
    seqs.append(np.full(400, ord("N"), dtype=np.uint8))     # all-N scaffold: 400 windows of one character
    lens.append(400)
    offsets = np.zeros(len(lens) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(lens)
    seq = np.concatenate(seqs)
    reads = []
    for _ in range(nsamples):
        recs = []
        for i, n in enumerate(lens):
            k = int(depth * n / 100 * rng.uniform(0.3, 1.5))
            rl = rng.choice([100, 100, 100, 100, 50, 150, 75, 300 if n == 400 else 100], k).astype(np.uint32)
            pos = rng.integers(0, n, k).astype(np.uint32)
            r = np.zeros(k, dtype=read_dtype)
            r["scaf"], r["pos0"], r["len"] = i, pos, rl
            r["flag_nsnps"] = np.where(rng.random(k) < 0.02, 4, 0) | (rng.integers(0, 4, k).astype(np.uint32) << 16)
            recs.append(r)
        r = np.concatenate(recs)
        rng.shuffle(r)
        reads.append(r)
    if cover_all_n:
        # every window needs a read in the LAST sample or the reference reads past a vector when it prints the row (quirk Q6): two reads that
        # cover all 400 one-character windows of the all-N scaffold
        extra = np.zeros(2, dtype=read_dtype)
        extra["scaf"], extra["pos0"], extra["len"] = len(lens) - 1, [0, 250], 300
        reads[-1] = np.concatenate([reads[-1], extra])
    return seq, offsets, reads


def _pack_names(has):
    """bool [S][G] (scaffold carries SCG name g) -> uint64 [S][ceil(G/64)] masks, name g in bit g % 64 of word g // 64"""
    S, G = has.shape
    W = (G + 63) // 64
    bits = np.zeros((S, 64 * W), dtype=bool)
    bits[:, :G] = has
    return np.packbits(bits, axis=1, bitorder="little").view("<u8").astype(np.uint64).reshape(S, W)


def _random_problem(rng, S, D, partial=False, ties=True, scg=True, nclus=3, G=70, carriers=None, contamination=0.0, dense=0, len_hi=400000):
    """Seeded random split-search problem of S scaffolds (T in 2..8 datapoints each, n = T unless partial) in D dimensions around nclus centres.

    SCG names 0..G-1 (masks of ceil(G/64) words): each name lands, with probability 0.8 per centre, on one scaffold of that centre.
    carriers: only that many scaffolds (drawn at random) carry names, and each of them carries at least one;
    contamination: every carrier also carries every name with this probability, whatever its centre;
    dense: that many carriers carry between 24 and 300 names (at most G) drawn at random.
    With these three at their defaults the draws are the ones the function always made."""
    T = rng.integers(2, 9, S).astype(np.uint32)
    n = T.copy()
    if partial:
        drop = rng.random(S) < 0.3
        n = np.where(drop, np.maximum(1, T - rng.integers(1, 4, S)), T).astype(np.uint32)
    dp2scaf = np.repeat(np.arange(S, dtype=np.uint32), n)
    N = dp2scaf.size
    grp = rng.integers(0, nclus, S)
    centers = rng.normal(0, 1.0, (nclus, D))
    vals = centers[grp[dp2scaf]].T + rng.normal(0, 0.35, (D, N))
    if ties:
        vals = np.round(vals, 1)             # heavy ties, negative values and +-0.0
        vals[vals == 0] = np.where(rng.random((vals == 0).sum()) < 0.5, 0.0, -0.0)
    length = rng.integers(2000, len_hi, S).astype(np.uint64)
    W = (G + 63) // 64
    mask = np.zeros((S, W), dtype=np.uint64)
    if scg:
        is_carrier = np.ones(S, dtype=bool)
        if carriers is not None:
            is_carrier[:] = False
            is_carrier[rng.choice(S, carriers, replace=False)] = True
        for g in range(G):
            for c in range(nclus):
                if rng.random() < 0.8:
                    cand = np.nonzero((grp == c) & is_carrier)[0]
                    if cand.size:
                        s = cand[rng.integers(0, cand.size)]
                        mask[s, g // 64] |= np.uint64(1) << np.uint64(g % 64)
        car = np.flatnonzero(is_carrier)
        extra = np.zeros((car.size, G), dtype=bool)
        if contamination > 0:
            extra |= rng.random((car.size, G)) < contamination
        for i in rng.choice(car.size, dense, replace=False) if dense else ():
            extra[i, rng.choice(G, int(rng.integers(min(24, G), min(300, G) + 1)), replace=False)] = True
        if carriers is not None:
            bare = ~mask[car].any(axis=1) & ~extra.any(axis=1)
            extra[bare, rng.integers(0, G, int(bare.sum()))] = True
        mask[car] |= _pack_names(extra)
    return np.ascontiguousarray(vals), dp2scaf, T, length, mask


def assert_search_matches_oracle(orecs, odp, osc, res):
    """A device search (pipeline.search) gives every cluster record, dp2cluster and scaf2cluster of the oracle's run (abwo.Search.run)."""
    assert len(orecs) == len(res.recs)
    for o, r in zip(orecs, res.recs):
        assert (o.id, o.parent, o.ndps, o.nscafs, o.split) == (r.id, r.parent, r.ndps, r.nscafs, r.split)
        assert (o.best.found, o.best.dim, o.best.value, o.best.a, o.best.legal) == (r.best.found, r.best.dim, r.best.value, r.best.a, r.best.legal), (o.id, o.best.b, r.best.b)
        assert o.best.b == r.best.b
        assert (o.child1, o.child2, o.child1_ndps, o.child2_ndps, o.child1_nscafs, o.child2_nscafs, o.child1_raw, o.child2_raw) == \
               (r.child1, r.child2, r.child1_ndps, r.child2_ndps, r.child1_nscafs, r.child2_nscafs, r.child1_raw, r.child2_raw)
        assert (o.total_size, o.scg_unique, o.scg_avg) == (r.total_size, r.scg_unique, r.scg_avg)
    assert odp.tolist() == res.dp2cluster.tolist()
    assert osc.tolist() == res.scaf2cluster.tolist()
