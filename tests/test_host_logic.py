"""Host-side logic of the drop-in path that needs no GPU: the read filter a host-side SAM parser may apply before it hands 8-byte records to
abw_coverage_batch (SURVEY.md section 8b(4); abawaca-build.cpp:546-551), the search problem derived from the window counts (ScafDpData.cpp:92-93), the
round-robin dimension shards, and the launch-list summariser used for profiles/."""
import gzip
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_host_side_read_filter_keeps_exactly_the_reads_the_reference_counts(oracle):
    """compact_reads drops unmapped reads, secondary alignments, reads with more than max_snps mismatches and reads on unknown scaffolds: the oracle
    (pinned on the reference) gives the same feature rows and the same per-scaffold read bases for the kept reads as for all reads."""
    from abawaca_b200 import capi, pipeline, synth
    mg = synth.make_metagenome(300, 2, 3, 17, shuffle_reads=True, bad_read_frac=0.2)
    reads = [r.copy() for r in mg.reads]
    reads[1]["scaf"][::53] = 0xFFFFFFFF                       # reference name not in the assembly
    reads[1]["len"] = np.random.default_rng(3).integers(30, 300, reads[1].size)
    full = oracle.build_features(mg.seq, mg.offsets, reads, this_sample=1)
    kept = []
    for r in reads:
        c = pipeline.compact_reads(r, mg.nscaf)
        back = np.zeros(c.n, dtype=capi.READ_DTYPE)
        back["scaf"], back["pos0"] = c.recs["scaf"], c.recs["pos0"]
        back["len"] = c.len16 if c.len16 is not None else c.length
        kept.append(back)                                       # flag 0, no mismatches: every kept read counts
        flag, nsnps = r["flag_nsnps"] & 0xFFFF, r["flag_nsnps"] >> 16
        assert c.n == int((((flag & 0x104) == 0) & (nsnps <= 15) & (r["scaf"] < mg.nscaf)).sum()) and 0 < c.n < r.size
    filtered = oracle.build_features(mg.seq, mg.offsets, kept, this_sample=1)
    assert np.array_equal(full["rows"], filtered["rows"]) and np.array_equal(full["info_cvg"], filtered["info_cvg"])
    # one length for the sample -> no per-read lengths travel; mixed lengths -> uint16 per read; too long -> the full format is demanded
    assert pipeline.compact_reads(reads[0], mg.nscaf).len16 is None and pipeline.compact_reads(reads[1], mg.nscaf).len16.dtype == np.uint16
    big = reads[0][:4].copy()
    big["flag_nsnps"] = 0
    big["len"] = [100, 70000, 100, 100]
    try:
        pipeline.compact_reads(big, mg.nscaf)
        raise AssertionError("a 70 kb read was accepted into the 16-bit length format")
    except ValueError:
        pass


def test_search_problem_drops_single_window_scaffolds():
    from abawaca_b200 import pipeline
    counts = np.array([3, 1, 2, 0, 5, 1])
    keep, dp2scaf, T, kept = pipeline.search_problem_from_counts(counts)
    assert kept.tolist() == [0, 2, 4] and T.tolist() == [3, 2, 5]
    assert keep.tolist() == [True] * 3 + [False] + [True] * 2 + [True] * 5 + [False]
    assert dp2scaf.tolist() == [0] * 3 + [1] * 2 + [2] * 5


def test_round_robin_shards_cover_every_dimension_once():
    for D in (1, 7, 180, 189, 229):
        for world in (1, 2, 3, 4, 8):
            owned = [list(range(r, D, world)) for r in range(world)]
            assert sorted(d for o in owned for d in o) == list(range(D))
            assert [len(o) for o in owned] == [(D - r + world - 1) // world if D > r else 0 for r in range(world)]     # cnt(q) of csrc/peer.cu
            assert max(len(o) for o in owned) - min(len(o) for o in owned) <= 1


def test_launch_shares_of_the_committed_launch_list(tmp_path):
    src = os.path.join(ROOT, "profiles", "r02_launches_ncu_gputime.csv.gz")
    csv = tmp_path / "launches.csv"
    csv.write_bytes(gzip.open(src).read())
    out = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "launch_shares.py"), str(csv), "1"], capture_output=True, text=True, check=True).stdout
    assert "launches," in out.splitlines()[0] and "| k_partition2 | 13 |" in out and "| k_sweep_ss | 13 |" in out
    shares = [float(l.split("|")[4]) for l in out.splitlines() if l.startswith("| k_")]
    assert 0.95 < sum(shares) < 1.02                        # shares are printed with three decimals


def test_run_ahead_rule_of_the_sharded_search_enqueues_the_same_levels_on_every_rank():
    """The rule of abw_search_run_sharded (csrc/search.cu): level l is enqueued iff the search had not ended by level l - lead, decided only after
    level l - lead has been reported.  Restated here and driven with ranks that observe the device's progress words (ticks, done_at) at arbitrary
    moments: whatever the timing, every rank enqueues exactly (index of the last level) + lead levels, so the collective counts match."""
    rng = np.random.default_rng(7)

    def levels_enqueued(last_level, lead, observe):
        # device: level i completes at time i + 1 (ticks = i + 1); done_at = last_level + 1 from then on
        lvl = 0
        while True:
            lvl += 1                                            # level lvl - 1 has just been enqueued
            if lvl < lead:
                continue
            need = lvl - lead + 1
            t = max(observe(), need)                            # the host polls until ticks >= need; it may look later than that
            done_at = last_level + 1 if t >= last_level + 1 else 0
            if done_at != 0 and done_at <= need:
                return lvl
    for lead in (1, 2, 3, 5, 8):
        for last_level in (0, 1, 2, 7, 12, 30):
            counts = {levels_enqueued(last_level, lead, lambda: int(rng.integers(0, 50))) for _ in range(200)}
            assert counts == {last_level + lead}, (lead, last_level, counts)


def test_random_problem_defaults_draw_what_they_always_drew():
    """_random_problem's SCG options (names, carriers, contamination, dense scaffolds) leave the problems of every seed the existing tests use as they
    were: the same arrays, and the generator left at the same state (digests taken before the options existed)."""
    import hashlib
    from golden_util import _random_problem

    def digest(rng, *args, **kw):
        h = hashlib.sha256()
        for a in _random_problem(rng, *args, **kw):
            h.update(np.ascontiguousarray(a).tobytes())
        h.update(np.int64(rng.integers(0, 2 ** 62)).tobytes())
        return h.hexdigest()[:16]

    expect = {1: "d2f8f94c78740395", 2: "f83ea99e16e7d2f1", 3: "497d2895c7b93285", 4: "919038c83ef0b061", 5: "c64fa1df96cbde5f", 6: "e018a0caaa61931f",
              7: "74ea0ebd7b5440fe"}
    for seed, partial, scg in [(1, False, True), (2, True, True), (3, False, False), (4, True, True), (5, False, True), (6, False, True), (7, True, False)]:
        rng = np.random.default_rng(seed)                   # test_gpu_parity.py: test_search_matches_oracle_on_random_problems
        S, D = int(rng.integers(150, 500)), int(rng.integers(3, 12))
        assert digest(rng, S, D, partial=partial, scg=scg, nclus=int(rng.integers(2, 5))) == expect[seed]
    rng = np.random.default_rng(11)                         # test_gpu_parity.py: test_small_and_degenerate_searches
    assert digest(rng, 20, 2) + digest(rng, 300, 3) == "d84b42ec405c059abe5490e3b22594f6"
    for seed, partial, h in [(21, False, "e0fef066441cbbed"), (22, True, "4945e952166bde9b"), (23, False, "7b97bc26196dd0a7")]:   # test_gpu_lookback_windows.py
        assert digest(np.random.default_rng(seed), 80000, 3, partial=partial) == h
    # test_gpu_sort_chunks.py's seeds (there with 30000 scaffolds in 400 dimensions), smaller
    assert digest(np.random.default_rng(31), 3000, 40, ties=True) == "fe7bc86683dce66f"
    assert digest(np.random.default_rng(32), 3000, 40, ties=False) == "0740f534a56494d7"


def test_oracle_cluster_scg_counts_a_repeated_scaffold_once(oracle):
    """abwo_cluster_scg takes its scaffold list as a set, like ClusterQuality::scg's std::set: repeats change nothing."""
    mask = np.array([[0b1011, 0], [0b0001, 1 << 63], [0, 0]], dtype=np.uint64)
    O = oracle.Search(np.zeros((1, 6)), np.repeat(np.arange(3, dtype=np.uint32), 2), np.full(3, 2, dtype=np.uint32), np.zeros(3, dtype=np.uint64), mask)
    assert O.cluster_scg([0, 1]) == (4, 5 / 4)
    assert O.cluster_scg([1, 0, 1, 1, 2, 0]) == (4, 5 / 4)
    assert O.cluster_scg([]) == (0, 0.0) and O.cluster_scg([2, 2]) == (0, 0.0)
