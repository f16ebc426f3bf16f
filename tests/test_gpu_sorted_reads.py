"""Coordinate-sorted read records (ABW_READS_SORTED, pipeline.sorted_reads, csrc/readcodec.cu).

On the CPU: a restatement of the format's decode rules in numpy round-trips the encoder's output back to compact_reads' records.
On the GPU: samples in the sorted format give the rows and .info coverage of the same reads as compact records and as the oracle, in both value
kinds; malformed samples get the behaviour the header defines; and one batch mixes all three record formats, staged behind h2d tickets, at sample
sizes around the tile boundaries of the coverage and decode kernels."""
import numpy as np
import pytest

SKIP = 0xFFFFFFFF


def ref_decode(n, delta, runs, exc):
    """(scaf, pos0) of every read, scaf = 0xFFFFFFFF for a skipped read, by the rules of include/abawaca_b200.h read for read"""
    run_scaf = np.full(n, SKIP, dtype=np.int64)
    start = np.zeros(n, dtype=bool)
    i = 0
    for s, c in runs.tolist():
        c = min(c, n - i)
        if c > 0:
            run_scaf[i:i + c] = s
            start[i] = True
        i += max(c, 0)
    scaf = np.full(n, SKIP, dtype=np.uint32)
    pos = np.zeros(n, dtype=np.uint32)
    prev = k = 0
    for i in range(n):
        d = int(delta[i])
        keep = run_scaf[i] != SKIP
        if d == 0xFFFF:
            keep = keep and k < len(exc)
            p = int(exc[k]) if k < len(exc) else 0
            k += 1
        else:
            p = ((0 if start[i] else prev) + d) & 0xFFFFFFFF
        prev = pos[i] = p
        if keep:
            scaf[i] = run_scaf[i]
    return scaf, pos


def decode_sample(s):
    return ref_decode(s.n, s.recs, s.runs, s.exc)


def as_full_records(s):
    """the decoded reads of a sorted sample as abw_read records (skipped reads keep scaf 0xFFFFFFFF), for the oracle and the compact format"""
    from abawaca_b200 import capi
    scaf, pos = decode_sample(s)
    r = np.zeros(s.n, dtype=capi.READ_DTYPE)
    r["scaf"], r["pos0"] = scaf, pos
    r["len"] = s.len16 if s.len16 is not None else s.length
    return r


def reads(n, nscaf, seed, max_pos=200000, order="coordinate"):
    from abawaca_b200 import capi
    rng = np.random.default_rng(seed)
    r = np.zeros(n, dtype=capi.READ_DTYPE)
    r["scaf"] = rng.integers(0, nscaf, n)
    r["pos0"] = rng.integers(0, max_pos, n)
    r["len"] = 150
    r["flag_nsnps"] = np.where(rng.random(n) < 0.05, 0x4, 0) | (rng.integers(0, 18, n).astype(np.uint32) << 16)
    return arrange(r, order, rng)


def arrange(r, order, rng):
    if order == "coordinate":                               # samtools sort: by reference, then by position
        return r[np.lexsort((r["pos0"], r["scaf"]))]
    if order == "grouped":                                  # grouped by scaffold, positions in no order
        return r[np.argsort(r["scaf"], kind="stable")]
    if order == "permuted":                                 # sorted, references in @SQ order rather than by name
        perm = rng.permutation(int(r["scaf"].max()) + 1)
        return r[np.lexsort((r["pos0"], perm[r["scaf"]]))]
    return r[rng.permutation(r.size)]


def check_round_trip(r, nscaf):
    from abawaca_b200 import capi, pipeline
    c, s = pipeline.compact_reads(r, nscaf), pipeline.sorted_reads(r, nscaf)
    assert s.fmt == capi.READS_SORTED and s.n == c.n and s.recs.dtype == np.uint16 and s.runs.dtype == capi.READ_RUN_DTYPE and s.exc.dtype == np.uint32
    scaf, pos = decode_sample(s)
    assert np.array_equal(scaf, c.recs["scaf"]) and np.array_equal(pos, c.recs["pos0"])
    assert s.length == c.length and ((s.len16 is None and c.len16 is None) or np.array_equal(s.len16, c.len16))
    assert int(s.runs["count"].sum()) == s.n and (s.runs["count"] > 0).all()
    return s


@pytest.mark.parametrize("order", ["coordinate", "grouped", "permuted", "shuffled"])
def test_round_trip_to_compact_records(order):
    check_round_trip(reads(5000, 40, 1, order=order), 40)


def test_round_trip_edge_cases():
    from abawaca_b200 import capi
    check_round_trip(np.zeros(0, dtype=capi.READ_DTYPE), 5)
    r = reads(300, 5, 2)
    r["flag_nsnps"] = 0x4                                   # every read filtered out
    s = check_round_trip(r, 5)
    assert s.n == 0 and s.runs.size == 0 and s.exc.size == 0
    # deltas of exactly 0xFFFE (literal) and 0xFFFF (escaped), negative deltas, positions up to 2^32 - 1, runs of one read, one scaffold over several runs
    r = np.zeros(10, dtype=capi.READ_DTYPE)
    r["len"] = 100
    r["scaf"] = [0, 0, 0, 0, 1, 0, 0, 2, 2, 2]
    r["pos0"] = [0xFFFE, 2 * 0xFFFE, 2 * 0xFFFE + 0xFFFF, 10, 5, 0xFFFFFFFF, 0xFFFFFFFE, 0xFFFF, 0xFFFF, 0xFFFE]
    s = check_round_trip(r, 3)
    assert s.recs.tolist() == [0xFFFE, 0xFFFE, 0xFFFF, 0xFFFF, 5, 0xFFFF, 0xFFFF, 0xFFFF, 0, 0xFFFF]
    assert s.exc.tolist() == [2 * 0xFFFE + 0xFFFF, 10, 0xFFFFFFFF, 0xFFFFFFFE, 0xFFFF, 0xFFFE]
    assert s.runs.tolist() == [(0, 4), (1, 1), (0, 2), (2, 3)]
    # per-read lengths travel as len16
    r = reads(700, 9, 3, order="grouped")
    r["len"] = np.random.default_rng(3).integers(30, 400, r.size)
    assert check_round_trip(r, 9).len16 is not None


def test_nbytes_is_about_two_bytes_per_read_on_sorted_input():
    from abawaca_b200 import pipeline
    r = reads(200000, 100, 4, max_pos=2_000_000)
    s, c = pipeline.sorted_reads(r, 100), pipeline.compact_reads(r, 100)
    assert s.nbytes == 2 * s.n + 8 * s.runs.size + 4 * s.exc.size
    assert s.runs.size == 100 and s.exc.size <= 100 and s.nbytes < 0.26 * c.nbytes


def test_reference_decoder_on_malformed_samples():
    """the decode rules the GPU tests hold the device to, on hand-made arrays"""
    delta = np.array([5, 1, 0xFFFF, 2, 0xFFFF, 3, 7], dtype=np.uint16)
    exc = np.array([100], dtype=np.uint32)
    runs = np.array([(4, 0), (7, 3), (8, 0), (9, 10)], dtype=[("scaf", "<u4"), ("count", "<u4")])
    scaf, pos = ref_decode(7, delta, runs, exc)
    assert scaf.tolist() == [7, 7, 7, 9, SKIP, 9, 9]        # counts past nreads are ignored; an escape past exc is skipped
    assert pos.tolist() == [5, 6, 100, 2, 0, 3, 10]         # and counts as 0 for the read after it
    scaf, pos = ref_decode(7, delta, runs[:2], exc)
    assert scaf.tolist() == [7, 7, 7] + [SKIP] * 4          # reads past the sum of the counts are skipped


# ---------------------------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def build(ctx, mg, samples, kind, this_sample=1, overlap_h2d=False):
    from abawaca_b200 import capi, pipeline
    fb = pipeline.build_features(ctx, mg.seq, mg.offsets, samples, this_sample=this_sample, kind=kind, skip_A=(kind == capi.FEAT_TRUNC3), overlap_h2d=overlap_h2d)
    try:
        return fb.rows_host(), fb.scaffold_stats_host(np.diff(mg.offsets.astype(np.int64)))["cvg"]
    finally:
        fb.close()


def expect(oracle, mg, full, kind, this_sample=1):
    from abawaca_b200 import capi
    f = oracle.build_features(mg.seq, mg.offsets, full, this_sample=this_sample, want_raw=(kind == capi.FEAT_RAW))
    return (f["raw"] if kind == capi.FEAT_RAW else f["rows"]), f["info_cvg"]


def compact_of(s):
    from abawaca_b200 import capi, pipeline
    scaf, pos = decode_sample(s)
    recs = np.zeros(s.n, dtype=capi.READ8_DTYPE)
    recs["scaf"], recs["pos0"] = scaf, pos
    return pipeline.ReadSample(capi.READS_COMPACT, s.n, recs, s.length, s.len16)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("order", ["coordinate", "grouped", "permuted", "shuffled"])
def test_sorted_samples_match_compact_records_and_the_oracle(ctx, oracle, order, kind):
    from abawaca_b200 import pipeline, synth
    mg = synth.make_metagenome(600, 3, 4, 31, n_run_frac=0.05)
    rng = np.random.default_rng(7)
    rd = [arrange(r.copy(), order, rng) for r in mg.reads]
    rd[1]["len"] = rng.integers(30, 400, rd[1].size)        # trimmed reads: len16, and the -c sample is this one
    samples = [pipeline.sorted_reads(r, mg.nscaf) for r in rd]
    runs = samples[2].runs
    runs["scaf"][runs.size // 2] = mg.nscaf + 3             # a run on a scaffold that is not in the assembly
    want = expect(oracle, mg, [as_full_records(s) for s in samples], kind)
    for name, smp in (("sorted", samples), ("compact", [compact_of(s) for s in samples])):
        rows, cvg = build(ctx, mg, smp, kind)
        assert np.array_equal(rows, want[0]), name
        assert np.array_equal(cvg, want[1]), name


def hand_sample(r, nscaf, cut_runs=None, extra_runs=None, drop_exc=0, zero_runs=False):
    """a sorted sample of reads r, made malformed: the runs cut to the first cut_runs, extra_runs appended, the last drop_exc escapes removed, zero
    count runs put between all others"""
    from abawaca_b200 import capi, pipeline
    s = pipeline.sorted_reads(r, nscaf)
    runs = s.runs
    if zero_runs:
        z = np.zeros(2 * runs.size + 1, dtype=capi.READ_RUN_DTYPE)
        z[1::2] = runs
        z["scaf"][0::2] = np.arange(runs.size + 1) % nscaf
        runs = z
    if cut_runs is not None:
        runs = runs[:cut_runs]
    if extra_runs is not None:
        runs["count"][-1] += 1000
        runs = np.concatenate([runs, np.array(extra_runs, dtype=capi.READ_RUN_DTYPE)])
    exc = s.exc[:s.exc.size - drop_exc]
    return pipeline.ReadSample(capi.READS_SORTED, s.n, s.recs, s.length, s.len16, runs=runs, exc=exc)


@pytest.mark.gpu
def test_malformed_samples_get_the_defined_behaviour(ctx, oracle):
    from abawaca_b200 import capi, synth
    mg = synth.make_metagenome(300, 3, 3, 32)
    rng = np.random.default_rng(9)
    rd = [arrange(r.copy(), "coordinate", rng) for r in mg.reads]
    rd[2] = arrange(arrange(rd[2], "shuffled", rng), "grouped", rng)    # negative deltas: escapes
    cases = {
        "sum of counts below nreads": [hand_sample(rd[0], mg.nscaf, cut_runs=20)] + [hand_sample(r, mg.nscaf) for r in rd[1:3]],
        "sum of counts above nreads": [hand_sample(rd[0], mg.nscaf, extra_runs=[(1, 5000), (2, 7)])] + [hand_sample(r, mg.nscaf) for r in rd[1:3]],
        "escape past exc": [hand_sample(r, mg.nscaf) for r in rd[:2]] + [hand_sample(rd[2], mg.nscaf, drop_exc=25)],
        "zero-count runs": [hand_sample(r, mg.nscaf, zero_runs=True) for r in rd[:3]],
    }
    for name, samples in cases.items():
        for s in samples:
            assert s.runs.dtype == capi.READ_RUN_DTYPE
        kept = [decode_sample(s)[0] for s in samples]
        assert name != "sum of counts below nreads" or (kept[0] == SKIP).sum() > 0
        assert name != "escape past exc" or (kept[2] == SKIP).sum() == 25
        want = expect(oracle, mg, [as_full_records(s) for s in samples], capi.FEAT_TRUNC3)
        rows, cvg = build(ctx, mg, samples, capi.FEAT_TRUNC3)
        assert np.array_equal(rows, want[0]), name
        assert np.array_equal(cvg, want[1]), name


@pytest.mark.gpu
def test_host_checked_cases_return_an_argument_error(ctx):
    from abawaca_b200 import capi, pipeline, synth
    mg = synth.make_metagenome(50, 1, 2, 33)
    s = pipeline.sorted_reads(arrange(mg.reads[0].copy(), "coordinate", None), mg.nscaf)
    d = ctx.alloc(1 << 20)
    bad = {
        "null runs": pipeline.ReadSample(capi.READS_SORTED, s.n, d_recs=d, length=150, d_runs=None, nruns=3, d_exc=d, nexc=1),
        "null exc": pipeline.ReadSample(capi.READS_SORTED, s.n, d_recs=d, length=150, d_runs=d, nruns=1, d_exc=None, nexc=1),
        "more escapes than reads": pipeline.ReadSample(capi.READS_SORTED, 10, d_recs=d, length=150, d_runs=d, nruns=1, d_exc=d, nexc=11),
        "2^32 runs": pipeline.ReadSample(capi.READS_SORTED, 10, d_recs=d, length=150, d_runs=d, nruns=1 << 32, d_exc=d, nexc=0),
    }
    for name, smp in bad.items():
        with pytest.raises(capi.AbwError, match="status 2:"):
            pipeline.build_features(ctx, mg.seq, mg.offsets, [smp], this_sample=0)
    ctx.free(d)


@pytest.mark.gpu
def test_one_batch_of_all_formats_behind_tickets_across_tile_boundaries(ctx, oracle):
    """FULL, COMPACT and SORTED samples in one abw_coverage_batch call, staged with h2d tickets; sample sizes on both sides of the 1024-read tile of
    the coverage kernels and of the 2048-read tile of the decode, and one run of one scaffold over many tiles"""
    from abawaca_b200 import capi, pipeline, synth
    mg = synth.make_metagenome(200, 1, 3, 34)
    seglen = np.diff(mg.offsets.astype(np.int64))
    big = int(np.argmax(seglen))
    raw = []
    for j, n in enumerate((1023, 1024, 1025, 2047, 2048, 2049)):
        r = reads(n, mg.nscaf, 40 + j, max_pos=int(seglen.min()) + 500, order="coordinate" if j % 2 else "permuted")
        r["flag_nsnps"] = 0                                 # every read passes the filter: the sizes are those of the sorted samples
        raw.append(r)
    long = reads(40000, 1, 50, max_pos=int(seglen[big]))
    long["scaf"], long["flag_nsnps"] = big, 0
    long["pos0"][20000:] += 70000                           # one run over about 20 decode tiles, with a gap of more than 0xFFFF in it
    raw.append(long)
    raw += [raw[1].copy(), raw[4].copy()]
    for kind in (capi.FEAT_TRUNC3, capi.FEAT_RAW):
        samples = [pipeline.sorted_reads(r, mg.nscaf) for r in raw[:7]] + [raw[7], pipeline.compact_reads(raw[8], mg.nscaf)]
        assert [s.n for s in samples[:6]] == [1023, 1024, 1025, 2047, 2048, 2049]
        assert samples[6].runs.size == 1 and samples[6].exc.size >= 1 and samples[8].fmt == capi.READS_COMPACT
        want = expect(oracle, mg, raw, kind, this_sample=2)
        rows, cvg = build(ctx, mg, samples, kind, this_sample=2, overlap_h2d=True)
        assert np.array_equal(rows, want[0]), kind
        assert np.array_equal(cvg, want[1]), kind
