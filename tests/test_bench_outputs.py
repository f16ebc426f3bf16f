"""bench.py --dump-outputs: what the timed path computed in its last step, written as float64 .npy files of at most 64 MB in all, on inputs that are the
same from run to run -- so that two builds of the project can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_writes_float64_and_samples_large_arrays_with_fixed_rows(tmp_path):
    import bench
    big = np.random.default_rng(1).integers(0, 1 << 40, (300_000, 40), dtype=np.uint64)     # 96 MB as float64
    small = np.arange(10, dtype=np.uint32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["big.npy", "big_rows.npy", "small.npy"] and sorted(os.listdir(tmp_path / "b")) == files
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    got = {f: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype == np.float64 for a in got.values())
    rows = got["big_rows.npy"].astype(np.int64)
    assert rows.size > 10_000 and np.all(np.diff(rows) > 0) and np.array_equal(got["big.npy"], big[rows].astype(np.float64))
    assert all(np.array_equal(got[f], np.load(tmp_path / "b" / f)) for f in files)
    assert np.array_equal(got["small.npy"], small.astype(np.float64))
    # a later dump that needs no sample leaves no stale row numbers behind
    bench.dump_outputs(str(tmp_path / "a"), {"big": big[:10], "small": small})
    assert sorted(os.listdir(tmp_path / "a")) == ["big.npy", "small.npy"]


def test_cluster_table_holds_every_record_field():
    import bench
    from abawaca_b200 import capi
    recs = (capi.ClusterRec * 2)()
    recs[0].id, recs[0].ndps, recs[0].split, recs[0].best.dim, recs[0].best.value = 1, 123456789012, 1, 181, 4.935
    recs[1].id, recs[1].parent, recs[1].scg_avg, recs[1].cvg_sd = 2, 1, 1.25, -1.0
    t = bench.cluster_table([recs[0], recs[1]])
    col = {f: i for i, f in enumerate(bench.CLUSTER_FIELDS)}
    assert t.shape == (2, len(capi.ClusterRec._fields_) + len(capi.Best._fields_) - 1) and t.dtype == np.float64
    assert (t[0, col["id"]], t[0, col["ndps"]], t[0, col["split"]], t[0, col["best.dim"]], t[0, col["best.value"]]) == (1, 123456789012, 1, 181, 4.935)
    assert (t[1, col["parent"]], t[1, col["scg_avg"]], t[1, col["cvg_sd"]]) == (1, 1.25, -1.0)
    assert bench.cluster_table([]).shape == (0, len(bench.CLUSTER_FIELDS))


@pytest.mark.gpu
def test_bench_dumps_the_outputs_of_its_last_timed_step(tmp_path, oracle):
    """A small workload through bench.py: the line reports the requested number of timed steps, and the dumped window table, feature rows and bins
    are those of the oracle on the same seeded inputs."""
    import bench
    from abawaca_b200 import pipeline, synth
    args = ["--scaffolds", "1500", "--samples", "3", "--genomes", "4"]
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1", "--no-cpu-baseline",
                        "--dump-outputs", str(out)] + args, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3 and len(line["step_ms"]["resident"]) == 3 and len(line["step_ms"]["e2e"]) == 3
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype == np.float64 for a in got.values()) and sum(a.nbytes for a in got.values()) <= 64_000_000

    mg = synth.make_metagenome(**dict(synth.CONFIGS["cfg2"], n_scaffolds=1500, n_samples=3, n_genomes=4), q6_reads=True)
    f = oracle.build_features(mg.seq, mg.offsets, mg.reads, this_sample=0)
    windows = np.stack([f[k].astype(np.float64) for k in ("seg_scaf", "seg_start", "seg_end", "seg_nonN")], axis=1)
    for name, ref in (("windows", windows), ("features", f["rows"])):
        rows = got[name + "_rows"].astype(np.int64) if name + "_rows" in got else np.arange(ref.shape[0])
        assert np.array_equal(got[name], ref[rows]), name
    keep, dp2scaf, T, kept = pipeline.search_problem_from_features(f["seg_scaf"], mg.nscaf)
    length = np.diff(mg.offsets.astype(np.int64)).astype(np.uint64)[kept]
    orecs, odp, osc = oracle.Search(np.ascontiguousarray(f["rows"][keep].T), dp2scaf, T, length, mg.scg_masks()[kept]).run()
    assert got["kept_scaffolds"].tolist() == np.asarray(kept).tolist()
    assert got["scaf2cluster"].tolist() == osc.tolist() and got["dp2cluster"].tolist() == odp.tolist()
    c = {name: got["clusters"][:, i] for i, name in enumerate(bench.CLUSTER_FIELDS)}
    assert [(int(i), int(s), int(d) if s else 0) for i, s, d in zip(c["id"], c["split"], c["best.dim"])] == \
        [(o.id, o.split, o.best.dim if o.split else 0) for o in orecs] and len(orecs) > 1
