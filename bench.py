#!/usr/bin/env python
"""bench.py -- scaffolds/s binned (feature build + split search) on N B200s, with roofline and CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--scaffolds S --samples M --genomes G] [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic metagenome: pack -> windows -> k-mer signature ->
per-sample coverage -> split search down to the final bins.  At N=1 the workload is BASELINE.json configs[1]
(50k scaffolds, 10 samples).  At N>1 the assembly has N x 50k scaffolds of ONE community (weak scaling): scaffolds are
sharded across the ranks for the feature build (no exchange), one NCCL all-to-all hands every rank its block of columns of all rows, and the split
search is sharded by dimension (abw_search_run_sharded: all-gather of per-cluster best records + one sum per level, enqueued on the device stream).

  value : whole-job scaffolds/s with the inputs (ASCII assembly, read records) already resident in HBM
  e2e   : the same through the C ABI with HOST buffers: H2D of assembly + compact read records and D2H of the .lrn matrix (integer thousandths),
          the window table and the bins inside the timed region
  roofline : algorithmic bytes of SURVEY.md section 8(d) over CUDA-event kernel time (one extra profiled step), for every kernel family the survey
          gives bytes for; the primary figure is the dominant family -- the split search, ALL its kernels (abw_search_create + abw_search_run)
  cpu_baseline : the UNMODIFIED reference binaries (oracle/_ref, -O2 build) on a bounded sample of the same workload, on this box's cores:
          full command lines (text in, text out), compute only (Bio::VectorReader-fed feature stage + work list, no text parsing), and the
          drop-in command lines of this repo on the same text files (e2e_cli)

`--impl reference` times only that reference arm (rank 0; other ranks exit 0).

`--dump-outputs DIR` writes, after the timed steps, what the last timed step of the resident path handed its caller (rank 0's) as DIR/<name>.npy in
float64, so that two builds can be compared output for output on the same seeded inputs (see dump_outputs()).
"""
import argparse
import gc
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from abawaca_b200 import synth  # noqa: E402

FALLBACK_HBM_GBS = 6650.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks and throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def workload_args(args):
    w = dict(synth.CONFIGS["cfg2"])
    if args.scaffolds:
        w["n_scaffolds"] = args.scaffolds
    if args.samples:
        w["n_samples"] = args.samples
    if args.genomes:
        w["n_genomes"] = args.genomes
    if getattr(args, "coverage_scale", 1.0) != 1.0:    # thinned reads for the large shapes (the host generator is the limit, not the GPU)
        w["cov_lo"], w["cov_hi"] = 0.5 * args.coverage_scale, 16.0 * args.coverage_scale
    return w


def workload_name(w):
    base = "BASELINE.json configs[1]: 50k scaffolds, 10 samples, feature build + split search" if (w["n_scaffolds"], w["n_samples"]) == (50000, 10) \
        and "cov_lo" not in w else "variant of configs[1]"
    thin = f", read depth x {w['cov_hi'] / 16.0:g}" if "cov_lo" in w else ""
    return f"{base} ({w['n_scaffolds']} scaffolds, {w['n_samples']} samples, {w['n_genomes']} synthetic genomes, seed {w['seed']}{thin})"


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference binaries on a bounded sample
# ------------------------------------------------------------------------------------------------------------------
def reference_sample(mg, per_genome=400, genomes=2):
    """The first `per_genome` scaffolds (name order) of each of the first `genomes` genomes, with their reads."""
    sel = []
    for g in sorted(set(mg.genome.tolist()))[:genomes]:
        sel.extend(np.nonzero(mg.genome == g)[0][:per_genome].tolist())
    sel = np.array(sorted(sel))
    remap = np.full(mg.nscaf, -1, dtype=np.int64)
    remap[sel] = np.arange(sel.size)
    lengths = np.diff(mg.offsets.astype(np.int64))[sel]
    offsets = np.zeros(sel.size + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(lengths)
    seq = np.concatenate([mg.scaffold(int(i)) for i in sel])
    reads = []
    for r in mg.reads:
        keep = remap[r["scaf"]] >= 0
        rr = r[keep].copy()
        rr["scaf"] = remap[rr["scaf"]].astype(np.uint32)
        reads.append(rr)
    names = [mg.names[int(i)] for i in sel]
    nameset = set(names)
    g2s = [(g, s) for g, s in mg.gene2scg if g[:g.rfind("_")] in nameset]
    return synth.Metagenome(names, mg.genome[sel], offsets, seq, reads, mg.scg_names, g2s, mg.read_len, mg.seed)


def run_command_lines(bindir, paths, workdir, ncpu, tag):
    """abawaca-build + abawaca of `bindir` on the text files of `paths`; returns (build seconds, bin seconds, bins, build directory)."""
    build = os.path.join(workdir, "build_" + tag)
    out = os.path.join(workdir, "out_" + tag)
    shutil.rmtree(build, ignore_errors=True)
    shutil.rmtree(out, ignore_errors=True)
    os.makedirs(build)
    t0 = time.perf_counter()
    subprocess.run([os.path.join(bindir, "abawaca-build"), "-f", paths["fasta"], "-o", build, "-s", os.path.join(workdir, "sample*.sam"), "-c", paths["sams"][0]],
                   check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    t1 = time.perf_counter()
    env = dict(os.environ, ABW_SCG_LIST=paths["scg_list"])
    subprocess.run([os.path.join(bindir, "abawaca"), "-u", build, "-o", out, "-c", paths["gene2scg"], "-p", str(ncpu)], check=True, env=env,
                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    t2 = time.perf_counter()
    bins = [int(l.split("\t")[1]) for l in open(os.path.join(out, "scaf2cluster.txt"))]
    return t1 - t0, t2 - t1, bins, build


def reference_compute_only(paths, build_dir, ncpu, workdir):
    """The reference's compute without text parsing: feature stage fed from memory (Bio::VectorReader, oracle/ref_compute_harness.cpp) and the
    work list alone (oracle/ref_search_harness.cpp prints its wall clock); both run the unmodified reference classes."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if not (os.path.exists(os.path.join(ref, "ref_compute")) and os.path.exists(os.path.join(ref, "ref_search"))):
        return None
    r = subprocess.run([os.path.join(ref, "ref_compute"), paths["fasta"]] + paths["sams"], check=True, capture_output=True, text=True)
    feat = json.loads(r.stdout.strip().splitlines()[-1])
    pre = os.path.join(build_dir, "abawaca")
    r = subprocess.run([os.path.join(ref, "ref_search"), pre + ".names", paths["fasta"], pre + ".info", pre + ".lrn", paths["gene2scg"], paths["scg_list"], "sensspec",
                        str(ncpu), os.path.join(workdir, "ref_search_dump.tsv")], check=True, capture_output=True, text=True)
    search_s = [float(l.split()[1]) for l in r.stderr.splitlines() if l.startswith("SEARCH_SECONDS")][-1]
    total = feat["scaf_s"] + feat["reads_s"] + search_s
    return {"windows_and_kmer_s": round(feat["scaf_s"], 3), "coverage_from_memory_s": round(feat["reads_s"], 3), "work_list_s": round(search_s, 3),
            "scaffolds_per_s": round(feat["scaffolds"] / total, 2),
            "what": "unmodified reference classes, no text parsing or writing: Scaf/Scaf_segment construction + add_mapped_read fed by Bio::VectorReader "
                    f"(1 thread, as abawaca-build), ClusterSeparator work list with {ncpu} threads"}


def reference_arm(mg, steps, warmup, per_genome, genomes, extra=None, with_compute_only=False, with_cli=False):
    ref = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(ref, "abawaca")):
        raise RuntimeError("oracle/_ref is not built (run __graft_entry__.build() where /root/reference is mounted)")
    sample = reference_sample(mg, per_genome, genomes)
    ncpu = max(1, min(40, os.cpu_count() or 1))       # abawaca -p is capped at 40 (abawaca.cpp:326-331)
    wd = tempfile.mkdtemp(prefix="abw_ref_")
    info = {}
    try:
        paths = synth.write_reference_inputs(sample, wd)
        tb, ts, bins, build_dir = [], [], None, None
        for i in range(warmup + steps):
            b, s, bins, build_dir = run_command_lines(ref, paths, wd, ncpu, "ref")
            if i >= warmup:
                tb.append(b); ts.append(s)
        if with_compute_only:
            try:
                info["compute_only"] = reference_compute_only(paths, build_dir, ncpu, wd)
            except Exception as e:
                info["compute_only"] = {"failed": repr(e)}
        if with_cli:
            # the drop-in command lines of this repo on the same text files: text in -> text out on both sides, CUDA start-up of two processes included
            try:
                mine = os.path.join(ROOT, "abawaca_b200", "bin")
                run_command_lines(mine, paths, wd, ncpu, "b200w")          # first process start on this box pages the library in
                b2, s2, bins2, _ = run_command_lines(mine, paths, wd, ncpu, "b200")
                info["e2e_cli"] = {"what": "abawaca-build + abawaca, text files in -> text files out, same sample, same box", "scaffolds": sample.nscaf,
                                   "reference_s": round(float(np.mean(tb) + np.mean(ts)), 3), "b200_s": round(b2 + s2, 3),
                                   "b200_build_s": round(b2, 3), "b200_bin_s": round(s2, 3), "ratio": round(float(np.mean(tb) + np.mean(ts)) / (b2 + s2), 2),
                                   "bins_identical": bool(bins2 == bins)}
            except Exception as e:
                info["e2e_cli"] = {"failed": repr(e)}
        extra_out = extra(paths, sample) if extra is not None else None
    finally:
        shutil.rmtree(wd, ignore_errors=True)
    t = float(np.mean(tb) + np.mean(ts))
    info.update(value=sample.nscaf / t, unit="scaffolds/s", cores=ncpu, kind="reference",
                sample=f"{sample.nscaf} scaffolds (first {per_genome} of each of {genomes} genomes) of the workload, {sum(r.size for r in sample.reads)} reads in "
                       f"{len(sample.reads)} SAM files, {len(set(bins)) - (1 if 0 in bins else 0)} bins; unmodified reference built -O2; abawaca-build (single-threaded by construction) "
                       f"{np.mean(tb):.2f} s + abawaca -p {ncpu} {np.mean(ts):.2f} s; the reference's cost per scaffold grows with the depth of the tree, "
                       f"so a small sample flatters it",
                build_s=float(np.mean(tb)), bin_s=float(np.mean(ts)))
    if extra_out is not None:
        info["_extra"] = extra_out
    return info, sample, bins


def reference_sample_size(steps, warmup):
    """Sample of the reference arm: sized so that steps + warmup runs end within a few minutes (about 115 scaffolds/s on this class of host)."""
    budget = 240.0 / max(1, steps + warmup)             # seconds per run
    if budget >= 24:
        return 400, 8                                   # 3200 scaffolds, 7 splits: about 27 s per run
    if budget >= 8:
        return 300, 4                                   # 1200 scaffolds, 3 splits: about 8 s per run
    return 400, 2                                       # 800 scaffolds, 1 split: about 4 s per run


# ------------------------------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------------------------------
def gpu_bins_for(ctx, mg, pipeline, capi):
    """One full pass from HOST buffers; returns (scaf2cluster over ALL scaffolds incl. dropped ones = 0, kept scaffolds)."""
    fb = pipeline.build_features(ctx, mg.seq, mg.offsets, mg.reads, this_sample=0)
    sg = fb.segments_host()
    keep, dp2scaf, T, kept = pipeline.search_problem_from_features(sg["seg_scaf"], mg.nscaf)
    length = np.diff(mg.offsets.astype(np.int64)).astype(np.uint64)[kept]
    mask = mg.scg_masks()[kept]
    rows = fb.rows_host()
    res = pipeline.search(ctx, rows, dp2scaf, T, length, mask, layout=capi.LAYOUT_ROWMAJOR, row_of_dp=np.nonzero(keep)[0])
    fb.close()
    bins = np.zeros(mg.nscaf, dtype=np.int64)
    bins[kept] = res.scaf2cluster
    return bins, kept


FEATURE_FAMILIES = {
    "k_kmer": ("k_kmer",),
    "coverage": ("k_cov_",),
}

DUMP_LIMIT_BYTES = 64_000_000
CLUSTER_FIELDS = ("id", "parent", "ndps", "nscafs", "split", "best.found", "best.dim", "best.value", "best.a", "best.b", "best.legal", "child1", "child2",
                  "child1_ndps", "child2_ndps", "child1_nscafs", "child2_nscafs", "child1_raw", "child2_raw", "total_size", "scg_unique", "scg_avg",
                  "gc_avg", "gc_sd", "cvg_avg", "cvg_sd")


def cluster_table(recs):
    """Cluster records as float64 [clusters][CLUSTER_FIELDS] (every integer field stays below 2**53, so the conversion is exact)."""
    def field(r, name):
        for part in name.split("."):
            r = getattr(r, part)
        return float(r)
    return np.array([[field(r, f) for f in CLUSTER_FIELDS] for r in recs], dtype=np.float64).reshape(-1, len(CLUSTER_FIELDS))


def dump_outputs(directory, arrays, seed=0):
    """Writes every array as <directory>/<name>.npy in float64, DUMP_LIMIT_BYTES in all.  An array larger than its share is replaced by the rows of a
    fixed, seeded sample (the same rows for the same shape), whose row numbers go beside it as <name>_rows.npy."""
    os.makedirs(directory, exist_ok=True)
    share = DUMP_LIMIT_BYTES // (2 * len(arrays)) - 4096          # room for an array, its row numbers and two .npy headers
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        rows_path = os.path.join(directory, f"{name}_rows.npy")
        if a.nbytes > share:
            k = max(1, share // (a.nbytes // a.shape[0]))
            rows = np.sort(np.random.default_rng(seed).choice(a.shape[0], k, replace=False))
            np.save(rows_path, rows.astype(np.float64))
            a = a[rows]
        elif os.path.exists(rows_path):
            os.remove(rows_path)
        np.save(os.path.join(directory, f"{name}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaffolds", type=int, default=0)
    ap.add_argument("--samples", type=int, default=0)
    ap.add_argument("--genomes", type=int, default=0)
    ap.add_argument("--coverage-scale", type=float, default=1.0, help="multiplies the read depth of the synthetic samples (large shapes: thinned reads)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="N > 1: skip the one-off comparison of the sharded search with the single-rank search")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    w = workload_args(args)

    if args.impl == "reference":
        if rank != 0:
            return 0
        mg = synth.make_metagenome(**w, q6_reads=True)
        per_genome, genomes = reference_sample_size(args.steps, max(args.warmup, 0))
        info, sample, _ = reference_arm(mg, args.steps, max(args.warmup, 0), per_genome, genomes)
        line = {"impl": "reference", "metric": "scaffolds/sec binned (feature build + split search)", "value": info["value"], "unit": "scaffolds/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sample.nscaf / info["value"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int64/f64", "data": "synthetic",
                "config": {"workload": workload_name(w), "timed": "bounded sample: " + info["sample"]},
                "cpu_baseline": {k: info[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": info["value"], "unit": "scaffolds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    from abawaca_b200 import capi, pipeline
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    mg = synth.make_metagenome(**w, q6_reads=True, shard=(rank if world > 1 else None))
    ctx = capi.Context(local_rank)
    L = ctx.lib
    import ctypes as C
    from abawaca_b200 import distributed
    nscaf = mg.nscaf
    lengths = np.diff(mg.offsets.astype(np.int64)).astype(np.uint64)
    masks = mg.scg_masks()
    if masks.shape[1] != 1:
        raise SystemExit("bench.py assumes at most 64 SCG names")
    total_bp = int(mg.seq.size)
    nreads = [int(r.size) for r in mg.reads]
    coll = None
    if world > 1:
        # the per-level collectives of the sharded search: NCCL from inside the library; ABW_TORCH_COLLECTIVES=1 selects the torch.distributed callbacks instead
        coll = distributed.TorchCollectives(local_rank) if os.environ.get("ABW_TORCH_COLLECTIVES") else distributed.NcclCollectives(ctx, local_rank)
    lengths_all = masks_all = None
    if world > 1:
        # static per-scaffold inputs of all ranks (sequence length, SCG mask), exchanged once: they are inputs, not results of a step
        st_local = torch.from_numpy(np.stack([lengths.astype(np.int64), masks[:, 0].astype(np.int64)], axis=1)).to(torch.device("cuda", local_rank))
        st_all = torch.empty((world * nscaf, 2), dtype=torch.int64, device=st_local.device)
        dist.all_gather_into_tensor(st_all, st_local)
        st_all = st_all.cpu().numpy()
        # pinned: abw_search_create uploads them every step
        pinned_np = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).pin_memory().numpy().view(np.uint64)   # noqa: E731
        lengths_all, masks_all = pinned_np(st_all[:, 0].astype(np.uint64)), pinned_np(st_all[:, 1].astype(np.uint64))

    # pinned host copies (e2e) and device-resident copies (value)
    h_seq = torch.from_numpy(mg.seq).pin_memory()
    h_reads = [torch.from_numpy(r.view(np.uint32).reshape(-1, 4)).pin_memory() for r in mg.reads[:1]]      # one sample, for the link measurement only
    # end-to-end path: what a host-side SAM parser hands over when it applies the read filter itself (abawaca-build.cpp:546-550, SURVEY.md section 8b(4)):
    # 8-byte records {scaffold, position} of the accepted reads in SAM order, one read length per sample (pipeline.compact_reads), in pinned memory
    h_compact = []
    for r in mg.reads:
        c = pipeline.compact_reads(r, mg.nscaf)
        t = torch.from_numpy(c.recs.view(np.uint32).reshape(-1, 2)).pin_memory()
        c.recs = t.numpy().view(capi.READ8_DTYPE).reshape(-1)
        c._pin = t
        if c.len16 is not None:
            t16 = torch.from_numpy(c.len16).pin_memory()
            c.len16, c._pin16 = t16.numpy(), t16
        h_compact.append(c)
    d_seq = ctx.alloc(total_bp + 64)
    ctx.to_device(d_seq, mg.seq)
    d_reads = []
    for r in mg.reads:
        p = ctx.alloc(max(r.nbytes, 16))
        ctx.to_device(p, r)
        d_reads.append(p)

    state = {}
    result_buffers = {}                                # records and bin arrays of the search, reused by every step
    dev = torch.device("cuda", local_rank)

    def exchange(fb, counts, timings=None, keep_doubles=False):
        """N > 1: the global scaffold table from all ranks' window counts, and this rank's block of columns of ALL datapoints (one NCCL all-to-all)."""
        t_x0 = time.perf_counter()
        # 1) windows per scaffold of every rank (the only per-scaffold quantity this step computed; lengths and SCG masks of all ranks were
        #    exchanged once at set-up): everybody derives the same global scaffold table, scaffold ids rank-major
        if state.get("h_cnt") is None:
            state["h_cnt"] = (torch.empty(nscaf, dtype=torch.int32).pin_memory(), torch.empty(world * nscaf, dtype=torch.int32).pin_memory(),
                              torch.empty(world * nscaf, dtype=torch.int32, device=dev))
        h_cnt, h_cnt_all, cnt_all = state["h_cnt"]
        h_cnt.numpy()[:] = counts
        dist.all_gather_into_tensor(cnt_all, h_cnt.to(dev, non_blocking=True))
        h_cnt_all.copy_(cnt_all, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        cnt_all = h_cnt_all.numpy()                                        # pinned, overwritten by the next step's exchange (the search of this step is over by then)
        memo = state.get("tables_memo")
        if memo is not None and np.array_equal(memo[0], cnt_all):         # the tables are a pure function of the counts: same counts, same tables
            keep_all, T_all, rows_per_rank = memo[1], memo[2], memo[3]
        else:
            if int(cnt_all.min()) >= 2:                                    # nothing to drop (every scaffold has two windows): no copies of the tables
                keep_all, T_all = slice(None), cnt_all.view(np.uint32).copy()
                rows_per_rank = cnt_all.reshape(world, nscaf).sum(axis=1).tolist()
            else:
                keep_all = cnt_all >= 2                                    # ScafDpData.cpp:92-93
                T_all = cnt_all[keep_all].astype(np.uint32)
                rows_per_rank = np.where(keep_all, cnt_all, 0).reshape(world, nscaf).sum(axis=1).tolist()
            state["tables_memo"] = (cnt_all.copy(), keep_all, T_all, rows_per_rank)
        if timings is not None:
            timings["exchange_tables_ms"] = 1000.0 * (time.perf_counter() - t_x0)
            t_x0 = time.perf_counter()
        # 2) every rank holds the rows of its own scaffolds and will search a block of COLUMNS of all datapoints (round-robin: rank q owns the dimensions
        #    q, q + world, ... so that every rank gets the same mix of k-mer and coverage dimensions, SURVEY.md 8e).  The columns travel as uint32
        #    thousandths (every value is int(1000 x) / 1000.0, abawaca-build.cpp:603): half the bytes of the doubles, and abw_search_create reads them as
        #    they are (ABW_LAYOUT_ROWMAJOR_MILLI32).
        ncol_of = [len(range(r, fb.ncols, world)) for r in range(world)]
        off, cnt = rank, ncol_of[rank]
        total_rows = int(sum(rows_per_rank))
        local64 = torch.as_tensor(distributed._DevArray(fb.d_rows, fb.nseg * fb.ncols * 8, "<f8", 8), device=dev).view(fb.nseg, fb.ncols)   # verify_sharded only
        def kept_rows():                                   # device index of the rows of the scaffolds that keep their windows (None: all); only the
            if not (counts < 2).any():                     # NCCL path and the one-off verification need it -- the peer kernel drops rows itself
                return None
            return torch.from_numpy(np.nonzero(np.repeat(counts >= 2, counts))[0]).to(dev)
        if keep_doubles:
            idx = kept_rows()
            if idx is not None:
                local64 = local64[idx]
        use_peer = not os.environ.get("ABW_NO_PEER") and coll is not None and getattr(coll.struct, "stream_ordered", 0)
        if os.environ.get("ABW_BENCH_DEBUG") and rank == 0:
            print("exchange: use_peer", bool(use_peer), "stream_ordered", getattr(coll.struct, "stream_ordered", None), file=sys.stderr, flush=True)
        if use_peer:
            # 2a) over NVLink peer memory (csrc/peer.cu): ONE kernel converts the local rows and stores every rank's columns straight into that rank's
            #     matrix (rows of scaffolds with a single window are left out on the way, ScafDpData.cpp:92-93); a one-word all-reduce on the context
            #     stream tells the receivers that everybody's rows have arrived.  Decided by global quantities only (buffer size from the global row
            #     count): every rank takes the same branch.
            need = total_rows * max(ncol_of) * 4
            px = state.get("peer")
            if px is None or (px.ok and px.half_bytes < need):
                if px is not None:
                    ctx.synchronize()
                    px.close()
                px = state["peer"] = distributed.PeerExchange(ctx, torch, dist, local_rank, int(need * 1.1) + 65536, coll)
            use_peer = px.ok
        if use_peer:
            if state.get("px_flag") is None:
                state["px_flag"] = ctx.alloc(16)
                ctx.memset(state["px_flag"], 0, 16)
            full_ptr = px.scatter(fb.d_rows, fb.nseg, fb.ncols, fb.ncols, int(sum(rows_per_rank[:rank])), d_inexact=state["px_flag"], segs=fb.segs)
            px.barrier()
            full = None
        else:
            # 2b) one NCCL all-to-all in which rank q receives from everybody the columns it owns -- 1/world of what an all-gather of whole rows would move
            d32 = fb.rows_milli32_device()
            ctx.synchronize()
            local = torch.as_tensor(distributed._DevArray(d32, fb.nseg * fb.ncols * 4, "<i4", 4), device=dev).view(fb.nseg, fb.ncols)
            idx = kept_rows()
            if idx is not None:
                local = local[idx]
            n_local = int(local.shape[0])
            send = torch.cat([local[:, r::world].reshape(-1) for r in range(world)])
            full = torch.empty((total_rows, cnt), dtype=torch.int32, device=dev)
            dist.all_to_all_single(full.view(-1), send, output_split_sizes=[n * cnt for n in rows_per_rank], input_split_sizes=[n_local * c for c in ncol_of])
            torch.cuda.synchronize(dev)
            full_ptr = full.data_ptr()
        if timings is not None:
            if use_peer:
                ctx.synchronize()
            timings["exchange_columns_ms"] = 1000.0 * (time.perf_counter() - t_x0)
        state["exchange_path"] = "peer memory (abw_scatter_columns_milli)" if use_peer else "NCCL all-to-all"
        return dict(full=full, full_ptr=full_ptr, total_rows=total_rows, off=off, cnt=cnt, T_all=T_all, keep_all=keep_all, rows_per_rank=rows_per_rank, local=local64)

    def step(resident, timings=None, on_features=None, keep_exchange=False, keep_features=False):
        if resident:
            fb = pipeline.build_features(ctx, d_seq, mg.offsets, d_reads, this_sample=0, seq_on_device=True, reads_on_device=True, nreads=nreads, timings=timings)
        else:
            fb = pipeline.build_features(ctx, h_seq.numpy(), mg.offsets, h_compact, this_sample=0, timings=timings, overlap_h2d=True)
        if on_features is not None:
            on_features()
        if world > 1:
            t_a = time.perf_counter()
            counts = np.diff(fb.seg_first_host().astype(np.int64))         # windows per scaffold: the ranks exchange them (exchange())
            if timings is not None:
                timings["segments_host_ms"] = 1000.0 * (time.perf_counter() - t_a)
        if not resident:
            # the .lrn matrix goes back to the host (pinned buffers) in the end-to-end path, while the split search runs: as integer thousandths
            # (uint16 k-mer columns, uint32 coverage columns; abw_rows_to_milli), which is what the text writer prints anyway
            ns_cov = fb.ncols - fb.nk
            if state.get("h_k16") is None or state["h_k16"].numel() < fb.nseg * fb.nk or state["h_k32"].numel() < fb.nseg * ns_cov:
                state["h_k16"] = torch.empty(int(fb.nseg * fb.nk * 1.05) + 1024, dtype=torch.int16).pin_memory()
                state["h_k32"] = torch.empty(int(fb.nseg * ns_cov * 1.05) + 1024, dtype=torch.int32).pin_memory()
            if state.get("h_seg") is None or state["h_seg"][0].numel() < fb.nseg:
                cap = int(fb.nseg * 1.05) + 1024
                state["h_seg"] = [torch.empty(cap, dtype=torch.int32).pin_memory()] + [torch.empty(cap, dtype=torch.int64).pin_memory() for _ in range(3)]
            fb.segments_async(state["h_seg"][0].numpy().view(np.uint32), *[t.numpy().view(np.uint64) for t in state["h_seg"][1:]])   # the .names columns
            fb.rows_milli(out16=state["h_k16"].numpy().view(np.uint16), out32=state["h_k32"].numpy().view(np.uint32), wait=False)
        if world == 1:
            # the search problem comes straight from the feature build on the device (windows per scaffold, scaffolds with a single window dropped as
            # ScafDpData.cpp:92-93 does, row index): abw_search_create_from_features
            res, kept = pipeline.search_features(ctx, fb, lengths, masks, timings=timings, buffers=result_buffers)
            ndps_total = int(res.dp2cluster.size)
        else:
            x = exchange(fb, counts, timings, keep_doubles=keep_exchange)
            kept = x["keep_all"]
            # dimension-sharded search: this rank sweeps columns [off, off+cnt) of every datapoint
            if isinstance(x["keep_all"], slice):
                len_kept, mask_kept = lengths_all, masks_all
            else:
                # lengths and SCG masks of the kept scaffolds: inputs, so the (pinned) subsets are reused as long as the step drops the same scaffolds
                kc = state.get("kept_cache")
                if kc is None or not (kc[0] is x["keep_all"] or np.array_equal(kc[0], x["keep_all"])):
                    kc = state["kept_cache"] = (x["keep_all"], pinned_np(lengths_all[x["keep_all"]]), pinned_np(masks_all[x["keep_all"]]))
                len_kept, mask_kept = kc[1], kc[2]
            res = pipeline.search(ctx, x["full_ptr"], None, x["T_all"], len_kept, mask_kept,
                                  layout=capi.LAYOUT_ROWMAJOR_MILLI32, values_on_device=True, nrows=x["total_rows"], D=x["cnt"], ld=x["cnt"], timings=timings,
                                  collectives=coll, dim_offset=x["off"], dim_stride=world, D_total=fb.ncols, buffers=result_buffers)
            ndps_total = x["total_rows"]
            if keep_exchange:
                state["exchange"] = x
            else:
                del x
        nbins = int(np.count_nonzero(np.bincount(res.scaf2cluster)[1:]))
        if world > 1:
            inexact = np.zeros(4, dtype=np.int32)
            if state.get("px_flag") is not None:
                ctx.to_host(inexact, state["px_flag"])
            if int(inexact[0]) or (fb._milli32 is not None and fb.milli_inexact()):
                raise SystemExit("bench.py: a feature value is not a multiple of 0.001")
        if not resident:
            ctx.synchronize()                          # the matrix has arrived on the host (copy stream) before the step counts as done
            if fb.milli_inexact():
                raise SystemExit("bench.py: a feature value is not a multiple of 0.001")
        state.update(ndps=ndps_total, nseg=fb.nseg, ncols=fb.ncols, prof=res.profile, nclusters=len(res.recs), nbins=nbins,
                     bins=res.scaf2cluster, res=res, kept=kept)
        if timings is not None:                        # window lengths: only needed for the algorithmic byte count of the k-mer kernel
            sg = fb.segments_host()
            state["seg_len"] = sg["seg_end"] - sg["seg_start"] + 1
        if keep_exchange or keep_features:
            state["fb"] = fb
        else:
            fb.close()
        return res

    ext = torch.cuda.ExternalStream(ctx.stream, device=local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(resident, steps, keep_last=False):
        """keep_last: the feature build of the last step stays open (state["fb"]) for last_step_outputs()."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launches
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        gc.collect()
        gc.disable()                                   # no interpreter garbage collection pause inside the timed region
        e0.record(ext)
        host = []
        for i in range(steps):
            m0, h0 = ctx.arena_misses, time.perf_counter()
            step(resident, keep_features=keep_last and i == steps - 1)
            host.append((round(1000.0 * (time.perf_counter() - h0), 3), ctx.arena_misses - m0))
            marks[i].record(ext)
        e1.record(ext)
        e1.synchronize()
        torch.cuda.synchronize()
        gc.enable()
        ms = e0.elapsed_time(e1)
        per_step = [round(([e0] + marks)[i].elapsed_time(marks[i]), 3) for i in range(steps)]
        t = torch.tensor([ms], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        state["host_ms_and_driver_allocations_" + ("resident" if resident else "e2e")] = host
        return float(t.item()), ctx.launches - l0, per_step

    def last_step_outputs():
        """What the last step handed its caller: the feature build (window table, .lrn matrix) and the split search (cluster records, bin of every
        datapoint and of every scaffold it kept, with the assembly index of those scaffolds).  Copied before the next step reuses the buffers."""
        fb, res, kept = state.pop("fb"), state["res"], state["kept"]
        if isinstance(kept, slice):                    # N > 1, no scaffold dropped
            kept = np.arange(world * nscaf)
        elif kept.dtype == bool:
            kept = np.nonzero(kept)[0]
        sg = fb.segments_host()
        out = {"windows": np.stack([sg[k].astype(np.float64) for k in ("seg_scaf", "seg_start", "seg_end", "seg_nonN")], axis=1),
               "features": fb.rows_host(), "clusters": cluster_table(res.recs), "dp2cluster": res.dp2cluster.astype(np.float64),
               "scaf2cluster": res.scaf2cluster.astype(np.float64), "kept_scaffolds": kept.astype(np.float64)}
        fb.close()
        return out

    def verify_sharded():
        """Once, outside the timed region: the NCCL-sharded search of this run against the single-rank search of the SAME gathered problem on rank 0 --
        every cluster record and every scaffold's bin must be identical (work list abawaca.cpp:98-197; merge order ClusterSeparator.cpp:11-16)."""
        res = step(True, keep_exchange=True)
        x, fb = state.pop("exchange"), state.pop("fb")
        rows_all = distributed.allgather_rows(torch, dist, x["local"].contiguous(), x["rows_per_rank"])
        verdict = torch.zeros(1, dtype=torch.int32, device=dev)
        if rank == 0:
            single = pipeline.search(ctx, rows_all.data_ptr(), None, x["T_all"], lengths_all[x["keep_all"]], masks_all[x["keep_all"]], layout=capi.LAYOUT_ROWMAJOR,
                                     values_on_device=True, nrows=int(rows_all.shape[0]), D=fb.ncols, ld=fb.ncols)
            key = lambda r: (r.id, r.parent, r.ndps, r.nscafs, r.split, r.best.found, r.best.dim, r.best.value, r.best.a, r.best.b, r.child1, r.child2,   # noqa: E731
                             r.child1_ndps, r.child2_ndps, r.child1_nscafs, r.child2_nscafs, r.child1_raw, r.child2_raw, r.total_size, r.scg_unique, r.scg_avg)
            same = [key(r) for r in res.recs] == [key(r) for r in single.recs] and np.array_equal(res.scaf2cluster, single.scaf2cluster) and \
                np.array_equal(res.dp2cluster, single.dp2cluster)
            verdict[0] = 1 if same else 2
        dist.all_reduce(verdict, op=dist.ReduceOp.MAX)
        fb.close()
        del x, rows_all
        return {"sharded_equals_single": bool(int(verdict.item()) == 1), "clusters": len(res.recs), "scaffolds": int(res.scaf2cluster.size),
                "what": "abw_search_run_sharded over NCCL on all ranks against abw_search_run on rank 0, same gathered matrix: records, scaffold bins and datapoint bins"}

    # the sampler is started BEFORE the warm-up: nvidia-smi takes driver locks while it starts and would otherwise stall the first timed launches
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("ABW_NO_CLOCK_SAMPLER"):   # one nvidia-smi poller per job: every query takes driver locks that all ranks' launches wait on
        sampler.start()
    for i in range(args.warmup):
        step(True)
        if i == 0 and "dp2c" in result_buffers:
            # the caller's result arrays (bin of every datapoint and scaffold) live in pinned memory from here on: the copies back are DMA transfers
            for k in ("dp2c", "s2c"):
                t = torch.empty(int(result_buffers[k].size * 1.05) + 1024, dtype=torch.int32).pin_memory()
                result_buffers[k + "_pinned"] = t
                result_buffers[k] = t.numpy().view(np.uint32)
            result_buffers["N"], result_buffers["S"] = int(result_buffers["dp2c"].size), int(result_buffers["s2c"].size)
    verify = None
    if world > 1 and not args.no_verify:
        verify = verify_sharded()
        if not verify["sharded_equals_single"]:
            raise SystemExit("bench.py: the sharded search differs from the single-rank search")
        step(True)                                     # the verification gathered whole matrices: one more untimed step so that the block caches hold the step's shapes again
    n_warm_samples = len(sampler.rows)                 # samples before this index were taken during the warm-up (same load)
    ms_res, launches, steps_res = timed(True, args.steps, keep_last=bool(args.dump_outputs))
    timed_rows = sampler.rows[n_warm_samples:]
    if len(timed_rows) >= 2:                           # enough samples inside the timed region itself; else keep the warm-up samples (same kernels, same load) as well
        sampler.rows = timed_rows
    clocks = sampler.stop()
    clocks["window"] = "timed region" if len(timed_rows) >= 2 else "warm-up + timed region"
    if args.dump_outputs:
        outputs = last_step_outputs()
        if rank == 0:
            dump_outputs(args.dump_outputs, outputs)
        del outputs
    for _ in range(max(1, args.warmup)):               # warm the host-buffer path (staging buffers enter the context's block cache)
        step(False)
    ms_e2e, _, steps_e2e = timed(False, args.steps)

    # what the host link gives on this box: the end-to-end step moves h2d_bytes_per_step over it (pinned read records of one sample, best of 3)
    pcie = None
    if h_reads and h_reads[0].numel():
        dst = torch.empty_like(h_reads[0], device=dev)
        best = None
        for _ in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); dst.copy_(h_reads[0], non_blocking=True); b.record(); b.synchronize()
            best = a.elapsed_time(b) if best is None else min(best, a.elapsed_time(b))
        nb = h_reads[0].numel() * h_reads[0].element_size()
        pcie = {"h2d_GBps": round(nb / best / 1e6, 2), "bytes": int(nb)}
        del dst

    # one extra profiled step: per-kernel CUDA-event durations (launches serialised while profiling), feature stage and split search reported apart
    phase_ms = {}
    t0 = time.perf_counter()
    step(True, timings=phase_ms)                       # host wall-clock per ABI phase of one (un-profiled) resident step
    phase_ms["step_total_ms"] = 1000.0 * (time.perf_counter() - t0)
    reports = {}

    def features_done():
        reports["features"] = ctx.profile_report()
        ctx.profile(True)                              # clears: what follows is the split search (create + run)
    ctx.profile(True)
    step(True, on_features=features_done)
    reports["search"] = ctx.profile_report()
    ctx.profile(False)
    prof = state["prof"]
    hbm, peak_src = peaks()
    seg_len = state["seg_len"].astype(np.int64)
    gbps = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0   # noqa: E731
    traffic_db = {}
    for f in ("r02_traffic.json", "r01_traffic.json"):
        try:
            for k, v in json.load(open(os.path.join(ROOT, "profiles", f))).items():
                traffic_db.setdefault(k, v)
        except Exception:
            pass
    # DESIGN.md section 5 / SURVEY.md section 8(d): algorithmic bytes per step
    alg_kmer = float(((seg_len + 3) // 4 + (seg_len + 7) // 8).sum() + state["nseg"] * 179 * 8)
    alg_cov = float(16 * sum(nreads) + 8 * state["nseg"] * len(nreads))
    alg_search = 12.0 * prof.sweep_elements
    ms_of = lambda rep, prefixes: sum(ms for k, (c, ms) in rep.items() if any(p in k for p in prefixes))   # noqa: E731
    ms_kmer = ms_of(reports["features"], FEATURE_FAMILIES["k_kmer"])
    ms_cov = ms_of(reports["features"], FEATURE_FAMILIES["coverage"]) + ms_of(reports["features"], ("k_rs_", "k_scan_"))   # sort and scans of the feature stage belong to the coverage
    ms_search = sum(ms for c, ms in reports["search"].values())
    ms_sweep = ms_of(reports["search"], ("k_sweep_ss", "k_sweep<"))
    families = {
        "split_search": {"kernels": "every kernel of abw_search_create + abw_search_run (" + str(len(reports["search"])) + " kernels)", "ms_per_step": round(ms_search, 4),
                         "algorithmic_bytes_per_step": alg_search, "achieved": round(gbps(alg_search, ms_search), 2), "frac": round(gbps(alg_search, ms_search) / hbm, 4)},
        "coverage": {"kernels": "every kernel of abw_coverage_batch incl. its sort", "ms_per_step": round(ms_cov, 4), "algorithmic_bytes_per_step": alg_cov,
                     "achieved": round(gbps(alg_cov, ms_cov), 2), "frac": round(gbps(alg_cov, ms_cov) / hbm, 4)},
        "k_kmer": {"kernels": "k_kmer", "ms_per_step": round(ms_kmer, 4), "algorithmic_bytes_per_step": alg_kmer, "achieved": round(gbps(alg_kmer, ms_kmer), 2),
                   "frac": round(gbps(alg_kmer, ms_kmer) / hbm, 4)},
    }
    # per kernel, beside the family figures: the sweep kernel alone against the same 12 B per (datapoint, dimension), with the DRAM bytes ncu saw it move
    sweep_traffic = None
    tj = traffic_db.get("k_sweep_ss")
    if tj:
        sweep_traffic = {"dram_bytes_per_step": round(tj["dram_bytes"] / tj["units"] * prof.sweep_elements), "source": tj["source"]}
    per_kernel = {"k_sweep_ss": {"ms_per_step": round(ms_sweep, 4), "achieved": round(gbps(alg_search, ms_sweep), 2), "frac": round(gbps(alg_search, ms_sweep) / hbm, 4),
                                 "note": "the sweep streams 4-byte elements; values and scaffold ids (the 12 B) are consumed by sort, packing, flip tables and partition, "
                                         "whose time the family figure includes", "traffic": sweep_traffic}}
    dom = max(families, key=lambda k: families[k]["ms_per_step"])
    launches_dom = sum(c for c, ms in reports["search"].values()) if dom == "split_search" else None
    fam_traffic = traffic_db.get("family:" + dom)
    roofline = {"bound": "hbm", "kernel": dom, "kernels": families[dom]["kernels"], "achieved": families[dom]["achieved"], "peak": hbm, "peak_source": peak_src, "unit": "GB/s",
                "frac": families[dom]["frac"], "traffic": (round(fam_traffic["dram_bytes"] / fam_traffic["units"] * prof.sweep_elements) if fam_traffic and dom == "split_search" else None),
                "traffic_source": fam_traffic["source"] if fam_traffic else None, "ms_per_step_in_kernels": families[dom]["ms_per_step"],
                "launches_per_step": launches_dom, "algorithmic_bytes_per_step": families[dom]["algorithmic_bytes_per_step"],
                "definition": "SURVEY.md 8(d): 12 B per (datapoint, dimension) of every evaluated cluster / CUDA-event time of ALL split-search kernels of a step",
                "families": families, "per_kernel": per_kernel}
    kernels = {}
    allrep = {}
    for rep in reports.values():
        for k, (c, ms) in rep.items():
            a = allrep.setdefault(k, [0, 0.0])
            a[0] += c; a[1] += ms
    total_ms = sum(v[1] for v in allrep.values())
    for k, (cnt, ms) in sorted(allrep.items(), key=lambda kv: -kv[1][1]):
        kernels[k] = {"launches": cnt, "ms": round(ms, 4), "share": round(ms / total_ms, 4) if total_ms else None}

    total_scaf = nscaf * world
    value = total_scaf * args.steps / (ms_res * 1e-3)
    e2e_value = total_scaf * args.steps / (ms_e2e * 1e-3)
    nrec_bytes = state["nclusters"] * C.sizeof(capi.ClusterRec)
    h2d = total_bp + sum(c.nbytes for c in h_compact) + mg.offsets.nbytes + nscaf * (4 + 8 + 8 * masks.shape[1])
    # .lrn matrix as integer thousandths (2 bytes per k-mer value, 4 per coverage value) + window table + window offsets + cluster records + per-scaffold and per-datapoint bins
    d2h = state["nseg"] * (179 * 2 + len(mg.reads) * 4) + state["nseg"] * (4 + 3 * 8) + (nscaf + 1) * 8 + nrec_bytes + nscaf * 4 + state["ndps"] * 4

    line = {"metric": "scaffolds/sec binned (feature build + split search)", "value": round(value, 2), "unit": "scaffolds/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_res / args.steps, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/int64/f64", "data": "synthetic",
            "config": {"workload": workload_name(w), "per_gpu": f"{nscaf} scaffolds, {total_bp} bp, {state['nseg']} windows x {state['ncols']} dimensions, {sum(nreads)} read records",
                       "parallelism": (f"one community of {world} x {nscaf} scaffolds: scaffold-sharded feature build, feature columns exchanged as uint32 thousandths over {state.get('exchange_path', 'NCCL all-to-all')}, "
                                       f"dimension-sharded split search ({state['ncols']} dimensions over {world} ranks)") if world > 1 else "1 GPU",
                       "l2": "inputs (assembly + read records, > 2 GB) are larger than the 126 MB L2; no explicit flush",
                       "e2e_inputs": "pinned host buffers: ASCII assembly + 8-byte read records of the reads that pass the host-side filter (abw_read8), one length per sample",
                       "clusters_evaluated": state["nclusters"], "bins": state["nbins"], "search_levels": prof.levels, "datapoints": state["ndps"],
                       "nccl": None if coll is None else {"search_collectives": type(coll).__name__, "callback_collectives_total": coll.calls, "callback_bytes_total": coll.bytes}},
            "e2e": {"value": round(e2e_value, 2), "unit": "scaffolds/s", "ms_per_step": round(ms_e2e / args.steps, 3), "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "pcie": pcie, "gpu_launches": int(launches), "step_ms": {"resident": steps_res, "e2e": steps_e2e,
                                                     "host_ms_and_driver_allocations": {"resident": state.get("host_ms_and_driver_allocations_resident"),
                                                                                        "e2e": state.get("host_ms_and_driver_allocations_e2e")}}, "clocks": clocks, "roofline": roofline, "kernels": kernels,
            "kernel_time_over_step_time": round(total_ms / (ms_res / args.steps), 3),
            "phase_wall_ms": {k: round(v, 3) for k, v in phase_ms.items()},
            "search_profile_ms": {"build": round(prof.build_ms, 3), "sweep": round(prof.sweep_ms, 3), "partition": round(prof.partition_ms, 3), "other": round(prof.other_ms, 3)}}
    if verify is not None:
        line["sharded_equals_single"] = verify["sharded_equals_single"]
        line["config"]["verification"] = verify

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            def ingest(paths, sample):
                # SAM text of one sample of the bounded workload -> records on the device (abw_parse_sam), text already resident in HBM
                text = np.fromfile(paths["sams"][0], dtype=np.uint8)
                sp = pipeline.SamParser(ctx, sample.names)
                d_text = ctx.alloc(text.size + 64)
                ctx.to_device(d_text, text)
                cap = int(np.count_nonzero(text == 10)) + 1
                d_rec = ctx.alloc(cap * 16)
                n = C.c_uint64()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                reps = 5
                for i in range(reps + 2):
                    if i == 2:
                        e0.record(ext)
                    ctx.check(L.abw_parse_sam(ctx.h, sp.h, C.c_void_p(d_text), text.size, 1, C.c_void_p(d_rec), cap, C.byref(n)))
                e1.record(ext)
                e1.synchronize()
                ms = e0.elapsed_time(e1) / reps
                got = np.zeros(int(n.value), dtype=capi.READ_DTYPE)
                ctx.to_host(got, d_rec)
                src = sample.reads[0]
                mapped = (src["flag_nsnps"] & 0x4) == 0
                ok = bool(got.size == src.size and np.array_equal(got[mapped], src[mapped]))
                ctx.free(d_text); ctx.free(d_rec); sp.close()
                return {"kernel_path": "abw_parse_sam", "text_bytes": int(text.size), "records": int(n.value), "ms": round(ms, 3),
                        "GBps": round(text.size / (ms * 1e-3) / 1e9, 2), "records_identical_to_generator": ok}
            # 4 genomes x 300 scaffolds: about 10 s of reference time, and the reference recurses (3 splits)
            info, sample, ref_bins = reference_arm(mg, 1, 0, 300, 4, extra=ingest, with_compute_only=True, with_cli=True)
            if "_extra" in info:
                line["ingest"] = info.pop("_extra")
            gbins, kept = gpu_bins_for(ctx, sample, pipeline, capi)
            # the reference lists only scaffolds with >= 2 windows (ScafDpData.cpp:92-93)
            info["gpu_bins_identical_on_sample"] = bool(ref_bins == [int(b) for b in gbins[kept]])
            if "e2e_cli" in info:
                line["e2e_cli"] = info.pop("e2e_cli")
            line["cpu_baseline"] = info
        except Exception as e:  # the baseline must never take the bench line down
            line["cpu_baseline"] = {"value": None, "unit": "scaffolds/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e!r}"}
    if rank == 0:
        print(json.dumps(line))
    if coll is not None and hasattr(coll, "close"):
        if state.get("peer") is not None:
            ctx.synchronize()
            dist.barrier()                              # nobody unmaps a buffer another rank may still be writing to
            state["peer"].close()
        coll.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
