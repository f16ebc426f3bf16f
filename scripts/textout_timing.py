"""Time of the .lrn text writers.

1. abw_format_lrn alone at the configs[1] shape (227 463 windows x 189 columns, 179 k-mer columns of thousandths <= 1 and 10 coverage columns),
   "%.3lf" and "%lf": per-kernel device time (CUDA events, abw_profile_enable) after a warm-up call, the 344 MB input being larger than L2; the
   whole call on the host clock; the device-to-host copy of the text into pageable memory, which is what the command lines do next.
2. The ABW_TIMING phases of both command lines on a sample of the configs[1] workload (--per-genome x --genomes scaffolds, every --thin-th read kept),
   for this tree's binaries and, with --parent BINDIR, another build's, alternating, --reps times; the outputs of the two must be identical.

python scripts/textout_timing.py [--per-genome 1000] [--genomes 8] [--thin 3] [--reps 3] [--parent BINDIR] [--json FILE]
"""
import argparse
import ctypes as C
import filecmp
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PEAK_MEASURED, PEAK_DATASHEET = 6459.6, 7700.0          # GB/s: DESIGN.md section 5, and NVIDIA's HGX B200 data sheet for one GPU


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def kernel_timing(reps=5):
    from abawaca_b200 import capi
    ctx = capi.Context(0)
    N, D = 227463, 189
    rng = np.random.default_rng(1)
    M = np.empty((N, D))
    M[:, :179] = rng.integers(0, 1001, (N, 179)) / 1000.0
    M[:, 179:] = rng.integers(0, 200000, (N, 10)) / 1000.0
    d = ctx.alloc(M.nbytes)
    ctx.to_device(d, M)
    cap = 1 << 30
    d_text = ctx.alloc(cap)
    done, nbytes = C.c_uint64(), C.c_uint64()
    call = lambda fmt: ctx.check(ctx.lib.abw_format_lrn(ctx.h, C.c_void_p(d), D, 0, D, None, 0, 0, N, fmt, C.c_void_p(d_text), cap, C.byref(done), C.byref(nbytes)))  # noqa: E731
    out = {}
    for fmt, name in ((capi.TEXT_3LF, "%.3lf"), (capi.TEXT_LF, "%lf")):
        call(fmt)
        host = []
        for _ in range(reps):
            t0 = time.perf_counter()
            call(fmt)
            host.append(time.perf_counter() - t0)
        text = np.empty(int(nbytes.value), dtype=np.uint8)
        copy = []
        for _ in range(reps):
            t0 = time.perf_counter()
            ctx.to_host(text, d_text)
            copy.append(time.perf_counter() - t0)
        ctx.profile(True)
        for _ in range(reps):
            call(fmt)
        prof = ctx.profile_report()
        ctx.profile(False)
        ms = {k.split("<")[0]: v[1] / v[0] for k, v in prof.items() if v[0]}
        t_write = ms["k_lrn_text_write"] / 1e3
        t_all = sum(ms.values()) / 1e3
        nb = int(nbytes.value)
        write_bytes = 8 * N * D + 8 * N + nb                      # matrix and line offsets read, text written
        all_bytes = 2 * 8 * N * D + 4 * N + 2 * 8 * N + nb        # length pass, scan, write pass
        out[name] = dict(lines=N, cols=D, text_bytes=nb, kernel_ms=ms, write_kernel_GBps=write_bytes / t_write / 1e9,
                         write_kernel_frac_of_measured_peak=write_bytes / t_write / 1e9 / PEAK_MEASURED, device_total_ms=t_all * 1e3,
                         device_total_GBps=all_bytes / t_all / 1e9, device_total_frac_of_measured_peak=all_bytes / t_all / 1e9 / PEAK_MEASURED,
                         frac_of_datasheet=all_bytes / t_all / 1e9 / PEAK_DATASHEET, call_host_ms=[1e3 * x for x in host], copy_to_pageable_host_ms=[1e3 * x for x in copy])
        print(name, json.dumps(out[name]), flush=True)
    ctx.free(d_text)
    ctx.free(d)
    ctx.close()
    return out


def phases(stderr):
    ph = {}
    for l in stderr.splitlines():
        m = re.match(r"\[abw timing\] (.*?)\s+([0-9.]+) s$", l)
        if m:
            ph[m.group(1)] = ph.get(m.group(1), 0.0) + float(m.group(2))
    return ph


def run_cli(bindir, paths, wd, tag):
    build, out = os.path.join(wd, "b_" + tag), os.path.join(wd, "o_" + tag)
    shutil.rmtree(build, ignore_errors=True)
    shutil.rmtree(out, ignore_errors=True)
    os.makedirs(build)
    env = dict(os.environ, ABW_SCG_LIST=paths["scg_list"], ABW_TIMING="1")
    t0 = time.perf_counter()
    r1 = subprocess.run([os.path.join(bindir, "abawaca-build"), "-f", paths["fasta"], "-o", build, "-s", os.path.join(wd, "sample*.sam"), "-c", paths["sams"][0]],
                        env=env, capture_output=True, text=True)
    t1 = time.perf_counter()
    r2 = subprocess.run([os.path.join(bindir, "abawaca"), "-u", build, "-o", out, "-c", paths["gene2scg"], "-p", "16"], env=env, capture_output=True, text=True)
    t2 = time.perf_counter()
    assert r1.returncode == 0 and r2.returncode == 0, (r1.stderr[-2000:], r2.stderr[-2000:])
    return dict(build_s=t1 - t0, abawaca_s=t2 - t1, build_phases=phases(r1.stderr), abawaca_phases=phases(r2.stderr)), build, out


def same_outputs(a_build, a_out, b_build, b_out):
    bad = [f for f in ("abawaca.lrn", "abawaca.names", "abawaca.info") if not filecmp.cmp(os.path.join(a_build, f), os.path.join(b_build, f), shallow=False)]
    for sub in ("", "clusters", "final-clusters"):
        da, db = os.path.join(a_out, sub), os.path.join(b_out, sub)
        fa = sorted(f for f in os.listdir(da) if os.path.isfile(os.path.join(da, f)) and f != "log")
        if fa != sorted(f for f in os.listdir(db) if os.path.isfile(os.path.join(db, f)) and f != "log"):
            bad.append(sub + ": file lists differ")
            continue
        bad += [os.path.join(sub, f) for f in fa if not filecmp.cmp(os.path.join(da, f), os.path.join(db, f), shallow=False)]
    return bad


def cli_timing(args):
    import bench
    from abawaca_b200 import synth
    mg = synth.make_metagenome(**synth.CONFIGS["cfg2"], q6_reads=True)
    sample = bench.reference_sample(mg, args.per_genome, args.genomes)
    sample.reads[:] = [r[::args.thin].copy() for r in sample.reads]
    wd = tempfile.mkdtemp(prefix="abw_textout_")
    try:
        paths = synth.write_reference_inputs(sample, wd)
        sam_bytes = sum(os.path.getsize(p) for p in paths["sams"])
        print(f"sample: {sample.nscaf} scaffolds, {len(paths['sams'])} SAM files, {sam_bytes / 1e9:.2f} GB of SAM text", flush=True)
        arms = [("this", os.path.join(ROOT, "abawaca_b200", "bin"))] + ([("parent", args.parent)] if args.parent else [])
        runs = {tag: [] for tag, _ in arms}
        diffs = None
        for rep in range(args.reps):
            dirs = {}
            for tag, bindir in (arms if rep % 2 == 0 else arms[::-1]):
                res, b, o = run_cli(bindir, paths, wd, tag)
                dirs[tag] = (b, o)
                runs[tag].append(res)
                print(f"rep {rep} {tag}: {json.dumps(res)}", flush=True)
            if args.parent and diffs is None:
                diffs = same_outputs(*dirs["this"], *dirs["parent"])
                print("outputs identical to the parent's" if not diffs else f"OUTPUTS DIFFER: {diffs[:20]}", flush=True)
        return dict(scaffolds=sample.nscaf, sam_bytes=sam_bytes, runs=runs, output_differences=diffs)
    finally:
        shutil.rmtree(wd, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--per-genome", type=int, default=1000)
    ap.add_argument("--genomes", type=int, default=8)
    ap.add_argument("--thin", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parent", default=None)
    ap.add_argument("--json", default=None)
    ap.add_argument("--skip-kernel", action="store_true")
    args = ap.parse_args()
    res = dict(gpu=gpu_info())
    print("gpu:", res["gpu"], flush=True)
    if not args.skip_kernel:
        res["kernel"] = kernel_timing()
    res["cli"] = cli_timing(args)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        json.dump(res, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
