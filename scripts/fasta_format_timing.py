"""Time of the FASTA writer on the device (abw_fasta_format, abw_twobit_format) and of abawaca with the assembly kept on the device.

1. The kernels: the FASTA text of all configs[1] scaffolds (0.5 Gbp) from a FASTA text (80 columns) and from a .2bit image, in one window; per-kernel
   device time (CUDA events, abw_profile_enable) after a warm-up call, output GB/s against the measured 6.46 TB/s; the base counts of both.
2. The ABW_TIMING phases of abawaca on the sample of scripts/textout_timing.py (one abawaca-build of this tree), for this tree's binary and, with
   --parent BINDIR, another build's, alternating, --reps times each, with -f on the FASTA assembly and on a .2bit of it; every output file of the two
   (all but the time-stamped log) must be identical.

python scripts/fasta_format_timing.py [--per-genome 1000] [--genomes 8] [--thin 3] [--reps 3] [--parent BINDIR] [--json FILE]
"""
import argparse
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import textout_timing as tt                      # noqa: E402  (gpu_info, phases, the sample of the command-line timing)

PEAK_MEASURED = tt.PEAK_MEASURED


def kernel_timing(mg, reps=5):
    from abawaca_b200 import capi, hostio, pipeline
    ctx = capi.Context(0)
    parts = []
    for i, name in enumerate(mg.names):
        s = mg.scaffold(i).tobytes()
        parts.append(b">" + name.encode() + b"\n" + b"".join(s[o:o + 80] + b"\n" for o in range(0, len(s), 80)))
    text = b"".join(parts)
    wd = tempfile.mkdtemp(prefix="abw_fafmt_")
    out = {}
    try:
        tb = os.path.join(wd, "a.2bit")
        hostio.write_twobit(tb, list(mg.names), [mg.scaffold(i).tobytes() for i in range(mg.nscaf)])
        for kind, data in (("fasta", text), ("2bit", open(tb, "rb").read())):
            asm = pipeline.AssemblyFile(ctx, data)
            recs = np.arange(asm.count, dtype=np.uint32)
            total, _ = asm.format_window(recs, 0, 0, 0)
            d_text = ctx.alloc(total)
            asm.format_window(recs, 0, d_text, total)            # warm-up
            host = []
            for _ in range(reps):
                t0 = time.perf_counter()
                asm.format_window(recs, 0, d_text, total)
                host.append(1e3 * (time.perf_counter() - t0))
            pipeline.base_counts(ctx, asm)
            ctx.profile(True)
            for _ in range(reps):
                asm.format_window(recs, 0, d_text, total)
                pipeline.base_counts(ctx, asm)
            prof = ctx.profile_report()
            ctx.profile(False)
            ms = {k: v[1] / v[0] for k, v in prof.items() if v[0]}
            wk = [k for k in ms if k.startswith("k_fasta_write")][0]
            bases = int(sum(mg.offsets[1:].astype(np.int64) - mg.offsets[:-1].astype(np.int64)))
            out[kind] = dict(records=asm.count, bases=bases, input_bytes=len(data), text_bytes=total, kernel_ms=ms,
                             write_kernel_output_GBps=total / (ms[wk] / 1e3) / 1e9,
                             write_kernel_output_frac_of_measured_peak=total / (ms[wk] / 1e3) / 1e9 / PEAK_MEASURED, call_host_ms=host)
            print(kind, json.dumps(out[kind]), flush=True)
            ctx.free(d_text)
            asm.close()
    finally:
        shutil.rmtree(wd, ignore_errors=True)
        ctx.close()
    return out


def run_abawaca(bindir, build, out, fasta, paths):
    shutil.rmtree(out, ignore_errors=True)
    env = dict(os.environ, ABW_SCG_LIST=paths["scg_list"], ABW_TIMING="1")
    t0 = time.perf_counter()
    r = subprocess.run([os.path.join(bindir, "abawaca"), "-u", build, "-f", fasta, "-o", out, "-c", paths["gene2scg"], "-p", "16"], env=env, capture_output=True,
                       text=True)
    t1 = time.perf_counter()
    assert r.returncode == 0, r.stderr[-2000:]
    return dict(abawaca_s=t1 - t0, phases=tt.phases(r.stderr))


def differences(a, b):
    bad = []
    for sub in ("", "clusters", "final-clusters"):
        da, db = os.path.join(a, sub), os.path.join(b, sub)
        fa = sorted(f for f in os.listdir(da) if os.path.isfile(os.path.join(da, f)) and f != "log")
        if fa != sorted(f for f in os.listdir(db) if os.path.isfile(os.path.join(db, f)) and f != "log"):
            bad.append(sub + ": file lists differ")
            continue
        bad += [os.path.join(sub, f) for f in fa if not filecmp.cmp(os.path.join(da, f), os.path.join(db, f), shallow=False)]
    return bad


def cli_timing(args, mg_cfg2):
    import bench
    from abawaca_b200 import hostio, synth
    sample = bench.reference_sample(mg_cfg2, args.per_genome, args.genomes)
    sample.reads[:] = [r[::args.thin].copy() for r in sample.reads]
    wd = tempfile.mkdtemp(prefix="abw_fafmt_cli_")
    try:
        paths = synth.write_reference_inputs(sample, wd)
        names, seqs = hostio.read_fasta(paths["fasta"])
        tb = os.path.join(wd, "assembly.2bit")
        hostio.write_twobit(tb, names, seqs)
        build = os.path.join(wd, "build")
        r = subprocess.run([os.path.join(ROOT, "abawaca_b200", "bin", "abawaca-build"), "-f", paths["fasta"], "-o", build, "-s", os.path.join(wd, "sample*.sam"),
                            "-c", paths["sams"][0]], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        print(f"sample: {sample.nscaf} scaffolds, assembly {os.path.getsize(paths['fasta']) / 1e6:.1f} MB FASTA, {os.path.getsize(tb) / 1e6:.1f} MB .2bit", flush=True)
        arms = [("this", os.path.join(ROOT, "abawaca_b200", "bin"))] + ([("parent", args.parent)] if args.parent else [])
        res = {}
        for kind, fasta in (("fasta", paths["fasta"]), ("2bit", tb)):
            runs = {tag: [] for tag, _ in arms}
            diffs = None
            for rep in range(args.reps):
                outs = {}
                for tag, bindir in (arms if rep % 2 == 0 else arms[::-1]):
                    outs[tag] = os.path.join(wd, "o_" + tag)
                    x = run_abawaca(bindir, build, outs[tag], fasta, paths)
                    runs[tag].append(x)
                    print(f"{kind} rep {rep} {tag}: {json.dumps(x)}", flush=True)
                if args.parent:
                    d = differences(outs["this"], outs["parent"])
                    diffs = d if diffs is None else diffs + d
                    nfiles = sum(len(fs) for _, _, fs in os.walk(outs["this"])) - 1
                    print(f"{kind} rep {rep}: {nfiles} output files, " + ("all identical to the parent's" if not d else f"OUTPUTS DIFFER: {d[:20]}"), flush=True)
            med = {tag: {ph: float(np.median([x["phases"].get(ph, 0.0) for x in v])) for ph in v[0]["phases"]} for tag, v in runs.items()}
            res[kind] = dict(runs=runs, median_phases_s=med, output_differences=diffs)
            print(f"{kind} median phases: {json.dumps(med)}", flush=True)
        return dict(scaffolds=sample.nscaf, **res)
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
    from abawaca_b200 import synth
    res = dict(gpu=tt.gpu_info())
    print("gpu:", res["gpu"], flush=True)
    mg = synth.make_metagenome(**synth.CONFIGS["cfg2"], q6_reads=True)
    if not args.skip_kernel:
        res["kernel"] = kernel_timing(mg)
    res["cli"] = cli_timing(args, mg)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        json.dump(res, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
