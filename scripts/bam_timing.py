"""Reads from BAM on the device (abw_bam_feed + abw_bam_finish) against the same reads as SAM text (abw_parse_sam).

The workload is sample 0 of bench.py's configs[1] stream (synth.CONFIGS["cfg2"], q6_reads=True), about 14.5 M reads, written by synth.write_bam
in htslib's block layout (a block starts at a record) and cut at random sizes (records cross blocks, as htsjdk writes them), zlib level 6, and as
the SAM text synth.write_reference_inputs writes.  The files are read into host memory first; each arm then hands them to the library in 64 MB
pieces, as abawaca-build does: the BAM arms through abw_bam_feed / abw_bam_finish, the SAM arm through abw_parse_sam on chunks cut at line
boundaries.  CUDA events on the context stream around the whole sample give its time (every call ends in a synchronize); the arms alternate after a
warm-up run of each.  One profiled run per BAM arm (abw_profile_enable) gives the time per kernel.  Single-thread host zlib inflate of every block of
the aligned file is timed as a reference point.  Last, abawaca-build runs on the cfg1 inputs as SAM and as BAM (aligned for even samples, cut for odd)
and the outputs are compared.

python scripts/bam_timing.py [--runs 3] [--json FILE] [--workdir DIR]
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CHUNK = 64 << 20


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def bgzf_blocks(data):
    o, out = 0, []
    while o < len(data):
        bsize = int.from_bytes(data[o + 16:o + 18], "little") + 1
        out.append((o, bsize))
        o += bsize
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--json", default=None)
    ap.add_argument("--workdir", default=None)
    a = ap.parse_args()
    import torch
    from abawaca_b200 import capi, pipeline, synth

    wd = a.workdir or tempfile.mkdtemp(prefix="bam_timing_")
    out = {"workload": "configs[1] (synth cfg2, q6_reads) sample 0", "gpu": gpu_info()}
    t0 = time.perf_counter()
    mg = synth.make_metagenome(**synth.CONFIGS["cfg2"], q6_reads=True)
    mg.reads = mg.reads[:1]
    out["generate_s"] = round(time.perf_counter() - t0, 1)
    out["reads"] = int(mg.reads[0].size)
    files = {}
    for arm, kw in (("bam_aligned", dict(aligned=True)), ("bam_cut", dict(aligned=False))):
        t0 = time.perf_counter()
        files[arm] = synth.write_bam(os.path.join(wd, arm + ".bam"), mg, 0, level=6, threads=os.cpu_count() or 8, **kw)
        out[f"write_{arm}_s"] = round(time.perf_counter() - t0, 1)
    t0 = time.perf_counter()
    files["sam"] = synth.write_reference_inputs(mg, wd)["sams"][0]
    out["write_sam_s"] = round(time.perf_counter() - t0, 1)
    data = {k: open(v, "rb").read() for k, v in files.items()}
    out["file_bytes"] = {k: len(v) for k, v in data.items()}

    # single-thread host zlib inflate of the aligned file, as a reference point
    blocks = bgzf_blocks(data["bam_aligned"])
    t0 = time.perf_counter()
    decoded = 0
    for o, n in blocks:
        decoded += len(zlib.decompress(data["bam_aligned"][o + 18:o + n - 8], -15))
    zs = time.perf_counter() - t0
    out["decoded_bytes"] = decoded
    out["bgzf_blocks"] = len(blocks)
    out["host_zlib_1thread"] = {"s": round(zs, 3), "GBps": round(decoded / zs / 1e9, 3)}
    print(json.dumps(out), flush=True)

    ctx = capi.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream, device=0)
    names = mg.names
    nrec = mg.reads[0].size
    d_sam = ctx.alloc(nrec * 16 + 16)
    sp = pipeline.SamParser(ctx, names)
    sam = np.frombuffer(data["sam"], dtype=np.uint8)
    # line-boundary cuts of the SAM text, as abawaca-build makes them
    cuts, o = [0], 0
    while o < sam.size:
        e = min(o + CHUNK, sam.size)
        if e < sam.size:
            e = o + int(np.flatnonzero(sam[o:e] == 10)[-1]) + 1
        cuts.append(e)
        o = e

    def run(arm, keep=False):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        if arm == "sam":
            n = 0
            for lo, hi in zip(cuts[:-1], cuts[1:]):
                n += sp.parse(sam[lo:hi], d_sam + 16 * n, nrec - n)
            res = (d_sam, n)
            r = None
        else:
            r = pipeline.BamReader(ctx, names)
            buf = data[arm]
            for o in range(0, len(buf), CHUNK):
                r.feed(memoryview(buf)[o:o + CHUNK])
            res = r.finish()
        ev1.record(stream)
        ev1.synchronize()
        ms = ev0.elapsed_time(ev1)
        host = None
        if keep:
            host = np.zeros(res[1], dtype=capi.READ_DTYPE)
            ctx.to_host(host, res[0])
        if r is not None:
            r.close()
        return ms, host

    arms = ["bam_aligned", "bam_cut", "sam"]
    recs = {}
    for arm in arms:                                   # warm-up, and the records for the comparison
        _, recs[arm] = run(arm, keep=True)
    out["identical_records"] = {arm: bool(np.array_equal(recs[arm], recs["sam"])) for arm in arms[:2]}
    out["records"] = int(recs["sam"].size)
    del recs
    times = {arm: [] for arm in arms}
    for _ in range(a.runs):
        for arm in arms:
            times[arm].append(run(arm)[0])
    out["device_ms_per_sample"] = {}
    for arm in arms:
        t = times[arm]
        med = statistics.median(t)
        src = decoded if arm != "sam" else len(data["sam"])
        out["device_ms_per_sample"][arm] = {"median": round(med, 1), "min": round(min(t), 1), "max": round(max(t), 1), "all": [round(x, 1) for x in t],
                                            "input_GBps" if arm == "sam" else "decoded_GBps": round(src / med / 1e6, 2),
                                            "Mrecords_per_s": round(nrec / med / 1e3, 1)}
    out["kernels_ms"] = {}
    for arm in arms[:2]:
        ctx.profile(True)
        run(arm)
        rep = ctx.profile_report()
        ctx.profile(False)
        out["kernels_ms"][arm] = {k: round(v[1], 2) for k, v in sorted(rep.items(), key=lambda kv: -kv[1][1]) if v[1] >= 0.05}
    sp.close()
    ctx.free(d_sam)
    ctx.close()
    print(json.dumps(out), flush=True)

    # abawaca-build on the cfg1 inputs: SAM against BAM
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "abawaca_b200", "host")], check=True)
    mg1 = synth.make_metagenome(**synth.CONFIGS["cfg1"])
    d1 = os.path.join(wd, "cfg1")
    p1 = synth.write_reference_inputs(mg1, d1)
    for j in range(len(mg1.reads)):
        synth.write_bam(os.path.join(d1, f"sample{j:02d}.bam"), mg1, j, aligned=(j % 2 == 0), level=6)
    wall, outs = {}, {}
    for rep_i in range(2):
        for kind in ("sam", "bam"):
            build = os.path.join(d1, f"build_{kind}")
            first = os.path.join(d1, f"sample00.{kind}")
            t0 = time.perf_counter()
            r = subprocess.run([os.path.join(ROOT, "abawaca_b200", "bin", "abawaca-build"), "-f", p1["fasta"], "-o", build, "-s", os.path.join(d1, f"sample*.{kind}"),
                                "-c", first], capture_output=True, text=True)
            wall.setdefault(kind, []).append(round(time.perf_counter() - t0, 2))
            assert r.returncode == 0, r.stderr[-2000:]
            outs[kind] = {f: open(os.path.join(build, f)).read() for f in ("abawaca.lrn", "abawaca.names", "abawaca.info")}
    norm = lambda t: re.sub(r"sample(\d+)\.(bam|sam)", r"sample\1", t)      # noqa: E731  (the paths of line 4 of the .lrn)
    out["abawaca_build_cfg1"] = {"wall_s": wall, "file_bytes": {k: sum(os.path.getsize(os.path.join(d1, f"sample{j:02d}.{k}")) for j in range(len(mg1.reads)))
                                                                for k in ("sam", "bam")},
                                 "identical_outputs": all(norm(outs["bam"][f]) == norm(outs["sam"][f]) for f in outs["bam"])}
    print(json.dumps(out), flush=True)
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
