"""End-to-end step with coordinate-sorted read records (ABW_READS_SORTED) against compact records (ABW_READS_COMPACT).

The workload is bench.py's configs[1] stream (synth.CONFIGS["cfg2"], q6_reads=True), every sample sorted by (scaffold, position) as `samtools sort`
leaves a SAM file.  Two arms are built from that one sorted stream: pipeline.compact_reads (8 bytes per read) and pipeline.sorted_reads (about 2).
Each arm runs bench.py's end-to-end step: pinned host buffers, every host-to-device copy enqueued up front and waited for by ticket, feature build,
the .lrn matrix back as integer thousandths while the split search (search_features) runs, the window table back, one synchronize.  The arms
alternate step by step after a warm-up; the host clock around a step that ends in a synchronize gives its time.  The host encode time of each arm
is reported on its own (it is not part of the step).  A separate profiled step of each arm (abw_profile_enable: CUDA events around every launch)
gives the decode kernels' device time; the run-start scans of the decode are the difference in k_scan_onepass time between the two arms.

python scripts/sorted_reads_timing.py [--steps 12] [--warmup 2] [--json FILE] [--dry-run]
(--dry-run: workload and both encodings on the host only, with their byte counts; no GPU is used)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PEAK_MEASURED, PEAK_DATASHEET = 6459.6, 7700.0          # GB/s: DESIGN.md section 5, and NVIDIA's HGX B200 data sheet for one GPU


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def encode(mg, pipeline):
    """both arms from the same coordinate-sorted stream, with the host time of each encoder"""
    arms, enc_ms = {"compact": [], "sorted": []}, {"compact": 0.0, "sorted": 0.0}
    for r in mg.reads:
        r = r[np.lexsort((r["pos0"], r["scaf"]))]
        for name, fn in (("compact", pipeline.compact_reads), ("sorted", pipeline.sorted_reads)):
            t0 = time.perf_counter()
            arms[name].append(fn(r, mg.nscaf))
            enc_ms[name] += 1000.0 * (time.perf_counter() - t0)
    return arms, enc_ms


def pin(torch, samples):
    """the host arrays of every sample in pinned memory (the tensors are kept on the sample)"""
    for s in samples:
        s._pinned = []
        for attr in ("recs", "len16", "runs", "exc"):
            a = getattr(s, attr)
            if a is None:
                continue
            t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).pin_memory()
            s._pinned.append(t)
            setattr(s, attr, t.numpy().view(a.dtype))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--json", default=None)
    ap.add_argument("--dry-run", action="store_true")
    args = ap.parse_args()
    from abawaca_b200 import pipeline, synth
    t0 = time.perf_counter()
    mg = synth.make_metagenome(**synth.CONFIGS["cfg2"], q6_reads=True)
    gen_s = time.perf_counter() - t0
    arms, enc_ms = encode(mg, pipeline)
    nreads = sum(s.n for s in arms["sorted"])
    nruns = sum(s.nruns for s in arms["sorted"])
    nexc = sum(s.nexc for s in arms["sorted"])
    fixed = int(mg.seq.size) + mg.offsets.nbytes         # the ASCII assembly and the scaffold offsets, the same in both arms
    res = dict(workload="configs[1] (synth cfg2, q6_reads), every sample sorted by (scaffold, position)", scaffolds=mg.nscaf, samples=len(mg.reads),
               reads_after_filter=nreads, runs=nruns, escapes=nexc, generate_s=round(gen_s, 1),
               host_encode_ms={k: round(v, 1) for k, v in enc_ms.items()},
               read_bytes_per_step={k: int(sum(s.nbytes for s in v)) for k, v in arms.items()},
               h2d_bytes_per_step={k: fixed + int(sum(s.nbytes for s in v)) for k, v in arms.items()})
    res["h2d_ratio_sorted_over_compact"] = round(res["h2d_bytes_per_step"]["sorted"] / res["h2d_bytes_per_step"]["compact"], 4)
    print(json.dumps(res), flush=True)
    if args.dry_run:
        return
    import torch
    from abawaca_b200 import capi
    res["gpu"] = gpu_info()
    ctx = capi.Context(0)
    for v in arms.values():
        pin(torch, v)
    h_seq = torch.from_numpy(mg.seq).pin_memory()
    lengths = np.diff(mg.offsets.astype(np.int64)).astype(np.uint64)
    masks = mg.scg_masks()
    bufs = {name: {} for name in arms}
    state = {}

    def step(name, keep=False):
        fb = pipeline.build_features(ctx, h_seq.numpy(), mg.offsets, arms[name], this_sample=0, overlap_h2d=True)
        if "h_k16" not in state:
            state["h_k16"] = torch.empty(fb.nseg * fb.nk, dtype=torch.int16).pin_memory()
            state["h_k32"] = torch.empty(fb.nseg * (fb.ncols - fb.nk), dtype=torch.int32).pin_memory()
            state["h_seg"] = [torch.empty(fb.nseg, dtype=torch.int32).pin_memory()] + [torch.empty(fb.nseg, dtype=torch.int64).pin_memory() for _ in range(3)]
        fb.segments_async(state["h_seg"][0].numpy().view(np.uint32), *[t.numpy().view(np.uint64) for t in state["h_seg"][1:]])
        fb.rows_milli(out16=state["h_k16"].numpy().view(np.uint16), out32=state["h_k32"].numpy().view(np.uint32), wait=False)
        r, kept = pipeline.search_features(ctx, fb, lengths, masks, buffers=bufs[name])
        ctx.synchronize()
        if fb.milli_inexact():
            raise SystemExit("a feature value is not a multiple of 0.001")
        out = None
        if keep:
            out = dict(k16=state["h_k16"].numpy().copy(), k32=state["h_k32"].numpy().copy(), bins=r.scaf2cluster.copy(), kept=np.array(kept), nclusters=len(r.recs))
        fb.close()
        return out

    order = ["compact", "sorted"]
    outs = {}
    for i in range(args.warmup):
        for name in order:
            o = step(name, keep=(i == 0))
            if o is not None:
                outs[name] = o
    ms = {name: [] for name in order}
    for i in range(args.steps):
        for name in (order if i % 2 == 0 else order[::-1]):
            t0 = time.perf_counter()
            step(name)
            ms[name].append(1000.0 * (time.perf_counter() - t0))
    a, b = outs["compact"], outs["sorted"]
    res["rows_identical"] = bool(np.array_equal(a["k16"], b["k16"]) and np.array_equal(a["k32"], b["k32"]))
    res["bins_identical"] = bool(np.array_equal(a["bins"], b["bins"]) and np.array_equal(a["kept"], b["kept"]) and a["nclusters"] == b["nclusters"])
    res["e2e_ms_per_step"] = {name: dict(median=round(statistics.median(v), 2), min=round(min(v), 2), max=round(max(v), 2), stdev=round(statistics.stdev(v), 2),
                                         steps=len(v), all=[round(x, 2) for x in v]) for name, v in ms.items()}
    res["e2e_gain_ms"] = round(res["e2e_ms_per_step"]["compact"]["median"] - res["e2e_ms_per_step"]["sorted"]["median"], 2)
    # profiled pass (launches serialised): one step of each arm
    prof = {}
    for name in order:
        ctx.profile(True)
        step(name)
        prof[name] = ctx.profile_report()
        ctx.profile(False)
    dec = {k: v for k, v in prof["sorted"].items() if k.startswith("k_sorted_")}
    scan_ms = prof["sorted"].get("k_scan_onepass<Tin>", (0, 0.0))[1] - prof["compact"].get("k_scan_onepass<Tin>", (0, 0.0))[1]
    dec_ms = sum(v[1] for v in dec.values()) + max(scan_ms, 0.0)
    alg_bytes = 2 * nreads + 8 * nreads + 8 * nruns + 4 * nexc
    res["decode"] = dict(kernels={k: dict(launches=v[0], ms=round(v[1], 4)) for k, v in dec.items()}, run_start_scans_ms=round(scan_ms, 4),
                         total_ms=round(dec_ms, 4), algorithmic_bytes=int(alg_bytes), GBps=round(alg_bytes / dec_ms / 1e6, 1),
                         frac_of_measured_peak=round(alg_bytes / dec_ms / 1e6 / PEAK_MEASURED, 4), frac_of_datasheet=round(alg_bytes / dec_ms / 1e6 / PEAK_DATASHEET, 4))
    res["profiled_step_kernels_ms"] = {name: {k: round(v[1], 4) for k, v in sorted(p.items(), key=lambda kv: -kv[1][1])[:12]} for name, p in prof.items()}
    ctx.close()
    print(json.dumps(res), flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        json.dump(res, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
