"""End-to-end step with the assembly in 2 bits per base (pipeline.packed_assembly, abw_pack_2bit) against the ASCII assembly (abw_pack_sequences).

The workload is bench.py's configs[1] stream (synth.CONFIGS["cfg2"], q6_reads=True), every sample sorted by (scaffold, position) as `samtools sort`
leaves a SAM file, with the reads as compact records (8 bytes per read) and as sorted records (about 2).  Each read format runs with the ASCII
assembly and with the 2-bit assembly: four arms.  Each arm runs bench.py's end-to-end step: pinned host buffers, every host-to-device copy enqueued
up front and waited for by ticket, feature build, the .lrn matrix back as integer thousandths while the split search (search_features) runs, the
window table back, one synchronize.  The arms alternate step by step after a warm-up; the host clock around a step that ends in a synchronize gives
its time.  The host encode time of each encoding is reported on its own (it is not part of the step).  A separate profiled step of each arm
(abw_profile_enable: CUDA events around every launch) gives the device time of the 2-bit decode kernels and of k_pack.

python scripts/twobit_timing.py [--steps 12] [--warmup 2] [--json FILE] [--dry-run]
(--dry-run: workload and encodings on the host only, with their byte counts; no GPU is used)
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
    """both read formats from the same coordinate-sorted stream, with the host time of each encoder"""
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
    reads, enc_ms = encode(mg, pipeline)
    t0 = time.perf_counter()
    pa = pipeline.packed_assembly(mg.seq, mg.offsets)
    enc_ms["2bit_assembly"] = 1000.0 * (time.perf_counter() - t0)
    nbases = int(mg.seq.size)
    asm_bytes = {"ascii": nbases + mg.offsets.nbytes, "2bit": pa.nbytes + pa.byte_off.nbytes + pa.lengths.nbytes}
    order = [(r, a) for r in ("compact", "sorted") for a in ("ascii", "2bit")]
    name = lambda r, a: r + "/" + a                        # noqa: E731
    res = dict(workload="configs[1] (synth cfg2, q6_reads), every sample sorted by (scaffold, position)", scaffolds=mg.nscaf, samples=len(mg.reads),
               bases=nbases, runs=int(pa.runs.size), runs_N=int((pa.runs["kind"] == 0).sum()), generate_s=round(gen_s, 1),
               host_encode_ms={k: round(v, 1) for k, v in enc_ms.items()},
               assembly_bytes_per_step=asm_bytes,
               h2d_bytes_per_step={name(r, a): asm_bytes[a] + int(sum(s.nbytes for s in reads[r])) for r, a in order})
    print(json.dumps(res), flush=True)
    if args.dry_run:
        return
    import torch
    from abawaca_b200 import capi
    res["gpu"] = gpu_info()
    ctx = capi.Context(0)
    for v in reads.values():
        pin(torch, v)
    h_seq = torch.from_numpy(mg.seq).pin_memory()
    pinned = []
    for attr in ("codes", "runs"):
        a = getattr(pa, attr)
        t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).pin_memory()
        pinned.append(t)
        setattr(pa, attr, t.numpy().view(a.dtype))
    lengths = np.diff(mg.offsets.astype(np.int64)).astype(np.uint64)
    masks = mg.scg_masks()
    bufs = {name(r, a): {} for r, a in order}
    state = {}

    def step(r, a, keep=False):
        seq = h_seq.numpy() if a == "ascii" else pa
        fb = pipeline.build_features(ctx, seq, mg.offsets, reads[r], this_sample=0, overlap_h2d=True)
        if "h_k16" not in state:
            state["h_k16"] = torch.empty(fb.nseg * fb.nk, dtype=torch.int16).pin_memory()
            state["h_k32"] = torch.empty(fb.nseg * (fb.ncols - fb.nk), dtype=torch.int32).pin_memory()
            state["h_seg"] = [torch.empty(fb.nseg, dtype=torch.int32).pin_memory()] + [torch.empty(fb.nseg, dtype=torch.int64).pin_memory() for _ in range(3)]
        fb.segments_async(state["h_seg"][0].numpy().view(np.uint32), *[t.numpy().view(np.uint64) for t in state["h_seg"][1:]])
        fb.rows_milli(out16=state["h_k16"].numpy().view(np.uint16), out32=state["h_k32"].numpy().view(np.uint32), wait=False)
        res_, kept = pipeline.search_features(ctx, fb, lengths, masks, buffers=bufs[name(r, a)])
        ctx.synchronize()
        if fb.milli_inexact():
            raise SystemExit("a feature value is not a multiple of 0.001")
        out = None
        if keep:
            out = dict(k16=state["h_k16"].numpy().copy(), k32=state["h_k32"].numpy().copy(), seg=[t.numpy().copy() for t in state["h_seg"]],
                       bins=res_.scaf2cluster.copy(), kept=np.array(kept), nclusters=len(res_.recs))
        fb.close()
        return out

    outs = {}
    for i in range(args.warmup):
        for r, a in order:
            o = step(r, a, keep=(i == 0))
            if o is not None:
                outs[name(r, a)] = o
    ms = {name(r, a): [] for r, a in order}
    for i in range(args.steps):
        for r, a in (order if i % 2 == 0 else order[::-1]):
            t0 = time.perf_counter()
            step(r, a)
            ms[name(r, a)].append(1000.0 * (time.perf_counter() - t0))
    ident = {}
    for r in ("compact", "sorted"):
        x, y = outs[r + "/ascii"], outs[r + "/2bit"]
        ident[r] = dict(rows=bool(np.array_equal(x["k16"], y["k16"]) and np.array_equal(x["k32"], y["k32"]) and all(np.array_equal(p, q) for p, q in zip(x["seg"], y["seg"]))),
                        bins=bool(np.array_equal(x["bins"], y["bins"]) and np.array_equal(x["kept"], y["kept"]) and x["nclusters"] == y["nclusters"]))
    res["identical_ascii_vs_2bit"] = ident
    res["e2e_ms_per_step"] = {k: dict(median=round(statistics.median(v), 2), min=round(min(v), 2), max=round(max(v), 2), stdev=round(statistics.stdev(v), 2),
                                      steps=len(v), all=[round(x, 2) for x in v]) for k, v in ms.items()}
    res["e2e_gain_ms"] = {r: round(res["e2e_ms_per_step"][r + "/ascii"]["median"] - res["e2e_ms_per_step"][r + "/2bit"]["median"], 2) for r in ("compact", "sorted")}
    # profiled pass (launches serialised): one step of each arm
    prof = {}
    for r, a in order:
        ctx.profile(True)
        step(r, a)
        prof[name(r, a)] = ctx.profile_report()
        ctx.profile(False)
    dec = {k: v for k, v in prof["sorted/2bit"].items() if k.startswith("k_2bit_")}
    dec_ms = sum(v[1] for v in dec.values())
    dec_bytes = nbases // 4 + 16 * int(pa.runs.size) + nbases // 2        # 0.25 B/base and 16 B per run in, 0.5 B/base (packed, valid, nmask) out
    pack = prof["sorted/ascii"].get("k_pack", (0, 0.0))
    pack_bytes = nbases + nbases // 2                                    # 1 B/base in, 0.5 B/base out
    rate = lambda b, t: dict(algorithmic_bytes=int(b), GBps=round(b / t / 1e6, 1), frac_of_measured_peak=round(b / t / 1e6 / PEAK_MEASURED, 4),   # noqa: E731
                             frac_of_datasheet=round(b / t / 1e6 / PEAK_DATASHEET, 4)) if t > 0 else {}
    res["decode_2bit"] = dict(kernels={k: dict(launches=v[0], ms=round(v[1], 4)) for k, v in dec.items()}, total_ms=round(dec_ms, 4), **rate(dec_bytes, dec_ms))
    res["k_pack"] = dict(launches=pack[0], ms=round(pack[1], 4), **rate(pack_bytes, pack[1]))
    res["profiled_step_kernels_ms"] = {k: {kk: round(v[1], 4) for kk, v in sorted(p.items(), key=lambda kv: -kv[1][1])[:12]} for k, p in prof.items()}
    ctx.close()
    print(json.dumps(res), flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        json.dump(res, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
