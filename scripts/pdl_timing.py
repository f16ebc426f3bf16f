"""bench.py against two builds of libabawaca_b200.so, run after run: the parent's (plain launches) and this tree's (programmatic dependent launch).

Each run is one `bench.py --gpus 1 --no-cpu-baseline` process with ABW_B200_LIB naming the library; the arms alternate (ABAB..., the first arm of a
round swapping every round) so that drift of the machine lands on both.  Per arm: ms_per_step of the resident step, e2e.ms_per_step,
kernel_time_over_step_time and the profiled per-kernel times (plain launches with CUDA events around each, bench.py's extra profiled step).  Before the
timed runs every arm runs once with --dump-outputs, and the .npy files of the two arms are compared bit for bit.  The card's name, power limit and SM
clocks are read at the start and at the end.

python scripts/pdl_timing.py --parent-lib PATH [--runs 5] [--steps 20] [--warmup 3] [--log FILE] [--json FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THIS_LIB = os.path.join(ROOT, "abawaca_b200", "libabawaca_b200.so")


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def bench(lib, args, extra=()):
    env = dict(os.environ, ABW_B200_LIB=lib)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(args.steps), "--warmup", str(args.warmup), "--no-cpu-baseline", *extra]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=tempfile.gettempdir())
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        raise SystemExit(f"bench.py failed with {lib}:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
    return json.loads(lines[-1])


def same_outputs(a, b):
    names = sorted(f for f in os.listdir(a) if f.endswith(".npy"))
    if not names or names != sorted(f for f in os.listdir(b) if f.endswith(".npy")):
        return False, names
    diff = []
    for f in names:
        x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
        if x.dtype != y.dtype or x.shape != y.shape or x.tobytes() != y.tobytes():
            diff.append(f)
    return not diff, {"files": names, "differing": diff}


def spread(v):
    return dict(median=round(statistics.median(v), 3), min=round(min(v), 3), max=round(max(v), 3), all=[round(x, 3) for x in v])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True, help="libabawaca_b200.so built from the parent commit")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--log", default=None)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    arms = {"parent": os.path.abspath(args.parent_lib), "pdl": THIS_LIB}
    res = {"gpu_start": gpu_info(), "runs_per_arm": args.runs, "steps": args.steps, "warmup": args.warmup, "libs": arms}
    print(json.dumps(res), flush=True)

    with tempfile.TemporaryDirectory(prefix="abw_pdl_") as tmp:
        for arm, lib in arms.items():
            bench(lib, args, ["--dump-outputs", os.path.join(tmp, arm)])
        same, detail = same_outputs(os.path.join(tmp, "parent"), os.path.join(tmp, "pdl"))
    res["outputs_identical"] = same
    res["outputs"] = detail
    print("outputs identical:", same, detail, flush=True)

    lines = {a: [] for a in arms}
    order = list(arms)
    for i in range(args.runs):
        for arm in (order if i % 2 == 0 else order[::-1]):
            d = bench(arms[arm], args)
            lines[arm].append(d)
            print(f"run {i} {arm}: ms_per_step {d['ms_per_step']}  e2e {d['e2e']['ms_per_step']}  kernel/step {d['kernel_time_over_step_time']}  "
                  f"launches {d['gpu_launches']}  sm {d['clocks'].get('sm_mhz')} MHz", flush=True)
    res["gpu_end"] = gpu_info()

    summary = {}
    for arm, ds in lines.items():
        kern = {}
        for d in ds:
            for k, v in d["kernels"].items():
                kern.setdefault(k, []).append(v["ms"])
        summary[arm] = {"ms_per_step": spread([d["ms_per_step"] for d in ds]), "e2e_ms_per_step": spread([d["e2e"]["ms_per_step"] for d in ds]),
                        "kernel_time_over_step_time": spread([d["kernel_time_over_step_time"] for d in ds]),
                        "profiled_kernel_ms": spread([sum(v["ms"] for v in d["kernels"].values()) for d in ds]),
                        "gpu_launches": sorted({d["gpu_launches"] for d in ds}), "sm_mhz": sorted({d["clocks"].get("sm_mhz") for d in ds}),
                        "kernels_median_ms": {k: round(statistics.median(v), 4) for k, v in kern.items()}}
    res["arms"] = summary
    p, q = summary["parent"]["ms_per_step"], summary["pdl"]["ms_per_step"]
    gain = p["median"] - q["median"]
    res["gain_ms_per_step"] = round(gain, 3)
    res["gain_exceeds_spread"] = bool(gain > max(p["max"] - p["min"], q["max"] - q["min"]))
    res["e2e_gain_ms_per_step"] = round(summary["parent"]["e2e_ms_per_step"]["median"] - summary["pdl"]["e2e_ms_per_step"]["median"], 3)
    top = sorted(summary["parent"]["kernels_median_ms"].items(), key=lambda kv: -kv[1])[:15]
    res["profiled_kernels_top"] = {k: {"parent": v, "pdl": summary["pdl"]["kernels_median_ms"].get(k)} for k, v in top}

    text = [f"gpu (start): {res['gpu_start']}", f"gpu (end):   {res['gpu_end']}",
            f"bench.py --gpus 1 --steps {args.steps} --warmup {args.warmup} --no-cpu-baseline, {args.runs} runs per arm, arms alternating",
            f"outputs of --dump-outputs identical bit for bit: {same} {detail}", "",
            "arm    | ms_per_step median (min-max) | e2e ms_per_step median (min-max) | kernel/step median | profiled kernel ms median | launches"]
    for arm, s in summary.items():
        m, e, k, pk = s["ms_per_step"], s["e2e_ms_per_step"], s["kernel_time_over_step_time"], s["profiled_kernel_ms"]
        text.append(f"{arm:6s} | {m['median']:.3f} ({m['min']:.3f}-{m['max']:.3f}) {m['all']} | {e['median']:.3f} ({e['min']:.3f}-{e['max']:.3f}) | "
                    f"{k['median']:.3f} | {pk['median']:.3f} | {s['gpu_launches']}")
    text.append(f"gain (parent - pdl), median ms_per_step: {res['gain_ms_per_step']}  exceeds both arms' max-min spread: {res['gain_exceeds_spread']}")
    text.append(f"e2e gain, median ms_per_step: {res['e2e_gain_ms_per_step']}")
    text.append("profiled per-kernel ms per step (plain launches), median over runs:")
    for k, v in res["profiled_kernels_top"].items():
        text.append(f"  {k:44s} parent {v['parent']:8.4f}  pdl {v['pdl'] if v['pdl'] is not None else float('nan'):8.4f}")
    print("\n".join(text), flush=True)
    for path, content in ((args.log, "\n".join(text) + "\n"), (args.json, json.dumps(res, indent=1))):
        if path:
            os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
            open(path, "w").write(content)


if __name__ == "__main__":
    main()
