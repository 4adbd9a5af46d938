"""Exact rescoring of the lower-bound survivors (rescore_merge_kernel) on the bench.py workload.

    python tools/rescore_perf.py [OUT_DIR] [--steps 60]

Builds the C3 index exactly as bench.py does (same seeds, weights and catalog projection) and runs CatalogIndex.rank:
one step under torch.profiler with CUDA activities (per-kernel times written to OUT_DIR/rescore_kernels.json), then
--steps steps timed with CUDA events without the profiler.  Prints the card, its power limit and the bytes the rescore
has to gather (survivors x 4d + kk x 4d per query, from rank_local_stats), so that the kernel time gives an achieved
GB/s.  Needs a GPU; there is no fallback."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "compatibility-family-learning_b200"))
import bench  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return name, r.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return name, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?", default="rescore_perf_out")
    ap.add_argument("--steps", type=int, default=60)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rescore_perf needs a GPU")
    os.makedirs(args.out, exist_ok=True)
    bench._ensure_library()
    from cfl import _native as nat
    from cfl.ranking import CatalogIndex

    dev = torch.device("cuda", 0)
    w = bench.synth_weights(dev)
    E = torch.empty(bench.N_PER_GPU, bench.D, device=dev)
    chunk = 1 << 18
    for lo in range(0, bench.N_PER_GPU, chunk):
        hi = min(bench.N_PER_GPU, lo + chunk)
        xb = bench.synth_features(hi - lo, dev, bench.SEED + 1 + lo // chunk)
        E[lo:hi] = nat.project_fwd(xb, w.V0, w.g0, w.b0, True, w.in_scale, None)[0]
        del xb
    index = CatalogIndex(w, E)
    xq = bench.synth_features(bench.Q, dev, bench.SEED + 7)
    for _ in range(5):
        index.rank(xq, bench.TOPK)
    torch.cuda.synchronize()

    # per-kernel times of one step (profiled in a run of its own: tracing slows the host, not the kernels)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        index.rank(xq, bench.TOPK)
        torch.cuda.synchronize()
    kernels = [{"name": e.name, "us": e.device_time} for e in prof.events()
               if e.device_type == torch.autograd.DeviceType.CUDA and e.device_time > 0]
    with open(os.path.join(args.out, "rescore_kernels.json"), "w") as fh:
        json.dump(kernels, fh, indent=1)
    rescore_us = [k["us"] for k in kernels if "rescore_merge_kernel" in k["name"]]

    # step time with CUDA events, profiler off
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        index.rank(xq, bench.TOPK)
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / args.steps

    filt = index.rank_local_stats(xq, bench.TOPK)[2]
    kk = bench.TOPK + 28
    gather_bytes = 4 * bench.D * (int(filt["survivors"]) + kk * bench.Q)
    first = rescore_us[0] if rescore_us else float("nan")
    name, power = card()
    res = {"card": name, "power_limit,max_sm_clock": power, "step_ms": step_ms, "steps": args.steps,
           "rescore_us": rescore_us, "survivors": int(filt["survivors"]), "queries": bench.Q, "d": bench.D,
           "gather_bytes": gather_bytes, "achieved_gbs": gather_bytes / (first * 1e-6) / 1e9,
           "datasheet_hbm_gbs": 7700.0, "filter": filt}
    print(json.dumps(res))
    with open(os.path.join(args.out, "rescore_perf.json"), "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
