"""Times the source direction of the monomer ranking (MonomerSourceCatalogIndex.rank, cfl_score_topk_monomer_source)
against the forward monomer ranking (MonomerCatalogIndex.rank) at the same shape: K = 4, d = 20, N = 2^20, Q = 1024,
k = 100 (the monomer configuration at a 1 M-row catalog).

    python tools/monomer_source_perf.py [--out FILE.jsonl] [--iters 20] [--profile DIR]

Both indexes are built from the same synthetic features through one set of random encoder weights (F = 128): the
forward catalog holds the targets' prototypes and its queries the sources' (a, gate); the source catalog holds the
sources' (a, gate) and its queries the targets' prototypes.  Each timed call is one rank() (query projection + the
four stages + merge) between device events; the two directions alternate call by call.  The card name and power limit
are read in the same run.  --profile DIR: a separate torch.profiler run (5 calls per direction) writes the per-kernel
tables to DIR and adds the kernel time of each stage (sample thresholds, filter, rescoring, redo) to the result line."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "compatibility-family-learning_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CFG = dict(K=4, d=20, N=1 << 20, Q=1024, k=100)
F = 128


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def build(seed=0):
    from cfl.ranking import EncoderWeights, MonomerCatalogIndex, MonomerSourceCatalogIndex
    from oracle import cfl_oracle as O
    rng = np.random.default_rng(seed)
    K, d = CFG["K"], CFG["d"]
    t = lambda a: torch.as_tensor(np.asarray(a, np.float32)).cuda()        # noqa: E731
    w = EncoderWeights(V0=t(O.xavier_uniform(rng, F, d)), Vp=t(O.xavier_uniform(rng, F, K * d)), g0=t(np.ones(d)),
                       gp=t(np.ones(K * d)), b0=t(0.1 * rng.normal(size=d)), bp=t(0.1 * rng.normal(size=K * d)),
                       weight_norm=True, act="tanh", Vg=t(O.xavier_uniform(rng, d, K)), gg=t(np.ones(K)))
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.relu(torch.randn(CFG["N"], F, device="cuda", generator=g))
    Xq = torch.relu(torch.randn(CFG["Q"], F, device="cuda", generator=g))
    src = MonomerSourceCatalogIndex.from_features(w, X)
    fwd = MonomerCatalogIndex.from_features(w, X)
    assert src.image is not None and fwd.image is not None
    del X
    return src, fwd, Xq


# kernels of each stage; the CUDA-core kernel and merge_plain_kernel run twice per call: sample, then redo
def stage_of(name, seen):
    if "score_monomer_src_kernel" in name or "score_monomer_kernel" in name:
        seen["exact"] += 1
        return "sample" if seen["exact"] == 1 else "redo"
    if "merge_plain_kernel" in name:
        seen["merge"] += 1
        return "sample" if seen["merge"] == 1 else "redo"
    if "mono_thresholds_kernel" in name:
        return "sample"
    if "prep_lb_kernel" in name or "score_lb_kernel" in name:
        return "filter"
    if "mono_rescore" in name:
        return "rescore"
    return "other"


def profile(fns, outdir, calls=5):
    from torch.profiler import ProfilerActivity, profile as prof
    os.makedirs(outdir, exist_ok=True)
    stages = {}
    for v, f in fns.items():
        torch.cuda.synchronize()
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            for _ in range(calls):
                f()
                torch.cuda.synchronize()
        with open(os.path.join(outdir, f"monomer_{v}_kernels.txt"), "w") as fh:
            fh.write(p.key_averages().table(sort_by="cuda_time_total", row_limit=25))
        evs = sorted((e for e in p.events() if str(e.device_type).endswith("CUDA") and "Memset" not in e.name
                      and "Memcpy" not in e.name), key=lambda e: e.time_range.start)
        # one call = the kernels between two projection launches; split the sequence by the rank() structure
        tot = {s: 0.0 for s in ("sample", "filter", "rescore", "redo", "other")}
        seen = {"exact": 0, "merge": 0}
        for e in evs:
            if "project" in e.name:                          # the query projection opens a new call
                seen = {"exact": 0, "merge": 0}
            tot[stage_of(e.name, seen)] += e.time_range.elapsed_us() / 1000.0
        stages[v] = {s: round(x / calls, 4) for s, x in tot.items()}
    return stages


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--profile", default=None, help="directory for a separate torch.profiler run")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("monomer_source_perf: needs a B200 (no CPU timing)")
    gpu, power = card()
    src, fwd, Xq = build()
    k = CFG["k"]
    fns = {"source": lambda: src.rank(Xq, k), "forward": lambda: fwd.rank(Xq, k)}
    for f in fns.values():                                   # warm-up: module loads, workspaces
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    ms = {v: [] for v in fns}
    for _ in range(args.iters):
        for v, f in fns.items():                             # alternating
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            b.synchronize()
            ms[v].append(a.elapsed_time(b))
    from cfl import _native as nat
    _, _, st = nat.score_topk_monomer_source(src.project_queries(Xq), src.a, src.gate, src.image, k, mu=src.mu,
                                             want_stats=True)
    K, d, N, Q = CFG["K"], CFG["d"], CFG["N"], CFG["Q"]
    res = dict(**CFG, gpu=gpu, power_limit_and_max_sm_clock=power,
               median_ms={v: float(np.median(x)) for v, x in ms.items()},
               min_ms={v: float(np.min(x)) for v, x in ms.items()},
               spread_ms={v: float(np.max(x) - np.min(x)) for v, x in ms.items()},
               gscores_per_s={v: Q * N / (float(np.median(x)) * 1e6) for v, x in ms.items()},
               source_stats=dict(zip(nat.SCORE_STAT_NAMES, st.tolist())),
               image_bytes_per_row=2 * ((K * (d + 1) + 15) // 16 * 16) + 8)
    if args.profile:
        res["stage_kernel_ms"] = profile(fns, args.profile)
    print(json.dumps(res), flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
