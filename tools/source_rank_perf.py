"""Times the source-direction ranking (SourceCatalogIndex.rank, cfl_score_topk_source) at the C3 and C4 shapes against the
forward ranking of the same shape (CatalogIndex.rank) and against the forward path under CFL_SCORE_NO_LB=1, which runs
the same exact-filter algorithm in the other direction.

    python tools/source_rank_perf.py [--out FILE.jsonl] [--iters 10] [--profile DIR]

Both indexes are built from the same synthetic features through one set of random encoder weights (F = 128), so the
queries lie where the catalog lies.  Each timed call is one rank() (query projection + scoring + merge) between device
events; the three variants are interleaved call by call.  The card name and power limit are read in the same run.
--profile DIR: a separate torch.profiler run (3 calls of each variant) writes the per-kernel table to DIR."""
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

CONFIGS = {"C3": dict(K=3, d=64, N=1 << 20, Q=1024, k=100), "C4": dict(K=4, d=20, N=2_000_000, Q=1024, k=100)}
F = 128


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def build(cfg, seed=0):
    from cfl.ranking import CatalogIndex, EncoderWeights, SourceCatalogIndex
    from oracle import cfl_oracle as O
    rng = np.random.default_rng(seed)
    K, d = cfg["K"], cfg["d"]
    t = lambda a: torch.as_tensor(np.asarray(a, np.float32)).cuda()        # noqa: E731
    w = EncoderWeights(V0=t(O.xavier_uniform(rng, F, d)), Vp=t(O.xavier_uniform(rng, F, K * d)), g0=t(np.ones(d)),
                       gp=t(np.ones(K * d)), b0=t(0.1 * rng.normal(size=d)), bp=t(0.1 * rng.normal(size=K * d)),
                       weight_norm=True, act="tanh")
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.relu(torch.randn(cfg["N"], F, device="cuda", generator=g))
    Xq = torch.relu(torch.randn(cfg["Q"], F, device="cuda", generator=g))
    src = SourceCatalogIndex.from_features(w, X)
    fwd = CatalogIndex.from_features(w, X)
    del X
    return src, fwd, Xq


def variants(src, fwd, Xq, k):
    def no_lb():
        os.environ["CFL_SCORE_NO_LB"] = "1"
        try:
            return fwd.rank(Xq, k)
        finally:
            del os.environ["CFL_SCORE_NO_LB"]
    return {"source": lambda: src.rank(Xq, k), "forward": lambda: fwd.rank(Xq, k), "forward_no_lb": no_lb}


def time_config(name, cfg, iters):
    src, fwd, Xq = build(cfg)
    fns = variants(src, fwd, Xq, cfg["k"])
    for f in fns.values():                                  # warm-up: module loads, workspaces, every shape
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    ms = {v: [] for v in fns}
    for _ in range(iters):
        for v, f in fns.items():                            # interleaved
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            b.synchronize()
            ms[v].append(a.elapsed_time(b))
    # the arithmetic of the two directions (bytes of the catalog image read per query tile, flops per pair)
    K, d, N = cfg["K"], cfg["d"], cfg["N"]
    dpad = (d + 7) // 8 * 8
    out = dict(config=name, **cfg, median_ms={v: float(np.median(x)) for v, x in ms.items()},
               min_ms={v: float(np.min(x)) for v, x in ms.items()},
               spread_ms={v: float(np.max(x) - np.min(x)) for v, x in ms.items()},
               catalog_image_bytes={"source": N * (8 * dpad * K + 4 * (K + K * (K + 1) // 2)),
                                    "forward_exact": N * (8 * dpad + 4)},
               gram_flops_per_pair=2 * K * d * 3)
    return out, fns


def profile(fns, outdir, name):
    from torch.profiler import ProfilerActivity, profile as prof
    os.makedirs(outdir, exist_ok=True)
    for v, f in fns.items():
        torch.cuda.synchronize()
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            for _ in range(3):
                f()
            torch.cuda.synchronize()
        table = p.key_averages().table(sort_by="cuda_time_total", row_limit=20)
        with open(os.path.join(outdir, f"{name}_{v}_kernels.txt"), "w") as fh:
            fh.write(table)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--configs", default="C3,C4")
    ap.add_argument("--profile", default=None, help="directory for a separate torch.profiler run")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("source_rank_perf: needs a B200 (no CPU timing)")
    gpu, power = card()
    lines = []
    for name in args.configs.split(","):
        res, fns = time_config(name, CONFIGS[name], args.iters)
        res.update(gpu=gpu, power_limit=power)
        lines.append(res)
        print(json.dumps(res), flush=True)
        if args.profile:
            profile(fns, args.profile, name)
        del fns
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
