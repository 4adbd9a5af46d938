"""Times the source-direction range queries and per-query AUC (SourceCatalogIndex.within / compatible / auc_per_query,
cfl_score_within and cfl_rank_counts_packed with CFL_PCD_SOURCE) at K = 3, d = 64, N = 2^20 sources, Q = 1024 target
queries, next to the forward CatalogIndex.within and the source rank(100) at the same shape.

    python tools/source_within_perf.py [--out FILE.jsonl] [--iters 10] [--profile DIR]

Both indexes are built from the same synthetic features through one set of random encoder weights (F = 64, tanh).
Radii: ~100 rows per query (each query's 100th distance from rank(100)) and ~10 000 rows per query (a quantile of 4096
sampled distances per query); compatible() at theta = the median 1000-row radius; auc_per_query with J = 8 random
positives per query, fused (tensor cores) and direct (CUDA cores).  Each timed call runs between device events after
two warm-up calls, the variants alternating call by call; the card name and power limit are read in the same run.
--profile DIR: a separate torch.profiler run (3 calls per variant) writes the per-kernel tables to DIR and adds the
kernel times per call to the result line.

The `large_kd` part times the shapes whose K*d-float source rows do not fit shared memory 128 at a time (K = 8,
d = 128, N = 2^16, Q = 256, random prototypes): the CUDA-core pcd_source count reads every row in place (VW = 0) and is
set against the forward CUDA-core count at the same K, d, N and Q -- the same pcd_direct arithmetic per pair, rows of d
floats staged in shared memory -- and the tensor-core count; the range query at ~100 rows per query on both routes,
whose rescore and fix kernels also read the rows in place, with per-kernel times from the profiler."""
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

CFG = dict(K=3, d=64, N=1 << 20, Q=1024, J=8)
F = 64


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def build(seed=0):
    from cfl.ranking import CatalogIndex, EncoderWeights, SourceCatalogIndex
    from oracle import cfl_oracle as O
    rng = np.random.default_rng(seed)
    K, d = CFG["K"], CFG["d"]
    t = lambda a: torch.as_tensor(np.asarray(a, np.float32)).cuda()        # noqa: E731
    w = EncoderWeights(V0=t(O.xavier_uniform(rng, F, d)), Vp=t(O.xavier_uniform(rng, F, K * d)), g0=t(np.ones(d)),
                       gp=t(np.ones(K * d)), b0=t(0.1 * rng.normal(size=d)), bp=t(0.1 * rng.normal(size=K * d)),
                       weight_norm=True, act="tanh")
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.relu(torch.randn(CFG["N"], F, device="cuda", generator=g))
    Xq = torch.relu(torch.randn(CFG["Q"], F, device="cuda", generator=g))
    src = SourceCatalogIndex.from_features(w, X)
    fwd = CatalogIndex.from_features(w, X)
    del X
    return src, fwd, Xq


def radius_for(nat, mode, query, catalog, rows):
    """Per query: the distance with about `rows` of N catalog rows below it (quantile of 4096 sampled rows)."""
    N = catalog.shape[0]
    samp = torch.randint(0, N, (query.shape[0], 4096), device="cuda")
    d = torch.cat([nat.pair_dist_rows(mode, query, catalog, samp[:, j:j + 32].contiguous()) for j in range(0, 4096, 32)], 1)
    return d.kthvalue(max(1, int(4096 * rows / N)), 1).values.contiguous()


def profile(fns, outdir, calls=3):
    from torch.profiler import ProfilerActivity, profile as prof
    os.makedirs(outdir, exist_ok=True)
    per = {}
    for v, f in fns.items():
        torch.cuda.synchronize()
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            for _ in range(calls):
                f()
                torch.cuda.synchronize()
        with open(os.path.join(outdir, f"source_within_{v}_kernels.txt"), "w") as fh:
            fh.write(p.key_averages().table(sort_by="cuda_time_total", row_limit=20))
        tot = {}
        for e in p.events():
            if str(e.device_type).endswith("CUDA") and "Memset" not in e.name and "Memcpy" not in e.name:
                n = e.name.split("(")[0].replace("void ", "")
                tot[n] = tot.get(n, 0.0) + e.time_range.elapsed_us() / 1000.0
        per[v] = {n: round(x / calls, 4) for n, x in sorted(tot.items(), key=lambda kv: -kv[1]) if x / calls >= 0.002}
    return per


def timed(f, iters=5):
    for _ in range(2):
        f()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        f()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return round(float(np.median(ms)), 4)


def large_kd(nat, profdir):
    K, d, N, Q = 8, 128, 1 << 16, 256
    g = torch.Generator(device="cuda").manual_seed(7)
    P = torch.randn(N, K, d, device="cuda", generator=g)
    Eq = P[torch.randint(0, N, (Q,), device="cuda", generator=g)].mean(1) + 0.5 * torch.randn(Q, d, device="cuda",
                                                                                              generator=g)
    Ef = torch.randn(N, d, device="cuda", generator=g)                    # forward: the same shapes, roles swapped
    Pf = torch.randn(Q, K, d, device="cuda", generator=g)
    mu = P.double().mean((0, 1)).float()
    img = nat.source_catalog_pack(P, mu)
    r = nat.score_topk_source(Eq, P, img, 100, mu=mu)[0][:, 99].contiguous()
    t1 = r[:, None].contiguous()
    tf = torch.full((Q, 1), float(r.median()), device="cuda")
    fns = {
        "count_source_cuda_cores_in_place": lambda: nat.rank_counts("pcd_source", Eq, P, t1),
        "count_forward_cuda_cores_staged": lambda: nat.rank_counts("pcd", Pf, Ef, tf),
        "count_source_tensor_cores": lambda: nat.rank_counts_packed(Eq, P, img, mu, t1, mode="pcd_source"),
        "within_source_tensor_cores": lambda: nat.score_within("pcd_source", Eq, P, r, image=img, mu=mu),
        "within_source_cuda_cores": lambda: nat.score_within("pcd_source", Eq, P, r),
    }
    res = dict(K=K, d=d, N=N, Q=Q, median_ms={v: timed(f) for v, f in fns.items()})
    if profdir:
        res["kernel_ms_per_call"] = profile({v: fns[v] for v in ("within_source_tensor_cores",
                                                                 "within_source_cuda_cores")}, profdir)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--profile", default=None, help="directory for a separate torch.profiler run")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("source_within_perf: needs a B200 (no CPU timing)")
    from cfl import _native as nat
    gpu, power = card()
    src, fwd, Xq = build()
    Q, N, J = CFG["Q"], CFG["N"], CFG["J"]
    Eq, Pq = src.project_queries(Xq), fwd.project_queries(Xq)
    r100 = src.rank(Xq, 100)[0][:, 99].contiguous()
    r10k = radius_for(nat, "pcd_source", Eq, src.P, 10_000)
    src.theta = float(radius_for(nat, "pcd_source", Eq, src.P, 1000).median())
    f100 = fwd.rank(Xq, 100)[0][:, 99].contiguous()
    rng = np.random.default_rng(1)
    pos = torch.as_tensor(np.stack([rng.choice(N, J, replace=False) for _ in range(Q)]), device="cuda")
    fns = {
        "source_within_100": lambda: src.within(Xq, r100),
        "source_within_10k": lambda: src.within(Xq, r10k),
        "source_compatible": lambda: src.compatible(Xq),
        "source_auc_fused": lambda: src.auc_per_query(Xq, pos),
        "source_auc_direct": lambda: src.auc_per_query(Xq, pos, method="direct"),
        "forward_within_100": lambda: fwd.within(Xq, f100),
        "source_rank_100": lambda: src.rank(Xq, 100),
    }
    rows = {}
    for v, f in fns.items():                                 # warm-up: module loads, workspaces
        for _ in range(2):
            out = f()
        if "within" in v or "compatible" in v:
            rows[v] = int(out[0][-1]) / Q
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
    _, st = nat.rank_counts_packed(Eq, src.P, src.image, src.mu, r100[:, None], want_stats=True, mode="pcd_source")
    res = dict(**CFG, gpu=gpu, power_limit_and_max_sm_clock=power,
               median_ms={v: round(float(np.median(x)), 4) for v, x in ms.items()},
               spread_ms={v: round(float(np.max(x) - np.min(x)), 4) for v, x in ms.items()},
               rows_per_query=rows, source_count_stats_r100=st)
    if args.profile:
        res["kernel_ms_per_call"] = profile(fns, args.profile)
    del src, fwd
    torch.cuda.empty_cache()
    res["large_kd"] = large_kd(nat, args.profile)
    print(json.dumps(res), flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
