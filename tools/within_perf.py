"""Timing of CatalogIndex.within() at the C3 shape (1024 queries x 2^20 catalog rows, K = 3, d = 64).

    python tools/within_perf.py [--out FILE] [--iters N]

Prints one JSON line per measurement (and writes them to --out): the card and its power limit; ms per within() call
(host clock around the call and a device synchronise; the call reads the result size back once) with radii chosen for
~100 and ~10 000 rows per query; the kernel time of each phase from a separate torch.profiler run -- count
(rank_count_umma_kernel + rank_fix_kernel, J = 1), emit (within_emit_umma_kernel + within_fix_kernel), rescore
(within_rescore_kernel), finish (within_finish_kernel); auc_per_query (J = 1) and rank(k = 100) on the same index; and
whether the tensor-core route's result equals the CUDA-core route's.  The catalog (256 MB of embeddings, 2x that of
image) is larger than the L2, so every pass reads it from HBM."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "compatibility-family-learning_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from cfl import _native as nat                      # noqa: E402
from cfl.ranking import CatalogIndex, EncoderWeights  # noqa: E402

PHASES = (("count", ("rank_count_umma_kernel", "rank_fix_kernel")),
          ("emit", ("within_emit_umma_kernel", "within_fix_kernel", "within_emit_kernel", "within_reset_flagged")),
          ("rescore", ("within_rescore_kernel",)),
          ("finish", ("within_finish_kernel",)))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                           # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return dict(what="card", device=name, nvidia_smi=q)


def build_index(N=1 << 20, Q=1024, K=3, d=64, F=64, seed=633):
    rng = np.random.default_rng(seed)
    def xavier(a, b):
        return torch.as_tensor(((rng.uniform(size=(a, b)) * 2 - 1) * (6 / (a + b)) ** 0.5).astype(np.float32)).cuda()
    w = EncoderWeights(V0=xavier(F, d), Vp=xavier(F, K * d), g0=torch.ones(d).cuda(), gp=torch.ones(K * d).cuda(),
                       b0=torch.zeros(d).cuda(), bp=torch.zeros(K * d).cuda())
    X = torch.relu(torch.randn(N, F, generator=torch.Generator().manual_seed(seed))).cuda()
    return CatalogIndex.from_features(w, X), X[:Q].contiguous()


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def phase_ms(fn, iters):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k, _ in PHASES}
    other = 0.0
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        hit = [k for k, names in PHASES if any(n in ev.key for n in names)]
        if hit:
            out[hit[0]] += t / 1e3 / iters
        else:
            other += t / 1e3 / iters
    out["other_kernels_and_copies"] = other
    return {k: round(v, 3) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    lines = []

    def emit(rec):
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    emit(card())
    index, xq = build_index()
    Pq = index.project_queries(xq)
    tv, _ = index.rank(xq, 101)
    samp = torch.randint(0, index.E.shape[0], (Pq.shape[0], 4096), device="cuda")
    sd = torch.cat([nat.pair_dist_rows("pcd", Pq, index.E, samp[:, i:i + 32].contiguous()) for i in range(0, 4096, 32)], 1)
    radii = {"~100": tv[:, 100].contiguous(),
             "~10000": torch.quantile(sd, 10000 / index.E.shape[0], dim=1).float().contiguous()}
    for name, r in radii.items():
        off, idx, val, st = nat.score_within("pcd", Pq, index.E, r, image=index.image, mu=index.mu, want_stats=True)
        n = (off[1:] - off[:-1]).double()
        core = nat.score_within("pcd", Pq, index.E, r)
        same = all(torch.equal(x, y) for x, y in zip((off, idx, val), core))
        med, best = timed(lambda: index.within(xq, r), a.iters)
        cnt_med, _ = timed(lambda: nat.within_counts("pcd", Pq, index.E, r, image=index.image, mu=index.mu), a.iters)
        ph = phase_ms(lambda: nat.score_within("pcd", Pq, index.E, r, image=index.image, mu=index.mu), a.iters)
        emit(dict(what="within", radius=name, Q=Pq.shape[0], N=index.E.shape[0], K=3, d=64,
                  rows_per_query_mean=round(float(n.mean()), 1), rows_min=int(n.min()), rows_max=int(n.max()),
                  total_rows=int(off[-1]), ms_within_call_median=round(med, 3), ms_within_call_min=round(best, 3),
                  ms_count_call_median=round(cnt_med, 3), kernel_ms_per_call=ph, stats=st,
                  equals_cuda_core_route=bool(same)))
    pos = torch.randint(0, index.E.shape[0], (Pq.shape[0], 1))
    med, _ = timed(lambda: index.auc_per_query(xq, pos), a.iters)
    emit(dict(what="auc_per_query", J=1, ms_call_median=round(med, 3)))
    med, _ = timed(lambda: index.rank(xq, 100), a.iters)
    emit(dict(what="rank", k=100, ms_call_median=round(med, 3)))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            for rec in lines:
                fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
