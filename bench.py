#!/usr/bin/env python
"""bench.py -- the CFL all-pairs compatibility-scoring hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], "Amazon dyadic co-purchase latents", SURVEY 8d C3):
F=1024 GoogLeNet-pool5-like features, FCPCD encoder K=3 prototypes, d=64, a 1M-item catalog
PER GPU (weak scaling: rank r holds catalog rows [r*1M,(r+1)*1M)), Q=1024 queries per step,
top-100.  One step = project the query batch onto its K prototypes (stage 1) -> soft-min
score against every catalog embedding + running top-k (stage 2) -> [N>1: NCCL all-gather of
the per-rank lists + merge kernel].  metric = query x candidate scores / second, whole job.

Synthetic data (seed 633 = reference default, cfl/utils.py:89), random-init Xavier weights.
The catalog (256 MB of embeddings per GPU) is larger than the 126 MB L2, so every step
streams it from HBM/L2 afresh (no explicit L2 flush needed; stated in config).

Besides the headline line (C3, weak scaling) the same JSON line carries, measured in the same run:
  "c5"       BASELINE configs[4]: 10 M catalog rows in TOTAL (strong scaling: 10 M / N rows per rank), K = 4,
             d in {64, 128}, Q = 2048 queries per step, embeddings generated directly (SURVEY 8d C5);
  "c4"       the ranking shape of BASELINE configs[3]: K = 4, d = 20, 2 M target rows in total (strong scaling), Q = 1024;
  "small_q"  Q = 16 queries against the C3 catalog: the HBM-bound regime (catalog GB/s against the measured copy peak);
  "filter"   survivors per query of the full filter pass and the queries that spilled / were redone (a regression to
             the slow paths shows up here);
  "per_rank" kernel_ms and survivors of every rank (stragglers);
  "auc"      per-query all-candidate AUC (J = 8 positives per query against the whole C3 catalog) with the rank counts
             taken in the tensor-core scoring kernel's epilogue, beside the CUDA-core route it must equal (N = 1 only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "compatibility-family-learning_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)
sys.dont_write_bytecode = True     # the tree may be read-only: the benchmark writes nothing into it

import numpy as np  # noqa: E402
import torch  # noqa: E402

F, K, D, N_PER_GPU, Q, TOPK = 1024, 3, 64, 1_000_000, 1024, 100
DATA_NORM = 31.9098            # experiments/dyadic/run.sh:15
SEED = 633
PASS_C_DRAM_BYTES = 145.0e6    # dram__bytes_read + write of score_lb_kernel<3> on this workload (profiles/r2_02_pass_c.md)
WORKLOAD = "C3 dyadic all-pairs: F=1024 K=3 d=64, 1M-item catalog per GPU, Q=1024 queries/step, top-100"


def config_dict(world):
    """The workload description both arms print (identical keys and values, so that the driver sees one config)."""
    return {"workload": WORKLOAD, "F": F, "K": K, "d": D, "catalog_per_gpu": N_PER_GPU,
            "catalog_total": N_PER_GPU * world, "queries_per_step": Q, "topk": TOPK,
            "l2": "catalog plane 128 MB/GPU (fp16) re-read per query tile from the 126 MB L2, first touch from HBM every "
                  "step; the exact planes (512 MB) and the rescoring rows stream from HBM: no flush needed",
            "sharding": "catalog rows by rank, queries replicated, NCCL all-gather + merge kernel"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm=j["hbm_gbs"], bf16=j["bf16_tflops"], bf16_sus=j["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sus=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q_ = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
          "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
          "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q_}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------
def synth_weights(device):
    """FCPCD weights: Xavier-uniform V, g=1, b=0 (cfl/layers.py:47-76 initialisers)."""
    from cfl.ranking import EncoderWeights
    g = torch.Generator(device="cpu").manual_seed(SEED)
    lim0, limp = (6.0 / (F + D)) ** 0.5, (6.0 / (F + K * D)) ** 0.5
    V0 = (torch.rand(F, D, generator=g) * 2 - 1) * lim0
    Vp = (torch.rand(F, K * D, generator=g) * 2 - 1) * limp
    return EncoderWeights(V0=V0.to(device), Vp=Vp.to(device), g0=torch.ones(D, device=device),
                          gp=torch.ones(K * D, device=device), b0=torch.zeros(D, device=device),
                          bp=torch.zeros(K * D, device=device), weight_norm=True, in_scale=1.0 / DATA_NORM)


def synth_features(n, device, seed):
    """relu(N(0,1))*10, GoogLeNet pool5-like (SURVEY 8d C3), generated on the device in chunks."""
    g = torch.Generator(device=device).manual_seed(seed)
    out = torch.empty(n, F, dtype=torch.float32, device=device)
    for lo in range(0, n, 1 << 17):
        hi = min(n, lo + (1 << 17))
        out[lo:hi] = torch.randn(hi - lo, F, generator=g, device=device).clamp_(min=0).mul_(10.0)
    return out


def c5_line(d, world, rank, device, steps=8, K5=4, Q5=2048, N5=10_000_000, label="C5"):
    """C5 (SURVEY 8d): N = 10 M rows in total, e ~ N(0,1)^d, p_k = e_anchor + 0.5 N(0,1), K = 4, Q = 2048, top-100.
    Strong scaling: rank r holds rows [r N/R, (r+1) N/R).  Scoring call only (the embeddings ARE the input).
    Also used for the C4 ranking shape (K = 4, d = 20, 2 M target rows in total, Q = 1024: BASELINE configs[3] /
    experiments/polyvore/run.sh -- its embeddings generated directly, the F = 2048 projection is stage 1's job)."""
    from cfl import _native as nat
    lo, hi = N5 * rank // world, N5 * (rank + 1) // world
    g = torch.Generator(device=device).manual_seed(SEED + 50 + d + 1000 * rank)
    E = torch.empty(hi - lo, d, dtype=torch.float32, device=device)
    for a in range(0, hi - lo, 1 << 20):
        b = min(hi - lo, a + (1 << 20))
        E[a:b] = torch.randn(b - a, d, generator=g, device=device)
    gq = torch.Generator(device=device).manual_seed(SEED + 51 + d)            # same queries on every rank
    anchors = torch.randn(Q5, d, generator=gq, device=device)
    Pq = anchors[:, None, :] + 0.5 * torch.randn(Q5, K5, d, generator=gq, device=device)
    s_ = E.sum(0, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(s_)
    mu = (s_ / N5).float()
    img = nat.catalog_pack(E, K5, mu)

    def step():
        tv, ti = nat.score_topk(Pq, E, TOPK, mu=mu, idx_base=lo, image=img)
        if world > 1:
            from cfl.ranking import _gather_merge
            tv, ti = _gather_merge(tv, ti, None, world)
        return tv, ti

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ks, ke = [], []
    e0.record()
    for _ in range(steps):
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nat.set_kernel_timer(a_, b_); ks.append(a_); ke.append(b_)
        step()
    e1.record()
    torch.cuda.synchronize()
    nat.set_kernel_timer(None, None)
    ms = e0.elapsed_time(e1) / steps
    kms = float(np.mean([a_.elapsed_time(b_) for a_, b_ in zip(ks, ke)]))
    if world > 1:
        t = torch.tensor([ms, kms], dtype=torch.float64, device=device)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms, kms = float(t[0]), float(t[1])
    st = dict(zip(nat.SCORE_STAT_NAMES, nat.score_topk(Pq, E, TOPK, mu=mu, idx_base=lo, image=img, want_stats=True)[2].tolist()))
    pk = peaks()
    flops = 2.0 * K5 * d * Q5 * (hi - lo)
    del E, img
    torch.cuda.empty_cache()
    return {"workload": f"{label}: {N5 // 1_000_000}M-item catalog in total, K={K5} d={d}, Q={Q5} queries/step, top-100", "scaling": "strong",
            "catalog_total": N5, "catalog_per_gpu": hi - lo, "value": Q5 * float(N5) / (ms / 1e3), "unit": "scores/s",
            "ms_per_step": ms, "filter_kernel_ms": kms, "filter_kernel_tflops": flops / (kms / 1e3) / 1e12,
            "filter_kernel_frac_of_bf16_burst": flops / (kms / 1e3) / 1e12 / pk["bf16"],
            "survivors_per_query": st["survivors"] / Q5, "redo_queries": st["redo_queries"],
            "exact_redo_queries": st["exact_redo_queries"]}


def small_q_line(index, device, q=16, steps=50):
    """Q = 16 queries against the resident C3 catalog: the HBM-bound regime.  The timed kernel is the full filter pass
    (score_lb_kernel), which streams the catalog's fp16 plane + (|e|^2, |e|) per row = 2d + 8 bytes per row once."""
    from cfl import _native as nat
    xq = synth_features(q, device, SEED + 99)

    def local_step():                      # this rank's shard only: no collective (the line is measured on rank 0 alone)
        return index.rank_local(index.project_queries(xq), TOPK)

    for _ in range(5):
        local_step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ks, ke = [], []
    e0.record()
    for _ in range(steps):
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nat.set_kernel_timer(a_, b_); ks.append(a_); ke.append(b_)
        local_step()
    e1.record()
    torch.cuda.synchronize()
    nat.set_kernel_timer(None, None)
    ms = e0.elapsed_time(e1) / steps
    kms = float(np.mean([a_.elapsed_time(b_) for a_, b_ in zip(ks, ke)]))
    st = index.rank_local_stats(xq, TOPK)[2]
    plane = N_PER_GPU * (2 * D + 8)
    pk = peaks()
    return {"queries": q, "ms_per_step": ms, "queries_per_s": q / (ms / 1e3), "kernel_ms": kms,
            "catalog_bytes_per_pass": plane, "catalog_gbs": plane / (kms / 1e3) / 1e9,
            "hbm_frac": plane / (kms / 1e3) / 1e9 / pk["hbm"], "lower_bound_pass": st["lower_bound_pass"],
            "kernel": "score_lb_kernel<3> over the whole catalog (fp16 plane + row norms, read once from HBM); the rest "
                      "of the step is launch-bound (16 small kernels)"}


def auc_line(index, device, j=8, steps=10):
    """Per-query all-candidate AUC on the resident C3 catalog (SURVEY 8d: J = 8 labelled positives per query, every
    other catalog row a negative): the rank counts are taken inside the tensor-core scoring kernel's epilogue
    (cfl_rank_counts_packed); checked against the CUDA-core direct route (same integers).  Two placements of the
    positives: among the query's best 64 catalog rows (what evaluating a trained model looks like: almost every row is
    farther than every threshold, whole query groups are skipped by the affine-hull bound) and uniformly random rows
    (AUC 0.5: every pair has to be counted against every threshold -- the worst case)."""
    from cfl import _native as nat
    xq = synth_features(Q, device, SEED + 7)
    g = torch.Generator(device=device).manual_seed(SEED + 55)
    n = index.E.shape[0]
    Pq = index.project_queries(xq)
    top64 = nat.score_topk(Pq, index.E, 64, mu=index.mu, image=index.image)[1]
    placements = {"positives_in_top64": top64[:, torch.randperm(64, generator=g, device=device)[:j]].contiguous() + index.idx_base,
                  "positives_random": torch.randint(0, n, (Q, j), generator=g, device=device) + index.idx_base}
    out = {"workload": f"per-query all-candidate AUC: Q={Q} queries x {n} catalog rows, J={j} positives each",
           "kernel": "rank_count_umma_kernel<3> (3xTF32 tcgen05 Gram + soft-min + packed threshold counters in the "
                     "epilogue, group skip by the affine-hull bound) + rank_fix_kernel (near-ties in fp32 direct form); "
                     "no Q x N matrix is written"}
    for name, pos in placements.items():
        fused = index.auc_per_query(xq, pos)
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        direct = index.auc_per_query(xq, pos, method="direct")
        d1.record()
        same = bool(torch.equal(fused.counts, direct.counts))
        _, st = nat.rank_counts_packed(Pq, index.E, index.image, index.mu, fused.pos_dist, want_stats=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ks, ke = [], []
        e0.record()
        for _ in range(steps):
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            nat.set_kernel_timer(a_, b_); ks.append(a_); ke.append(b_)
            index.auc_per_query(xq, pos)
        e1.record()
        torch.cuda.synchronize()
        nat.set_kernel_timer(None, None)
        ms = e0.elapsed_time(e1) / steps
        kms = float(np.mean([a_.elapsed_time(b_) for a_, b_ in zip(ks, ke)]))
        out[name] = {"ms_per_call": ms, "scores_per_s": Q * n / (ms / 1e3), "count_kernels_ms": kms,
                     "count_kernels_tflops": 2.0 * K * D * Q * n / (kms / 1e3) / 1e12,
                     "cuda_core_route_ms": d0.elapsed_time(d1), "counts_equal_cuda_core_route": same,
                     "ambiguous_records": st["records"], "worst_deviation_over_band": round(st["worst_ratio"], 4),
                     "recounted_queries": st["recounted_queries"], "mean_auc": float(torch.nanmean(fused.auc))}
    return out


def _ensure_library():
    """The in-tree C-ABI library, built by nvcc when it is missing or older than its sources (a no-op on a snapshot that
    carries the prebuilt .so; ranks of one job take turns on a file lock).  There is no fallback: without nvcc and
    without the library this raises."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("cfl_build", os.path.join(PKG, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def dump_outputs(out_dir, arrays):
    """Writes every tensor as out_dir/<name>.npy, floating point as float32 and integers (the global catalog indices)
    as float64, which holds them exactly: the files of two builds can be compared array for array."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype.kind == "f" else np.float64))


def run_ours(args):
    _ensure_library()
    from cfl import _native as nat
    from cfl.ranking import CatalogIndex

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=device)
    nat.lib()
    w = synth_weights(device)

    # --- setup (untimed): project this rank's catalog shard, chunked to bound memory ---
    t0 = time.time()
    n_total = N_PER_GPU * world
    E = torch.empty(N_PER_GPU, D, dtype=torch.float32, device=device)
    chunk = 1 << 18
    proj_ms = 0.0
    for lo in range(0, N_PER_GPU, chunk):
        hi = min(N_PER_GPU, lo + chunk)
        xb = synth_features(hi - lo, device, SEED + 1 + rank * 1000 + lo // chunk)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        y, _, _ = nat.project_fwd(xb, w.V0, w.g0, w.b0, True, w.in_scale, None)
        e1.record()
        E[lo:hi] = y
        torch.cuda.synchronize()
        proj_ms += e0.elapsed_time(e1)
        del xb, y
    index = CatalogIndex(w, E, idx_base=rank * N_PER_GPU, n_total=n_total)
    setup_s = time.time() - t0

    # --- query batches: device-resident copies (value) and pinned host copies (e2e) ---
    nb = 4
    xq_dev = [synth_features(Q, device, SEED + 7 + i) for i in range(nb)]     # same on every rank
    xq_host = [x.cpu().pin_memory() for x in xq_dev]
    out_v = torch.empty(Q, TOPK, dtype=torch.float32).pin_memory()
    out_i = torch.empty(Q, TOPK, dtype=torch.int64).pin_memory()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    inflight = []
    INFLIGHT = int(os.environ.get("CFL_BENCH_INFLIGHT", "4"))

    def step_device(i):
        # independent query batches: with several ranks the exchange (all-gather + merge) of batch i runs on a side
        # stream under the scoring of the following batches; at most INFLIGHT results are outstanding (the survivor
        # counts, hence the step times, differ from rank to rank and batch to batch: a deeper queue keeps a rank that
        # waits for a slower peer's all-gather fed), every one is waited for inside the timed region (the closing drain)
        if world == 1:
            return index.rank(xq_dev[i % nb], TOPK)
        if len(inflight) >= INFLIGHT:
            inflight.pop(0)[2].synchronize()
        inflight.append(index.rank_async(xq_dev[i % nb], TOPK))
        return inflight[-1][:2]

    out_ring = [(out_v, out_i), (torch.empty_like(out_v).pin_memory(), torch.empty_like(out_i).pin_memory())]
    pending = []

    def step_e2e(i):
        # the call a user with HOST buffers makes: pinned features in, pinned top-k out.  H2D of this
        # batch, scoring and D2H of its result are all inside the timed region; consecutive batches
        # overlap (copy / compute / copy-back streams), the loop's closing synchronize waits for all.
        ov, oi = out_ring[i & 1]
        if len(pending) >= 2:
            pending.pop(0).synchronize()                          # the ring slot's previous result was delivered
        pending.append(index.rank_host(xq_host[i % nb], TOPK, ov, oi))
        return ov, oi

    def timed(step_fn, steps, warmup, kernel_events=False):
        # -> (ms, kernel ms per step, clocks, what the last timed step returned).  The warm-up holds a step's result
        # across the next step as the timed loop does, so the allocator is in the same state when the timing starts.
        for i in range(warmup):
            last = step_fn(i)
        barrier()
        ks, ke = [], []
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            if kernel_events:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                nat.set_kernel_timer(a, b)
                ks.append(a); ke.append(b)
            last = step_fn(i)
        for ev_ in pending:
            ev_.synchronize()
        pending.clear()
        for r_ in inflight:
            r_[2].synchronize()
        inflight.clear()
        e1.record()
        barrier()
        nat.set_kernel_timer(None, None)
        clocks = sampler.stop() if sampler else None
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=device)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t.item())
        kms = [a.elapsed_time(b) for a, b in zip(ks, ke)] if kernel_events else []
        return ms, kms, clocks, last

    ms_dev, kernel_ms, clocks, out_dev = timed(step_device, args.steps, args.warmup, kernel_events=True)
    ms_e2e, _, _, out_e2e = timed(step_e2e, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        # the last timed step's results of both entry points (the same query batch): device tensors from rank() and
        # the pinned host buffers rank_host() filled
        dump_outputs(args.dump_outputs, {"topk_dist": out_dev[0], "topk_index": out_dev[1],
                                         "e2e_topk_dist": out_e2e[0], "e2e_topk_index": out_e2e[1]})

    # survivor statistics of one more (untimed) step and every rank's kernel time: stragglers / slow paths
    filt = index.rank_local_stats(xq_dev[0], TOPK)[2]
    k_ms_rank = float(np.mean(kernel_ms)) if kernel_ms else float("nan")
    per_rank = None
    if world > 1:
        t = torch.tensor([k_ms_rank, float(filt["survivors"]), float(filt["redo_queries"]), float(filt["spill_queries"])],
                         dtype=torch.float64, device=device)
        allr = [torch.zeros_like(t) for _ in range(world)]
        torch.distributed.all_gather(allr, t)
        per_rank = {"kernel_ms": [round(float(a[0]), 4) for a in allr], "survivors": [int(a[1]) for a in allr],
                    "redo_queries": [int(a[2]) for a in allr], "spill_queries": [int(a[3]) for a in allr]}

    scores_per_step = float(Q) * float(n_total)
    value = scores_per_step / (ms_dev / args.steps / 1e3)
    e2e_value = scores_per_step / (ms_e2e / args.steps / 1e3)

    # --- roofline of the dominant kernel (the lower-bound filter pass), per launch on this rank ---
    pk = peaks()
    k_ms = k_ms_rank
    flops = 2.0 * K * D * Q * N_PER_GPU                           # SURVEY 8d: 2*K*d per score; one MMA per product
    achieved = flops / (k_ms / 1e3) / 1e12
    # The kernel issues kind::f16 MMAs (fp16 operands, fp32 accumulate): the peak is the measured dense 16-bit rate.
    # Burst figure when the whole timed region is shorter than a second (the clocks never leave their maximum: see
    # "clocks"), the sustained one otherwise -- stated in peak_source.
    burst = ms_dev < 1000.0
    f16_peak = pk["bf16"] if burst else pk["bf16_sus"]
    # traffic: dram__bytes_read.sum + dram__bytes_write.sum of this launch from the committed ncu --set full capture
    # of the same kernel on the same workload (profiles/r2_02_pass_c.md); None for other shapes.
    traffic = PASS_C_DRAM_BYTES if (N_PER_GPU, D, K, Q) == (1_000_000, 64, 3, 1024) else None
    alg_bytes = N_PER_GPU * (2 * D + 8)                           # fp16 plane + (|e|^2, |e|) per row, read once
    roofline = dict(bound="tensor", achieved=round(achieved, 2), peak=round(f16_peak, 1), unit="TFLOP/s",
                    frac=round(achieved / f16_peak, 4), traffic=traffic,
                    kernel="score_lb_kernel<3>: tcgen05.mma.kind::f16 (fp32 accumulators in TMEM) of the catalog's fp16 "
                           "plane against the queries' affine-hull basis + lower-bound test in the epilogue (the dominant "
                           "launch of cfl_score_topk_packed; every survivor is rescored exactly in fp32)",
                    kernel_ms=round(k_ms, 4), algorithmic_flops_per_launch=flops,
                    algorithmic_bytes_per_launch=alg_bytes,
                    peak_source=f"{pk['src']} bf16_tflops{'' if burst else '_sustained'} (dense 16-bit cuBLAS rate; "
                                f"{'burst: timed region %.2f s at full clocks' % (ms_dev / 1e3) if burst else 'sustained: long timed region'}); "
                                f"fraction of the sustained figure: {achieved / pk['bf16_sus']:.4f}",
                    hbm_gbs=round((traffic or alg_bytes) / (k_ms / 1e3) / 1e9, 1))

    small_q = small_q_line(index, device) if (rank == 0 and not args.quick) else None
    # catalog projection (stage 1 of an index build) at steady clocks: one 262144-item chunk of features, repeated.
    # (The setup loop above runs right after process start, before the clocks have ramped: its own time is kept as
    # "setup_ms" only.)
    proj = None
    if rank == 0:
        xb = synth_features(1 << 18, device, SEED + 5)
        for _ in range(3):
            nat.project_fwd(xb, w.V0, w.g0, w.b0, True, w.in_scale, None)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        for _ in range(10):
            nat.project_fwd(xb, w.V0, w.g0, w.b0, True, w.in_scale, None)
        p1.record()
        torch.cuda.synchronize()
        pms = p0.elapsed_time(p1) / 10
        nb_ = xb.shape[0]
        proj = {"items": nb_, "ms": pms, "items_per_s": nb_ / (pms / 1e3), "gbs": nb_ * (4 * F + 4 * D) / (pms / 1e3) / 1e9,
                "hbm_frac": nb_ * (4 * F + 4 * D) / (pms / 1e3) / 1e9 / pk["hbm"], "setup_ms": proj_ms,
                "kernel": "project_umma_tma_kernel (3xTF32 tcgen05, x tiles by tensor-map TMA): F=1024 -> d=64, x read once"}
        del xb
    auc = auc_line(index, device) if (world == 1 and not args.quick) else None
    if world > 1:
        torch.distributed.barrier()
    del index, E
    torch.cuda.empty_cache()
    c5 = None if args.quick else [c5_line(64, world, rank, device), c5_line(128, world, rank, device)]
    c4 = None if args.quick else c5_line(20, world, rank, device, steps=20, K5=4, Q5=1024, N5=2_000_000, label="C4")
    line = None
    if rank == 0:
        # the CPU arms are timed on rank 0 at N=1 only (torchrun pins OMP threads and the other ranks spin)
        cpu = cpu_baseline_sample(target_s=10.0) if (world == 1 and not args.no_cpu_baseline) else None
        cpu_gram = cpu_gram_sample(target_s=5.0) if (world == 1 and not args.no_cpu_baseline) else None
        line = {
            "metric": "query x candidate scores/sec (fused soft-min scoring + top-100)",
            "value": value, "unit": "scores/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "dtype_note": "fp32 in/out. Projections and sample passes: error-compensated 3xTF32 tcgen05 MMA; full pass: one fp16-operand MMA (kind::f16, fp32 accumulate) used only as a rigorous lower-bound filter, every survivor rescored in fp32 direct form (results identical to the 3xTF32 path)",
            "data": "synthetic",
            "config": config_dict(world),
            "topk_queries_per_s": Q / (ms_dev / args.steps / 1e3),
            "e2e": {"value": e2e_value, "unit": "scores/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": Q * F * 4, "d2h_bytes_per_step": Q * TOPK * 12},
            "gpu_launches": launches_per_step(world) * args.steps,
            "roofline": roofline, "cpu_baseline": cpu, "cpu_baseline_gram": cpu_gram, "clocks": clocks,
            "filter": {"survivors_per_query": filt["survivors"] / Q, "redo_queries": filt["redo_queries"],
                       "exact_redo_queries": filt["exact_redo_queries"],
                       "spill_queries": filt["spill_queries"], "probe_dropped_queries": filt["probe_dropped_queries"],
                       "lower_bound_pass": filt["lower_bound_pass"]},
            "per_rank": per_rank, "small_q": small_q, "auc": auc, "c5": c5, "c4": c4,
            "catalog_projection": proj,
            "setup_s": setup_s,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return line


def launches_per_step(world):
    # colnorm, project_fwd_splitk + its finalize (1024 queries = 8 tcgen05 tiles: split-F CUDA-core kernel), prep_queries, pack_queries, score_umma x2 (passes A/B), select_threshold x2,
    # prep_lb, score_lb (probe) + probe_classify, score_lb (pass C), rescore_merge, score_lb + rescore_merge (second
    # round under the safe threshold: both leave at once when every query was verified), redo_compact + score_umma
    # (compact exact redo: what still needs the exact kernel, gathered into one query tile), score_umma (in-place exact
    # redo of what did not fit; both exit when nothing is left to redo), merge_rescore (redone queries only)
    # (+ topk_merge after the all-gather for N>1)
    return 20 + (1 if world > 1 else 0)


# ------------------------------------------------------------------------------------------
# CPU arm: the reference's own op sequence (torch-CPU port, oracle/torch_port.py) on host cores
# ------------------------------------------------------------------------------------------
def _cpu_inputs(nq, nc):
    g = torch.Generator().manual_seed(SEED)
    lim0, limp = (6.0 / (F + D)) ** 0.5, (6.0 / (F + K * D)) ** 0.5
    V0 = (torch.rand(F, D, generator=g) * 2 - 1) * lim0
    Vp = (torch.rand(F, K * D, generator=g) * 2 - 1) * limp
    xq = torch.randn(nq, F, generator=g).clamp_(min=0) * 10
    E = torch.randn(nc, D, generator=g)
    return V0, Vp, xq, E


def cpu_step(Vp, xq, E, pair_batch):
    """One step of the reference CPU path on a bounded sample: project the queries, push the
    cross product through the pair scorer in batches (cfl/bin/predict.py:195), stable top-k."""
    from oracle import torch_port as T
    P = T.fc_weight_norm(xq / DATA_NORM, Vp, torch.ones(K * D), torch.zeros(K * D)).reshape(-1, K, D)
    S = T.all_pairs_scores_blocked(P, E, torch.tensor(1.0), cand_block=pair_batch)
    k = min(TOPK, E.shape[0])
    torch.topk(S, k, dim=1)
    return S.numel()


def cpu_baseline_sample(target_s=12.0, pair_batch=65536):
    """Times the oracle port on this box's host cores; sample sized for ~target_s of CPU work."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    nq, nc = 4, 100_000
    V0, Vp, xq, E = _cpu_inputs(nq, nc)
    cpu_step(Vp, xq, E, pair_batch)                       # warm-up
    t0 = time.time()
    n = cpu_step(Vp, xq, E, pair_batch)
    dt = time.time() - t0
    rate = n / dt
    reps = max(1, int(target_s / max(dt, 1e-3)))
    t0 = time.time()
    tot = 0
    for _ in range(reps):
        tot += cpu_step(Vp, xq, E, pair_batch)
        if time.time() - t0 > 2 * target_s:
            break
    dt = time.time() - t0
    rate = tot / dt
    return dict(value=rate, unit="scores/s", cores=cores, kind="port",
                sample=f"{tot / (nq * nc):.0f} passes of Q={nq} x N={nc} (K={K}, d={D}) through the op-for-op torch-CPU "
                       f"port of base.py:125-146 in candidate blocks of {pair_batch}; {dt:.1f} s",
                cpu=_cpu_model())


def cpu_gram_sample(target_s=5.0):
    """The strongest honest CPU line (BASELINE.md section 3 item 2; NOT what the reference does): Gram form through
    MKL SGEMM + softmax + top-k on all host cores, bounded sample."""
    from oracle import torch_port as T
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    nq, nc = 64, 200_000
    V0, Vp, xq, E = _cpu_inputs(nq, nc)
    P = T.fc_weight_norm(xq / DATA_NORM, Vp, torch.ones(K * D), torch.zeros(K * D)).reshape(-1, K, D)

    def step():
        S = T.all_pairs_scores_gram(P, E, torch.tensor(1.0))
        torch.topk(S, TOPK, dim=1)
        return S.numel()

    step()
    t0 = time.time()
    tot = 0
    while time.time() - t0 < target_s:
        tot += step()
    dt = time.time() - t0
    return dict(value=tot / dt, unit="scores/s", cores=cores, kind="port",
                sample=f"{tot / (nq * nc):.0f} passes of Q={nq} x N={nc} (K={K}, d={D}): Gram form (MKL SGEMM) + softmax + "
                       f"top-{TOPK}; {dt:.1f} s; stronger than the reference's own op sequence", cpu=_cpu_model())


def _cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (TensorFlow cannot be
    installed: oracle port, kind "port") with all host threads, same metric/config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    nq, nc, pair_batch = 4, 100_000, 65536
    V0, Vp, xq, E = _cpu_inputs(nq, nc)
    for _ in range(max(args.warmup, 1)):
        cpu_step(Vp, xq, E, pair_batch)
    t0 = time.time()
    tot = 0
    for _ in range(args.steps):
        tot += cpu_step(Vp, xq, E, pair_batch)
    dt = time.time() - t0
    value = tot / dt
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cb = dict(value=value, unit="scores/s", cores=cores, kind="port", cpu=_cpu_model(),
              sample=f"each step = Q={nq} queries x N={nc} candidates (bounded sample of the {Q} x {N_PER_GPU} step)")
    print(json.dumps({
        "impl": "reference", "metric": "query x candidate scores/sec (fused soft-min scoring + top-100)",
        "value": value, "unit": "scores/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_dict(world),
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "scores/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU arms (kernel experiments only)")
    ap.add_argument("--quick", action="store_true", help="headline line only: no C5 / small-Q side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the top-k distances and indices of the last timed step (device and host-buffer entry "
                         "points, 2.5 MB in all) as DIR/<name>.npy; the inputs are seeded, identical from run to run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
