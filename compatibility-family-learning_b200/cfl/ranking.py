"""All-candidates ranking with the CFL compatibility score (SURVEY App. A.6).

The reference only scores labelled pairs (cfl/utils.py:227-274); ranking a catalog is the
pair scorer (DistBase.build_dist, cfl/models/base.py:125-146; Thresholder,
cfl/models/blocks.py:21-22) applied to the query x catalog cross product, followed by a stable
sort.  ``CatalogIndex`` keeps one shard of projected catalog embeddings resident in HBM and
answers ``rank(query_features, k)``; with ``torch.distributed`` initialised every rank holds
one contiguous shard, ranks locally, all-gathers the [Q,k] lists (NCCL) and merges them with
``cfl_topk_merge`` -- the result is independent of the number of ranks.
"""
from __future__ import annotations

from dataclasses import dataclass
from types import SimpleNamespace
from typing import Optional

import numpy as np
import torch

from . import _native as nat


@dataclass
class EncoderWeights:
    """Weights of one encoder head pair, names as in the reference's variable scopes
    (``outputs/fully_connected/{V,g,biases}``, ``prototype_outputs/...``; for the Dist model
    ``latent_outputs/...``, ``pcd_outputs/...`` with ``weight_norm=False``)."""
    V0: torch.Tensor                      # [F, d]
    Vp: torch.Tensor                      # [F, K*d]
    g0: Optional[torch.Tensor] = None
    gp: Optional[torch.Tensor] = None
    b0: Optional[torch.Tensor] = None
    bp: Optional[torch.Tensor] = None
    weight_norm: bool = True
    in_scale: float = 1.0                 # 1/normalize_value (cfl/ops.py:198) or 1/data_norm
    act: Optional[str] = None             # --act-type
    Vg: Optional[torch.Tensor] = None     # monomer gate head [d, K] (monomer_outputs/fully_connected/V)
    gg: Optional[torch.Tensor] = None     # its weight-norm scaler g [K] (the gate never has a bias, base.py:96-103)

    @property
    def d(self):
        return self.V0.shape[1]

    @property
    def K(self):
        return self.Vp.shape[1] // self.V0.shape[1]


def shard_bounds(n_total: int, world: int, rank: int):
    """Contiguous catalog rows [lo, hi) of ``rank`` (SURVEY 8e)."""
    return n_total * rank // world, n_total * (rank + 1) // world


class CatalogIndex:
    """One catalog shard of e0 embeddings, resident on the GPU."""

    def __init__(self, weights: EncoderWeights, embeddings: torch.Tensor, idx_base: int = 0,
                 n_total: Optional[int] = None, mu: Optional[torch.Tensor] = None,
                 theta: float = 1e-6, group=None):
        if not embeddings.is_cuda:
            raise nat.CflNativeError("CatalogIndex needs CUDA embeddings (there is no CPU path)")
        self.w = weights
        self.E = embeddings
        self.idx_base = int(idx_base)
        self.n_total = int(n_total if n_total is not None else embeddings.shape[0])
        self.group = group
        self.theta = float(theta)
        self.mu = mu if mu is not None else self._global_mean()
        # tensor-core operand image of the (static) catalog, built once
        self.image = nat.catalog_pack(self.E, self.w.K, self.mu) if self.E.shape[0] else None

    # -- construction -------------------------------------------------------------------
    @classmethod
    def from_features(cls, weights: EncoderWeights, features: torch.Tensor, idx_base: int = 0,
                      n_total: Optional[int] = None, chunk: int = 1 << 16, **kw):
        """Projects this rank's catalog rows (host or device features) through the e0 head in
        chunks (stage 1 over the catalog shards by rows with no communication)."""
        dev = weights.V0.device
        n = features.shape[0]
        E = torch.empty(n, weights.d, dtype=torch.float32, device=dev)
        for lo in range(0, n, chunk):
            xb = features[lo:lo + chunk]
            if not xb.is_cuda:
                xb = xb.to(dev, non_blocking=True)
            y, _, _ = nat.project_fwd(xb, weights.V0, weights.g0, weights.b0, weights.weight_norm,
                                      weights.in_scale, weights.act)
            E[lo:lo + chunk] = y
        return cls(weights, E, idx_base=idx_base, n_total=n_total, **kw)

    def _global_mean(self):
        """Centring vector = mean of the WHOLE catalog (sum over shards), so every rank uses
        the same mu and per-candidate values do not depend on the sharding."""
        mu = nat.col_mean(self.E) if self.E.shape[0] else torch.zeros(self.w.d, device=self.E.device)
        if self._world() > 1:
            s = mu.double() * self.E.shape[0]
            torch.distributed.all_reduce(s, group=self.group)
            mu = (s / self.n_total).float()
        return mu

    def _world(self):
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            return torch.distributed.get_world_size(self.group)
        return 1

    # -- queries ------------------------------------------------------------------------
    def project_queries(self, xq: torch.Tensor) -> torch.Tensor:
        """Query side of pcd = the K prototypes of the source item (base.py:126-131)."""
        if not xq.is_cuda:
            xq = xq.to(self.E.device, non_blocking=True)
        P, _, _ = nat.project_fwd(xq, self.w.Vp, self.w.gp, self.w.bp, self.w.weight_norm,
                                  self.w.in_scale, self.w.act)
        return P.view(xq.shape[0], self.w.K, self.w.d)

    def rank_local(self, Pq: torch.Tensor, k: int):
        return nat.score_topk(Pq, self.E, k, mu=self.mu, mode="pcd", idx_base=self.idx_base,
                              image=self.image)

    def rank_local_stats(self, xq: torch.Tensor, k: int = 100):
        """One local ranking call plus the counters of cfl_score_topk_stats as a dict (survivors of the
        filter pass, queries that spilled / were dropped by the probe / were redone exactly)."""
        Pq = self.project_queries(xq)
        tv, ti, st = nat.score_topk(Pq, self.E, k, mu=self.mu, mode="pcd", idx_base=self.idx_base,
                                    image=self.image, want_stats=True)
        return tv, ti, dict(zip(nat.SCORE_STAT_NAMES, st.tolist()))

    def rank(self, xq: torch.Tensor, k: int = 100):
        """-> (dist [Q,k] ascending, index [Q,k] int64 global).  score = theta+ - dist."""
        Pq = self.project_queries(xq)
        tv, ti = self.rank_local(Pq, k)
        world = self._world()
        if world == 1:
            return tv, ti
        return _gather_merge(tv, ti, self.group, world)

    def rank_async(self, xq: torch.Tensor, k: int = 100):
        """As ``rank`` for a stream of independent query batches: the local scoring runs on the current stream, the
        exchange (all-gather + merge kernel) on a side stream, so that batch i's exchange overlaps batch i+1's
        scoring.  -> (dist, index, event); the tensors are valid once ``event`` has fired (wait for it, or make the
        consuming stream wait: ``stream.wait_event(event)``)."""
        Pq = self.project_queries(xq)
        tv, ti = self.rank_local(Pq, k)
        dev = tv.device
        cur = torch.cuda.current_stream(dev)
        done = torch.cuda.Event()
        world = self._world()
        if world == 1:
            done.record(cur)
            return tv, ti, done
        if not hasattr(self, "_xchg"):
            self._xchg = torch.cuda.Stream(dev)
        scored = torch.cuda.Event()
        scored.record(cur)
        with torch.cuda.stream(self._xchg):
            self._xchg.wait_event(scored)
            tv.record_stream(self._xchg)
            ti.record_stream(self._xchg)
            mv, mi = _gather_merge(tv, ti, self.group, world)
            done.record(self._xchg)
        return mv, mi, done

    def rank_host(self, xq_host: torch.Tensor, k: int, out_val: torch.Tensor, out_idx: torch.Tensor):
        """Host-buffer entry point: pinned query features in, pinned results out, nothing blocks.

        The batch is copied on a copy stream into one of two device staging slots while the previous
        batch is still being scored; scoring waits for its copy, the results go back on a third stream.
        Returns a ``torch.cuda.Event`` that fires when ``out_val`` / ``out_idx`` are complete."""
        dev = self.E.device
        if not hasattr(self, "_h2d"):
            self._h2d, self._d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
            self._slots, self._slot_free, self._turn = [None, None], [None, None], 0
        s = self._turn
        self._turn ^= 1
        if self._slots[s] is None or self._slots[s].shape != xq_host.shape:
            self._slots[s] = torch.empty(xq_host.shape, dtype=torch.float32, device=dev)
        cur = torch.cuda.current_stream(dev)
        with torch.cuda.stream(self._h2d):
            if self._slot_free[s] is not None:
                self._h2d.wait_event(self._slot_free[s])           # the batch that used this slot has been projected
            self._slots[s].copy_(xq_host, non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(self._h2d)
        cur.wait_event(ready)
        Pq = self.project_queries(self._slots[s])
        self._slot_free[s] = torch.cuda.Event()
        self._slot_free[s].record(cur)
        tv, ti = self.rank_local(Pq, k)
        world = self._world()
        scored = torch.cuda.Event()
        scored.record(cur)
        if world > 1:
            # exchange + merge on their own stream: they overlap the next batch's scoring
            if not hasattr(self, "_xchg"):
                self._xchg = torch.cuda.Stream(dev)
            with torch.cuda.stream(self._xchg):
                self._xchg.wait_event(scored)
                tv.record_stream(self._xchg)
                ti.record_stream(self._xchg)
                tv, ti = _gather_merge(tv, ti, self.group, world)
                scored = torch.cuda.Event()
                scored.record(self._xchg)
        with torch.cuda.stream(self._d2h):
            self._d2h.wait_event(scored)
            out_val.copy_(tv, non_blocking=True)
            out_idx.copy_(ti, non_blocking=True)
            tv.record_stream(self._d2h)
            ti.record_stream(self._d2h)
            done = torch.cuda.Event()
            done.record(self._d2h)
        return done

    def auc_per_query(self, xq: torch.Tensor, pos_idx: torch.Tensor, method: str = "fused"):
        """All-candidate AUC of every query: ``pos_idx`` [Q,J] int64 = GLOBAL catalog rows of the query's
        labelled positives (unique per query; -1 pads), every other catalog row is a negative.  Exact
        integer rank counts, independent of the sharding.  -> namespace(auc, two_u, n_pos, n_neg, ...).

        ``method="fused"`` (default; "gram" is an alias): the counts are taken inside the tensor-core scoring kernel's
        epilogue (``cfl_rank_counts_packed``) -- no Q x N matrix is ever written; near-ties are re-evaluated in the
        direct form, so the integers equal the direct route's.
        ``method="direct"``: every pair in fp32 direct-difference form on the CUDA cores (``cfl_rank_counts``)."""
        Pq = self.project_queries(xq)
        if method == "gram":
            method = "fused"
        if method not in ("direct", "fused"):
            raise ValueError("auc_per_query: method must be 'direct' or 'fused'")
        packed = (self.image, self.mu) if method == "fused" else None
        return _auc_per_query("pcd", Pq, self.E, None, pos_idx, self.idx_base, self.n_total, self.group, self._world(),
                              packed=packed)

    def within(self, xq: torch.Tensor, radius, max_results: int = nat.WITHIN_MAX_RESULTS):
        """Every catalog row closer than ``radius`` (a scalar or one per query): ``{c : dist(q, c) < r_q}``, exact.
        -> CSR lists (offsets [Q+1] int64, index [T] int64 global, dist [T] float32), each query's rows ordered by
        (distance, index); the distances are the direct-form values of ``pair_dist_rows``.  The rows are emitted from
        the tensor-core scoring epilogue (near-ties checked in the direct form), on the CUDA cores for shapes without
        a tcgen05 tiling.  Sharded: every rank lists its shard, the lists are all-gathered and merged (the result does
        not depend on the rank count).  One device->host read of the result size per call; more than ``max_results``
        rows raise CflNativeError before anything is allocated for them."""
        Pq = self.project_queries(xq)
        return _within("pcd", Pq, self.E, None, radius, self.idx_base, self.group, self._world(), max_results,
                       image=self.image, mu=self.mu)

    def compatible(self, xq: torch.Tensor, max_results: int = nat.WITHIN_MAX_RESULTS):
        """The rows the model calls compatible with each query: Thresholder score max(theta, 1e-6) - dist > 0
        (blocks.py:21-22; the accuracy counts of cfl/utils.py:247,264), i.e. ``within`` at r = max(theta, 1e-6)."""
        return self.within(xq, compatible_radius(self.theta), max_results=max_results)

    def scores(self, dist: torch.Tensor) -> torch.Tensor:
        """Thresholder (blocks.py:21-22): max(theta, 1e-6) - dist."""
        return max(self.theta, 1e-6) - dist


def compatible_radius(theta: float) -> float:
    """r with (score > 0  <=>  dist < r) for fp32 distances: max(float32(theta), float32(1e-6))."""
    return float(max(np.float32(theta), np.float32(1e-6)))


def _within(mode, query, catalog, gate, radius, idx_base, group, world, max_results, image=None, mu=None):
    """Range query over this shard, then (sharded) the exchange: per-query counts first (all-gather, so the size guard
    sees the whole result before anything is emitted), then every rank's lists padded to the longest one, one
    all-gather each for indices and distances, and the merge kernel."""
    Q = query.shape[0]
    r = nat.within_radius(radius, Q, catalog.device)
    if catalog.shape[0] == 0:
        image = None
    counts = nat.within_counts(mode, query, catalog, r, w=gate, image=image, mu=mu)
    if world == 1:
        return nat.score_within(mode, query, catalog, r, w=gate, image=image, mu=mu, idx_base=idx_base,
                                max_results=max_results, counts=counts)
    cnt = torch.empty(world * Q, dtype=torch.int64, device=counts.device)
    torch.distributed.all_gather_into_tensor(cnt, counts.contiguous(), group=group)
    cnt = cnt.view(world, Q)
    per_rank = cnt.sum(1).cpu()
    if int(per_rank.sum()) > max_results:
        raise nat.CflNativeError(f"within: the result has {int(per_rank.sum())} rows, more than max_results = "
                                 f"{max_results}")
    off, idx, dist = nat.score_within(mode, query, catalog, r, w=gate, image=image, mu=mu, idx_base=idx_base,
                                      max_results=max_results, counts=counts)
    offs = torch.zeros(world, Q + 1, dtype=torch.int64, device=cnt.device)
    offs[:, 1:] = torch.cumsum(cnt, 1)
    out_off = torch.zeros(Q + 1, dtype=torch.int64, device=cnt.device)
    out_off[1:] = torch.cumsum(cnt.sum(0), 0)
    ld = int(per_rank.max())
    if ld == 0:
        return out_off, idx, dist
    pi = torch.zeros(ld, dtype=torch.int64, device=idx.device)
    pd = torch.zeros(ld, dtype=torch.float32, device=idx.device)
    pi[:idx.shape[0]] = idx
    pd[:dist.shape[0]] = dist
    gi = torch.empty(world * ld, dtype=torch.int64, device=idx.device)
    gd = torch.empty(world * ld, dtype=torch.float32, device=idx.device)
    torch.distributed.all_gather_into_tensor(gi, pi, group=group)
    torch.distributed.all_gather_into_tensor(gd, pd, group=group)
    mi, md = nat.within_merge(offs, gi.view(world, ld), gd.view(world, ld), out_off)
    return out_off, mi, md


def auc_from_rank_counts(counts: torch.Tensor, pos_dist: torch.Tensor, n_total: int):
    """Per-query AUC from the exact rank counts of ``cfl_rank_counts`` (integer arithmetic; any device).

    counts [Q,J,2] int64 = (#{c: dist(q,c) < t_qj}, #{c: dist(q,c) == t_qj}) over ALL ``n_total`` candidates
    (positives included), pos_dist [Q,J] = t (NaN = no positive in that slot).  The positives of a query are
    removed from its counts, the rest are its negatives:  2U_q = sum_j 2 #{neg: dist > t_j} + #{neg: dist == t_j}
    -- the rank statistic of ``roc_auc_score`` on scores theta+ - dist (cfl/utils.py:267-268).
    Returns (auc [Q] float64 (NaN when a query has no positive or no negative), two_u [Q], n_pos [Q], n_neg [Q])."""
    valid = ~torch.isnan(pos_dist)
    t = pos_dist
    both = valid[:, :, None] & valid[:, None, :]
    lt_pos = ((t[:, None, :] < t[:, :, None]) & both).sum(-1)          # [Q,J]: positives j' strictly closer than j
    eq_pos = ((t[:, None, :] == t[:, :, None]) & both).sum(-1)         # includes j itself
    n_pos = valid.sum(-1)
    n_neg = int(n_total) - n_pos
    neg_lt = counts[..., 0] - lt_pos
    neg_eq = counts[..., 1] - eq_pos
    neg_gt = n_neg[:, None] - neg_lt - neg_eq
    two_u = ((2 * neg_gt + neg_eq) * valid).sum(-1)
    den = (2 * n_pos * n_neg).double()
    auc = torch.where(den > 0, two_u.double() / den.clamp(min=1), torch.full_like(den, float("nan")))
    return auc, two_u, n_pos, n_neg


def _auc_per_query(mode, query, catalog, gate, pos_idx, idx_base, n_total, group, world, packed=None):
    """Positives' distances where they live, summed over shards; exact counts per shard, summed (SURVEY 8e).
    packed = (catalog image, mu): count on the tensor cores (pcd, pcd_source)."""
    n_local = catalog.shape[0]
    pos_idx = pos_idx.to(catalog.device)
    local = pos_idx - idx_base
    local = torch.where((pos_idx >= 0) & (local >= 0) & (local < n_local), local, torch.full_like(local, -1))
    pos_dist = nat.pair_dist_rows(mode, query, catalog, local, w=gate)
    if world > 1:
        have = (~torch.isnan(pos_dist)).to(torch.int32)
        val = torch.nan_to_num(pos_dist, nan=0.0)
        torch.distributed.all_reduce(have, group=group)
        torch.distributed.all_reduce(val, group=group)               # one owner per positive: the sum is its value
        pos_dist = torch.where(have > 0, val, torch.full_like(val, float("nan")))
    if packed is not None and n_local > 0:
        counts = nat.rank_counts_packed(query, catalog, packed[0], packed[1], pos_dist,
                                        mode="pcd_source" if mode == "pcd_source" else None)
    else:
        counts = nat.rank_counts(mode, query, catalog, pos_dist, w=gate)
    if world > 1:
        torch.distributed.all_reduce(counts, group=group)
    auc, two_u, n_pos, n_neg = auc_from_rank_counts(counts, pos_dist, n_total)
    return SimpleNamespace(auc=auc, two_u=two_u, n_pos=n_pos, n_neg=n_neg, counts=counts, pos_dist=pos_dist)


_XCHG_BUFS = {}


def _gather_merge(tv, ti, group, world):
    """The one exchange step of the sharded ranking: every rank packs its [Q,k] lists into one record (one kernel), ONE
    all-gather of the records -- the latency-bound collective is paid once -- and the merge kernel reads the gathered
    records in place.  The buffers are kept per (device, stream, shape) in a ring of four (the exchange of batch i runs
    while batches i+1.. are scored), so a step allocates nothing but its two result tensors: the host time to enqueue
    a step is what limits the sharded throughput (DESIGN section 5)."""
    Q, k = tv.shape
    if not tv.is_cuda:                                         # CPU tensors (gloo tests of the host logic)
        n = Q * k
        rec = torch.empty(12 * n, dtype=torch.uint8)
        rec[:8 * n].view(torch.int64).copy_(ti.reshape(-1))
        rec[8 * n:].view(torch.float32).copy_(tv.reshape(-1))
        out = torch.empty(world * 12 * n, dtype=torch.uint8)
        torch.distributed.all_gather_into_tensor(out, rec, group=group)
        out = out.view(world, 12 * n)
        gi = out[:, :8 * n].contiguous().view(torch.int64).view(world, Q, k)
        gv = out[:, 8 * n:].contiguous().view(torch.float32).view(world, Q, k)
        return nat.topk_merge(gv, gi)
    rb = nat.topk_record_bytes(Q, k)
    key = (tv.device.index, torch.cuda.current_stream(tv.device).cuda_stream, Q, k, world)
    ring = _XCHG_BUFS.get(key)
    if ring is None:
        ring = [[torch.empty(rb, dtype=torch.uint8, device=tv.device),
                 torch.empty(world * rb, dtype=torch.uint8, device=tv.device)] for _ in range(4)] + [0]
        if len(_XCHG_BUFS) >= 8:                               # ragged batch sizes: keep the eight most recent shapes (the
            _XCHG_BUFS.pop(next(iter(_XCHG_BUFS)))             # freed blocks go back to this stream's pool, in stream order)
        _XCHG_BUFS[key] = ring
    rec, out = ring[ring[4]]
    ring[4] = (ring[4] + 1) % 4
    nat.topk_pack_records(tv.contiguous(), ti.contiguous(), rec)
    torch.distributed.all_gather_into_tensor(out, rec, group=group)
    return nat.topk_merge_records(out, world, Q, k)


def _monomer_source_side(w: EncoderWeights, x: torch.Tensor):
    """The monomer SOURCE side of items x (base.py:94-105): a = act(e0) from the embedding head ``V0/g0/b0`` and the
    gate softmax of ``pre @ Vg`` (weight norm with ``gg``, no bias), pre = the embedding head's pre-activation."""
    a, pre, _ = nat.project_fwd(x, w.V0, w.g0, w.b0, w.weight_norm, w.in_scale, w.act, want_pre=True)
    logits, _, _ = nat.project_fwd(pre, w.Vg, w.gg, None, True, 1.0, None)
    return a, torch.softmax(logits, dim=-1)


class MonomerCatalogIndex:
    """Monomer ranking (``--dist-type monomer``): the pair scorer's monomer branch
    (DistBase.build_dist, cfl/models/base.py:109-117) on the query x catalog cross product.

    The roles are the reference's: the SOURCE (query) item supplies ``a = act(e0)`` and the gate
    ``w = softmax(FC_wn(e0 pre-activation -> K, no bias))`` (base.py:94-105); the TARGET (catalog)
    item supplies its K prototypes, so one shard holds ``[N, K, d]`` resident on the GPU.
    Sharding, the all-gather + merge and the tie rule are those of ``CatalogIndex``."""

    def __init__(self, weights: EncoderWeights, prototypes: torch.Tensor, idx_base: int = 0,
                 n_total: Optional[int] = None, theta: float = 1e-6, group=None):
        if not prototypes.is_cuda:
            raise nat.CflNativeError("MonomerCatalogIndex needs CUDA prototypes (there is no CPU path)")
        if weights.Vg is None:
            raise nat.CflNativeError("MonomerCatalogIndex needs the gate head (EncoderWeights.Vg)")
        self.w = weights
        self.P = prototypes.view(prototypes.shape[0], weights.K, weights.d)
        self.idx_base = int(idx_base)
        self.n_total = int(n_total if n_total is not None else prototypes.shape[0])
        self.theta = float(theta)
        self.group = group
        # tensor-core image of the (static) catalog: augmented fp16 vectors centred on the global mean of all prototypes
        # (None when K(d+1) > 128: the CUDA-core kernel serves those shapes)
        self.mu = self._global_mean() if self.P.shape[0] else None
        self.image = nat.monomer_pack(self.P, self.mu) if self.P.shape[0] else None

    def _global_mean(self):
        s = self.P.double().sum(dim=(0, 1))
        n = torch.tensor([float(self.P.shape[0] * self.P.shape[1])], dtype=torch.float64, device=self.P.device)
        if self._world() > 1:
            torch.distributed.all_reduce(s, group=self.group)
            torch.distributed.all_reduce(n, group=self.group)
        return (s / n).float()

    @classmethod
    def from_features(cls, weights: EncoderWeights, features: torch.Tensor, idx_base: int = 0,
                      n_total: Optional[int] = None, chunk: int = 1 << 16, **kw):
        """Projects this rank's catalog rows through the prototype head (no communication)."""
        dev = weights.Vp.device
        n = features.shape[0]
        P = torch.empty(n, weights.K * weights.d, dtype=torch.float32, device=dev)
        for lo in range(0, n, chunk):
            xb = features[lo:lo + chunk]
            if not xb.is_cuda:
                xb = xb.to(dev, non_blocking=True)
            y, _, _ = nat.project_fwd(xb, weights.Vp, weights.gp, weights.bp, weights.weight_norm,
                                      weights.in_scale, weights.act)
            P[lo:lo + chunk] = y
        return cls(weights, P, idx_base=idx_base, n_total=n_total, **kw)

    def _world(self):
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            return torch.distributed.get_world_size(self.group)
        return 1

    def project_queries(self, xq: torch.Tensor):
        """-> (a [Q,d], w [Q,K]): embedding and gate softmax of the source items (base.py:94-105)."""
        if not xq.is_cuda:
            xq = xq.to(self.P.device, non_blocking=True)
        return _monomer_source_side(self.w, xq)

    def rank_local(self, a: torch.Tensor, gate: torch.Tensor, k: int):
        if self.image is not None:
            return nat.score_topk_monomer_packed(a, gate, self.P, self.image, k, mu=self.mu, idx_base=self.idx_base)
        return nat.score_topk_monomer(a, gate, self.P, k, idx_base=self.idx_base)

    def rank(self, xq: torch.Tensor, k: int = 100):
        """-> (dist [Q,k] ascending, index [Q,k] int64 global).  score = theta+ - dist."""
        a, gate = self.project_queries(xq)
        tv, ti = self.rank_local(a, gate, k)
        world = self._world()
        return (tv, ti) if world == 1 else _gather_merge(tv, ti, self.group, world)

    def auc_per_query(self, xq: torch.Tensor, pos_idx: torch.Tensor):
        """As ``CatalogIndex.auc_per_query`` with the monomer distance."""
        a, gate = self.project_queries(xq)
        return _auc_per_query("monomer", a, self.P, gate, pos_idx, self.idx_base, self.n_total, self.group,
                              self._world())

    def within(self, xq: torch.Tensor, radius, max_results: int = nat.WITHIN_MAX_RESULTS):
        """As ``CatalogIndex.within`` with the monomer distance (direct form on the CUDA cores)."""
        a, gate = self.project_queries(xq)
        return _within("monomer", a, self.P, gate, radius, self.idx_base, self.group, self._world(), max_results)

    def compatible(self, xq: torch.Tensor, max_results: int = nat.WITHIN_MAX_RESULTS):
        """As ``CatalogIndex.compatible``: ``within`` at the Thresholder radius max(theta, 1e-6)."""
        return self.within(xq, compatible_radius(self.theta), max_results=max_results)

    def scores(self, dist: torch.Tensor) -> torch.Tensor:
        return max(self.theta, 1e-6) - dist


class SourceCatalogIndex:
    """The other direction of pcd: rank the SOURCE items of a catalog for TARGET queries.

    pcd is not symmetric (DistBase.build_dist, cfl/models/base.py:125-139): dist = |v - sum_k s_k p_k|^2 takes v = e0 of
    the target item and p_k = the K prototypes of the source item.  ``CatalogIndex`` answers "which targets go with
    this source"; this index answers "which sources is this target compatible with" -- e.g. which existing items
    should now recommend a newly added item.  One shard holds the sources' prototypes ``[N, K, d]`` resident on the GPU
    with their tensor-core image (``source_catalog_pack``), centred on the mean of all prototypes of all shards;
    sharding, the all-gather + merge and the tie rule are those of ``CatalogIndex``.

    ``weights``: the catalog side goes through the prototype head ``Vp/gp/bp`` (``from_features``), the queries through
    the embedding head ``V0/g0/b0`` (``project_queries``).  For a directed model (e.g. Polyvore ``top_to_other``, where
    ``DistEncoderSrc`` encodes the source side and ``DistEncoderDst`` the target side) build ``EncoderWeights`` with
    ``Vp, gp, bp`` from the Src encoder's prototype head and ``V0, g0, b0`` from the Dst encoder's embedding head."""

    def __init__(self, weights: EncoderWeights, prototypes: torch.Tensor, idx_base: int = 0,
                 n_total: Optional[int] = None, theta: float = 1e-6, group=None):
        if not prototypes.is_cuda:
            raise nat.CflNativeError("SourceCatalogIndex needs CUDA prototypes (there is no CPU path)")
        self.w = weights
        self.P = prototypes.view(prototypes.shape[0], weights.K, weights.d)
        self.idx_base = int(idx_base)
        self.n_total = int(n_total if n_total is not None else prototypes.shape[0])
        self.theta = float(theta)
        self.group = group
        self.mu = self._global_mean()
        self.image = nat.source_catalog_pack(self.P, self.mu)

    def _global_mean(self):
        """Mean of every prototype of every shard, so that all ranks centre on the same vector."""
        s = self.P.double().sum(dim=(0, 1))
        n = torch.tensor([float(self.P.shape[0] * self.P.shape[1])], dtype=torch.float64, device=self.P.device)
        if self._world() > 1:
            torch.distributed.all_reduce(s, group=self.group)
            torch.distributed.all_reduce(n, group=self.group)
        return (s / n.clamp(min=1)).float()

    @classmethod
    def from_features(cls, weights: EncoderWeights, features: torch.Tensor, idx_base: int = 0,
                      n_total: Optional[int] = None, chunk: int = 1 << 16, **kw):
        """Projects this rank's source rows through the prototype head (no communication)."""
        dev = weights.Vp.device
        n = features.shape[0]
        P = torch.empty(n, weights.K * weights.d, dtype=torch.float32, device=dev)
        for lo in range(0, n, chunk):
            xb = features[lo:lo + chunk]
            if not xb.is_cuda:
                xb = xb.to(dev, non_blocking=True)
            y, _, _ = nat.project_fwd(xb, weights.Vp, weights.gp, weights.bp, weights.weight_norm,
                                      weights.in_scale, weights.act)
            P[lo:lo + chunk] = y
        return cls(weights, P, idx_base=idx_base, n_total=n_total, **kw)

    def _world(self):
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            return torch.distributed.get_world_size(self.group)
        return 1

    def project_queries(self, xq: torch.Tensor) -> torch.Tensor:
        """Query side = e0 of the target item (base.py:47-57)."""
        if not xq.is_cuda:
            xq = xq.to(self.P.device, non_blocking=True)
        e, _, _ = nat.project_fwd(xq, self.w.V0, self.w.g0, self.w.b0, self.w.weight_norm, self.w.in_scale, self.w.act)
        return e

    def rank_local(self, Eq: torch.Tensor, k: int):
        return nat.score_topk_source(Eq, self.P, self.image, k, mu=self.mu, idx_base=self.idx_base)

    def rank(self, xq: torch.Tensor, k: int = 100):
        """-> (dist [Q,k] ascending, index [Q,k] int64 global source rows).  score = theta+ - dist."""
        tv, ti = self.rank_local(self.project_queries(xq), k)
        world = self._world()
        return (tv, ti) if world == 1 else _gather_merge(tv, ti, self.group, world)

    def auc_per_query(self, xq: torch.Tensor, pos_idx: torch.Tensor, method: str = "fused"):
        """All-candidate AUC of every target query over the SOURCE rows: ``pos_idx`` [Q,J] int64 = GLOBAL source rows
        of the query's labelled positives (unique per query; -1 pads), every other source row is a negative.  As
        ``CatalogIndex.auc_per_query``: ``method="fused"`` counts inside the tensor-core scoring epilogue over the
        source image, ``method="direct"`` evaluates every pair on the CUDA cores; the integers are the same."""
        if method not in ("direct", "fused"):
            raise ValueError("auc_per_query: method must be 'direct' or 'fused'")
        packed = (self.image, self.mu) if method == "fused" else None
        return _auc_per_query("pcd_source", self.project_queries(xq), self.P, None, pos_idx, self.idx_base,
                              self.n_total, self.group, self._world(), packed=packed)

    def within(self, xq: torch.Tensor, radius, max_results: int = nat.WITHIN_MAX_RESULTS):
        """Every source row closer than ``radius`` (a scalar or one per query) to each target query, exact: CSR lists
        as ``CatalogIndex.within``, distances bit-identical to those ``rank`` reports.  Emitted from the tensor-core
        scoring epilogue over the source image; sharding and the size guard as ``CatalogIndex.within``."""
        return _within("pcd_source", self.project_queries(xq), self.P, None, radius, self.idx_base, self.group,
                       self._world(), max_results, image=self.image, mu=self.mu)

    def compatible(self, xq: torch.Tensor, max_results: int = nat.WITHIN_MAX_RESULTS):
        """The sources whose Thresholder calls each target compatible (score max(theta, 1e-6) - dist > 0): e.g. every
        existing item that should now recommend a newly added one.  ``within`` at r = max(theta, 1e-6)."""
        return self.within(xq, compatible_radius(self.theta), max_results=max_results)

    def scores(self, dist: torch.Tensor) -> torch.Tensor:
        """Thresholder (blocks.py:21-22): max(theta, 1e-6) - dist."""
        return max(self.theta, 1e-6) - dist


class MonomerSourceCatalogIndex:
    """The other direction of the monomer distance: rank the SOURCE items of a catalog for TARGET queries.

    The monomer distance is directed (DistBase.build_dist, cfl/models/base.py:109-117): dist = sum_k w_k |a - P'_k|^2
    takes a and the gate w of the source item (base.py:94-105) and the K prototypes P' of the target item.
    ``MonomerCatalogIndex`` answers "which targets go with this source"; this index answers "which sources is this
    target compatible with" -- e.g. which existing items should now recommend a newly added item.  One shard holds the
    sources' ``a`` [N, d] and gate ``w`` [N, K] resident on the GPU with their tensor-core image
    (``monomer_source_pack``; None when K(d+1) > 128, where the CUDA-core kernel serves the shape), centred on the
    mean of ``a`` over all shards; sharding, the all-gather + merge and the tie rule are those of ``CatalogIndex``.

    ``weights``: the catalog side goes through the embedding head ``V0/g0/b0`` and the gate ``Vg/gg``
    (``from_features``), the queries through the prototype head ``Vp/gp/bp`` (``project_queries``).  For a directed
    model (e.g. Polyvore ``top_to_other``, where ``DistEncoderSrc`` encodes the source side and ``DistEncoderDst`` the
    target side) build ``EncoderWeights`` with ``V0, g0, b0`` and ``Vg, gg`` from the Src encoder's embedding and gate
    heads and ``Vp, gp, bp`` from the Dst encoder's prototype head."""

    def __init__(self, weights: EncoderWeights, a: torch.Tensor, gate: torch.Tensor, idx_base: int = 0,
                 n_total: Optional[int] = None, theta: float = 1e-6, group=None):
        if not a.is_cuda or not gate.is_cuda:
            raise nat.CflNativeError("MonomerSourceCatalogIndex needs CUDA embeddings and gates (there is no CPU path)")
        self.w = weights
        self.a = a.view(a.shape[0], weights.d)
        self.gate = gate.view(gate.shape[0], weights.K)
        self.idx_base = int(idx_base)
        self.n_total = int(n_total if n_total is not None else a.shape[0])
        self.theta = float(theta)
        self.group = group
        self.mu = self._global_mean()
        self.image = nat.monomer_source_pack(self.a, self.gate, self.mu) if self.a.shape[0] else None

    def _global_mean(self):
        """Mean of the sources' a over every shard, so that all ranks centre on the same vector."""
        s = self.a.double().sum(dim=0)
        n = torch.tensor([float(self.a.shape[0])], dtype=torch.float64, device=self.a.device)
        if self._world() > 1:
            torch.distributed.all_reduce(s, group=self.group)
            torch.distributed.all_reduce(n, group=self.group)
        return (s / n.clamp(min=1)).float()

    @classmethod
    def from_features(cls, weights: EncoderWeights, features: torch.Tensor, idx_base: int = 0,
                      n_total: Optional[int] = None, chunk: int = 1 << 16, **kw):
        """Projects this rank's source rows through the embedding head and the gate (no communication)."""
        if weights.Vg is None:
            raise nat.CflNativeError("MonomerSourceCatalogIndex needs the gate head (EncoderWeights.Vg)")
        dev = weights.V0.device
        n = features.shape[0]
        a = torch.empty(n, weights.d, dtype=torch.float32, device=dev)
        gate = torch.empty(n, weights.K, dtype=torch.float32, device=dev)
        for lo in range(0, n, chunk):
            xb = features[lo:lo + chunk]
            if not xb.is_cuda:
                xb = xb.to(dev, non_blocking=True)
            a[lo:lo + chunk], gate[lo:lo + chunk] = _monomer_source_side(weights, xb)
        return cls(weights, a, gate, idx_base=idx_base, n_total=n_total, **kw)

    def _world(self):
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            return torch.distributed.get_world_size(self.group)
        return 1

    def project_queries(self, xq: torch.Tensor) -> torch.Tensor:
        """-> [Q, K, d]: the K prototypes of the target items (base.py:47-57)."""
        if not xq.is_cuda:
            xq = xq.to(self.a.device, non_blocking=True)
        w = self.w
        P, _, _ = nat.project_fwd(xq, w.Vp, w.gp, w.bp, w.weight_norm, w.in_scale, w.act)
        return P.view(P.shape[0], w.K, w.d)

    def rank_local(self, Pq: torch.Tensor, k: int):
        return nat.score_topk_monomer_source(Pq, self.a, self.gate, self.image, k, mu=self.mu, idx_base=self.idx_base)

    def rank(self, xq: torch.Tensor, k: int = 100):
        """-> (dist [Q,k] ascending, index [Q,k] int64 global source rows).  score = theta+ - dist."""
        tv, ti = self.rank_local(self.project_queries(xq), k)
        world = self._world()
        return (tv, ti) if world == 1 else _gather_merge(tv, ti, self.group, world)

    def auc_per_query(self, xq: torch.Tensor, pos_idx: torch.Tensor):
        """As ``SourceCatalogIndex.auc_per_query`` with the monomer distance (direct form on the CUDA cores);
        ``pos_idx`` holds GLOBAL source rows."""
        return _auc_per_query("monomer_source", self.project_queries(xq), self.a, self.gate, pos_idx, self.idx_base,
                              self.n_total, self.group, self._world())

    def within(self, xq: torch.Tensor, radius, max_results: int = nat.WITHIN_MAX_RESULTS):
        """As ``SourceCatalogIndex.within`` with the monomer distance (direct form on the CUDA cores); the distances
        are bit-identical to those ``rank`` reports."""
        return _within("monomer_source", self.project_queries(xq), self.a, self.gate, radius, self.idx_base, self.group,
                       self._world(), max_results)

    def compatible(self, xq: torch.Tensor, max_results: int = nat.WITHIN_MAX_RESULTS):
        """As ``SourceCatalogIndex.compatible``: ``within`` at the Thresholder radius max(theta, 1e-6)."""
        return self.within(xq, compatible_radius(self.theta), max_results=max_results)

    def scores(self, dist: torch.Tensor) -> torch.Tensor:
        """Thresholder (blocks.py:21-22): max(theta, 1e-6) - dist."""
        return max(self.theta, 1e-6) - dist
