"""Range queries and per-query AUC in the source direction: cfl_pair_dist_rows / cfl_rank_counts /
cfl_rank_counts_packed / cfl_score_within with CFL_PCD_SOURCE and CFL_MONOMER_SOURCE, and
SourceCatalogIndex / MonomerSourceCatalogIndex .within, .compatible and .auc_per_query.

The queries are TARGET items, the candidates SOURCE items.  The fp64 oracle is the forward one transposed:
pcd_source = all_pairs_dist(P_src, E_tgt).T, monomer_source = all_pairs_monomer_dist(a_src, w_src, P_tgt).T.

CPU: the SASS of the new tensor-core kernels, the no-GPU failure mode, the sharded assembly on a gloo world-2 group with
oracle-backed kernel doubles.  GPU: distances against the oracle, definition parity of score_within on both routes,
packed counts against the CUDA-core counts (ties, several threshold chunks, the record overflow), which kernel ran,
agreement with rank(), compatible(), AUC against the oracle, the 2^20-row shape and two GPUs."""
import collections
import ctypes as C
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import cfl_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "compatibility-family-learning_b200", "cfl", "_lib", "libcfl_b200.so")


def src_dist(Eq, P):
    """fp64 pcd_source matrix [Q, N]: e = Eq[q] (target e0), p = P[c] (source prototypes [N,K,d])."""
    return O.all_pairs_dist(P.astype(np.float64), Eq.astype(np.float64)).T.copy()


def msrc_dist(Pq, A, W):
    """fp64 monomer_source matrix [Q, N]: the target's prototypes Pq[q], the source's a = A[c] and gate W[c]."""
    return O.all_pairs_monomer_dist(A.astype(np.float64), W.astype(np.float64), Pq.astype(np.float64)).T.copy()


def _csr_reference(D, r, idx_base=0):
    """(offsets, index, dist) of {c : D[q, c] < r[q]} ordered by (D, index)."""
    off, idx, val = [0], [], []
    for q in range(D.shape[0]):
        with np.errstate(invalid="ignore"):
            sel = np.nonzero(D[q] < r[q])[0]
        sel = sel[np.lexsort((sel, D[q, sel]))]
        idx.append(sel + idx_base)
        val.append(D[q, sel])
        off.append(off[-1] + len(sel))
    return (np.array(off, np.int64), np.concatenate(idx).astype(np.int64) if idx else np.zeros(0, np.int64),
            np.concatenate(val).astype(np.float32) if val else np.zeros(0, np.float32))


# ------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def census():
    """{demangled kernel name: Counter of SASS mnemonics} of the built library (method of test_sass_static.py)."""
    cuobjdump = next((c for c in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump") if c and os.path.exists(c)),
                     None)
    filt = shutil.which("c++filt")
    if cuobjdump is None or filt is None:
        pytest.skip("cuobjdump / c++filt not available")
    ops = ("UTCHMMA", "LDTM", "UBLKCP", "STL", "LDL")
    sass = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, timeout=600, check=True).stdout
    per, fn = collections.defaultdict(collections.Counter), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            fn = m.group(1)
            per[fn]["_"] += 0
            continue
        if fn is not None:
            for op in ops:
                if op in line and re.search(r"\b%s\b" % op, line):
                    per[fn][op] += 1
    names = subprocess.run([filt], input="\n".join(per), capture_output=True, text=True, check=True).stdout.splitlines()
    return {re.sub(r"\(.*", "", re.sub(r"^void ", "", nice)): per[m] for m, nice in zip(per, names)}


def test_source_count_and_emit_kernels_are_tcgen05_code_without_local_memory(census):
    for name in ("rank_count_src_umma_kernel", "within_emit_src_umma_kernel"):
        for K in range(1, 9):
            k = f"cfl::{name}<{K}>"
            assert k in census, f"{k} not in the library"
            for op in ("UTCHMMA", "LDTM", "UBLKCP"):
                assert census[k][op] > 0, f"{k}: no {op} in its SASS"
            assert census[k]["STL"] == 0 and census[k]["LDL"] == 0, (k, census[k])
    for K in range(1, 9):
        for name in ("rank_fix_src_kernel", "within_fix_src_kernel"):
            assert f"cfl::{name}<{K}>" in census


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_source_modes_fail_loudly_without_a_gpu():
    from cfl import _native
    lib = _native.lib()
    for mode in (3, 4):
        assert lib.cfl_pair_dist_rows(mode, None, 1, 2, 4, 8, None, None, 8, 8, None, 1, None, None) == -5
        assert lib.cfl_rank_counts(mode, None, 1, 2, 4, 8, None, None, 8, 8, None, 1, None, None) == -5
        assert lib.cfl_score_within(mode, None, 1, 2, 4, 8, None, None, None, 8, 8, None, None, None, 0, None, None,
                                    None, 0, None) == -5
        assert lib.cfl_pair_loss_fwd(mode, None, 4, None, 8, None, 2, 2, 4, None, 0, 0.0, None, None, None, None, None,
                                     0, None) != 0
    assert lib.cfl_rank_counts_packed(3, None, 1, 2, 4, 8, None, None, 8, 8, None, None, 1, None, None, 0, None) == -5
    fwd = lib.cfl_rank_counts_packed_workspace_bytes(1024, 3, 64, 1 << 20)
    src = lib.cfl_rank_counts_packed_source_workspace_bytes(1024, 3, 64, 1 << 20)
    assert src == fwd                                          # the forward layout, its query regions reused
    for Q, K, d in ((1, 2, 128), (1, 8, 64), (70, 5, 20), (65536, 8, 128)):
        assert (lib.cfl_rank_counts_packed_source_workspace_bytes(Q, K, d, 1 << 20)
                >= lib.cfl_rank_counts_packed_workspace_bytes(Q, K, d, 1 << 20))
    assert lib.cfl_score_within_workspace_bytes(3, 1024, 3, 64, 1 << 20) > lib.cfl_score_within_workspace_bytes(
        4, 1024, 3, 64, 1 << 20)                               # pcd_source reserves the tensor-core workspace
    with pytest.raises(_native.CflNativeError):
        _native.score_within("pcd_source", torch.zeros(2, 4), torch.zeros(5, 3, 4), 1.0)
    with pytest.raises(_native.CflNativeError):
        _native.rank_counts("monomer_source", torch.zeros(2, 3, 4), torch.zeros(5, 4), torch.zeros(2, 1),
                            w=torch.full((5, 3), 1.0 / 3))


def _case():
    rng = np.random.default_rng(19)
    N, K, d, Q = 257, 3, 6, 9
    P = np.round(rng.normal(size=(N, K, d)), 1).astype(np.float32)
    Eq = np.round(rng.normal(size=(Q, d)), 1).astype(np.float32)
    D = src_dist(Eq, P).astype(np.float32)
    r = np.sort(D, 1)[np.arange(Q), rng.integers(0, 60, Q)]        # radii on a row's distance: ties on the boundary
    r[2] = np.nan
    r[3] = 0.0
    pos = np.full((Q, 4), -1, np.int64)
    for q in range(Q):
        pos[q, :1 + q % 4] = rng.choice(N, 1 + q % 4, replace=False)
    return Eq, P, r, pos


def _doubles(nat):
    """Oracle-backed stand-ins for the pcd_source kernels (fp64 distances rounded to fp32; the kernels' contracts)."""
    def dense(mode, query, catalog):
        assert mode == "pcd_source"
        if catalog.shape[0] == 0:
            return np.zeros((query.shape[0], 0), np.float32)
        return src_dist(query.numpy(), catalog.numpy()).astype(np.float32)

    def within_counts(mode, query, catalog, radius, w=None, image=None, mu=None):
        with np.errstate(invalid="ignore"):
            return torch.as_tensor((dense(mode, query, catalog) < radius.numpy()[:, None]).sum(1).astype(np.int64))

    def score_within(mode, query, catalog, radius, w=None, image=None, mu=None, idx_base=0,
                     max_results=nat.WITHIN_MAX_RESULTS, want_stats=False, counts=None):
        off, idx, val = _csr_reference(dense(mode, query, catalog), radius.numpy(), idx_base)
        if off[-1] > max_results:
            raise nat.CflNativeError(f"score_within: the result has {off[-1]} rows, more than max_results")
        return torch.as_tensor(off), torch.as_tensor(idx), torch.as_tensor(val)

    def within_merge(offsets, idx, dist_, out_offsets):
        R, Q = offsets.shape[0], offsets.shape[1] - 1
        oi, od = [], []
        for q in range(Q):
            ii = np.concatenate([idx[r, offsets[r, q]:offsets[r, q + 1]].numpy() for r in range(R)])
            dd = np.concatenate([dist_[r, offsets[r, q]:offsets[r, q + 1]].numpy() for r in range(R)])
            o = np.lexsort((ii, dd))
            oi.append(ii[o]); od.append(dd[o])
        return torch.as_tensor(np.concatenate(oi)), torch.as_tensor(np.concatenate(od))

    def pair_dist_rows(mode, query, catalog, pos_idx, w=None):
        D = dense(mode, query, catalog)
        p = pos_idx.numpy()
        out = np.full(p.shape, np.nan, np.float32)
        ok = (p >= 0) & (p < D.shape[1])
        out[ok] = D[np.nonzero(ok)[0], p[ok]]
        return torch.as_tensor(out)

    def rank_counts(mode, query, catalog, pos_dist, w=None):
        D, t = dense(mode, query, catalog), pos_dist.numpy()
        lt = (D[:, None, :] < t[:, :, None]).sum(-1)
        eq = (D[:, None, :] == t[:, :, None]).sum(-1)
        return torch.as_tensor(np.stack([lt, eq], -1).astype(np.int64))

    def rank_counts_packed(query, catalog, image, mu, pos_dist, want_stats=False, mode=None):
        assert mode == "pcd_source"
        return rank_counts(mode, query, catalog, pos_dist)

    nat.within_counts, nat.score_within, nat.within_merge = within_counts, score_within, within_merge
    nat.pair_dist_rows, nat.rank_counts, nat.rank_counts_packed = pair_dist_rows, rank_counts, rank_counts_packed


def _sharded_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    for p in (ROOT, os.path.join(ROOT, "compatibility-family-learning_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from cfl import ranking
    _doubles(ranking.nat)
    Eq, P, r, pos = _case()
    lo, hi = ranking.shard_bounds(P.shape[0], world, rank)
    off, idx, val = ranking._within("pcd_source", torch.as_tensor(Eq), torch.as_tensor(P[lo:hi]), None,
                                    torch.as_tensor(r), lo, None, world, 1 << 20)
    res = ranking._auc_per_query("pcd_source", torch.as_tensor(Eq), torch.as_tensor(P[lo:hi]), None,
                                 torch.as_tensor(pos), lo, P.shape[0], None, world, packed=(object(), None))
    if rank == 0:
        np.savez(os.path.join(out_dir, "w.npz"), off=off.numpy(), idx=idx.numpy(), val=val.numpy(),
                 two_u=res.two_u.numpy(), n_pos=res.n_pos.numpy(), n_neg=res.n_neg.numpy())
    dist.destroy_process_group()


def test_sharded_source_within_and_auc_world2_gloo_match_the_oracle(tmp_path):
    """SourceCatalogIndex's assembly (_within / _auc_per_query with mode "pcd_source"): counts all-gathered, lists
    merged, the positives' distances and the counts all-reduced -- the oracle's CSR and AUC integers over all sources."""
    port = 33700 + os.getpid() % 2000
    mp.spawn(_sharded_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    got = np.load(tmp_path / "w.npz")
    Eq, P, r, pos = _case()
    D = src_dist(Eq, P).astype(np.float32)
    off, idx, val = _csr_reference(D, r)
    np.testing.assert_array_equal(got["off"], off)
    np.testing.assert_array_equal(got["idx"], idx)
    np.testing.assert_array_equal(got["val"], val)
    assert off[3] - off[2] == 0 and off[4] - off[3] == 0                # NaN and r = 0: empty lists
    two_u, n_pos, n_neg = O.per_query_auc(D, pos)
    assert got["two_u"].tolist() == two_u and got["n_pos"].tolist() == n_pos and got["n_neg"].tolist() == n_neg


# ------------------------------------------------------------------------------------ GPU
def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).cuda()


@pytest.fixture(scope="module")
def nat():
    from cfl import _native
    _native.lib()
    _, major, _ = _native.device_info()
    assert major == 10, "these tests need a B200 (sm_100)"
    return _native


def _pair_dense(nat, mode, query, catalog, w=None, chunk=32):
    """[Q, N] direct-form distances through pair_dist_rows, 32 rows (its largest J) per call."""
    Q, N = query.shape[0], catalog.shape[0]
    out = torch.empty(Q, N, dtype=torch.float32, device="cuda")
    for lo in range(0, N, chunk):
        hi = min(N, lo + chunk)
        pos = torch.arange(lo, hi, device="cuda")[None, :].expand(Q, hi - lo).contiguous()
        out[:, lo:hi] = nat.pair_dist_rows(mode, query, catalog, pos, w=w)
    return out


def _check_definition(res, D, r, idx_base=0):
    """res == the CSR of {c : D[q, c] < r_q}: sets, distance bits, (dist, index) order."""
    off, idx, val = (t.cpu().numpy() for t in res[:3])
    woff, widx, wval = _csr_reference(D, r, idx_base)
    np.testing.assert_array_equal(off - off[0], woff)
    np.testing.assert_array_equal(idx, widx)
    assert val.view(np.uint32).tolist() == wval.view(np.uint32).tolist()


def _planted_radii(rng, D, hi=300):
    Q, N = D.shape
    return np.sort(D, 1)[np.arange(Q), rng.integers(0, min(hi, N), Q)]   # a row's distance: ties on the boundary


def _pcd_src_data(rng, Q, K, d, N):
    P = rng.normal(size=(N, K, d)).astype(np.float32)
    Eq = (P[rng.integers(0, N, Q)].mean(1) + 0.5 * rng.normal(size=(Q, d))).astype(np.float32)
    return Eq, P


def _msrc_data(rng, Q, K, d, N):
    A = rng.normal(size=(N, d)).astype(np.float32)
    W = rng.random(size=(N, K)).astype(np.float32)
    W /= W.sum(1, keepdims=True)
    Pq = (A[rng.integers(0, N, Q)][:, None, :] + 0.5 * rng.normal(size=(Q, K, d))).astype(np.float32)
    return Pq, A, W


@pytest.mark.gpu
@pytest.mark.parametrize("K,d", [(1, 10), (2, 20), (3, 64), (5, 128), (8, 128)])
def test_pair_dist_rows_pcd_source_against_the_oracle(nat, K, d):
    rng = np.random.default_rng(K * 31 + d)
    Q, N, J = 40, 900, 6
    Eq, P = _pcd_src_data(rng, Q, K, d, N)
    pos = rng.integers(-1, N, size=(Q, J))
    got = nat.pair_dist_rows("pcd_source", dev(Eq), dev(P), dev(pos, torch.int64)).cpu().numpy()
    D = src_dist(Eq, P)
    want = np.where(pos >= 0, D[np.arange(Q)[:, None], np.maximum(pos, 0)], np.nan)
    np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4)
    assert np.isnan(got[pos < 0]).all()
    if K == 1:                                                 # the forward call with the roles swapped, bit for bit
        fwd = _pair_dense(nat, "pcd", dev(P), dev(Eq)).T
        src = _pair_dense(nat, "pcd_source", dev(Eq), dev(P))
        assert torch.equal(fwd.contiguous(), src)


@pytest.mark.gpu
@pytest.mark.parametrize("K,d", [(1, 10), (2, 20), (4, 31), (8, 64)])
def test_pair_dist_rows_monomer_source_against_the_oracle(nat, K, d):
    rng = np.random.default_rng(K * 37 + d)
    Q, N, J = 30, 700, 5
    Pq, A, W = _msrc_data(rng, Q, K, d, N)
    pos = rng.integers(-1, N, size=(Q, J))
    got = nat.pair_dist_rows("monomer_source", dev(Pq), dev(A), dev(pos, torch.int64), w=dev(W)).cpu().numpy()
    D = msrc_dist(Pq, A, W)
    want = np.where(pos >= 0, D[np.arange(Q)[:, None], np.maximum(pos, 0)], np.nan)
    np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("K,d,Q,N", [(1, 10, 17, 3001), (2, 20, 70, 5003), (3, 64, 130, 7001), (4, 128, 1, 4099),
                                     (5, 20, 70, 2050), (8, 10, 17, 3333), (8, 128, 70, 2000), (3, 20, 1, 1000)])
def test_source_within_definition_parity(nat, K, d, Q, N):
    """Both routes (the source image and image=None: CUDA cores; K*d = 1024 reads the rows in place) give the CSR of
    the dense pair_dist_rows matrix, bit for bit, with no count mismatch and no re-emitted query."""
    rng = np.random.default_rng(K * 100 + d + Q)
    Eq, P = _pcd_src_data(rng, Q, K, d, N)
    Ed, Pd = dev(Eq), dev(P)
    D = _pair_dense(nat, "pcd_source", Ed, Pd).cpu().numpy()
    r = _planted_radii(rng, D)
    mu = Pd.double().mean((0, 1)).float()
    img = nat.source_catalog_pack(Pd, mu)
    res = nat.score_within("pcd_source", Ed, Pd, dev(r), image=img, mu=mu, idx_base=7, want_stats=True)
    _check_definition(res, D, r, 7)
    assert res[3]["count_mismatch_queries"] == 0 and res[3]["reemitted_queries"] == 0, res[3]
    assert res[3]["worst_ratio"] < 0.5, res[3]
    sizes = nat.rank_counts("pcd_source", Ed, Pd, dev(r)[:, None])[:, 0, 0]
    assert torch.equal(res[0][1:] - res[0][:-1], sizes)
    core = nat.score_within("pcd_source", Ed, Pd, dev(r), idx_base=7, want_stats=True)
    for a, b in zip(res[:3], core[:3]):
        assert torch.equal(a, b)
    assert core[3]["count_mismatch_queries"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("K,d,Q,N", [(1, 10, 17, 3001), (2, 20, 70, 2003), (4, 31, 130, 1500), (8, 64, 33, 1200),
                                     (4, 20, 1, 999)])
def test_monomer_source_within_definition_parity(nat, K, d, Q, N):
    rng = np.random.default_rng(K * 1000 + d + Q)
    Pq, A, W = _msrc_data(rng, Q, K, d, N)
    Pd, Ad, Wd = dev(Pq), dev(A), dev(W)
    D = _pair_dense(nat, "monomer_source", Pd, Ad, w=Wd).cpu().numpy()
    r = _planted_radii(rng, D)
    res = nat.score_within("monomer_source", Pd, Ad, dev(r), w=Wd, idx_base=3, want_stats=True)
    _check_definition(res, D, r, 3)
    assert res[3]["count_mismatch_queries"] == 0, res[3]
    np.testing.assert_allclose(D, msrc_dist(Pq, A, W), rtol=1e-4, atol=1e-4)


def _counts_case(rng, kind, Q, K, d, N, J):
    if kind == "integer":                                      # integer-valued: exact ties everywhere
        P = rng.integers(-2, 3, size=(N, K, d)).astype(np.float32)
        Eq = rng.integers(-2, 3, size=(Q, d)).astype(np.float32)
    else:
        Eq, P = _pcd_src_data(rng, Q, K, d, N)
    D = src_dist(Eq, P)
    if kind == "top":                                          # positives near the top of the ranking
        pos = np.argsort(D, 1)[:, :J * 3][:, ::3].copy()
    else:
        pos = np.stack([rng.choice(N, J, replace=False) for _ in range(Q)])
    pos[0, J // 2:] = -1                                       # padding slots
    return Eq, P, pos


@pytest.mark.gpu
@pytest.mark.parametrize("kind,K,d,Q,N,J", [("top", 3, 64, 70, 20000, 8), ("random", 2, 20, 130, 9000, 5),
                                            ("integer", 4, 10, 33, 5000, 8), ("random", 8, 128, 17, 3000, 32),
                                            ("top", 1, 128, 65, 12000, 32), ("integer", 5, 20, 48, 4000, 12)])
def test_packed_source_counts_equal_the_cuda_core_counts(nat, kind, K, d, Q, N, J):
    rng = np.random.default_rng(K * 7 + d + J)
    Eq, P, pos = _counts_case(rng, kind, Q, K, d, N, J)
    Ed, Pd = dev(Eq), dev(P)
    t = nat.pair_dist_rows("pcd_source", Ed, Pd, dev(pos, torch.int64))
    mu = Pd.double().mean((0, 1)).float()
    img = nat.source_catalog_pack(Pd, mu)
    packed, st = nat.rank_counts_packed(Ed, Pd, img, mu, t, want_stats=True, mode="pcd_source")
    direct = nat.rank_counts("pcd_source", Ed, Pd, t)
    assert torch.equal(packed, direct)
    assert st["worst_ratio"] < 0.5, st
    assert st["recounted_queries"] == 0, st


@pytest.mark.gpu
def test_packed_source_counts_record_overflow_recounts(nat, monkeypatch):
    rng = np.random.default_rng(5)
    Eq, P, pos = _counts_case(rng, "integer", 70, 3, 16, 6000, 8)
    Ed, Pd = dev(Eq), dev(P)
    t = nat.pair_dist_rows("pcd_source", Ed, Pd, dev(pos, torch.int64))
    mu = Pd.double().mean((0, 1)).float()
    img = nat.source_catalog_pack(Pd, mu)
    want = nat.rank_counts("pcd_source", Ed, Pd, t)
    monkeypatch.setenv("CFL_EXPERIMENTS", "1")
    monkeypatch.setenv("CFL_RANK_REC_CAP", "64")
    got, st = nat.rank_counts_packed(Ed, Pd, img, mu, t, want_stats=True, mode="pcd_source")
    assert st["recounted_queries"] > 0, st
    assert torch.equal(got, want)
    r = t[:, 0].nan_to_num(0.0).contiguous()
    res = nat.score_within("pcd_source", Ed, Pd, r, image=img, mu=mu, want_stats=True)
    assert res[3]["reemitted_queries"] > 0 and res[3]["count_mismatch_queries"] == 0, res[3]
    monkeypatch.delenv("CFL_RANK_REC_CAP")
    ref = nat.score_within("pcd_source", Ed, Pd, r)
    for a, b in zip(res[:3], ref):
        assert torch.equal(a, b)


def _kernels_of(fn, expect):
    """Names of the kernels fn launches.  In long test processes a trace can come back without some kernel records
    (tests/test_monomer_source_ranking.py), so fn (deterministic) is traced again, up to four times, until every
    expected name has appeared; the result is the union of the traces."""
    fn()                                                       # untraced first call: modules loaded
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    names = set()
    for _ in range(4):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names |= {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
        if all(any(x in n for n in names) for x in expect):
            break
    return names


@pytest.mark.gpu
def test_profiler_shows_which_source_kernel_ran(nat):
    rng = np.random.default_rng(9)
    Eq, P = _pcd_src_data(rng, 40, 3, 32, 5000)
    Ed, Pd = dev(Eq), dev(P)
    mu = Pd.double().mean((0, 1)).float()
    img = nat.source_catalog_pack(Pd, mu)
    r = torch.full((40,), float(np.median(src_dist(Eq[:2], P))), device="cuda")
    want = ("rank_count_src_umma_kernel<3>", "within_emit_src_umma_kernel<3>", "within_rescore_src_kernel<3, false, true>")
    tc = _kernels_of(lambda: nat.score_within("pcd_source", Ed, Pd, r, image=img, mu=mu), want)
    for x in want:
        assert any(x in n for n in tc), (x, tc)
    assert not any("within_emit_kernel" in n or "within_emit_umma_kernel" in n for n in tc), tc
    want = ("rank_count_src_kernel<3, false", "within_emit_src_kernel<3, false")
    core = _kernels_of(lambda: nat.score_within("pcd_source", Ed, Pd, r), want)
    for x in want:
        assert any(x in n for n in core), (x, core)
    assert not any("umma" in n for n in core), core
    Pq, A, W = _msrc_data(rng, 20, 4, 20, 3000)
    want = ("rank_count_src_kernel<4, true", "within_emit_src_kernel<4, true", "within_rescore_src_kernel<4, true, false>")
    mono = _kernels_of(lambda: nat.score_within("monomer_source", dev(Pq), dev(A), 5.0, w=dev(W)), want)
    for x in want:
        assert any(x in n for n in mono), (x, mono)
    Eb, Pb = dev(rng.normal(size=(40, 128))), dev(rng.normal(size=(500, 8, 128)))
    want = ("rank_count_src_kernel<8, false, 0>",)              # K*d = 1024: rows read in place
    big = _kernels_of(lambda: nat.rank_counts("pcd_source", Eb, Pb, torch.ones(40, 1, device="cuda")), want)
    assert any(want[0] in n for n in big), big


def _weights(rng, F, K, d, gate=False):
    from cfl.ranking import EncoderWeights
    return EncoderWeights(V0=dev(O.xavier_uniform(rng, F, d)), Vp=dev(O.xavier_uniform(rng, F, K * d)),
                          g0=dev(np.ones(d)), gp=dev(np.ones(K * d)), b0=dev(0.1 * rng.normal(size=d)),
                          bp=dev(0.1 * rng.normal(size=K * d)), weight_norm=True, act="tanh",
                          Vg=dev(O.xavier_uniform(rng, d, K)) if gate else None, gg=dev(np.ones(K)) if gate else None)


def _agreement(index, xq, k=100):
    """within(r = k-th distance of rank(k)) has rank's index set except rows within 1e-5 relative of r; shared rows
    carry rank's distance bits."""
    tv, ti = index.rank(xq, k)
    off, idx, val = index.within(xq, tv[:, k - 1].contiguous())
    offc, idxc, valc = off.cpu().numpy(), idx.cpu().numpy(), val.cpu().numpy()
    tvc, tic = tv.cpu().numpy(), ti.cpu().numpy()
    for q in range(tvc.shape[0]):
        mine = dict(zip(idxc[offc[q]:offc[q + 1]].tolist(), valc[offc[q]:offc[q + 1]].tolist()))
        theirs = dict(zip(tic[q].tolist(), tvc[q].tolist()))
        rq = float(tvc[q, k - 1])
        for c in set(mine) ^ set(theirs):
            v = mine.get(c, theirs.get(c))
            assert abs(v - rq) <= 1e-5 * rq, (q, c, v, rq)
        for c in set(mine) & set(theirs):
            assert np.float32(mine[c]).view(np.uint32) == np.float32(theirs[c]).view(np.uint32), (q, c)
    return tv


def _compatible(nat, index, xq, tv, mode, query, catalog, w=None):
    from cfl.ranking import compatible_radius
    index.theta = float(tv[:, 40].median())
    off, idx, val = index.compatible(xq)
    assert (index.scores(val) > 0).all()
    assert int(off[-1]) > 0
    samp = torch.randint(0, catalog.shape[0], (query.shape[0], 32), device="cuda")
    sd = nat.pair_dist_rows(mode, query, catalog, samp, w=w)
    offc, idxc = off.cpu().numpy(), idx.cpu().numpy()
    for q in range(query.shape[0]):
        inside = set(idxc[offc[q]:offc[q + 1]].tolist())
        for j in range(32):
            if int(samp[q, j]) not in inside:
                assert float(index.scores(sd[q, j])) <= 0
    ref = index.within(xq, compatible_radius(index.theta))
    for a, b in zip((off, idx, val), ref):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_source_index_within_compatible_and_rank_agree(nat):
    from cfl.ranking import SourceCatalogIndex
    rng = np.random.default_rng(21)
    F, K, d, N, Q = 96, 3, 32, 60000, 50
    w = _weights(rng, F, K, d)
    idx = SourceCatalogIndex.from_features(w, dev(np.maximum(rng.normal(size=(N, F)), 0)))
    xq = dev(np.maximum(rng.normal(size=(Q, F)), 0))
    tv = _agreement(idx, xq)
    _compatible(nat, idx, xq, tv, "pcd_source", idx.project_queries(xq), idx.P)


@pytest.mark.gpu
def test_monomer_source_index_within_compatible_and_rank_agree(nat):
    from cfl.ranking import MonomerSourceCatalogIndex
    rng = np.random.default_rng(22)
    F, K, d, N, Q = 64, 4, 20, 40000, 40
    w = _weights(rng, F, K, d, gate=True)
    idx = MonomerSourceCatalogIndex.from_features(w, dev(np.maximum(rng.normal(size=(N, F)), 0)))
    xq = dev(np.maximum(rng.normal(size=(Q, F)), 0))
    tv = _agreement(idx, xq)
    _compatible(nat, idx, xq, tv, "monomer_source", idx.project_queries(xq), idx.a, w=idx.gate)


def _positives(rng, Q, N, J):
    pos = np.stack([rng.choice(N, J, replace=False) for _ in range(Q)]).astype(np.int64)
    pos[1, 2:] = -1
    return pos


@pytest.mark.gpu
def test_source_auc_per_query_against_the_oracle_and_across_shards(nat):
    from cfl.ranking import SourceCatalogIndex
    rng = np.random.default_rng(23)
    F, K, d, N, Q, J = 64, 2, 20, 8000, 24, 6
    w = _weights(rng, F, K, d)
    X = dev(np.maximum(rng.normal(size=(N, F)), 0))
    xq = dev(np.maximum(rng.normal(size=(Q, F)), 0))
    pos = _positives(rng, Q, N, J)
    idx = SourceCatalogIndex.from_features(w, X)
    fused = idx.auc_per_query(xq, dev(pos, torch.int64))
    direct = idx.auc_per_query(xq, dev(pos, torch.int64), method="direct")
    assert torch.equal(fused.counts, direct.counts) and torch.equal(fused.two_u, direct.two_u)
    D = src_dist(idx.project_queries(xq).cpu().numpy(), idx.P.cpu().numpy())
    two_u, n_pos, n_neg = O.per_query_auc(D.astype(np.float32), pos)
    assert fused.two_u.cpu().tolist() == two_u
    assert fused.n_pos.cpu().tolist() == n_pos and fused.n_neg.cpu().tolist() == n_neg
    # two shards, each with its own image, centred on the one global mean: the counts add up to one index's
    n1 = 3001
    a = SourceCatalogIndex(w, idx.P[:n1].reshape(n1, -1), idx_base=0, n_total=N)
    b = SourceCatalogIndex(w, idx.P[n1:].reshape(N - n1, -1), idx_base=n1, n_total=N)
    a.mu = b.mu = idx.mu
    a.image, b.image = nat.source_catalog_pack(a.P, idx.mu), nat.source_catalog_pack(b.P, idx.mu)
    ra, rb = a.auc_per_query(xq, dev(pos, torch.int64)), b.auc_per_query(xq, dev(pos, torch.int64))
    t = torch.where(torch.isnan(ra.pos_dist), rb.pos_dist, ra.pos_dist)
    assert torch.equal(t.nan_to_num(-1.0), fused.pos_dist.nan_to_num(-1.0))
    ca = nat.rank_counts_packed(idx.project_queries(xq), a.P, a.image, idx.mu, t, mode="pcd_source")
    cb = nat.rank_counts_packed(idx.project_queries(xq), b.P, b.image, idx.mu, t, mode="pcd_source")
    assert torch.equal(ca + cb, fused.counts)


@pytest.mark.gpu
def test_monomer_source_auc_per_query_against_the_oracle(nat):
    from cfl.ranking import MonomerSourceCatalogIndex
    rng = np.random.default_rng(24)
    F, K, d, N, Q, J = 64, 3, 16, 6000, 20, 5
    w = _weights(rng, F, K, d, gate=True)
    idx = MonomerSourceCatalogIndex.from_features(w, dev(np.maximum(rng.normal(size=(N, F)), 0)))
    xq = dev(np.maximum(rng.normal(size=(Q, F)), 0))
    pos = _positives(rng, Q, N, J)
    res = idx.auc_per_query(xq, dev(pos, torch.int64))
    D = msrc_dist(idx.project_queries(xq).cpu().numpy(), idx.a.cpu().numpy(), idx.gate.cpu().numpy())
    two_u, n_pos, n_neg = O.per_query_auc(D.astype(np.float32), pos)
    assert res.n_pos.cpu().tolist() == n_pos and res.n_neg.cpu().tolist() == n_neg
    # fp32 direct form against fp64 rounded: equal integers unless a positive sits within rounding of a negative
    assert np.abs(np.array(res.two_u.cpu().tolist()) - np.array(two_u)).max() <= 2


@pytest.mark.gpu
@pytest.mark.parametrize("rank_k", [100, 5000])
def test_source_within_one_million_rows(nat, rank_k):
    """2^20 sources, K = 3, d = 64, Q = 1024 targets, radii at the rank_k-th distance: sizes equal the packed counts,
    sampled distances equal pair_dist_rows, two calls are bit-identical."""
    rng = np.random.default_rng(633)
    N, K, d, Q = 1 << 20, 3, 64, 1024
    Pd = torch.randn(N, K, d, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    Ed = (Pd[torch.as_tensor(rng.integers(0, N, Q), device="cuda")].mean(1) + 0.5 * torch.randn(Q, d, device="cuda"))
    mu = Pd.double().mean((0, 1)).float()
    img = nat.source_catalog_pack(Pd, mu)
    probe = nat.score_topk_source(Ed, Pd, img, 128, mu=mu)[0]
    # radius with about rank_k rows: the 100th distance, or a quantile of sampled distances for 5000
    if rank_k <= 128:
        r = probe[:, rank_k - 1].contiguous()
    else:
        samp = torch.randint(0, N, (Q, 4096), device="cuda")
        sd = torch.cat([nat.pair_dist_rows("pcd_source", Ed, Pd, samp[:, j:j + 32].contiguous())
                        for j in range(0, 4096, 32)], 1)
        r = sd.kthvalue(int(4096 * rank_k / N) + 1, 1).values.contiguous()
    res = nat.score_within("pcd_source", Ed, Pd, r, image=img, mu=mu, want_stats=True)
    off, idx, val, st = res
    assert st["count_mismatch_queries"] == 0 and st["reemitted_queries"] == 0, st
    sizes = nat.rank_counts_packed(Ed, Pd, img, mu, r[:, None], mode="pcd_source")[:, 0, 0]
    assert torch.equal(off[1:] - off[:-1], sizes)
    mean = float(sizes.double().mean())
    assert 0.5 * rank_k <= mean <= 2.0 * rank_k, mean
    q = torch.searchsorted(off, torch.arange(int(off[-1]), device="cuda"), right=True) - 1
    pick = torch.randint(0, int(off[-1]), (4096,), device="cuda")
    qs, rows = q[pick], idx[pick]
    want = nat.pair_dist_rows("pcd_source", Ed[qs], Pd, rows[:, None]).squeeze(1)
    assert torch.equal(want, val[pick])
    again = nat.score_within("pcd_source", Ed, Pd, r, image=img, mu=mu)
    for a, b in zip(res[:3], again):
        assert torch.equal(a, b)


def _mgpu_worker(rank, world, port, out):
    for p in (ROOT, os.path.join(ROOT, "compatibility-family-learning_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from cfl import ranking
    X, w, Q, pos = _mgpu_data()
    lo, hi = ranking.shard_bounds(len(X), world, rank)
    idx = ranking.SourceCatalogIndex.from_features(w, X[lo:hi].cuda(), idx_base=lo, n_total=len(X))
    tv, _ = idx.rank(X[:Q].cuda(), 100)
    off, ii, vv = idx.within(X[:Q].cuda(), tv[:, 60].contiguous())
    auc = idx.auc_per_query(X[:Q].cuda(), pos.cuda())
    if rank == 0:
        torch.save(dict(off=off.cpu(), idx=ii.cpu(), val=vv.cpu(), r=tv[:, 60].cpu(), two_u=auc.two_u.cpu()), out)
    dist.destroy_process_group()


def _mgpu_data():
    rng = np.random.default_rng(4)
    N, F, K, d, Q = 60_000, 64, 3, 32, 50
    X = torch.as_tensor(np.maximum(rng.normal(size=(N, F)), 0).astype(np.float32))
    w = _weights(rng, F, K, d)
    return X, w, Q, torch.as_tensor(_positives(rng, Q, N, 4))


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_source_within_and_auc_two_gpus_equal_one(tmp_path):
    out = str(tmp_path / "w.pt")
    mp.spawn(_mgpu_worker, args=(2, 29300 + os.getpid() % 500, out), nprocs=2, join=True)
    got = torch.load(out)
    from cfl import ranking
    X, w, Q, pos = _mgpu_data()
    idx = ranking.SourceCatalogIndex.from_features(w, X.cuda())
    off, ii, vv = idx.within(X[:Q].cuda(), got["r"].cuda())
    assert torch.equal(off.cpu(), got["off"]) and torch.equal(ii.cpu(), got["idx"]) and torch.equal(vv.cpu(), got["val"])
    assert torch.equal(idx.auc_per_query(X[:Q].cuda(), pos.cuda()).two_u.cpu(), got["two_u"])


@pytest.mark.gpu
def test_pair_loss_and_topk_reject_the_source_modes(nat):
    """The source modes exist only for the rank-count and range-query entry points."""
    lib = nat.lib()
    B, K, d = 8, 2, 4
    a = torch.zeros(B, d, device="cuda")
    P = torch.zeros(B, K * d, device="cuda")
    out = torch.zeros(B, device="cuda")
    w = torch.full((B, K), 0.5, device="cuda")
    theta = torch.ones(1, device="cuda")
    ws = torch.zeros(lib.cfl_pair_workspace_bytes(B), dtype=torch.uint8, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    for mode in (3, 4):
        st = lib.cfl_pair_loss_fwd(mode, p(a), d, p(P), K * d, p(w), B, K, d, p(theta), 1, 0.0, p(out), None, None,
                                   None, p(ws), ws.numel(), None)
        assert st == -1, st
        tv = torch.zeros(1, 1, device="cuda")
        ti = torch.zeros(1, 1, dtype=torch.int64, device="cuda")
        wst = torch.zeros(lib.cfl_score_topk_workspace_bytes(1, K, d, 8, 1), dtype=torch.uint8, device="cuda")
        st = lib.cfl_score_topk(mode, p(P), 1, K, d, K * d, p(a), 8, d, None, 1, 0, p(tv), p(ti), None, p(wst),
                                wst.numel(), None)
        assert st == -3, st
