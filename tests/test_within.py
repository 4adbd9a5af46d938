"""Catalog range queries (cfl_score_within, CatalogIndex.within / compatible): every row with dist(q, c) < r_q, exact, as
CSR lists ordered by (distance, index).

CPU: the SASS of the emitting tensor-core kernel, the sharded assembly on a gloo world-2 group with oracle-backed kernel
doubles, the size guard, and the no-GPU failure mode of the new entry points.  GPU: the definition (sets, bits, order,
sizes) against pair_dist_rows / rank_counts on both routes, exact ties, monomer, the overflow and large-segment paths,
edges, the 1 M-row shape, compatible(), agreement with rank(), and two GPUs."""
import collections
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


def test_emitting_kernel_is_tcgen05_code_without_spills(census):
    for K in range(1, 9):
        k = f"cfl::within_emit_umma_kernel<{K}>"
        assert k in census, f"{k} not in the library"
        for op in ("UTCHMMA", "LDTM", "UBLKCP"):
            assert census[k][op] > 0, f"{k}: no {op} in its SASS"
    k3 = census["cfl::within_emit_umma_kernel<3>"]
    assert k3["STL"] == 0 and k3["LDL"] == 0, k3


def _dense(query, catalog):
    return O.all_pairs_dist(query.numpy().astype(np.float64), catalog.numpy().astype(np.float64)).astype(np.float32)


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


def _doubles(nat):
    """Oracle-backed stand-ins for the kernels (fp64 distances rounded to fp32; same CSR contract)."""
    def within_counts(mode, query, catalog, radius, w=None, image=None, mu=None):
        if catalog.shape[0] == 0:
            return torch.zeros(query.shape[0], dtype=torch.int64)
        with np.errstate(invalid="ignore"):
            return torch.as_tensor((_dense(query, catalog) < radius.numpy()[:, None]).sum(1).astype(np.int64))

    def score_within(mode, query, catalog, radius, w=None, image=None, mu=None, idx_base=0,
                     max_results=nat.WITHIN_MAX_RESULTS, want_stats=False, counts=None):
        D = _dense(query, catalog) if catalog.shape[0] else np.zeros((query.shape[0], 0), np.float32)
        off, idx, val = _csr_reference(D, radius.numpy(), idx_base)
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

    nat.within_counts, nat.score_within, nat.within_merge = within_counts, score_within, within_merge


def _case():
    rng = np.random.default_rng(12)
    N, K, d, Q = 301, 3, 6, 9
    E = np.round(rng.normal(size=(N, d)), 1).astype(np.float32)
    Pq = np.round(rng.normal(size=(Q, K, d)), 1).astype(np.float32)
    D = O.all_pairs_dist(Pq.astype(np.float64), E.astype(np.float64)).astype(np.float32)
    r = np.sort(D, 1)[np.arange(Q), rng.integers(0, 60, Q)]        # radii on a row's distance: ties on the boundary
    r[2] = np.nan
    r[3] = 0.0
    return E, Pq, r


def _within_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    for p in (ROOT, os.path.join(ROOT, "compatibility-family-learning_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from cfl import ranking
    _doubles(ranking.nat)
    E, Pq, r = _case()
    lo, hi = ranking.shard_bounds(E.shape[0], world, rank)
    off, idx, val = ranking._within("pcd", torch.as_tensor(Pq), torch.as_tensor(E[lo:hi]), None, torch.as_tensor(r),
                                    lo, None, world, 1 << 20)
    try:
        ranking._within("pcd", torch.as_tensor(Pq), torch.as_tensor(E[lo:hi]), None, torch.as_tensor(r), lo, None,
                        world, int(off[-1]) - 1)
        guard = False
    except ranking.nat.CflNativeError as e:
        guard = str(int(off[-1])) in str(e)
    if rank == 0:
        np.savez(os.path.join(out_dir, "w.npz"), off=off.numpy(), idx=idx.numpy(), val=val.numpy(), guard=guard)
    dist.destroy_process_group()


def test_sharded_within_world2_gloo_matches_single_process(tmp_path):
    """Counts all-gathered, per-rank lists padded, gathered and merged: the same CSR as one process, and the size guard
    sees the whole result."""
    port = 31700 + os.getpid() % 2000
    mp.spawn(_within_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    got = np.load(tmp_path / "w.npz")
    E, Pq, r = _case()
    D = O.all_pairs_dist(Pq.astype(np.float64), E.astype(np.float64)).astype(np.float32)
    off, idx, val = _csr_reference(D, r)
    np.testing.assert_array_equal(got["off"], off)
    np.testing.assert_array_equal(got["idx"], idx)
    np.testing.assert_array_equal(got["val"], val)
    assert off[3] - off[2] == 0 and off[4] - off[3] == 0                # NaN and r = 0: empty lists
    assert bool(got["guard"])


def test_single_process_within_and_size_guard():
    from cfl import ranking
    saved = (ranking.nat.within_counts, ranking.nat.score_within, ranking.nat.within_merge)
    try:
        _doubles(ranking.nat)
        E, Pq, r = _case()
        off, idx, val = ranking._within("pcd", torch.as_tensor(Pq), torch.as_tensor(E), None, torch.as_tensor(r), 5,
                                        None, 1, 1 << 20)
        D = O.all_pairs_dist(Pq.astype(np.float64), E.astype(np.float64)).astype(np.float32)
        want = _csr_reference(D, r, 5)
        for a, b in zip((off, idx, val), want):
            np.testing.assert_array_equal(a.numpy(), b)
        with pytest.raises(ranking.nat.CflNativeError, match=str(int(off[-1]))):
            ranking._within("pcd", torch.as_tensor(Pq), torch.as_tensor(E), None, torch.as_tensor(r), 5, None, 1,
                            int(off[-1]) - 1)
    finally:
        ranking.nat.within_counts, ranking.nat.score_within, ranking.nat.within_merge = saved


def test_compatible_radius_is_the_thresholder_boundary():
    from cfl.ranking import compatible_radius
    for theta in (1e-9, 1e-6, 0.3, 2.5, 17.0):
        r = np.float32(compatible_radius(theta))
        d = np.array([np.nextafter(r, np.float32(0)), r, np.nextafter(r, np.float32(np.inf))], np.float32)
        score = np.float32(max(theta, 1e-6)) - d                      # CatalogIndex.scores in fp32
        assert ((score > 0) == (d < r)).all()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_within_entry_points_fail_loudly_without_a_gpu():
    from cfl import _native
    lib = _native.lib()
    assert lib.cfl_score_within(0, None, 1, 2, 4, 8, None, None, None, 8, 4, None, None, None, 0, None, None, None, 0,
                                None) == -5
    assert lib.cfl_score_within_stats(None, 0, None, None) == -5
    assert lib.cfl_within_merge(None, None, None, 4, 2, 1, None, None, None, None) == -5
    assert lib.cfl_score_within_workspace_bytes(0, 1024, 3, 64, 1 << 20) > 0
    with pytest.raises(_native.CflNativeError):
        _native.score_within("pcd", torch.zeros(2, 3, 4), torch.zeros(5, 4), 1.0)


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
    """[Q, N] direct-form distances through pair_dist_rows, 32 rows per call."""
    Q, N = query.shape[0], catalog.shape[0]
    out = torch.empty(Q, N, dtype=torch.float32, device="cuda")
    for lo in range(0, N, chunk):
        hi = min(N, lo + chunk)
        pos = torch.arange(lo, hi, device="cuda")[None, :].expand(Q, hi - lo).contiguous()
        out[:, lo:hi] = nat.pair_dist_rows(mode, query, catalog, pos, w=w)
    return out


def _check_definition(nat, res, D, r, idx_base=0):
    """res == the CSR of {c : D[q, c] < r_q}: sets, distance bits, (dist, index) order."""
    off, idx, val = (t.cpu().numpy() for t in res[:3])
    woff, widx, wval = _csr_reference(D, r, idx_base)
    np.testing.assert_array_equal(off - off[0], woff)
    np.testing.assert_array_equal(idx, widx)
    assert val.view(np.uint32).tolist() == wval.view(np.uint32).tolist()


def _planted_radii(rng, D, hi=300):
    Q, N = D.shape
    srt = np.sort(D, 1)
    return srt[np.arange(Q), rng.integers(0, min(hi, N), Q)]         # the distance of a row: ties sit on the boundary


@pytest.mark.gpu
@pytest.mark.parametrize("K,d,Q,N", [(1, 10, 37, 3001), (2, 20, 70, 5003), (3, 64, 70, 7001), (4, 128, 33, 4099),
                                     (8, 20, 19, 2050), (3, 10, 65, 3333), (2, 64, 130, 1000)])
def test_within_definition_parity(nat, K, d, Q, N):
    rng = np.random.default_rng(K * 100 + d + Q)
    E = rng.normal(size=(N, d)).astype(np.float32)
    Pq = (E[rng.integers(0, N, Q)][:, None, :] + 0.5 * rng.normal(size=(Q, K, d))).astype(np.float32)
    Ed, Pd = dev(E), dev(Pq)
    D = _pair_dense(nat, "pcd", Pd, Ed).cpu().numpy()
    r = _planted_radii(rng, D)
    mu = nat.col_mean(Ed)
    img = nat.catalog_pack(Ed, K, mu)
    res = nat.score_within("pcd", Pd, Ed, dev(r), image=img, mu=mu, idx_base=7, want_stats=True)
    _check_definition(nat, res, D, r, 7)
    assert res[3]["count_mismatch_queries"] == 0 and res[3]["reemitted_queries"] == 0, res[3]
    if img is not None:
        assert res[3]["worst_ratio"] < 0.5, res[3]
    sizes = nat.rank_counts("pcd", Pd, Ed, dev(r)[:, None])[:, 0, 0]
    assert torch.equal(res[0][1:] - res[0][:-1], sizes)
    core = nat.score_within("pcd", Pd, Ed, dev(r), idx_base=7)          # the CUDA-core route: the same result
    for a, b in zip(res[:3], core):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_within_exact_ties_on_integer_inputs(nat):
    """Integer-valued inputs: every fp32 distance is an exact integer, the radius sits on a tie value, strict < leaves
    every tied row out -- bit-exact against numpy, on both routes."""
    rng = np.random.default_rng(5)
    N, d, Q = 5000, 10, 40
    E = rng.integers(-2, 3, size=(N, d)).astype(np.float32)
    for K in (1, 2, 4):
        p = rng.integers(-2, 3, size=(Q, 1, d)).astype(np.float32)
        Pq = np.repeat(p, K, axis=1)
        D = O.all_pairs_dist(Pq.astype(np.float64), E.astype(np.float64))
        assert (D == np.round(D)).all()
        r = np.sort(D, 1)[np.arange(Q), rng.integers(0, 400, Q)].astype(np.float32)
        Ed, Pd = dev(E), dev(Pq)
        mu = nat.col_mean(Ed)
        img = nat.catalog_pack(Ed, K, mu)
        got = nat.score_within("pcd", Pd, Ed, dev(r), image=img, mu=mu)
        _check_definition(nat, got, D.astype(np.float32), r)
        core = nat.score_within("pcd", Pd, Ed, dev(r))
        for a, b in zip(got, core):
            assert torch.equal(a, b)


@pytest.mark.gpu
def test_within_against_the_fp64_oracle(nat):
    """Sets equal the fp64 oracle's except rows within 1e-5 relative of r_q."""
    rng = np.random.default_rng(6)
    K, d, Q, N = 3, 64, 50, 20000
    E = rng.normal(size=(N, d)).astype(np.float32)
    Pq = (E[rng.integers(0, N, Q)][:, None, :] + 0.5 * rng.normal(size=(Q, K, d))).astype(np.float32)
    D = O.all_pairs_dist(Pq.astype(np.float64), E.astype(np.float64))
    r = np.sort(D, 1)[:, 500].astype(np.float32)
    Ed = dev(E)
    mu = nat.col_mean(Ed)
    off, idx, _ = (t.cpu().numpy() for t in nat.score_within("pcd", dev(Pq), Ed, dev(r), image=nat.catalog_pack(Ed, K, mu),
                                                             mu=mu))
    for q in range(Q):
        got = set(idx[off[q]:off[q + 1]].tolist())
        want = set(np.nonzero(D[q] < r[q])[0].tolist())
        for c in got ^ want:
            assert abs(D[q, c] - r[q]) <= 1e-5 * r[q]


@pytest.mark.gpu
@pytest.mark.parametrize("K,d,Q,N", [(4, 20, 21, 3001), (3, 8, 9, 1000), (2, 32, 66, 2049)])
def test_within_monomer(nat, K, d, Q, N):
    rng = np.random.default_rng(K + d + Q + N)
    Pt = rng.normal(size=(N, K, d)).astype(np.float32)
    a = (Pt[rng.integers(0, N, Q), 0] + 0.5 * rng.normal(size=(Q, d))).astype(np.float32)
    w = O.softmax(rng.normal(size=(Q, K))).astype(np.float32)
    ad, Ptd, wd = dev(a), dev(Pt), dev(w)
    D = _pair_dense(nat, "monomer", ad, Ptd, w=wd).cpu().numpy()
    r = _planted_radii(rng, D)
    res = nat.score_within("monomer", ad, Ptd, dev(r), w=wd, idx_base=11, want_stats=True)
    _check_definition(nat, res, D, r, 11)
    assert res[3]["count_mismatch_queries"] == 0
    sizes = nat.rank_counts("monomer", ad, Ptd, dev(r)[:, None], w=wd)[:, 0, 0]
    assert torch.equal(res[0][1:] - res[0][:-1], sizes)


@pytest.mark.gpu
def test_within_record_overflow_and_large_segments(nat, monkeypatch):
    """A record list too small for the band pairs: the affected queries are re-emitted on the CUDA cores, the result is
    unchanged.  Segments beyond the shared-memory sort (one query selects every row) are sorted in global memory."""
    rng = np.random.default_rng(9)
    K, d, Q, N = 3, 16, 40, 40000
    E = rng.integers(-2, 3, size=(N, d)).astype(np.float32)
    Pq = rng.integers(-2, 3, size=(Q, K, d)).astype(np.float32)
    Ed, Pd = dev(E), dev(Pq)
    D = _pair_dense(nat, "pcd", Pd, Ed).cpu().numpy()
    r = _planted_radii(rng, D, hi=3000)
    r[0] = np.inf                                                    # 40000 rows: the global-memory sort
    r[1] = np.sort(D[1])[20000]                                      # ~20000 rows
    r[2] = np.sort(D[2])[5000]                                       # a segment for the 1024-thread shared-memory sort
    mu = nat.col_mean(Ed)
    img = nat.catalog_pack(Ed, K, mu)
    base = nat.score_within("pcd", Pd, Ed, dev(r), image=img, mu=mu, want_stats=True)
    _check_definition(nat, base, D, r)
    assert int(base[0][1] - base[0][0]) == N
    monkeypatch.setenv("CFL_EXPERIMENTS", "1")
    monkeypatch.setenv("CFL_RANK_REC_CAP", "64")
    small = nat.score_within("pcd", Pd, Ed, dev(r), image=img, mu=mu, want_stats=True)
    assert small[3]["reemitted_queries"] > 0 and small[3]["count_mismatch_queries"] == 0, small[3]
    for a, b in zip(base[:3], small[:3]):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_within_edges(nat):
    rng = np.random.default_rng(4)
    K, d, Q, N = 3, 32, 10, 2000
    E = rng.normal(size=(N, d)).astype(np.float32)
    Pq = rng.normal(size=(Q, K, d)).astype(np.float32)
    Ed, Pd = dev(E), dev(Pq)
    mu = nat.col_mean(Ed)
    img = nat.catalog_pack(Ed, K, mu)
    for image in (img, None):
        for r in (0.0, -1.0, float("nan")):                          # below every distance / NaN: empty lists
            off, idx, val = nat.score_within("pcd", Pd, Ed, r, image=image, mu=mu)
            assert off.tolist() == [0] * (Q + 1) and idx.numel() == 0 and val.numel() == 0
    off, idx, val = nat.score_within("pcd", Pd, Ed[:0], 1e30)        # an empty shard
    assert off.tolist() == [0] * (Q + 1) and idx.numel() == 0
    off, idx, val = nat.score_within("pcd", Pd[:0], Ed, 1e30, image=img, mu=mu)   # Q = 0
    assert off.tolist() == [0] and idx.numel() == 0
    with pytest.raises(nat.CflNativeError, match=str(Q * N)):        # the size guard, before any output exists
        nat.score_within("pcd", Pd, Ed, float("inf"), image=img, mu=mu, max_results=Q * N - 1)


def _c3_index(nat, N=1 << 20, Q=1024, K=3, d=64, F=64, seed=633):
    from cfl.ranking import CatalogIndex, EncoderWeights
    rng = np.random.default_rng(seed)
    w = EncoderWeights(V0=dev(O.xavier_uniform(rng, F, d)), Vp=dev(O.xavier_uniform(rng, F, K * d)),
                       g0=torch.ones(d).cuda(), gp=torch.ones(K * d).cuda(), b0=torch.zeros(d).cuda(),
                       bp=torch.zeros(K * d).cuda())
    X = torch.relu(torch.randn(N, F, generator=torch.Generator().manual_seed(seed))).cuda()
    return CatalogIndex.from_features(w, X), X[:Q].contiguous()


@pytest.mark.gpu
def test_within_one_million_rows(nat):
    """C3 shape (1024 queries x 2^20 rows, K = 3, d = 64) at ~100 and ~5000 rows per query: sizes equal the counts of
    rank_counts_packed, no count mismatch, sampled distances equal pair_dist_rows, two calls are bit-identical."""
    index, xq = _c3_index(nat)
    Pq = index.project_queries(xq)
    tv, _ = index.rank(xq, 100)
    samp = torch.randint(0, index.E.shape[0], (Pq.shape[0], 2048), device="cuda")
    sd = torch.cat([nat.pair_dist_rows("pcd", Pq, index.E, samp[:, i:i + 32].contiguous()) for i in range(0, 2048, 32)], 1)
    for r in (tv[:, 99].contiguous(), torch.quantile(sd, 5000 / index.E.shape[0], dim=1).float().contiguous()):
        off, idx, val, st = nat.score_within("pcd", Pq, index.E, r, image=index.image, mu=index.mu, want_stats=True)
        assert st["count_mismatch_queries"] == 0, st
        cnt = nat.rank_counts_packed(Pq, index.E, index.image, index.mu, r[:, None])[:, 0, 0]
        assert torch.equal(off[1:] - off[:-1], cnt)
        n = off[1:] - off[:-1]
        print("rows per query: mean %.1f min %d max %d" % (n.double().mean(), n.min(), n.max()))
        q = torch.arange(Pq.shape[0], device="cuda")
        have = n > 0
        pick = off[:-1] + (torch.randint(0, 1 << 30, (Pq.shape[0],), device="cuda") % n.clamp(min=1))
        pos = torch.where(have, idx[pick.clamp(max=max(idx.numel() - 1, 0))], torch.full_like(q, -1))
        t = nat.pair_dist_rows("pcd", Pq, index.E, pos[:, None])[:, 0]
        assert torch.equal(t[have], val[pick[have]])
        again = nat.score_within("pcd", Pq, index.E, r, image=index.image, mu=index.mu)
        for a, b in zip((off, idx, val), again):
            assert torch.equal(a, b)


@pytest.mark.gpu
def test_compatible_and_agreement_with_rank(nat):
    """compatible(): every returned row scores > 0, sampled other rows <= 0.  within(r = k-th distance of rank(k))
    agrees with rank's index set except rows within 1e-5 relative of r."""
    from cfl.ranking import compatible_radius
    index, xq = _c3_index(nat, N=200003, Q=70)
    Pq = index.project_queries(xq)
    tv, ti = index.rank(xq, 100)
    index.theta = float(tv[:, 40].median())
    off, idx, val = index.compatible(xq)
    assert (index.scores(val) > 0).all()
    n = (off[1:] - off[:-1]).cpu()
    assert n.sum() > 0
    samp = torch.randint(0, index.E.shape[0], (Pq.shape[0], 32), device="cuda")
    sd = nat.pair_dist_rows("pcd", Pq, index.E, samp)
    offc, idxc = off.cpu().numpy(), idx.cpu().numpy()
    for q in range(Pq.shape[0]):
        inside = set(idxc[offc[q]:offc[q + 1]].tolist())
        for j in range(32):
            if int(samp[q, j]) not in inside:
                assert float(index.scores(sd[q, j])) <= 0
    r = np.float32(compatible_radius(index.theta))
    assert (val < torch.tensor(r, device="cuda")).all()
    k = 100
    off, idx, val = index.within(xq, tv[:, k - 1].contiguous())
    offc, idxc, valc = off.cpu().numpy(), idx.cpu().numpy(), val.cpu().numpy()
    tvc, tic = tv.cpu().numpy(), ti.cpu().numpy()
    for q in range(Pq.shape[0]):
        dist_of = dict(zip(tic[q].tolist(), tvc[q].tolist()))
        dist_of.update(zip(idxc[offc[q]:offc[q + 1]].tolist(), valc[offc[q]:offc[q + 1]].tolist()))
        got, want = set(idxc[offc[q]:offc[q + 1]].tolist()), set(tic[q].tolist())
        rq = float(tvc[q, k - 1])
        for c in got ^ want:
            assert abs(dist_of[c] - rq) <= 1e-5 * rq, (q, c, dist_of[c], rq)


def _mgpu_worker(rank, world, port, out):
    for p in (ROOT, os.path.join(ROOT, "compatibility-family-learning_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from cfl import ranking
    X, w, Q = _mgpu_data()
    lo, hi = ranking.shard_bounds(len(X), world, rank)
    idx = ranking.CatalogIndex.from_features(w, X[lo:hi].cuda(), idx_base=lo, n_total=len(X))
    tv, _ = idx.rank(X[:Q].cuda(), 100)
    off, ii, vv = idx.within(X[:Q].cuda(), tv[:, 60].contiguous())
    if rank == 0:
        torch.save(dict(off=off.cpu(), idx=ii.cpu(), val=vv.cpu(), r=tv[:, 60].cpu(), mu=idx.mu.cpu()), out)
    dist.destroy_process_group()


def _mgpu_data():
    from cfl.ranking import EncoderWeights
    rng = np.random.default_rng(3)
    N, F, K, d, Q = 60_000, 64, 3, 32, 50
    X = torch.as_tensor(np.maximum(rng.normal(size=(N, F)), 0).astype(np.float32))
    c = lambda a: torch.as_tensor(a).cuda()
    w = EncoderWeights(V0=c(O.xavier_uniform(rng, F, d)), Vp=c(O.xavier_uniform(rng, F, K * d)),
                       g0=torch.ones(d).cuda(), gp=torch.ones(K * d).cuda(), b0=torch.zeros(d).cuda(),
                       bp=torch.zeros(K * d).cuda())
    return X, w, Q


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_within_two_gpus_equals_one(tmp_path):
    out = str(tmp_path / "w.pt")
    mp.spawn(_mgpu_worker, args=(2, 29800 + os.getpid() % 1000, out), nprocs=2, join=True)
    got = torch.load(out)
    from cfl import ranking
    X, w, Q = _mgpu_data()
    idx = ranking.CatalogIndex.from_features(w, X.cuda(), mu=got["mu"].cuda())
    off, ii, vv = idx.within(X[:Q].cuda(), got["r"].cuda())
    assert torch.equal(off.cpu(), got["off"]) and torch.equal(ii.cpu(), got["idx"]) and torch.equal(vv.cpu(), got["val"])
