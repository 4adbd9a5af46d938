"""The other direction of the pcd distance: target e0 queries ranked against a catalog of source prototypes
(cfl_score_topk_source, cfl.ranking.SourceCatalogIndex), against the fp64 oracle with the roles swapped
(``all_pairs_dist_source`` below, on the oracle's ``all_pairs_dist``).

Bars are those of ``_check_topk`` in test_kernels_gpu.py with the roles swapped: the un-rescored Gram values within
1e-4*D + 8 eps32 (|e_q - mu|^2 + max_k |p_ck - mu|^2), the reported (direct-form) distances within 1e-4, index sets
equal except for near-ties of the k-th distance.  The SASS check at the end needs no GPU."""
import collections
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import cfl_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "compatibility-family-learning_b200", "cfl", "_lib", "libcfl_b200.so")
gpu = pytest.mark.gpu


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).cuda()


def host(t):
    return t.detach().cpu().numpy().astype(np.float64)


@pytest.fixture(scope="module")
def nat():
    from cfl import _native
    _native.lib()
    assert _native.device_info()[1] == 10, "these tests need a B200 (sm_100)"
    return _native


def all_pairs_dist_source(Eq, Pc, block=256):
    """dist[q,c] = pcd_dist(v=Eq[q], P=Pc[c]) -- cfl/models/base.py:125-139 with the roles of ``O.all_pairs_dist``
    swapped: the query is the TARGET item (its e0 ``Eq`` [Q,d]), the candidate the SOURCE item (its K prototypes
    ``Pc`` [N,K,d]).  ``O.all_pairs_dist(Pq, E)`` is pcd(v=E[c], P=Pq[q]) for every pair, so the transpose of
    ``O.all_pairs_dist(Pc, Eq)`` is this matrix.  pcd is not symmetric: for K > 1 it is not all_pairs_dist(Eq[:,None], ...)."""
    return O.all_pairs_dist(Pc, Eq, block=block).T.copy()


def _check_result(D, tv, ti, k):
    """Reported values are the exact distances of the reported rows (1e-4), listed in (value, index) order; index sets
    equal up to near-ties of the k-th distance.  Two reported values each within 1e-4 of the oracle may invert the
    oracle's order by at most 2e-4 of the distance."""
    kk = min(k, D.shape[1])
    want_v, want_i = O.rank_topk(D, kk)
    got = np.take_along_axis(D, ti[:, :kk], 1)
    np.testing.assert_allclose(tv[:, :kk], got, rtol=1e-4, atol=0, err_msg="rescored values")
    dv, di = np.diff(tv[:, :kk], axis=1), np.diff(ti[:, :kk], axis=1)
    assert ((dv > 0) | ((dv == 0) & (di > 0))).all(), "not in (value, index) order"
    for q in range(D.shape[0]):
        if (ti[q, :kk] == want_i[q]).all():
            continue
        kth = want_v[q, -1]
        for c in set(ti[q, :kk].tolist()) ^ set(want_i[q].tolist()):
            assert abs(D[q, c] - kth) <= 2e-6 * max(kth, 1.0) + 1e-7, f"q={q} cand {c} is not a near-tie"
        assert (np.diff(D[q, ti[q, :kk]]) >= -2e-4 * max(kth, 1.0)).all()
    if kk < k:
        assert (ti[:, kk:] == -1).all() and np.isinf(tv[:, kk:]).all()


def _check_source_topk(nat, Eq, Pc, k, mu=None, D=None):
    """Dense call (single adaptive pass): Gram bar and result; then the plain call (the sampled cascade on long
    catalogs): result.  Returns the plain call's (values, indices)."""
    if D is None:
        D = all_pairs_dist_source(Eq.astype(np.float64), Pc.astype(np.float64))
    mud = None if mu is None else dev(mu)
    image = nat.source_catalog_pack(dev(Pc), mud)
    tv, ti, dense = nat.score_topk_source(dev(Eq), dev(Pc), image, k, mu=mud, want_dense=True)
    c = np.zeros(Eq.shape[1]) if mu is None else mu.astype(np.float64)
    e2 = ((Eq - c) ** 2).sum(-1)
    p2 = ((Pc - c) ** 2).sum(-1).max(-1)
    tol = 1e-4 * D + 8 * np.finfo(np.float32).eps * (e2[:, None] + p2[None, :])
    dense = host(dense)
    assert (np.abs(dense - D) <= tol).all(), f"gram-form error {np.max(np.abs(dense - D) / tol):.2f}x tolerance"
    _check_result(D, host(tv), ti.cpu().numpy(), k)
    tv, ti = nat.score_topk_source(dev(Eq), dev(Pc), image, k, mu=mud)
    tv, ti = host(tv), ti.cpu().numpy()
    _check_result(D, tv, ti, k)
    return tv, ti


def _data(rng, Q, K, d, N, offset=0.0):
    Pc = (rng.normal(size=(N, K, d)) + offset).astype(np.float32)
    # targets near some source's prototype hull, so that the soft-min is not one-hot everywhere
    Eq = (Pc[rng.integers(0, N, Q)].mean(1) + 0.5 * rng.normal(size=(Q, d))).astype(np.float32)
    return Eq, Pc


# Single-pass / two-pass: the sampled cascade runs when a catalog part has >= 16 tiles of 128 rows (parts = 148 / query
# tiles): (1, 1, 64, 400000), (33, 1, 128, 320000) and (2, 8, 64, 320000) have 21, 16 and 16 tiles per part,
# (1024, 5, 20, 20000) 26 (and a ragged last query tile: QT = 48), the others one pass.  (3, 4, 20, 50, 100) has N < k.
@gpu
@pytest.mark.parametrize("Q,K,d,N,k", [(1, 1, 64, 400000, 100), (33, 1, 128, 320000, 100), (33, 2, 20, 5000, 100),
                                       (130, 3, 64, 2500, 1), (130, 3, 64, 40000, 128), (1024, 5, 20, 20000, 100),
                                       (5, 8, 128, 3000, 50), (20, 5, 10, 129, 128), (3, 4, 20, 50, 100),
                                       (64, 4, 10, 7000, 128), (2, 8, 64, 320000, 100)])
def test_source_topk_shapes(nat, Q, K, d, N, k):
    rng = np.random.default_rng(Q * 7 + K * 11 + d + N)
    Eq, Pc = _data(rng, Q, K, d, N)
    _check_source_topk(nat, Eq, Pc, k)


@gpu
def test_source_duplicates_rank_lower_index_first_and_calls_are_deterministic(nat):
    rng = np.random.default_rng(31)
    Eq, Pc = _data(rng, 40, 3, 20, 6000)
    Pc[100] = Pc[7]
    Pc[650] = Pc[7]
    Eq[::4] = Pc[7, 0] + 0.01 * rng.normal(size=(10, 20)).astype(np.float32)     # on a prototype of the duplicates
    tv, ti = _check_source_topk(nat, Eq, Pc, 100)
    seen = 0
    for q in range(ti.shape[0]):
        pos = {c: int(np.where(ti[q] == c)[0][0]) for c in (7, 100, 650) if c in ti[q]}
        if len(pos) == 3:
            assert pos[7] < pos[100] < pos[650]
            seen += 1
    assert seen == 10
    image = nat.source_catalog_pack(dev(Pc))
    a = nat.score_topk_source(dev(Eq), dev(Pc), image, 100)
    b = nat.score_topk_source(dev(Eq), dev(Pc), image, 100)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@gpu
def test_source_offset_catalog_with_centring(nat):
    """+10 common offset on both sides: the Gram form holds its bar once both sides are centred on mu."""
    rng = np.random.default_rng(99)
    Eq, Pc = _data(rng, 16, 4, 64, 4000, offset=10.0)
    mu = Pc.astype(np.float64).reshape(-1, 64).mean(0).astype(np.float32)
    _check_source_topk(nat, Eq, Pc, 100, mu=mu)


@pytest.fixture(scope="module")
def knob_case():
    rng = np.random.default_rng(8)
    Eq, Pc = _data(rng, 40, 3, 20, 400000)              # 21 tiles per catalog part: the sampled cascade
    return Eq, Pc, all_pairs_dist_source(Eq.astype(np.float64), Pc.astype(np.float64))


@gpu
@pytest.mark.parametrize("env", [{"CFL_SCORE_NO_CASCADE": "1"}, {"CFL_SCORE_NO_OPTIMISTIC": "1"},
                                 {"CFL_SCORE_OPT_MULT": "1"}])
def test_source_knobs_force_the_redo_path(nat, monkeypatch, knob_case, env):
    """The knobs steer the cascade, never the result.  Under CFL_SCORE_OPT_MULT=1 the optimistic threshold lets only
    about kk/8 rows through, so queries fail verification and are redone exactly (stats prove it)."""
    for kv in env.items():
        monkeypatch.setenv(*kv)
    Eq, Pc, D = knob_case
    image = nat.source_catalog_pack(dev(Pc))
    tv, ti, st = nat.score_topk_source(dev(Eq), dev(Pc), image, 100, want_stats=True)
    _check_result(D, host(tv), ti.cpu().numpy(), 100)
    stats = dict(zip(nat.SCORE_STAT_NAMES, st.tolist()))
    assert stats["survivors"] > 0 and stats["lower_bound_pass"] == 0
    if "CFL_SCORE_OPT_MULT" in env:
        assert stats["redo_queries"] > 0, stats


@gpu
def test_source_k1_equals_forward_with_roles_swapped(nat):
    """K = 1: pcd(v = e_q, p = p_c) = |e_q - p_c|^2 = the forward call with catalog = prototypes and queries =
    embeddings; both rescore the same rows in the same arithmetic, so values and indices agree bit for bit."""
    rng = np.random.default_rng(12)
    Eq, Pc = _data(rng, 300, 1, 64, 200000)
    mu = dev(Pc[:, 0].astype(np.float64).mean(0).astype(np.float32))
    P2 = dev(Pc[:, 0])
    fv, fi = nat.score_topk(dev(Eq)[:, None, :], P2, 100, mu=mu, image=nat.catalog_pack(P2, 1, mu))
    sv, si = nat.score_topk_source(dev(Eq), dev(Pc), nat.source_catalog_pack(dev(Pc), mu), 100, mu=mu)
    assert torch.equal(fi, si)
    assert torch.equal(fv.view(torch.int32), sv.view(torch.int32))


@gpu
def test_source_c3_shape_sampled_queries(nat):
    """C3 shape: 1024 target queries against 2^20 source rows, K = 3, d = 64, k = 100; 8 queries checked against the
    oracle over the whole catalog."""
    Q, K, d, N, k = 1024, 3, 64, 1 << 20, 100
    g = torch.Generator(device="cuda").manual_seed(3)
    Pc = torch.randn(N, K, d, device="cuda", generator=g)
    Eq = Pc[torch.randint(0, N, (Q,), device="cuda", generator=g)].mean(1) + 0.5 * torch.randn(Q, d, device="cuda",
                                                                                                 generator=g)
    mu = Pc.view(-1, d).double().mean(0).float()
    tv, ti = nat.score_topk_source(Eq, Pc, nat.source_catalog_pack(Pc, mu), k, mu=mu)
    sample = np.arange(0, Q, Q // 8)
    Pn, Es = Pc.cpu().numpy(), Eq.cpu().numpy()[sample].astype(np.float64)
    D = np.empty((len(sample), N))
    for lo in range(0, N, 1 << 17):
        D[:, lo:lo + (1 << 17)] = all_pairs_dist_source(Es, Pn[lo:lo + (1 << 17)].astype(np.float64))
    _check_result(D, host(tv)[sample], ti.cpu().numpy()[sample], k)


@gpu
def test_source_catalog_index_from_features_and_shards(nat):
    from cfl.ranking import EncoderWeights, SourceCatalogIndex
    rng = np.random.default_rng(21)
    F, K, d, N, Q, k = 96, 3, 32, 30000, 50, 100
    w = EncoderWeights(V0=dev(O.xavier_uniform(rng, F, d)), Vp=dev(O.xavier_uniform(rng, F, K * d)),
                       g0=dev(np.ones(d)), gp=dev(np.ones(K * d)), b0=dev(0.1 * rng.normal(size=d)),
                       bp=dev(0.1 * rng.normal(size=K * d)), weight_norm=True, act="tanh")
    Xc = dev(np.maximum(rng.normal(size=(N, F)), 0))
    Xq = dev(np.maximum(rng.normal(size=(Q, F)), 0))
    idx = SourceCatalogIndex.from_features(w, Xc)
    tv, ti = idx.rank(Xq, k)
    # the oracle on the projected features: target e0 of the queries, source prototypes of the catalog
    E, P = host(idx.project_queries(Xq)), host(idx.P)
    D = all_pairs_dist_source(E, P)
    _check_result(D, host(tv), ti.cpu().numpy(), k)
    n1 = 11111
    a = SourceCatalogIndex.from_features(w, Xc[:n1], idx_base=0, n_total=N)
    b = SourceCatalogIndex.from_features(w, Xc[n1:], idx_base=n1, n_total=N)
    va, ia = a.rank(Xq, k)
    vb, ib = b.rank(Xq, k)
    mv, mi = nat.topk_merge(torch.stack([va, vb]), torch.stack([ia, ib]))
    assert torch.equal(mi, ti) and torch.equal(mv, tv)


# ---------------------------------------------------------------------------------------------- no GPU
def test_source_kernel_is_tcgen05_code_and_spill_free_for_small_K():
    """score_src_umma_kernel<K>: tcgen05.mma (UTCHMMA), tcgen05.ld (LDTM), bulk TMA (UBLKCP) for every K, no
    local-memory traffic (STL / LDL) for K <= 4."""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    filt = shutil.which("c++filt")
    if not os.path.exists(cuobjdump) or filt is None:
        pytest.skip("cuobjdump / c++filt not available")
    sass = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, timeout=600, check=True).stdout
    per, fn = collections.defaultdict(collections.Counter), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            fn = m.group(1) if "score_src_umma_kernel" in m.group(1) else None
            continue
        if fn is not None:
            for op in ("UTCHMMA", "LDTM", "UBLKCP", "STL", "LDL"):
                if re.search(r"\b%s\b" % op, line):
                    per[fn][op] += 1
    names = subprocess.run([filt], input="\n".join(per), capture_output=True, text=True, check=True).stdout.splitlines()
    census = {re.sub(r"\(.*", "", re.sub(r"^void ", "", nice)): per[m] for m, nice in zip(per, names)}
    for K in range(1, 9):
        kern = f"cfl::score_src_umma_kernel<{K}>"
        assert kern in census, f"{kern} not in the library"
        for op in ("UTCHMMA", "LDTM", "UBLKCP"):
            assert census[kern][op] > 0, f"{kern}: no {op} in its SASS"
        if K <= 4:
            assert census[kern]["STL"] == 0 and census[kern]["LDL"] == 0, f"{kern}: local-memory traffic"
