"""The other direction of the monomer distance: target queries (K prototypes each) ranked against a catalog of source
items (a, gate w) -- cfl_score_topk_monomer_source, cfl.ranking.MonomerSourceCatalogIndex -- against the fp64 oracle
with the roles swapped: ``O.all_pairs_monomer_dist(a_src, w_src, P_tgt).T``.

Bars are those of test_monomer_allpairs.py: reported distances within 1e-4 of the oracle, index sets equal except for
near-ties of the k-th distance.  Both routes (the tensor-core filter over the packed image, and the CUDA-core kernel
with image = None) rescore in the same fp32 arithmetic, so they must agree bit for bit; which route ran is read from a
torch.profiler trace.  The SASS check at the end needs no GPU."""
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
RTOL = 1e-4
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


def kernel_name(raw):
    """Profiler kernel name -> 'cfl::kernel<args>' (no return type, no parameter list)."""
    if raw.startswith("_Z") and shutil.which("c++filt"):
        raw = subprocess.run(["c++filt", raw], capture_output=True, text=True).stdout.strip()
    raw = re.sub(r"^void ", "", raw)
    return re.sub(r"\([^()]*\)$", "", raw)


def traced(fn):
    """(fn's result, set of kernel names it launched).  A profiler session that delivered no GPU kernel record at all
    (only the CPU-side runtime calls came back) is run again, up to three times; fn is deterministic, so the result of
    the last run is the result."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        names = {kernel_name(e.name) for e in prof.events()}
        if any(n.startswith("cfl::") for n in names):
            break
    return out, names


def oracle_source(a, w, Pq):
    """dist[q,c] = monomer_dist(a = a[c], Pt = Pq[q], w = w[c]): cfl/models/base.py:109-117 with the SOURCE item as
    the candidate (its a [N,d] and gate w [N,K]) and the TARGET item as the query (its K prototypes Pq [Q,K,d])."""
    block = max(1, int(2e7 // Pq.size))                        # sources per block of the oracle's [b,Q,K,d] difference
    return O.all_pairs_monomer_dist(a.astype(np.float64), w.astype(np.float64), Pq.astype(np.float64), block=block).T


def check_result(D, tv, ti, k):
    """Reported values within 1e-4 of the oracle's distances of the reported rows, listed in (value, index) order;
    index sets equal up to near-ties of the k-th distance; -1 / +inf padding when N < k."""
    kk = min(k, D.shape[1])
    want_v, want_i = O.rank_topk(D, kk)
    got = np.take_along_axis(D, ti[:, :kk], 1)
    np.testing.assert_allclose(tv[:, :kk], got, rtol=RTOL, atol=0, err_msg="reported values")
    dv, di = np.diff(tv[:, :kk], axis=1), np.diff(ti[:, :kk], axis=1)
    assert ((dv > 0) | ((dv == 0) & (di > 0))).all(), "not in (value, index) order"
    for q in range(D.shape[0]):
        kth = want_v[q, -1]
        for c in set(ti[q, :kk].tolist()) ^ set(want_i[q].tolist()):
            assert abs(D[q, c] - kth) <= 2e-6 * max(kth, 1.0) + 1e-7, f"q={q} cand {c} is not a near-tie"
    if kk < k:
        assert (ti[:, kk:] == -1).all() and np.isinf(tv[:, kk:]).all()


def _data(rng, Q, K, d, N, offset=0.0):
    A = (rng.normal(size=(N, d)) + offset).astype(np.float32)
    W = O.softmax(2.0 * rng.normal(size=(N, K))).astype(np.float32)
    # targets whose prototypes lie near some source's embedding, so that the k nearest are not all far away
    Pq = (A[rng.integers(0, N, (Q, K))] + 0.5 * rng.normal(size=(Q, K, d))).astype(np.float32)
    return Pq, A, W


def _mean(A):
    return dev(A.astype(np.float64).mean(0).astype(np.float32))


PACKED = ["cfl::score_monomer_src_kernel", "cfl::mono_src_prep_lb_kernel", "cfl::score_lb_kernel<1>"]
FORWARD = ["cfl::score_monomer_kernel<1>", "cfl::score_monomer_kernel<2>", "cfl::score_monomer_kernel<4>",
           "cfl::mono_prep_lb_kernel"]


def run_both_routes(nat, Pq, A, W, k, mu=None):
    """Packed route (when the shape has one) and CUDA-core route on the same inputs; asserts which route ran and that
    the two agree bit for bit.  -> (values, indices, stats of the packed call or None)."""
    K, d = Pq.shape[1], Pq.shape[2]
    Pd, Ad, Wd = dev(Pq), dev(A), dev(W)
    # CUDA-core route: proven by its counters (the call zeroes them; the packed route always sets lower_bound_pass).
    # Its profiler traces came back without the score_monomer_src_kernel record in long test processes (the merge
    # after it was recorded), so the kernel names are asserted on the packed route, which runs the same kernel.
    ev, ei, st = nat.score_topk_monomer_source(Pd, Ad, Wd, None, k, want_stats=True)
    assert (st == 0).all(), st
    image = nat.monomer_source_pack(Ad, Wd, mu) if A.shape[0] else None
    if K * (d + 1) > 128:
        assert image is None
        return host(ev), ei.cpu().numpy(), None
    assert (image is not None) == (A.shape[0] > 0)
    if image is None:
        return host(ev), ei.cpu().numpy(), None
    (tv, ti, st), names = traced(lambda: nat.score_topk_monomer_source(Pd, Ad, Wd, image, k, mu=mu, want_stats=True))
    assert dict(zip(nat.SCORE_STAT_NAMES, st.tolist()))["lower_bound_pass"] == 1
    for n in PACKED + [f"cfl::mono_rescore_src_kernel<{K}>", "cfl::merge_plain_kernel"]:
        assert n in names, f"packed route did not launch {n}: {sorted(x for x in names if x.startswith('cfl::'))}"
    for n in FORWARD + [f"cfl::mono_rescore_kernel<{K}>"]:
        assert n not in names, f"packed route launched {n}"
    assert torch.equal(ei, ti) and torch.equal(ev.view(torch.int32), tv.view(torch.int32)), "routes differ"
    return host(tv), ti.cpu().numpy(), dict(zip(nat.SCORE_STAT_NAMES, st.tolist()))


# K(d+1) <= 128 takes the packed route (and is compared with the CUDA-core route); (4, 64) and (8, 20) have only the
# CUDA-core route.  Q = 15 / 17 leave ragged query tiles (16 per CUDA-core tile, 192 per filter tile at K = 1); N < k
# pads.  N >= 28 672 gives the full sampled cascade (every 32nd tile) at k = 100.
@gpu
@pytest.mark.parametrize("Q,K,d,N,k", [(1, 1, 64, 60000, 100), (15, 2, 10, 30000, 100), (17, 3, 31, 40000, 128),
                                       (1000, 4, 20, 30000, 100), (17, 4, 31, 20000, 1), (15, 8, 10, 20000, 100),
                                       (17, 1, 31, 3000, 100), (15, 2, 20, 50, 100), (1, 3, 10, 129, 128),
                                       (33, 4, 64, 20000, 100), (17, 8, 20, 10000, 128), (15, 2, 64, 5000, 100)])
def test_monomer_source_topk_shapes(nat, Q, K, d, N, k):
    rng = np.random.default_rng(Q * 7 + K * 11 + d + N)
    Pq, A, W = _data(rng, Q, K, d, N)
    tv, ti, _ = run_both_routes(nat, Pq, A, W, k, mu=_mean(A))
    check_result(oracle_source(A, W, Pq), tv, ti, k)


@gpu
def test_monomer_source_k1_unit_gate_equals_forward_with_roles_swapped(nat):
    """K = 1, w = 1: sum_k w_k |a_c - p_q|^2 = |p_q - a_c|^2, the forward call with query a := p and catalog := a.
    The two differences are exact negatives, so their squares -- and the reported lists -- agree bit for bit."""
    rng = np.random.default_rng(12)
    Q, d, N = 300, 64, 200000
    Pq, A, _ = _data(rng, Q, 1, d, N)
    mu = _mean(A)
    Ad, Pd = dev(A), dev(Pq)
    ones_c, ones_q = torch.ones(N, 1, device="cuda"), torch.ones(Q, 1, device="cuda")
    sv, si = nat.score_topk_monomer_source(Pd, Ad, ones_c, nat.monomer_source_pack(Ad, ones_c, mu), 100, mu=mu)
    cat = Ad[:, None, :]
    fv, fi = nat.score_topk_monomer_packed(Pd[:, 0], ones_q, cat, nat.monomer_pack(cat, mu), 100, mu=mu)
    assert torch.equal(fi, si)
    assert torch.equal(fv.view(torch.int32), sv.view(torch.int32))


@gpu
def test_monomer_source_duplicates_rank_lower_index_first_and_calls_are_deterministic(nat):
    rng = np.random.default_rng(31)
    Pq, A, W = _data(rng, 40, 3, 20, 40000)
    for r in (100, 650):
        A[r], W[r] = A[7], W[7]
    Pq[::4] = A[7] + 0.01 * rng.normal(size=(10, 3, 20)).astype(np.float32)      # every prototype near the duplicates
    tv, ti, _ = run_both_routes(nat, Pq, A, W, 100, mu=_mean(A))
    check_result(oracle_source(A, W, Pq), tv, ti, 100)
    for q in range(0, 40, 4):
        assert ti[q, :3].tolist() == [7, 100, 650], ti[q, :5]
    Ad, Wd, Pd = dev(A), dev(W), dev(Pq)
    image = nat.monomer_source_pack(Ad, Wd, _mean(A))
    a = nat.score_topk_monomer_source(Pd, Ad, Wd, image, 100, mu=_mean(A))
    b = nat.score_topk_monomer_source(Pd, Ad, Wd, image, 100, mu=_mean(A))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@gpu
def test_monomer_source_offset_catalog_with_centring(nat):
    """+10 common offset on both sides, centred on the sources' mean: the filter's margin holds after centring."""
    rng = np.random.default_rng(99)
    Pq, A, W = _data(rng, 16, 4, 20, 40000, offset=10.0)
    tv, ti, st = run_both_routes(nat, Pq, A, W, 100, mu=_mean(A))
    check_result(oracle_source(A, W, Pq), tv, ti, 100)
    assert st["lower_bound_pass"] == 1, st


@gpu
def test_monomer_source_fp16_range_flag_redoes_every_query_exactly(nat):
    """A source embedding far outside the fp16 range raises the image's range flag: the filter declines and every query
    is redone by the CUDA-core kernel; the result is still exact (and the CUDA-core route's bits)."""
    rng = np.random.default_rng(77)
    Q = 40
    Pq, A, W = _data(rng, Q, 4, 20, 50000)
    A[123, 5] = 3.0e5
    tv, ti, st = run_both_routes(nat, Pq, A, W, 50, mu=_mean(A))
    assert st["redo_queries"] == Q, st
    check_result(oracle_source(A, W, Pq), tv, ti, 50)


@gpu
def test_monomer_source_failed_optimistic_threshold_is_redone_exactly(nat):
    """A clustered catalog: every row near the queries sits in a tile the threshold sample visits (every 32nd tile),
    every other row is far away.  The sample's optimistic threshold then admits about 4k/32 rows of the whole catalog,
    fewer than k: verification fails, the queries are redone, and the result is still exact."""
    rng = np.random.default_rng(5)
    Q, K, d, k = 24, 4, 20, 100
    N = 320 * 128                                              # 320 tiles: the sample takes tiles 0, 32, ..., 288
    A = (20.0 + rng.normal(size=(N, d))).astype(np.float32)
    near = (np.arange(N) // 128) % 32 == 0
    cen = rng.normal(size=(3, d)).astype(np.float32)
    A[near] = cen[rng.integers(0, 3, near.sum())] + 0.05 * rng.normal(size=(near.sum(), d)).astype(np.float32)
    W = O.softmax(rng.normal(size=(N, K))).astype(np.float32)
    Pq = (cen[rng.integers(0, 3, (Q, 1))] + 0.1 * rng.normal(size=(Q, K, d))).astype(np.float32)
    tv, ti, st = run_both_routes(nat, Pq, A, W, k, mu=_mean(A))
    assert st["redo_queries"] > 0, st
    check_result(oracle_source(A, W, Pq), tv, ti, k)


@gpu
def test_monomer_source_empty_queries_empty_shard_and_bad_shapes(nat):
    rng = np.random.default_rng(3)
    Pq, A, W = _data(rng, 5, 2, 10, 1000)
    Pd, Ad, Wd = dev(Pq), dev(A), dev(W)
    image = nat.monomer_source_pack(Ad, Wd)
    tv, ti = nat.score_topk_monomer_source(Pd[:0], Ad, Wd, image, 10)
    assert tv.shape == (0, 10) and ti.shape == (0, 10)
    assert nat.monomer_source_pack(Ad[:0], Wd[:0]) is None
    tv, ti = nat.score_topk_monomer_source(Pd, Ad[:0], Wd[:0], None, 10)
    assert (ti == -1).all() and torch.isinf(tv).all()
    with pytest.raises(nat.CflNativeError):                  # K = 9
        nat.score_topk_monomer_source(dev(np.zeros((2, 9, 4))), dev(np.zeros((10, 4))), dev(np.ones((10, 9))), None, 5)
    with pytest.raises(nat.CflNativeError):                  # d = 129
        nat.score_topk_monomer_source(dev(np.zeros((2, 1, 129))), dev(np.zeros((10, 129))), dev(np.ones((10, 1))),
                                      None, 5)
    for k in (0, 129):
        with pytest.raises(nat.CflNativeError):
            nat.score_topk_monomer_source(Pd, Ad, Wd, image, k)
    with pytest.raises(nat.CflNativeError):                  # K(d+1) > 128 has no packed image
        nat.score_topk_monomer_source(dev(np.zeros((2, 4, 64))), dev(np.zeros((10, 64))), dev(np.ones((10, 4))),
                                      image, 5)
    with pytest.raises(nat.CflNativeError):                  # gate does not match the prototypes' K
        nat.score_topk_monomer_source(Pd, Ad, Wd[:, :1], None, 5)


@gpu
def test_monomer_source_1m_row_shape_sampled_queries(nat):
    """The monomer configuration (K = 4, d = 20) at 2^20 source rows, Q = 1024 target queries, k = 100: the packed
    route equals the CUDA-core route bit for bit, and 8 queries match the oracle over the whole catalog."""
    Q, K, d, N, k = 1024, 4, 20, 1 << 20, 100
    g = torch.Generator(device="cuda").manual_seed(3)
    A = torch.randn(N, d, device="cuda", generator=g)
    W = torch.softmax(2 * torch.randn(N, K, device="cuda", generator=g), -1)
    Pq = A[torch.randint(0, N, (Q, K), device="cuda", generator=g)] + 0.5 * torch.randn(Q, K, d, device="cuda",
                                                                                         generator=g)
    mu = A.double().mean(0).float()
    tv, ti, st = nat.score_topk_monomer_source(Pq, A, W, nat.monomer_source_pack(A, W, mu), k, mu=mu, want_stats=True)
    ev, ei = nat.score_topk_monomer_source(Pq, A, W, None, k)
    assert torch.equal(ei, ti) and torch.equal(ev.view(torch.int32), tv.view(torch.int32))
    stats = dict(zip(nat.SCORE_STAT_NAMES, st.tolist()))
    assert stats["lower_bound_pass"] == 1 and stats["redo_queries"] <= Q // 20, stats
    sample = np.arange(0, Q, Q // 8)
    D = oracle_source(A.cpu().numpy(), W.cpu().numpy(), Pq.cpu().numpy()[sample])
    check_result(D, host(tv)[sample], ti.cpu().numpy()[sample], k)


@gpu
def test_monomer_source_index_from_features_and_shards(nat):
    from cfl.ranking import EncoderWeights, MonomerSourceCatalogIndex
    rng = np.random.default_rng(21)
    F, K, d, N, Q, k = 96, 4, 20, 30000, 50, 100
    w = EncoderWeights(V0=dev(O.xavier_uniform(rng, F, d)), Vp=dev(O.xavier_uniform(rng, F, K * d)),
                       g0=dev(1.0 + 0.1 * rng.normal(size=d)), gp=dev(np.ones(K * d)), b0=dev(0.1 * rng.normal(size=d)),
                       bp=dev(0.1 * rng.normal(size=K * d)), weight_norm=True, act="tanh",
                       Vg=dev(O.xavier_uniform(rng, d, K)), gg=dev(1.0 + 0.1 * rng.normal(size=K)))
    Xc = np.maximum(rng.normal(size=(N, F)), 0).astype(np.float32)
    Xq = np.maximum(rng.normal(size=(Q, F)), 0).astype(np.float32)
    idx = MonomerSourceCatalogIndex.from_features(w, dev(Xc))
    assert idx.image is not None
    # the catalog side against the oracle's projection and gate (cfl/models/base.py:94-105)
    V0, g0, b0, Vg, gg = (host(t) for t in (w.V0, w.g0, w.b0, w.Vg, w.gg))
    a64, pre64, _ = O.fc_weight_norm(Xc.astype(np.float64), V0, g0, b0, act="tanh", return_pre=True)
    w64 = O.softmax(O.fc_weight_norm(pre64, Vg, gg))
    np.testing.assert_allclose(host(idx.a), a64, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(host(idx.gate), w64, rtol=1e-4, atol=1e-5)
    P64 = O.fc_weight_norm(Xq.astype(np.float64), host(w.Vp), host(w.gp), host(w.bp), act="tanh").reshape(Q, K, d)
    Pq = idx.project_queries(dev(Xq))
    np.testing.assert_allclose(host(Pq), P64, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(host(idx.mu), host(idx.a).mean(0), rtol=1e-5, atol=1e-6)
    tv, ti = idx.rank(dev(Xq), k)
    check_result(oracle_source(host(idx.a), host(idx.gate), host(Pq)), host(tv), ti.cpu().numpy(), k)
    n1 = N // 2
    a = MonomerSourceCatalogIndex.from_features(w, dev(Xc[:n1]), idx_base=0, n_total=N)
    b = MonomerSourceCatalogIndex.from_features(w, dev(Xc[n1:]), idx_base=n1, n_total=N)
    va, ia = a.rank(dev(Xq), k)
    vb, ib = b.rank(dev(Xq), k)
    mv, mi = nat.topk_merge(torch.stack([va, vb]), torch.stack([ia, ib]))
    assert torch.equal(mi, ti) and torch.equal(mv, tv)


# ---------------------------------------------------------------------------------------------- no GPU
def test_monomer_source_kernel_is_packed_fp32x2_without_local_memory():
    """score_monomer_src_kernel: packed FP32x2 adds and FMAs (FADD2 / FFMA2, two queries per instruction) and no
    local-memory traffic (STL / LDL) -- the kernel is not templated on K, so this holds for every K.  The packed
    route's filter is score_lb_kernel<1>, which tests/test_sass_static.py already covers."""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, timeout=600, check=True).stdout
    ops, fn = collections.Counter(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            fn = m.group(1)
            continue
        if fn is not None and "score_monomer_src_kernel" in fn:
            for op in ("FADD2", "FFMA2", "STL", "LDL"):
                if re.search(r"\b%s\b" % op, line):
                    ops[op] += 1
    assert ops["FFMA2"] > 0 and ops["FADD2"] > 0, ops
    assert ops["STL"] == 0 and ops["LDL"] == 0, ops
