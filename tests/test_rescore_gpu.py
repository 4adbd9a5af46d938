"""rescore_merge_kernel (the exact rescoring of the lower-bound pass's survivors) in the regimes the other cascade tests
reach only by chance: queries that admit far more survivors than the candidate buffer holds (every survivor under the
safe threshold is a candidate, so the buffer is compacted again and again), a query whose survivors overflow a part
buffer into its spill list, rows without 16-byte alignment (the 4-byte gather), and a SASS check that every
instantiation keeps its registers (no local memory)."""
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


def test_rescore_kernel_has_no_local_memory():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    filt = shutil.which("c++filt")
    if not os.path.exists(cuobjdump) or filt is None:
        pytest.skip("cuobjdump / c++filt not available")
    sass = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, timeout=600, check=True).stdout
    per, fn = collections.Counter(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            fn = m.group(1) if "rescore_merge_kernel" in m.group(1) else None
            if fn:
                per[fn] += 0
            continue
        if fn is not None and re.search(r"\b(STL|LDL)\b", line):
            per[fn] += 1
    names = subprocess.run([filt], input="\n".join(per), capture_output=True, text=True, check=True).stdout.splitlines()
    found = {re.sub(r"\(.*", "", n.replace("void ", "")): per[m] for m, n in zip(per, names)}
    for K in range(1, 9):
        name = f"cfl::rescore_merge_kernel<{K}>"
        assert name in found, f"{name} not in the library"
        assert found[name] == 0, f"{name}: {found[name]} local-memory instructions"


@pytest.fixture(scope="module")
def nat():
    from cfl import _native
    _native.lib()
    assert _native.device_info()[1] == 10, "these tests need a B200 (sm_100)"
    return _native


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).cuda()


def _check(nat, monkeypatch, Pq, E, qs, env):
    """The lower-bound cascade under `env` returns the single adaptive pass's bits, and the oracle's top-100 on qs."""
    mu = nat.col_mean(E)
    monkeypatch.setenv("CFL_SCORE_MIN_TILES", "100000000")
    a = nat.score_topk(Pq, E, 100, mu=mu)
    monkeypatch.setenv("CFL_SCORE_MIN_TILES", "2")
    monkeypatch.setenv("CFL_SCORE_SAMPLE_STRIDE", "8")
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    tv, ti, st = nat.score_topk(Pq, E, 100, mu=mu, want_stats=True)
    stats = dict(zip(nat.SCORE_STAT_NAMES, st.tolist()))
    assert stats["lower_bound_pass"] == 1, stats
    assert torch.equal(a[1], ti) and torch.equal(a[0], tv)
    D = O.all_pairs_dist(Pq[qs].cpu().numpy().astype(np.float64), E.cpu().numpy().astype(np.float64), block=1)
    wv, wi = O.rank_topk(D, 100)
    np.testing.assert_allclose(tv[qs].cpu().numpy().astype(np.float64), wv, rtol=1e-4)
    got = ti[qs].cpu().numpy()
    for r in range(len(qs)):
        for c_ in set(got[r].tolist()) ^ set(wi[r].tolist()):
            assert abs(D[r, c_] - wv[r, -1]) <= 1e-5 * max(wv[r, -1], 1.0) + 1e-7
    return stats


@pytest.mark.gpu
@pytest.mark.parametrize("K,d", [(3, 64), (2, 30), (4, 128)])
def test_every_survivor_a_candidate(nat, monkeypatch, K, d):
    """Without the optimistic threshold every survivor under the safe threshold enters the candidate buffer: with a
    1/8 sample that is over a thousand rows per query, so the buffer is compacted several times (sorts of 512 and 1024
    keys).  d = 30 gathers with 4-byte loads (rows not 16-byte aligned); d = 128 stages the kk rows in two passes."""
    rng = np.random.default_rng(300 + 10 * K + d)
    N, Q = 150_000, 96
    E = rng.normal(size=(N, d)).astype(np.float32)
    Pq = (E[rng.integers(0, N, Q)][:, None, :] + 0.5 * rng.normal(size=(Q, K, d))).astype(np.float32)
    stats = _check(nat, monkeypatch, _dev(Pq), _dev(E), [0, 47, Q - 1], {"CFL_SCORE_NO_OPTIMISTIC": "1"})
    assert stats["survivors"] > 1024 * Q, stats


@pytest.mark.gpu
def test_spill_list_query(nat, monkeypatch):
    """6000 near-copies of one row, stored together: the query sitting on them keeps most of them through the lower
    bound, more than a part buffer holds (a part is about 8000 rows here), so the rest goes to its spill list and the
    rescoring reads both."""
    rng = np.random.default_rng(911)
    N, Q, K, d = 1_200_000, 64, 3, 64
    E = rng.normal(size=(N, d)).astype(np.float32)
    E[400_000:406_000] = E[400_000] + 0.05 * rng.normal(size=(6000, d)).astype(np.float32)
    Pq = (E[rng.integers(0, N, Q)][:, None, :] + 0.5 * rng.normal(size=(Q, K, d))).astype(np.float32)
    Pq[5] = E[400_000] + 0.05 * rng.normal(size=(K, d)).astype(np.float32)
    stats = _check(nat, monkeypatch, _dev(Pq), _dev(E), [5, 0, Q - 1], {})
    assert stats["spill_queries"] >= 1, stats
