"""Static check of the built library (no GPU): the hot kernels really are tcgen05 / TMEM / TMA code -- `cuobjdump -sass` of
cfl/_lib/libcfl_b200.so must show UTCHMMA (tcgen05.mma), LDTM (tcgen05.ld), UBLKCP / UTMALDG (bulk and tensor-map TMA) in
them -- and the kernels the bench step launches carry no local-memory spills (STL / LDL).  Guards against a build that
silently loses the tensor-core path (the profiling guide's SASS mnemonics)."""
import collections
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "compatibility-family-learning_b200", "cfl", "_lib", "libcfl_b200.so")
OPS = ("UTCHMMA", "LDTM", "UBLKCP", "UTMALDG", "UTCBAR", "SYNCS", "FFMA2", "STL", "LDL")


def _tool(name):
    for c in (shutil.which(name), os.path.join("/usr/local/cuda/bin", name)):
        if c and os.path.exists(c):
            return c
    return None


@pytest.fixture(scope="module")
def census():
    cuobjdump, filt = _tool("cuobjdump"), shutil.which("c++filt")
    if cuobjdump is None or filt is None:
        pytest.skip("cuobjdump / c++filt not available")
    sass = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, timeout=600, check=True).stdout
    per, fn = collections.defaultdict(collections.Counter), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            fn = m.group(1)
            per[fn]["_"] += 0
            continue
        if fn is not None:
            for op in OPS:
                if op in line and re.search(r"\b%s\b" % op, line):
                    per[fn][op] += 1
    names = subprocess.run([filt], input="\n".join(per), capture_output=True, text=True, check=True).stdout.splitlines()
    out = {}
    for mangled, nice in zip(per, names):
        nice = re.sub(r"^void ", "", nice)
        out[re.sub(r"\(.*", "", nice)] = per[mangled]
    return out


def test_hot_kernels_are_tcgen05_and_tma_code(census):
    def has(kernel, *ops):
        assert kernel in census, f"{kernel} not in the library"
        for op in ops:
            assert census[kernel][op] > 0, f"{kernel}: no {op} in its SASS"

    for K in range(1, 9):
        has(f"cfl::score_lb_kernel<{K}>", "UTCHMMA", "LDTM", "UBLKCP", "UTCBAR")        # pass C (lower-bound filter)
        has(f"cfl::score_umma_kernel<{K}>", "UTCHMMA", "LDTM", "UBLKCP")                # exact 3xTF32 scoring
        has(f"cfl::rank_count_umma_kernel<{K}>", "UTCHMMA", "LDTM", "UBLKCP")           # fused rank counts
    has("cfl::project_umma_tma_kernel", "UTCHMMA", "LDTM", "UTMALDG")                    # projection, x by tensor-map TMA
    has("cfl::project_umma_kernel", "UTCHMMA", "LDTM", "UBLKCP")
    for S in (1, 2, 4):
        for wn in ("false", "true"):
            has(f"cfl::project_bwd_umma_tma_kernel<{S}, {wn}>", "UTCHMMA", "LDTM", "UTMALDG")   # dV = x^T dpre
    # packed FP32x2 epilogues (two queries per instruction)
    assert census["cfl::score_umma_kernel<3>"]["FFMA2"] > 0 and census["cfl::score_monomer_kernel<4>"]["FFMA2"] > 0


def test_bench_step_kernels_do_not_spill(census):
    spill_free = ["cfl::score_umma_kernel<3>", "cfl::score_umma_kernel<4>", "cfl::rank_count_umma_kernel<3>",
                  "cfl::project_umma_tma_kernel", "cfl::project_umma_kernel"]
    spill_free += [f"cfl::score_lb_kernel<{K}>" for K in range(1, 9)]
    spill_free += [f"cfl::project_bwd_umma_tma_kernel<{S}, {wn}>" for S in (1, 2, 4) for wn in ("false", "true")]
    for k in spill_free:
        assert census[k]["STL"] == 0 and census[k]["LDL"] == 0, f"{k}: local-memory traffic (STL {census[k]['STL']}, LDL {census[k]['LDL']})"


def test_every_projection_and_pair_kernel_has_a_path_test(census):
    """Every projection / paired-loss kernel in the library is reached by a case of tests/test_kernel_paths_gpu.py (its
    KERNEL_TABLE) or allowed there with a reason: a dispatch path added without a parity case fails here, without a GPU."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("kernel_paths", os.path.join(ROOT, "tests", "test_kernel_paths_gpu.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    family = re.compile(r"cfl::(project_\w+|pair_\w+|colnorm_kernel|colstats_\w+)(<.*>)?$")
    ours = sorted(k for k in census if family.match(k))
    assert len(ours) >= 60, f"census found only {ours}"
    missing = [k for k in ours if k not in mod.KERNEL_TABLE and not any(p.fullmatch(k) for p in mod.KERNEL_ALLOW)]
    assert not missing, f"kernels without a path case in test_kernel_paths_gpu.py: {missing}"
    stale = [k for k in mod.KERNEL_TABLE if k not in census]
    assert not stale, f"KERNEL_TABLE names kernels the library does not have: {stale}"
