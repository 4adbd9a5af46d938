"""Every dispatch path of the projection (``cfl_project_fwd/_bwd``) and paired-loss (``cfl_pair_loss_fwd/_bwd``) kernels
against the fp64 oracle, with proof of the kernel that ran.

Path proof: ``launched(fn)`` runs ``fn`` once under ``torch.profiler`` (CUDA activity) and returns the demangled names of
the kernels it launched (``cfl::project_bwd_umma_tma_kernel<2, false>``).  Every case names the kernels it must reach
and the competing kernels it must not; a case that lands on another path fails.  ``KERNEL_TABLE`` maps each kernel to
the first case that reaches it; ``tests/test_sass_static.py`` checks that every projection / paired kernel in the built
library is in it (or in ``KERNEL_ALLOW`` with a reason), so a path added later without a case fails without a GPU.

Bars (derived, not tuned):
- projection forward, z and pre:  |got - want| <= 1e-4 |want| + 1.5e-6 S + 1e-7 with S = in_scale (|x| @ |V|) scaler
  (scaler = g / |V_col| under weight norm, else 1).  1e-4 is the project's fp32 bar; 1.5e-6 S is twice the error of
  the 3xTF32 split (3 * 2^-22 of each |x_f V_fn| term; the fp32 CUDA-core kernels stay far below it).
- projection forward, y:  the same with the S term multiplied by L = max |act'| over the row, act' taken at the
  oracle pre-activation and at both ends of its error interval (the activation's local Lipschitz constant: an error
  e in pre moves y by at most L e).
- projection backward:  atol 3e-5 max|ref| (with the default 1e-4 relative term), the bar of test_project_bwd_shapes;
  the oracle takes act' and the weight-norm term from the saved y, z the backward is given (``bwd_oracle``).
- paired kernels:  1e-4 relative on distances and statistics; gradients at atol 2e-5 max|ref|, the bar of
  test_pair_random_shapes.  Counts of correct decisions are exact except for pairs whose score is within 1e-5 |dist|
  of zero, where the fp32 and fp64 decisions may differ.

Bit equality where the code makes it so: the TMA and the register-prefetch forward kernels issue the same tcgen05 MMAs
in the same order on the same tf32 splits (split_tf32_fast reproduces cvt.rna.tf32 for finite values) into the same
accumulator rotation and share the epilogue; the same holds for the two weight-gradient kernels, which also share the
slab reduction.  Those pairs are compared bit for bit; the fp32 CUDA-core kernels sum in another order and are compared
with the tensor-core result within the oracle bar."""
import re
import shutil
import subprocess
import zlib

import numpy as np
import pytest
import torch

from oracle import cfl_oracle as O

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).cuda()


def host(t):
    return t.detach().cpu().numpy().astype(np.float64)


def assert_close(got, want, rtol=1e-4, atol=0.0, msg=""):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    scale = np.maximum(np.abs(want), atol / rtol if rtol else 0)
    err = np.abs(got - want)
    bad = err > rtol * scale + atol
    assert not bad.any(), f"{msg} max rel err {np.max(err / np.maximum(np.abs(want), 1e-30)):.3e} at {np.argmax(bad)}"


def kernel_name(raw):
    """Profiler kernel name -> 'cfl::kernel<args>' (no return type, no parameter list)."""
    if raw.startswith("_Z") and shutil.which("c++filt"):
        raw = subprocess.run(["c++filt", raw], capture_output=True, text=True).stdout.strip()
    raw = re.sub(r"^void ", "", raw)
    raw = re.sub(r"\([^()]*\)$", "", raw)
    return raw.replace("(bool)0", "false").replace("(bool)1", "true")


def traced(fn):
    """(fn's result, set of kernel names it launched)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {kernel_name(e.name) for e in prof.events()}
    return out, names


def launched(fn):
    return traced(fn)[1]


def assert_path(names, expect, forbid=(), case=""):
    ours = sorted(n for n in names if n.startswith("cfl::"))
    for k in expect:
        assert k in names, f"{case}: expected {k} to run; launched {ours}"
    for k in forbid:
        if k not in expect:
            assert k not in names, f"{case}: {k} ran but the case is for {sorted(expect)}"


@pytest.fixture(scope="module")
def nat():
    from cfl import _native
    _native.lib()
    sms, major, _ = _native.device_info()
    assert major == 10, "these tests need a B200 (sm_100)"
    return _native


ACTS = ("linear", "tanh", "sigmoid", "relu", "lrelu")


# ---------------------------------------------------------------------------------------------------------------------
# projection forward
# ---------------------------------------------------------------------------------------------------------------------
F_SPLIT = ("cfl::project_fwd_splitk", "cfl::project_fwd_splitk_final")
F_TMA, F_REG, F_SIMT = ("cfl::project_umma_tma_kernel",), ("cfl::project_umma_kernel",), ("cfl::project_fwd_simt",)
F_ALL = F_SPLIT + F_TMA + F_REG + F_SIMT
ROUTE_FWD = {"split": F_SPLIT, "tma": F_TMA, "reg": F_REG, "simt": F_SIMT}


def _fc(route, B, F, N, **kw):
    return dict(route=route, B=B, F=F, N=N, **kw)


# (case id, parameters); kw: act, wn, g, bias, in_scale, x ('dense' | 'off4': pointer + 4 B | 'ld3': ldx % 4 == 3),
# V ('dense' | 'slice': ldV > N), env
FWD_CASES = [
    ("split-B1", _fc("split", 1, 512, 64)),
    ("split-B100", _fc("split", 100, 4096, 80, act="tanh")),
    ("split-B1024", _fc("split", 1024, 1000, 200, act="sigmoid")),
    ("tma-N5", _fc("tma", 4096, 512, 5)),
    ("tma-N64", _fc("tma", 2048, 256, 64, act="tanh")),
    ("tma-N80", _fc("tma", 1500, 1024, 80)),
    ("tma-N96", _fc("tma", 3000, 512, 96, act="relu")),
    ("tma-N128", _fc("tma", 2100, 384, 128)),
    ("tma-N144", _fc("tma", 1200, 512, 144, act="tanh")),
    ("tma-N256", _fc("tma", 2048, 256, 256)),
    ("tma-C5-d64-query", _fc("tma", 2048, 2048, 256)),
    ("reg-N64", _fc("reg", 2048, 512, 64, env={"CFL_PROJECT_NO_TMA": "1"})),
    ("reg-N128", _fc("reg", 2048, 512, 128, act="tanh", env={"CFL_PROJECT_NO_TMA": "1"})),
    ("reg-N256", _fc("reg", 2048, 512, 256, env={"CFL_PROJECT_NO_TMA": "1"})),
    ("simt-F7", _fc("simt", 1500, 7, 64)),
    ("simt-F1001", _fc("simt", 1100, 1001, 100, act="tanh")),
    ("simt-C5-d128-query", _fc("simt", 2048, 2048, 512)),
    ("simt-x-off4", _fc("simt", 1300, 256, 64, x="off4")),
    ("simt-x-ld3", _fc("simt", 1300, 256, 64, x="ld3")),
    ("simt-forced", _fc("simt", 2048, 512, 128, env={"CFL_FORCE_SIMT": "1"})),
    ("tma-B1025", _fc("tma", 1025, 256, 64)),
    ("tma-B1151", _fc("tma", 1151, 128, 130, act="sigmoid")),
    ("tma-B65613", _fc("tma", 65536 + 77, 256, 64, act="tanh")),          # >= 3 tiles per CTA: both TMEM buffers wrap
    ("tma-noWN", _fc("tma", 1500, 512, 100, wn=False)),
    ("tma-WN-g-None", _fc("tma", 1500, 512, 100, g=False)),
    ("tma-bias-None", _fc("tma", 1500, 512, 100, bias=False, act="tanh")),
    ("tma-in-scale", _fc("tma", 1500, 512, 100, in_scale=0.37, act="sigmoid")),
    ("tma-in-scale-noWN", _fc("tma", 1500, 512, 100, in_scale=0.37, wn=False)),
    ("tma-V-slice", _fc("tma", 1500, 512, 100, V="slice", act="relu")),
    ("split-V-slice", _fc("split", 300, 512, 100, V="slice")),
]
FWD_CASES += [(f"tma-F{F}-N{N}", _fc("tma", 1300, F, N, act="tanh")) for F in (8, 16, 24, 40) for N in (64, 200)]
FWD_CASES += [(f"{r}-{a}", _fc(r, B, 256, N, act=a)) for a in ACTS
              for r, B, N in (("split", 100, 48), ("tma", 2048, 48), ("simt", 2048, 300))]


def _fwd_inputs(rng, c):
    B, F, N = c["B"], c["F"], c["N"]
    x = rng.normal(size=(B, F)).astype(np.float32)
    V = O.xavier_uniform(rng, F, N)
    g = rng.uniform(0.5, 1.5, N).astype(np.float32) if c.get("g", True) else None
    b = (0.1 * rng.normal(size=N)).astype(np.float32) if c.get("bias", True) else None
    return x, V, g, b


def _x_on_device(x, layout):
    B, F = x.shape
    if layout == "dense":
        return dev(x)
    if layout == "off4":                                     # ldx % 4 == 0, base pointer 4 B past a 16-B boundary
        big = torch.zeros(B, F + 4, device="cuda")
        t = big[:, 1:F + 1]
    else:                                                    # aligned base, ldx = F + 3
        big = torch.zeros(B, F + 3, device="cuda")
        t = big[:, :F]
    t.copy_(dev(x))
    return t


def _V_on_device(V, layout):
    if layout == "dense":
        return dev(V)
    F, N = V.shape
    big = torch.zeros(F, N + 7, device="cuda")
    big[:, :N] = dev(V)
    return big[:, :N]


def fwd_oracle(x, V, g, b, wn, in_scale, act):
    """(y, pre, z, S): fp64 oracle and the error scale S = in_scale (|x| @ |V|) scaler."""
    x6, V6 = in_scale * x.astype(np.float64), V.astype(np.float64)
    g6 = None if g is None else g.astype(np.float64)
    b6 = None if b is None else b.astype(np.float64)
    if wn:
        y, pre, z = O.fc_weight_norm(x6, V6, g6, b6, act, return_pre=True)
        sc = (1.0 if g6 is None else g6) / np.sqrt((V6 ** 2).sum(0))
    else:
        z = x6 @ V6
        pre = z if b6 is None else z + b6
        y = O.activation(pre, act)
        sc = np.ones(V.shape[1])
    S = (np.abs(x6) @ np.abs(V6)) * sc[None, :]
    return y, pre, z, S


def fwd_bars(want_y, want_pre, want_z, S, act):
    """Element-wise bars on (y, pre, z) -- the rule of the module docstring."""
    e = 1.5e-6 * S + 1e-7
    bz = 1e-4 * np.abs(want_z) + e
    bp = 1e-4 * np.abs(want_pre) + e
    lip = np.maximum.reduce([np.abs(O.activation_grad(O.activation(p, act), p, act))
                             for p in (want_pre, want_pre - bp, want_pre + bp)])
    by = 1e-4 * np.abs(want_y) + 1.5e-6 * S * lip.max(1, keepdims=True) + 1e-7
    return by, bp, bz


def check_fwd(got, want, bars, case):
    for name, gt, wt, bar in zip(("y", "pre", "z"), got, want, bars):
        err = np.abs(host(gt) - wt)
        assert (err <= bar).all(), f"{case} {name}: worst {np.max(err / bar):.2f}x bar"


@pytest.mark.parametrize("case,c", FWD_CASES, ids=[i for i, _ in FWD_CASES])
def test_project_fwd_path(nat, monkeypatch, case, c):
    for k, v in c.get("env", {}).items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    x, V, g, b = _fwd_inputs(rng, c)
    wn, sc, act = c.get("wn", True), c.get("in_scale", 1.0), c.get("act", "linear")
    xd, Vd = _x_on_device(x, c.get("x", "dense")), _V_on_device(V, c.get("V", "dense"))
    gd, bd = (None if g is None else dev(g)), (None if b is None else dev(b))
    out, names = traced(lambda: nat.project_fwd(xd, Vd, gd, bd, wn, sc, act, want_pre=True, want_z=True))
    expect = ROUTE_FWD[c["route"]] + (("cfl::colnorm_kernel",) if wn else ())
    assert_path(names, expect, F_ALL + ("cfl::colnorm_kernel",), case)
    y, pre, z, S = fwd_oracle(x, V, g, b, wn, sc, act)
    check_fwd(out, (y, pre, z), fwd_bars(y, pre, z, S, act), case)


SCALAR_EPI = [("split", 100, 256, 200), ("tma", 1500, 256, 200), ("tma", 1500, 16, 64), ("simt", 1500, 7, 200)]


@pytest.mark.parametrize("route,B,F,N", SCALAR_EPI)
def test_project_fwd_c_abi_ldy_scalar_epilogue(nat, route, B, F, N):
    """Direct C-ABI call with ldy = N + 3 (rows not 16-byte aligned: the scalar epilogue); the 3 padding columns of y,
    pre and z keep their sentinel."""
    import ctypes as C
    rng = np.random.default_rng(B + F + N)
    x, V, g, b = _fwd_inputs(rng, dict(B=B, F=F, N=N))
    xd, Vd, gd, bd = dev(x), dev(V), dev(g), dev(b)
    ldy, sent = N + 3, -1234.5
    y, pre, z = (torch.full((B, ldy), sent, device="cuda") for _ in range(3))
    nws = nat.lib().cfl_project_fwd_workspace_bytes(B, F, N)
    ws = torch.empty(max(nws, 1), dtype=torch.uint8, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    names = launched(lambda: nat._check(nat.lib().cfl_project_fwd(
        p(xd), B, F, F, p(Vd), N, N, p(gd), p(bd), 1, 0.8, nat.ACTS["tanh"], p(y), ldy, p(pre), p(z), p(ws), ws.numel(),
        st), "cfl_project_fwd"))
    assert_path(names, ROUTE_FWD[route], F_ALL, f"ldy {route}")
    for t in (y, pre, z):
        assert (t[:, N:] == sent).all(), "padding columns were written"
    want = fwd_oracle(x, V, g, b, True, 0.8, "tanh")
    check_fwd((y[:, :N], pre[:, :N], z[:, :N]), want[:3], fwd_bars(*want, "tanh"), f"ldy {route}")


@pytest.mark.parametrize("B,F,N,act", [(2048, 512, 64, "tanh"), (2048, 512, 128, "linear"), (2048, 512, 256, "sigmoid"),
                                       (1300, 40, 200, "relu"), (1300, 8, 64, "lrelu")])
def test_project_fwd_paths_agree(nat, monkeypatch, B, F, N, act):
    """One shape on the TMA, register-prefetch and CUDA-core forward kernels: TMA == register bit for bit, CUDA cores
    within the oracle bar of them."""
    rng = np.random.default_rng(B * 3 + F + N)
    x, V, g, b = _fwd_inputs(rng, dict(B=B, F=F, N=N))
    xd, Vd, gd, bd = dev(x), dev(V), dev(g), dev(b)
    run = lambda: nat.project_fwd(xd, Vd, gd, bd, True, 1.0, act, want_pre=True, want_z=True)
    res = {}
    for route, env in (("tma", None), ("reg", "CFL_PROJECT_NO_TMA"), ("simt", "CFL_FORCE_SIMT")):
        if env:
            monkeypatch.setenv(env, "1")
        res[route], names = traced(run)
        assert_path(names, ROUTE_FWD[route], F_ALL, route)
        if env:
            monkeypatch.delenv(env)
    for a, r in zip(res["tma"], res["reg"]):
        assert torch.equal(a, r), "TMA and register-prefetch forward kernels differ"
    want = fwd_oracle(x, V, g, b, True, 1.0, act)
    bars = fwd_bars(*want, act)
    check_fwd(res["tma"], want[:3], bars, "tma")
    for name, a, s, bar in zip(("y", "pre", "z"), res["tma"], res["simt"], bars):
        err = np.abs(host(a) - host(s))
        assert (err <= bar).all(), f"{name}: tensor-core vs CUDA-core forward {np.max(err / bar):.2f}x bar"


# ---------------------------------------------------------------------------------------------------------------------
# projection backward
# ---------------------------------------------------------------------------------------------------------------------
B_GEMM = ("cfl::project_bwd_gemm",)
B_UMMA = tuple(f"cfl::project_bwd_umma{t}_kernel<{nbi}, {ny}>" for t in ("", "_tma") for nbi in (1, 2, 4)
               for ny in ("false", "true"))
B_ALL = B_GEMM + B_UMMA
B_COMMON = ("cfl::colstats_kernel", "cfl::colstats_final", "cfl::project_bwd_final")


def _bwd_kernel(route, N, act):
    if route == "gemm":
        return B_GEMM
    npad = (N + 15) // 16 * 16
    nbi = 1 if npad <= 64 else (2 if npad <= 128 else 4)
    needy = "false" if act in (None, "linear") else "true"
    return (f"cfl::project_bwd_umma{'_tma' if route == 'tma' else ''}_kernel<{nbi}, {needy}>",)


def _bc(route, B, F, N, act, wn=True, **kw):
    return dict(route=route, B=B, F=F, N=N, act=act, wn=wn, **kw)


NO_TMA_B = {"CFL_PROJECT_BWD_NO_TMA": "1"}
# nh (accumulator sets) = min(3, 512 / Npad - 1): 3 for Npad <= 128, 2 for Npad 144..160, 1 above
BWD_CASES = [
    ("tma<1,false>", _bc("tma", 4096, 256, 64, "linear")),
    ("tma<1,true>", _bc("tma", 3000, 300, 60, "tanh", wn=False)),
    ("tma<2,false>-nh3", _bc("tma", 4100, 512, 100, None)),
    ("tma<2,true>", _bc("tma", 2500, 256, 128, "sigmoid")),
    ("tma<4,false>-nh1", _bc("tma", 3000, 384, 200, "linear", wn=False)),
    ("tma<4,true>-nh2-N160", _bc("tma", 2600, 256, 160, "relu")),
    ("tma<4,true>-nh2-N144", _bc("tma", 2600, 256, 144, "lrelu", wn=False)),
    ("reg<4,true>-Npad176", _bc("reg", 2048, 256, 176, "tanh")),
    ("reg<4,false>-Npad256", _bc("reg", 3000, 200, 250, "linear", wn=False)),
    ("reg<1,false>-ldx3", _bc("reg", 2000, 128, 64, "linear", x="ld3")),
    ("reg<1,true>-noTMA", _bc("reg", 2000, 256, 64, "relu", env=NO_TMA_B)),
    ("reg<2,false>-noTMA", _bc("reg", 2000, 256, 112, "linear", env=NO_TMA_B)),
    ("reg<2,true>-ldx3", _bc("reg", 2000, 200, 128, "tanh", x="ld3")),
    ("gemm-B200", _bc("gemm", 200, 512, 64, "tanh")),
    ("gemm-N300", _bc("gemm", 1000, 256, 300, "sigmoid")),
    ("gemm-forced", _bc("gemm", 3000, 256, 100, "linear", env={"CFL_FORCE_SIMT": "1"})),
    ("tma-in-scale", _bc("tma", 3000, 256, 64, "tanh", in_scale=0.37)),
    ("tma-in-scale-noWN", _bc("tma", 3000, 256, 64, "linear", wn=False, in_scale=0.37)),
    ("tma-WN-g-None", _bc("tma", 3000, 256, 80, "linear", g=False)),
    ("tma-accumulate", _bc("tma", 3000, 256, 100, "tanh", acc=True)),
    ("gemm-accumulate", _bc("gemm", 200, 64, 20, "linear", acc=True)),
    ("reg-accumulate-noWN", _bc("reg", 3000, 256, 176, "sigmoid", wn=False, acc=True)),
]


def bwd_oracle(x, V, g, b, wn, in_scale, act, dy, reg_c, y, z):
    """(dV, dg or None, db) in fp64, with the L2 terms reg_c * V and reg_c * b, of the backward given the saved
    forward outputs y, z it is called with: act' and q = sum_b dpre z are taken from them, as the kernels do.  (From
    the fp64 pre-activation instead, an element within rounding of a relu / lrelu kink can take the other branch and
    move dV by |x dy| -- not an error of the backward.)"""
    x6, V6, dy6 = in_scale * x.astype(np.float64), V.astype(np.float64), dy.astype(np.float64)
    g6 = None if g is None else g.astype(np.float64)
    b6 = np.zeros(V.shape[1]) if b is None else b.astype(np.float64)
    ys, zo = host(y), host(z)
    dpre = dy6 * O.activation_grad(ys, ys, act)             # relu / lrelu: y > 0 exactly where pre > 0
    if wn:
        dV, dg, db = O.fc_weight_norm_bwd(x6, V6, g6, zo, dpre)
        dg = None if g is None else dg
    else:
        dV, dg, db = x6.T @ dpre, None, dpre.sum(0)
    return dV + reg_c * V6, dg, db + reg_c * b6


@pytest.mark.parametrize("case,c", BWD_CASES, ids=[i for i, _ in BWD_CASES])
def test_project_bwd_path(nat, monkeypatch, case, c):
    for k, v in c.get("env", {}).items():
        monkeypatch.setenv(k, v)
    B, F, N, act, wn = c["B"], c["F"], c["N"], c["act"], c["wn"]
    sc, reg_c = c.get("in_scale", 1.0), 0.01
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    x, V, g, b = _fwd_inputs(rng, dict(B=B, F=F, N=N, g=c.get("g", True) and wn))
    dy = rng.normal(size=(B, N)).astype(np.float32)
    xd, Vd, gd, bd = _x_on_device(x, c.get("x", "dense")), dev(V), (None if g is None else dev(g)), dev(b)
    y, _, z = nat.project_fwd(xd, Vd, gd, bd, wn, sc, act, want_pre=True, want_z=True)
    acc = c.get("acc", False)
    if acc:                                                  # known values the kernel must add to
        dV0 = rng.normal(size=(F, N)).astype(np.float32)
        dg0, db0 = rng.normal(size=N).astype(np.float32), rng.normal(size=N).astype(np.float32)
        bufs = dict(dV=dev(dV0), dg=dev(dg0) if g is not None else None, dbias=dev(db0))
    else:
        bufs = {}
    (dV, dg, db), names = traced(lambda: nat.project_bwd(xd, Vd, gd, bd, wn, sc, act, y, z, dev(dy), reg_c=reg_c,
                                                         accumulate=acc, **bufs))
    assert_path(names, _bwd_kernel(c["route"], N, act) + B_COMMON + (("cfl::colnorm_kernel",) if wn else ()),
                B_ALL, case)
    dVo, dgo, dbo = bwd_oracle(x, V, g, b, wn, sc, act, dy, reg_c, y, z)
    tol = lambda r: 3e-5 * np.abs(r).max()
    base = (dV0, dg0, db0) if acc else (0.0, 0.0, 0.0)
    assert_close(host(dV), base[0] + dVo, atol=tol(dVo), msg=f"{case} dV")
    assert_close(host(db), base[2] + dbo, atol=tol(dbo), msg=f"{case} db")
    if dgo is not None:
        assert_close(host(dg), base[1] + dgo, atol=tol(dgo), msg=f"{case} dg")
    else:
        assert dg is None


@pytest.mark.parametrize("B,F,N,act", [(3000, 256, 64, "linear"), (3000, 256, 128, "tanh"), (3000, 256, 200, "linear"),
                                       (2600, 128, 160, "sigmoid")])
def test_project_bwd_paths_agree(nat, monkeypatch, B, F, N, act):
    """One shape on the TMA, register-prefetch and fp32 dV kernels: TMA == register bit for bit (same MMAs, same slab
    reduction), fp32 within the oracle bar of them."""
    rng = np.random.default_rng(B + 5 * F + N)
    x, V, g, b = _fwd_inputs(rng, dict(B=B, F=F, N=N))
    dy = rng.normal(size=(B, N)).astype(np.float32)
    xd, Vd, gd, bd, dyd = dev(x), dev(V), dev(g), dev(b), dev(dy)
    y, _, z = nat.project_fwd(xd, Vd, gd, bd, True, 1.0, act, want_pre=True, want_z=True)
    res = {}
    for route, env in (("tma", None), ("reg", "CFL_PROJECT_BWD_NO_TMA"), ("gemm", "CFL_FORCE_SIMT")):
        if env:
            monkeypatch.setenv(env, "1")
        res[route], names = traced(lambda: nat.project_bwd(xd, Vd, gd, bd, True, 1.0, act, y, z, dyd, reg_c=0.01))
        assert_path(names, _bwd_kernel(route, N, act), B_ALL, route)
        if env:
            monkeypatch.delenv(env)
    for a, r in zip(res["tma"], res["reg"]):
        assert torch.equal(a, r), "TMA and register-prefetch weight-gradient kernels differ"
    want = bwd_oracle(x, V, g, b, True, 1.0, act, dy, 0.01, y, z)
    for name, a, s, w in zip(("dV", "dg", "db"), res["tma"], res["gemm"], want):
        assert_close(host(a), w, atol=3e-5 * np.abs(w).max(), msg=f"tma {name}")
        assert_close(host(s), host(a), atol=3e-5 * np.abs(w).max(), msg=f"fp32 vs tensor-core {name}")


# ---------------------------------------------------------------------------------------------------------------------
# paired kernels
# ---------------------------------------------------------------------------------------------------------------------
def pick_group(d):
    """(G, MAXE) of csrc/pair.cu: G = smallest power of two with 4 G >= d (d <= 128), else (32, 8)."""
    if d > 128:
        return 32, 8
    G = 1
    while 4 * G < d:
        G *= 2
    return G, 4


# one d <= 128 (MAXE = 4; every lane group G in 1..32 appears) and one d in 129..256 (MAXE = 8) per K
PAIR_KD = [(1, 3), (2, 7), (3, 13), (4, 29), (5, 50), (6, 128), (7, 2), (8, 6),
           (1, 129), (2, 160), (3, 200), (4, 255), (5, 256), (6, 137), (7, 250), (8, 256)]
PAIR_B = (1, 7, 4097)
PAIR_CASES = [(K, d, B) for K, d in PAIR_KD for B in PAIR_B]


def _strided(arr, pad, fill=0.0):
    """A device copy of 2-D ``arr`` as a column slice of a wider buffer (leading dimension > width)."""
    B, n = arr.shape
    big = torch.full((B, n + pad), fill, device="cuda")
    big[:, :n] = dev(arr)
    return big, big[:, :n]


def _pair_inputs(rng, B, K, d):
    v = rng.normal(size=(B, d)).astype(np.float32)
    P = (v[:, None, :] + rng.normal(size=(B, K, d))).astype(np.float32)
    w = O.softmax(rng.normal(size=(B, K))).astype(np.float32)
    up = rng.normal(size=B).astype(np.float32)
    return v, P, w, up


def _pair_dev(v, P):
    B, K, d = P.shape
    _, a = _strided(v, 3)
    _, P2 = _strided(P.reshape(B, K * d), 5)
    return a, P2.view(B, K, d)


def _grad_out(B, K, d, sent=-777.0):
    da_big, da = _strided(np.zeros((B, d), np.float32), 2, sent)
    dP_big, dP = _strided(np.zeros((B, K * d), np.float32), 1, sent)
    return da_big, da, dP_big, dP


@pytest.mark.parametrize("K,d,B", PAIR_CASES)
def test_pair_paths(nat, K, d, B):
    """pcd, monomer (and siamese at K = 1), forward and backward, strided a / P in and strided da / dP out."""
    G, maxe = pick_group(d)
    rng = np.random.default_rng(K * 1000 + d * 10 + B)
    v, P, w, up = _pair_inputs(rng, B, K, d)
    a, Pd = _pair_dev(v, P)
    v6, P6, w6, up6 = (t.astype(np.float64) for t in (v, P, w, up))
    expect = (f"cfl::pair_fwd_kernel<{K}, {maxe}>", f"cfl::pair_bwd_kernel<{K}, {maxe}>")
    others = tuple(f"cfl::pair_{s}_kernel<{k}, {m}>" for s in ("fwd", "bwd") for k in range(1, 9) for m in (4, 8))
    modes = [("pcd", None), ("monomer", dev(w))] + ([("siamese", None)] if K == 1 else [])
    for mode, wd in modes:
        da_big, da, dP_big, dP = _grad_out(B, K, d)

        def run():
            dist, _, s, _ = nat.pair_loss_fwd(mode, a, Pd, w=wd, want_s=mode == "pcd")
            g = nat.pair_loss_bwd(mode, a, Pd, w=wd, ddist=dev(up), da=da, dP=dP)
            return dist, s, g

        (dist, s, (ga, gP, gw, _)), names = traced(run)
        assert_path(names, expect, others, f"{mode} K={K} d={d} (G={G})")
        assert ga is da
        assert (da_big[:, d:] == -777.0).all() and (dP_big[:, K * d:] == -777.0).all(), "padding columns written"
        if mode == "monomer":
            want = O.monomer_dist(v6, P6, w6)
            dao, dPo, dwo = O.monomer_dist_bwd(v6, P6, w6, up6)
            assert_close(host(gw), dwo, atol=2e-5 * np.abs(dwo).max(), msg="monomer dw")
        elif mode == "siamese":
            want = O.siamese_dist(v6, P6[:, 0])
            dao, dPo = O.pcd_dist_bwd(v6, P6, up6)
        else:
            want, so, _ = O.pcd_dist(v6, P6, return_aux=True)
            assert_close(host(s), so, rtol=1e-4, atol=1e-6, msg="softmax weights")
            dao, dPo = O.pcd_dist_bwd(v6, P6, up6)
        assert_close(host(dist), want, msg=f"{mode} dist")
        assert_close(host(da), dao, atol=2e-5 * np.abs(dao).max(), msg=f"{mode} da")
        assert_close(host(dP).reshape(B, K, d), dPo, atol=2e-5 * np.abs(dPo).max(), msg=f"{mode} dP")


@pytest.mark.parametrize("K,d", [(2, 24), (5, 7), (8, 130)])
@pytest.mark.parametrize("label", [0, 1])
def test_pair_loss_statistics_and_dtheta(nat, K, d, label):
    """Fused label statistics (softplus, correct, dist, sqrt, hinge sums) and the fused upstream gradient with dtheta,
    with a margin, against the Thresholder / loss oracle."""
    B = 4097
    rng = np.random.default_rng(K * 31 + d + label)
    v, P, _, _ = _pair_inputs(rng, B, K, d)
    a, Pd = _pair_dev(v, P)
    v6, P6 = v.astype(np.float64), P.astype(np.float64)
    dist = O.pcd_dist(v6, P6)
    theta, margin = float(np.median(dist)), float(1.1 * np.median(dist))
    th = dev(np.array([theta], np.float32))
    th6 = float(np.float32(theta))
    (_, score, _, st), names = traced(lambda: nat.pair_loss_fwd("pcd", a, Pd, theta=th, label=label, margin=margin,
                                                                 want_score=True, want_stats=True))
    maxe = pick_group(d)[1]
    assert_path(names, (f"cfl::pair_fwd_kernel<{K}, {maxe}>", "cfl::pair_stats_final"), (), "stats")
    st = host(st)
    sc = O.thresholder(dist, th6)
    assert_close(host(score), sc, atol=1e-4 * np.abs(dist).max(), msg="score")
    assert_close(st[0], O.softplus(-sc if label else sc).sum(), msg="softplus sum")
    correct = (sc > 0) if label else (sc <= 0)
    near = np.abs(sc) <= 1e-5 * np.abs(dist)
    assert abs(st[1] - correct.sum()) <= near.sum(), "correct count"
    assert_close(st[2], dist.sum(), msg="dist sum")
    assert_close(st[3], np.sqrt(dist + 1e-7).sum(), msg="sqrt sum")
    assert_close(st[4], np.maximum(0.0, np.float32(margin) - dist).sum(), msg="hinge sum")
    assert st[5] == B
    c_ce, c_lin, c_mar = 1.0 / B, 0.3 / B, 0.5 / B
    da_big, da, dP_big, dP = _grad_out(B, K, d)
    (_, _, _, dth), names = traced(lambda: nat.pair_loss_bwd("pcd", a, Pd, theta=th, label=label, margin=margin,
                                                             c_ce=c_ce, c_lin=c_lin, c_margin=c_mar, want_dtheta=True,
                                                             da=da, dP=dP))
    assert_path(names, (f"cfl::pair_bwd_kernel<{K}, {maxe}>", "cfl::pair_stats_final"), (), "dtheta")
    if label:
        ce = c_ce * O.sigmoid(dist - th6)
        dd = ce + c_lin
    else:
        ce = -c_ce * O.sigmoid(th6 - dist)
        dd = ce - np.where(dist < np.float32(margin), c_mar, 0.0)
    assert_close(host(dth)[0], -ce.sum(), msg="dtheta")
    dao, dPo = O.pcd_dist_bwd(v6, P6, dd)
    keep = np.abs(dist - margin) > 1e-4 * margin            # the hinge step is ambiguous within rounding of dist
    assert_close(host(da)[keep], dao[keep], atol=2e-5 * np.abs(dao).max(), msg="da")
    assert_close(host(dP).reshape(B, K, d)[keep], dPo[keep], atol=2e-5 * np.abs(dPo).max(), msg="dP")


# ---------------------------------------------------------------------------------------------------------------------
# output buffers the kernels cannot write in place
# ---------------------------------------------------------------------------------------------------------------------
def test_project_bwd_output_buffers(nat):
    """Caller-supplied dV / dg / dbias that are not dense float32 receive the result (accumulated onto their values);
    a wrong dtype or shape raises."""
    B, F, N = 700, 96, 40
    rng = np.random.default_rng(7)
    x, V, g, b = _fwd_inputs(rng, dict(B=B, F=F, N=N))
    xd, Vd, gd, bd, dyd = dev(x), dev(V), dev(g), dev(b), dev(rng.normal(size=(B, N)))
    y, _, z = nat.project_fwd(xd, Vd, gd, bd, True, 1.0, "tanh", want_pre=True, want_z=True)
    dV0, dg0, db0 = (rng.normal(size=s).astype(np.float32) for s in ((F, N), N, N))
    for acc in (False, True):
        ref = nat.project_bwd(xd, Vd, gd, bd, True, 1.0, "tanh", y, z, dyd, dV=dev(dV0), dg=dev(dg0), dbias=dev(db0),
                              accumulate=acc, reg_c=0.01)
        dV = torch.empty(N, F, device="cuda").t()           # column-major
        dV.copy_(dev(dV0))
        dg = torch.empty(2 * N, device="cuda")[::2]          # stride 2
        dg.copy_(dev(dg0))
        db = torch.empty(N, 3, device="cuda")[:, 1]
        db.copy_(dev(db0))
        out = nat.project_bwd(xd, Vd, gd, bd, True, 1.0, "tanh", y, z, dyd, dV=dV, dg=dg, dbias=db,
                              accumulate=acc, reg_c=0.01)
        assert out[0] is dV and out[1] is dg and out[2] is db
        for got, want, n in zip((dV, dg, db), ref, ("dV", "dg", "dbias")):
            assert torch.equal(got, want), f"{n} (accumulate={acc}) was not written"
    with pytest.raises(nat.CflNativeError):
        nat.project_bwd(xd, Vd, gd, bd, True, 1.0, "tanh", y, z, dyd, dV=torch.zeros(F, N, dtype=torch.float64,
                                                                                     device="cuda"))
    with pytest.raises(nat.CflNativeError):
        nat.project_bwd(xd, Vd, gd, bd, True, 1.0, "tanh", y, z, dyd, dg=torch.zeros(N + 1, device="cuda"))


def test_pair_bwd_output_buffers(nat):
    """Caller-supplied da / dP that the kernel cannot write in place (transposed, or a dP with no [B, K*d] view) receive
    the result; strided row-major ones are written in place; a wrong dtype or shape raises."""
    B, K, d = 301, 3, 20
    rng = np.random.default_rng(11)
    v, P, _, up = _pair_inputs(rng, B, K, d)
    a, Pd, upd = dev(v), dev(P), dev(up)
    ref_da, ref_dP, _, _ = nat.pair_loss_bwd("pcd", a, Pd, ddist=upd)
    da = torch.zeros(d, B, device="cuda").t()                # column-major [B, d]
    dP = torch.zeros(B, d, K, device="cuda").permute(0, 2, 1)   # [B, K, d] with no [B, K*d] view
    out_da, out_dP, _, _ = nat.pair_loss_bwd("pcd", a, Pd, ddist=upd, da=da, dP=dP)
    assert out_da is da and out_dP is dP
    assert torch.equal(da, ref_da) and torch.equal(dP, ref_dP)
    dPt = torch.zeros(K * d, B, device="cuda").t()           # column-major [B, K*d]
    _, out_dP, _, _ = nat.pair_loss_bwd("pcd", a, Pd, ddist=upd, dP=dPt)
    assert torch.equal(dPt.reshape(B, K, d), ref_dP) and torch.equal(out_dP, ref_dP)
    with pytest.raises(nat.CflNativeError):
        nat.pair_loss_bwd("pcd", a, Pd, ddist=upd, da=torch.zeros(B, d, dtype=torch.float64, device="cuda"))
    with pytest.raises(nat.CflNativeError):
        nat.pair_loss_bwd("pcd", a, Pd, ddist=upd, dP=torch.zeros(B, K, d + 1, device="cuda"))


# ---------------------------------------------------------------------------------------------------------------------
# the expected-kernel table (read by tests/test_sass_static.py without a GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _table():
    t = {}

    def add(names, case):
        for n in names:
            t.setdefault(n, case)

    for case, c in FWD_CASES:
        add(ROUTE_FWD[c["route"]] + (("cfl::colnorm_kernel",) if c.get("wn", True) else ()), f"test_project_fwd_path[{case}]")
    for case, c in BWD_CASES:
        add(_bwd_kernel(c["route"], c["N"], c["act"]) + B_COMMON, f"test_project_bwd_path[{case}]")
    for K, d, B in PAIR_CASES:
        m = pick_group(d)[1]
        add((f"cfl::pair_fwd_kernel<{K}, {m}>", f"cfl::pair_bwd_kernel<{K}, {m}>"), f"test_pair_paths[{K}-{d}-{B}]")
    add(("cfl::pair_stats_final",), "test_pair_loss_statistics_and_dtheta")
    return t


KERNEL_TABLE = _table()
# kernels of the same families that the scoring side owns (tested there)
KERNEL_ALLOW = {
    re.compile(r"cfl::pair_dist_rows_kernel<\d, (true|false)>"):
        "rank-count / range-query positive distances (tests/test_rank_counts.py, tests/test_within.py)",
}
