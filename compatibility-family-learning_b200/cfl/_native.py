"""ctypes binding of libcfl_b200.so (the C ABI declared in include/cfl_b200.h).

There is no fallback: if the library is missing or a call fails, a ``CflNativeError`` is
raised.  torch is used only for device memory, streams and (elsewhere) torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libcfl_b200.so")

MODES = {"pcd": 0, "monomer": 1, "siamese": 2, "pcd_source": 3, "monomer_source": 4}
ACTS = {None: 0, "linear": 0, "tanh": 1, "sigmoid": 2, "relu": 3, "lrelu": 4}
MAX_K, MAX_D, MAX_TOPK = 8, 256, 128


class CflNativeError(RuntimeError):
    pass


_lib = None
_lock = threading.Lock()

_i64, _int, _f32, _sz, _vp = C.c_int64, C.c_int, C.c_float, C.c_size_t, C.c_void_p

# name -> (restype, argtypes); mirrors include/cfl_b200.h one to one
SIGNATURES = {
    "cfl_last_error": (C.c_char_p, []),
    "cfl_version": (_int, []),
    "cfl_device_info": (_int, [C.POINTER(_int)] * 3),
    "cfl_project_fwd_workspace_bytes": (_sz, [_i64, _int, _int]),
    "cfl_project_fwd": (_int, [_vp, _i64, _int, _i64, _vp, _int, _i64, _vp, _vp, _int, _f32, _int,
                               _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "cfl_project_bwd_workspace_bytes": (_sz, [_i64, _int, _int]),
    "cfl_project_bwd": (_int, [_vp, _i64, _int, _i64, _vp, _int, _i64, _vp, _vp, _int, _f32, _int,
                               _vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _int, _f32, _vp, _sz, _vp]),
    "cfl_pair_workspace_bytes": (_sz, [_i64]),
    "cfl_pair_loss_fwd": (_int, [_int, _vp, _i64, _vp, _i64, _vp, _i64, _int, _int, _vp, _int, _f32,
                                 _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cfl_pair_loss_bwd": (_int, [_int, _vp, _i64, _vp, _i64, _vp, _i64, _int, _int, _vp, _int, _f32,
                                 _f32, _f32, _f32, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "cfl_score_topk_workspace_bytes": (_sz, [_i64, _int, _int, _i64, _int]),
    "cfl_score_topk": (_int, [_int, _vp, _i64, _int, _int, _i64, _vp, _i64, _i64, _vp, _int, _i64,
                              _vp, _vp, _vp, _vp, _sz, _vp]),
    "cfl_catalog_pack_bytes": (_sz, [_i64, _int, _int]),
    "cfl_catalog_pack": (_int, [_vp, _i64, _int, _int, _i64, _vp, _vp, _sz, _vp]),
    "cfl_score_topk_packed_workspace_bytes": (_sz, [_i64, _int, _int, _i64, _int]),
    "cfl_score_topk_packed": (_int, [_int, _vp, _i64, _int, _int, _i64, _vp, _vp, _i64, _i64, _vp, _int, _i64,
                                     _vp, _vp, _vp, _vp, _sz, _vp]),
    "cfl_score_topk_stats": (_int, [_i64, _int, _int, _i64, _int, _int, _vp, _sz, _vp, _vp, _vp]),
    "cfl_source_catalog_pack_bytes": (_sz, [_i64, _int, _int]),
    "cfl_source_catalog_pack": (_int, [_vp, _i64, _int, _int, _i64, _vp, _vp, _sz, _vp]),
    "cfl_score_topk_source_workspace_bytes": (_sz, [_i64, _int, _int, _i64, _int]),
    "cfl_score_topk_source": (_int, [_vp, _i64, _i64, _int, _int, _vp, _vp, _i64, _i64, _vp, _int, _i64,
                                     _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cfl_score_topk_monomer_workspace_bytes": (_sz, [_i64, _int, _int, _i64, _int]),
    "cfl_score_topk_monomer": (_int, [_vp, _i64, _vp, _i64, _int, _int, _vp, _i64, _i64, _int, _i64,
                                      _vp, _vp, _vp, _vp, _sz, _vp]),
    "cfl_monomer_pack_bytes": (_sz, [_i64, _int, _int]),
    "cfl_monomer_pack": (_int, [_vp, _i64, _int, _int, _i64, _vp, _vp, _sz, _vp]),
    "cfl_score_topk_monomer_packed_workspace_bytes": (_sz, [_i64, _int, _int, _i64, _int]),
    "cfl_score_topk_monomer_packed": (_int, [_vp, _i64, _vp, _i64, _int, _int, _vp, _vp, _i64, _i64, _vp, _int, _i64,
                                             _vp, _vp, _vp, _vp, _sz, _vp]),
    "cfl_monomer_source_pack_bytes": (_sz, [_i64, _int, _int]),
    "cfl_monomer_source_pack": (_int, [_vp, _i64, _vp, _i64, _int, _int, _vp, _vp, _sz, _vp]),
    "cfl_score_topk_monomer_source_workspace_bytes": (_sz, [_i64, _int, _int, _i64, _int]),
    "cfl_score_topk_monomer_source": (_int, [_vp, _i64, _i64, _int, _int, _vp, _vp, _i64, _vp, _i64, _vp, _int, _i64,
                                             _vp, _vp, _vp, _vp, _sz, _vp]),
    "cfl_topk_merge": (_int, [_vp, _vp, _int, _i64, _int, _vp, _vp, _vp]),
    "cfl_topk_record_bytes": (_sz, [_i64, _int]),
    "cfl_topk_pack_records": (_int, [_vp, _vp, _i64, _int, _vp, _vp]),
    "cfl_topk_merge_records": (_int, [_vp, _int, _i64, _int, _vp, _vp, _vp]),
    "cfl_col_mean_workspace_bytes": (_sz, [_i64, _int]),
    "cfl_col_mean": (_int, [_vp, _i64, _int, _i64, _vp, _vp, _sz, _vp]),
    "cfl_pair_dist_rows": (_int, [_int, _vp, _i64, _int, _int, _i64, _vp, _vp, _i64, _i64, _vp, _int, _vp, _vp]),
    "cfl_rank_counts": (_int, [_int, _vp, _i64, _int, _int, _i64, _vp, _vp, _i64, _i64, _vp, _int, _vp, _vp]),
    "cfl_dense_rank_counts": (_int, [_vp, _i64, _i64, _i64, _vp, _int, _vp, _vp]),
    "cfl_rank_counts_packed_workspace_bytes": (_sz, [_i64, _int, _int, _i64]),
    "cfl_rank_counts_packed_source_workspace_bytes": (_sz, [_i64, _int, _int, _i64]),
    "cfl_rank_counts_packed": (_int, [_int, _vp, _i64, _int, _int, _i64, _vp, _vp, _i64, _i64, _vp, _vp, _int,
                                      _vp, _vp, _sz, _vp]),
    "cfl_rank_counts_packed_stats": (_int, [_i64, _int, _int, _i64, _vp, _sz, _vp, _vp]),
    "cfl_score_within_workspace_bytes": (_sz, [_int, _i64, _int, _int, _i64]),
    "cfl_score_within": (_int, [_int, _vp, _i64, _int, _int, _i64, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _i64,
                                _vp, _vp, _vp, _sz, _vp]),
    "cfl_score_within_stats": (_int, [_vp, _sz, _vp, _vp]),
    "cfl_within_merge": (_int, [_vp, _vp, _vp, _i64, _int, _i64, _vp, _vp, _vp, _vp]),
    "cfl_auc_workspace_bytes": (_sz, [_i64, _i64]),
    "cfl_auc": (_int, [_vp, _i64, _vp, _i64, _vp, _vp, _sz, _vp]),
    "cfl_adam_step": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _f32, _f32, _f32, _f32, _f32, _vp]),
    "cfl_adam_step_dev": (_int, [_vp, _vp, _vp, _vp, _i64, _vp, _f32, _f32, _f32, _f32, _f32, _vp]),
    "cfl_set_kernel_timer": (_int, [_vp, _vp]),
    "cfl_selftest_umma": (_int, [_vp, _vp, _vp, _int, _int, _vp]),
    "cfl_selftest_umma_f16": (_int, [_vp, _vp, _vp, _int, _int, _vp]),
}


def lib():
    """Loads the library once; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise CflNativeError(
                    f"{LIB_PATH} not found: build it with "
                    "`python compatibility-family-learning_b200/build.py` (there is no CPU fallback)")
            l = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(l, name)          # AttributeError if the .so lacks a declared symbol
                fn.restype, fn.argtypes = res, args
            _lib = l
    return _lib


def _check(status: int, what: str):
    if status != 0:
        msg = lib().cfl_last_error().decode("utf-8", "replace")
        raise CflNativeError(f"{what} failed (status {status}): {msg}")


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, name):
    if t is None:
        return None
    if not t.is_cuda:
        raise CflNativeError(f"{name} must be a CUDA tensor (no CPU path)")
    if t.dtype != torch.float32:
        raise CflNativeError(f"{name} must be float32, got {t.dtype}")
    return t


def _rows(t, name):
    """2-D view with unit inner stride; returns (tensor, leading dimension)."""
    t = _f32c(t, name)
    if t.dim() != 2 or t.stride(1) != 1 or (t.shape[0] > 1 and t.stride(0) < t.shape[1]):
        t = t.contiguous()
    return t, (t.stride(0) if t.shape[0] > 1 else t.shape[1])


def _out(t, shape, name, dense=False):
    """A caller's output buffer -> (buffer the kernel writes, caller's tensor or None).

    The kernel writes the first of the pair.  When the caller's tensor cannot be written in place (not row-major with
    unit inner stride, or not dense where ``dense``), the first is a dense copy of it (so accumulating kernels see its
    values) and the second is the tensor that ``_copy_back`` refreshes after the call.  A wrong dtype, device or shape
    raises: the buffer would otherwise be left stale or written out of bounds."""
    t = _f32c(t, name)
    shape = tuple(int(s) for s in shape)
    if tuple(t.shape) != shape:
        raise CflNativeError(f"{name} must have shape {shape}, got {tuple(t.shape)}")
    if dense:
        ok = t.is_contiguous()
    else:
        ok = t.dim() == 2 and (t.numel() == 0 or (t.stride(1) == 1 and (t.shape[0] <= 1 or t.stride(0) >= t.shape[1])))
    return (t, None) if ok else (t.contiguous(), t)


def _copy_back(buf, caller):
    if caller is not None:
        caller.copy_(buf.view(caller.shape))


class _WorkspaceCache:
    """One growing byte buffer per (device, stream) -- the C ABI never allocates."""

    def __init__(self):
        self.bufs = {}

    def get(self, nbytes: int, device) -> torch.Tensor:
        key = (device.index, torch.cuda.current_stream(device).cuda_stream)
        b = self.bufs.get(key)
        if b is None or b.numel() < nbytes:
            b = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
            self.bufs[key] = b
        return b


_ws = _WorkspaceCache()


def device_info():
    a, b, c = _int(), _int(), _int()
    _check(lib().cfl_device_info(C.byref(a), C.byref(b), C.byref(c)), "cfl_device_info")
    return a.value, b.value, c.value


# ------------------------------------------------------------------------------------------
# Stage 1
# ------------------------------------------------------------------------------------------
def project_fwd(x, V, g=None, bias=None, weight_norm=True, in_scale=1.0, act=None,
                want_pre=False, want_z=False):
    """y = act((in_scale*x @ V) * g/|V_col| + bias)  -- cfl/layers.py:80-94."""
    x, ldx = _rows(x, "x")
    V, ldV = _rows(V, "V")
    B, F = x.shape
    N = V.shape[1]
    if V.shape[0] != F:
        raise CflNativeError(f"project_fwd: x is [*, {F}] but V is {tuple(V.shape)}")
    y = torch.empty(B, N, dtype=torch.float32, device=x.device)
    pre = torch.empty_like(y) if want_pre else None
    z = torch.empty_like(y) if want_z else None
    g = _f32c(g, "g")
    bias = _f32c(bias, "bias")
    nws = lib().cfl_project_fwd_workspace_bytes(B, F, N)
    ws = _ws.get(nws, x.device)
    _check(lib().cfl_project_fwd(_ptr(x), B, F, ldx, _ptr(V), N, ldV, _ptr(g), _ptr(bias),
                                 1 if weight_norm else 0, float(in_scale), ACTS[act], _ptr(y), N,
                                 _ptr(pre), _ptr(z), _ptr(ws), ws.numel(), _stream()), "cfl_project_fwd")
    return y, pre, z


def project_bwd(x, V, g, bias, weight_norm, in_scale, act, y, z, dy, dV=None, dg=None, dbias=None,
                accumulate=False, reg_c=0.0, want_dg=True, want_dbias=True):
    x, ldx = _rows(x, "x")
    V, ldV = _rows(V, "V")
    dy, lddy = _rows(dy, "dy")
    B, F = x.shape
    N = V.shape[1]
    # y and z share one leading dimension in the C ABI: pass both dense
    y = None if y is None else _f32c(y, "y").contiguous()
    z = None if z is None else _f32c(z, "z").contiguous()
    ldy = N
    dev = x.device
    if dV is None:
        dV = torch.empty(F, N, dtype=torch.float32, device=dev)
        accumulate = False
    if dg is None and want_dg and weight_norm and g is not None:
        dg = torch.empty(N, dtype=torch.float32, device=dev)
    if dbias is None and want_dbias:
        dbias = torch.empty(N, dtype=torch.float32, device=dev)
    # the kernels write dense [F, N] / [N] float32 buffers (and read them back when accumulating)
    dV_k, dV_c = _out(dV, (F, N), "dV", dense=True)
    dg_k, dg_c = (None, None) if dg is None else _out(dg, (N,), "dg", dense=True)
    db_k, db_c = (None, None) if dbias is None else _out(dbias, (N,), "dbias", dense=True)
    nws = lib().cfl_project_bwd_workspace_bytes(B, F, N)
    ws = _ws.get(nws, dev)
    _check(lib().cfl_project_bwd(_ptr(x), B, F, ldx, _ptr(V), N, ldV, _ptr(g), _ptr(bias),
                                 1 if weight_norm else 0, float(in_scale), ACTS[act], _ptr(y), ldy,
                                 _ptr(z), _ptr(dy), lddy, _ptr(dV_k), _ptr(dg_k), _ptr(db_k),
                                 1 if accumulate else 0, float(reg_c), _ptr(ws), ws.numel(), _stream()),
           "cfl_project_bwd")
    _copy_back(dV_k, dV_c)
    _copy_back(dg_k, dg_c)
    _copy_back(db_k, db_c)
    return dV, dg, dbias


# ------------------------------------------------------------------------------------------
# Stage 2, paired
# ------------------------------------------------------------------------------------------
def _pair_views(a, P, K, d):
    a, lda = _rows(a, "a")
    P = _f32c(P, "P")
    B = a.shape[0]
    P2 = P.reshape(B, K * d)
    P2, ldP = _rows(P2, "P")
    return a, lda, P2, ldP, B


def pair_loss_fwd(mode, a, P, w=None, theta=None, label=-1, margin=0.0, want_dist=True,
                  want_score=False, want_s=False, want_stats=False):
    """dist / score / softmax weights / batch statistics of paired rows."""
    K = P.shape[1] if P.dim() == 3 else 1
    d = a.shape[1]
    a, lda, P2, ldP, B = _pair_views(a, P, K, d)
    dev = a.device
    dist = torch.empty(B, dtype=torch.float32, device=dev) if want_dist else None
    score = torch.empty(B, dtype=torch.float32, device=dev) if want_score else None
    s = torch.empty(B, K, dtype=torch.float32, device=dev) if want_s else None
    stats = torch.empty(8, dtype=torch.float64, device=dev) if want_stats else None
    w = None if w is None else _f32c(w, "w").contiguous()
    ws = _ws.get(lib().cfl_pair_workspace_bytes(B), dev)
    _check(lib().cfl_pair_loss_fwd(MODES[mode], _ptr(a), lda, _ptr(P2), ldP, _ptr(w), B, K, d,
                                   _ptr(theta), int(label), float(margin), _ptr(dist), _ptr(score),
                                   _ptr(s), _ptr(stats), _ptr(ws), ws.numel(), _stream()),
           "cfl_pair_loss_fwd")
    return dist, score, s, stats


def pair_loss_bwd(mode, a, P, w=None, theta=None, label=1, margin=0.0, c_ce=0.0, c_lin=0.0,
                  c_margin=0.0, ddist=None, want_dtheta=False, da=None, dP=None):
    K = P.shape[1] if P.dim() == 3 else 1
    d = a.shape[1]
    a, lda, P2, ldP, B = _pair_views(a, P, K, d)
    dev = a.device
    if da is None:
        da = torch.empty(B, d, dtype=torch.float32, device=dev)
    if dP is None:
        dP = torch.empty(B, K * d, dtype=torch.float32, device=dev)
    # caller buffers the kernel cannot write in place (e.g. transposed) receive the result by copy-back
    da2, da_c = _out(da, (B, d), "da")
    dP = _f32c(dP, "dP")
    if tuple(dP.shape) not in ((B, K, d), (B, K * d)):
        raise CflNativeError(f"dP must have shape {(B, K, d)} or {(B, K * d)}, got {tuple(dP.shape)}")
    try:
        dP2, dP_c = _out(dP.view(B, K * d), (B, K * d), "dP")
    except RuntimeError:                                     # no [B, K*d] view of the caller's buffer
        dP2, dP_c = dP.reshape(B, K * d).contiguous(), dP
    ldda = da2.stride(0) if B > 1 else d
    lddP = dP2.stride(0) if B > 1 else K * d
    dw = torch.empty(B, K, dtype=torch.float32, device=dev) if mode == "monomer" else None
    dth = torch.empty(1, dtype=torch.float64, device=dev) if want_dtheta else None
    w = None if w is None else _f32c(w, "w").contiguous()
    ddist = None if ddist is None else _f32c(ddist, "ddist").contiguous()
    ws = _ws.get(lib().cfl_pair_workspace_bytes(B), dev)
    _check(lib().cfl_pair_loss_bwd(MODES[mode], _ptr(a), lda, _ptr(P2), ldP, _ptr(w), B, K, d,
                                   _ptr(theta), int(label), float(margin), float(c_ce), float(c_lin),
                                   float(c_margin), _ptr(ddist), _ptr(da2), ldda, _ptr(dP2), lddP,
                                   _ptr(dw), _ptr(dth), _ptr(ws), ws.numel(), _stream()),
           "cfl_pair_loss_bwd")
    _copy_back(da2, da_c)
    _copy_back(dP2, dP_c)
    return da, dP.reshape(B, K, d) if dP.dim() == 2 else dP, dw, dth


# ------------------------------------------------------------------------------------------
# Stage 2, all pairs
# ------------------------------------------------------------------------------------------
def col_mean(E):
    E, lde = _rows(E, "E")
    N, d = E.shape
    mu = torch.empty(d, dtype=torch.float32, device=E.device)
    ws = _ws.get(lib().cfl_col_mean_workspace_bytes(N, d), E.device)
    _check(lib().cfl_col_mean(_ptr(E), N, d, lde, _ptr(mu), _ptr(ws), ws.numel(), _stream()),
           "cfl_col_mean")
    return mu


def catalog_pack(E, K, mu=None):
    """Builds the tensor-core operand image of a catalog once (None when (K, d) has no tcgen05
    tiling -- score_topk then uses the CUDA-core kernel on the raw rows)."""
    E, lde = _rows(E, "E")
    N, d = E.shape
    nbytes = lib().cfl_catalog_pack_bytes(N, K, d)
    if nbytes == 0:
        return None
    img = torch.empty(nbytes + 1024, dtype=torch.uint8, device=E.device)
    off = (-img.data_ptr()) % 1024
    img = img[off:off + nbytes]
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    _check(lib().cfl_catalog_pack(_ptr(E), N, K, d, lde, _ptr(mu), _ptr(img), nbytes, _stream()),
           "cfl_catalog_pack")
    return img


def score_topk(Pq, E, k, mu=None, mode="pcd", idx_base=0, want_dense=False, image=None, want_stats=False):
    """Top-k candidates of every query by soft-min distance; exact (rescored) values.
    ``image`` = catalog_pack(E, K, mu) skips the per-call packing of the catalog.  ``want_stats`` appends the int64
    counters of cfl_score_topk_stats (SCORE_STAT_NAMES) for this call."""
    Pq = _f32c(Pq, "Pq")
    if Pq.dim() == 2:
        Pq = Pq[:, None, :]
    Q, K, d = Pq.shape
    Pq2, ldq = _rows(Pq.reshape(Q, K * d), "Pq")
    E, lde = _rows(E, "E")
    N = E.shape[0]
    if E.shape[1] != d:
        raise CflNativeError(f"score_topk: Pq has d={d} but E is {tuple(E.shape)}")
    dev = E.device
    top_val = torch.empty(Q, k, dtype=torch.float32, device=dev)
    top_idx = torch.empty(Q, k, dtype=torch.int64, device=dev)
    dense = torch.empty(Q, N, dtype=torch.float32, device=dev) if want_dense else None
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    if image is not None:
        ws = _ws.get(lib().cfl_score_topk_packed_workspace_bytes(Q, K, d, N, k), dev)
        _check(lib().cfl_score_topk_packed(MODES[mode], _ptr(Pq2), Q, K, d, ldq, _ptr(image), _ptr(E), N, lde,
                                           _ptr(mu), int(k), int(idx_base), _ptr(top_val), _ptr(top_idx),
                                           _ptr(dense), _ptr(ws), ws.numel(), _stream()), "cfl_score_topk_packed")
    else:
        ws = _ws.get(lib().cfl_score_topk_workspace_bytes(Q, K, d, N, k), dev)
        _check(lib().cfl_score_topk(MODES[mode], _ptr(Pq2), Q, K, d, ldq, _ptr(E), N, lde, _ptr(mu),
                                    int(k), int(idx_base), _ptr(top_val), _ptr(top_idx), _ptr(dense),
                                    _ptr(ws), ws.numel(), _stream()), "cfl_score_topk")
    if want_stats:
        stats = torch.zeros(SCORE_NSTATS, dtype=torch.int64, device=dev)
        thr = torch.zeros(3, Q, dtype=torch.float32, device=dev) if want_stats == "thresholds" else None
        _check(lib().cfl_score_topk_stats(Q, K, d, N, int(k), 1 if image is not None else 0, _ptr(ws), ws.numel(),
                                          _ptr(stats), _ptr(thr), _stream()), "cfl_score_topk_stats")
        return (top_val, top_idx, stats, thr) if thr is not None else (top_val, top_idx, stats)
    return (top_val, top_idx, dense) if want_dense else (top_val, top_idx)


SCORE_NSTATS = 8
SCORE_STAT_NAMES = ("survivors", "spill_queries", "probe_dropped_queries", "redo_queries", "lower_bound_pass",
                    "exact_redo_queries")


def source_catalog_pack(P, mu=None):
    """Tensor-core image of a SOURCE catalog P [N,K,d] (the K prototypes of every source item), centred on mu, for
    score_topk_source; built once per shard.  None for an empty catalog."""
    P = _f32c(P, "P")
    if P.dim() != 3:
        raise CflNativeError("source_catalog_pack: P must be [N,K,d]")
    N, K, d = P.shape
    if N == 0:
        return None
    nbytes = lib().cfl_source_catalog_pack_bytes(N, K, d)
    if nbytes == 0:
        raise CflNativeError(f"source_catalog_pack: K={K} d={d} outside K <= {MAX_K}, d <= 128")
    P2, ldp = _rows(P.reshape(N, K * d), "P")
    img = torch.empty(nbytes + 1024, dtype=torch.uint8, device=P.device)
    off = (-img.data_ptr()) % 1024
    img = img[off:off + nbytes]
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    _check(lib().cfl_source_catalog_pack(_ptr(P2), N, K, d, ldp, _ptr(mu), _ptr(img), nbytes, _stream()),
           "cfl_source_catalog_pack")
    return img


def score_topk_source(Eq, P, image, k, mu=None, idx_base=0, want_dense=False, want_stats=False):
    """The other direction of pcd: top-k SOURCE items (catalog P [N,K,d], image = source_catalog_pack(P, mu)) of every
    TARGET query Eq [Q,d], dist(q,c) = pcd(v = Eq[q], P = P[c]) (base.py:125-139); exact (rescored) values, ties ->
    lower index.  ``want_dense`` appends the un-rescored Gram values [Q,N], ``want_stats`` the int64 counters
    (SCORE_STAT_NAMES) of this call."""
    Eq, ldq = _rows(Eq, "Eq")
    P = _f32c(P, "P")
    if P.dim() != 3:
        raise CflNativeError("score_topk_source: P must be [N,K,d]")
    N, K, d = P.shape
    Q = Eq.shape[0]
    if Eq.shape[1] != d:
        raise CflNativeError(f"score_topk_source: Eq is {tuple(Eq.shape)} but P is {tuple(P.shape)}")
    if N > 0 and image is None:
        raise CflNativeError("score_topk_source: a non-empty catalog needs its image (source_catalog_pack)")
    P2, ldp = _rows(P.reshape(N, K * d), "P")
    dev = P.device
    top_val = torch.empty(Q, k, dtype=torch.float32, device=dev)
    top_idx = torch.empty(Q, k, dtype=torch.int64, device=dev)
    dense = torch.empty(Q, N, dtype=torch.float32, device=dev) if want_dense else None
    stats = torch.zeros(SCORE_NSTATS, dtype=torch.int64, device=dev) if want_stats else None
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    ws = _ws.get(lib().cfl_score_topk_source_workspace_bytes(Q, K, d, N, k), dev)
    _check(lib().cfl_score_topk_source(_ptr(Eq), ldq, Q, K, d, _ptr(image), _ptr(P2), N, ldp, _ptr(mu), int(k),
                                       int(idx_base), _ptr(top_val), _ptr(top_idx), _ptr(dense), _ptr(stats),
                                       _ptr(ws), ws.numel(), _stream()), "cfl_score_topk_source")
    out = (top_val, top_idx)
    if want_dense:
        out += (dense,)
    if want_stats:
        out += (stats,)
    return out


def score_topk_monomer(a, w, P, k, idx_base=0, want_dense=False):
    """Monomer mode on the cross product (base.py:109-117): a [Q,d] and w [Q,K] of the query
    (source) items, P [N,K,d] prototypes of the catalog (target) items -> top-k per query."""
    a, lda = _rows(a, "a")
    w = _f32c(w, "w").contiguous()
    P = _f32c(P, "P")
    if P.dim() != 3:
        raise CflNativeError("score_topk_monomer: P must be [N,K,d]")
    N, K, d = P.shape
    Q = a.shape[0]
    if a.shape[1] != d or tuple(w.shape) != (Q, K):
        raise CflNativeError(f"score_topk_monomer: a {tuple(a.shape)}, w {tuple(w.shape)} do not match P {tuple(P.shape)}")
    P2, ldp = _rows(P.reshape(N, K * d), "P")
    dev = P.device
    top_val = torch.empty(Q, k, dtype=torch.float32, device=dev)
    top_idx = torch.empty(Q, k, dtype=torch.int64, device=dev)
    dense = torch.empty(Q, N, dtype=torch.float32, device=dev) if want_dense else None
    ws = _ws.get(lib().cfl_score_topk_monomer_workspace_bytes(Q, K, d, N, k), dev)
    _check(lib().cfl_score_topk_monomer(_ptr(a), lda, _ptr(w), Q, K, d, _ptr(P2), N, ldp, int(k), int(idx_base),
                                        _ptr(top_val), _ptr(top_idx), _ptr(dense), _ptr(ws), ws.numel(), _stream()),
           "cfl_score_topk_monomer")
    return (top_val, top_idx, dense) if want_dense else (top_val, top_idx)


def monomer_pack(P, mu=None):
    """Tensor-core image of a monomer catalog P [N,K,d] (None when K(d+1) > 128: CUDA-core kernel only)."""
    P = _f32c(P, "P")
    if P.dim() != 3:
        raise CflNativeError("monomer_pack: P must be [N,K,d]")
    N, K, d = P.shape
    nbytes = lib().cfl_monomer_pack_bytes(N, K, d)
    if nbytes == 0:
        return None
    P2, ldp = _rows(P.reshape(N, K * d), "P")
    img = torch.empty(nbytes + 1024, dtype=torch.uint8, device=P.device)
    off = (-img.data_ptr()) % 1024
    img = img[off:off + nbytes]
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    _check(lib().cfl_monomer_pack(_ptr(P2), N, K, d, ldp, _ptr(mu), _ptr(img), nbytes, _stream()), "cfl_monomer_pack")
    return img


def score_topk_monomer_packed(a, w, P, image, k, mu=None, idx_base=0, want_stats=False):
    """Monomer top-k through the tensor-core path (image = monomer_pack(P, mu)); values and indices as
    score_topk_monomer (the survivors are rescored in its arithmetic)."""
    a, lda = _rows(a, "a")
    w = _f32c(w, "w").contiguous()
    P = _f32c(P, "P")
    N, K, d = P.shape
    Q = a.shape[0]
    if a.shape[1] != d or tuple(w.shape) != (Q, K):
        raise CflNativeError(f"score_topk_monomer_packed: a {tuple(a.shape)}, w {tuple(w.shape)} do not match P {tuple(P.shape)}")
    P2, ldp = _rows(P.reshape(N, K * d), "P")
    dev = P.device
    top_val = torch.empty(Q, k, dtype=torch.float32, device=dev)
    top_idx = torch.empty(Q, k, dtype=torch.int64, device=dev)
    stats = torch.zeros(SCORE_NSTATS, dtype=torch.int64, device=dev) if want_stats else None
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    ws = _ws.get(lib().cfl_score_topk_monomer_packed_workspace_bytes(Q, K, d, N, k), dev)
    _check(lib().cfl_score_topk_monomer_packed(_ptr(a), lda, _ptr(w), Q, K, d, _ptr(image), _ptr(P2), N, ldp, _ptr(mu),
                                               int(k), int(idx_base), _ptr(top_val), _ptr(top_idx), _ptr(stats), _ptr(ws),
                                               ws.numel(), _stream()), "cfl_score_topk_monomer_packed")
    return (top_val, top_idx, stats) if want_stats else (top_val, top_idx)


def _monomer_source_catalog(A, W, what):
    A, lda = _rows(A, "A")
    W = _f32c(W, "W").contiguous()
    if W.dim() != 2 or W.shape[0] != A.shape[0]:
        raise CflNativeError(f"{what}: A {tuple(A.shape)} and W {tuple(W.shape)} must be [N,d] and [N,K]")
    return A, lda, W


def monomer_source_pack(A, W, mu=None):
    """Tensor-core image of a monomer SOURCE catalog: A [N,d] = the sources' act(e0), W [N,K] = their gate softmax,
    centred on mu; for score_topk_monomer_source, built once per shard.  None when K(d+1) > 128 (CUDA-core route only)
    or for an empty catalog."""
    A, lda, W = _monomer_source_catalog(A, W, "monomer_source_pack")
    (N, d), K = A.shape, W.shape[1]
    nbytes = lib().cfl_monomer_source_pack_bytes(N, K, d)
    if nbytes == 0:
        return None
    img = torch.empty(nbytes + 1024, dtype=torch.uint8, device=A.device)
    off = (-img.data_ptr()) % 1024
    img = img[off:off + nbytes]
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    _check(lib().cfl_monomer_source_pack(_ptr(A), lda, _ptr(W), N, K, d, _ptr(mu), _ptr(img), nbytes, _stream()),
           "cfl_monomer_source_pack")
    return img


def score_topk_monomer_source(Pq, A, W, image, k, mu=None, idx_base=0, want_stats=False):
    """The other direction of the monomer distance: top-k SOURCE items (catalog A [N,d], W [N,K], image =
    monomer_source_pack(A, W, mu), or None for the CUDA-core route) of every TARGET query Pq [Q,K,d] (its K
    prototypes), dist(q,c) = sum_k W[c,k] |A[c] - Pq[q,k]|^2 (base.py:109-117); exact values, ties -> lower index.
    ``want_stats`` appends the int64 counters (SCORE_STAT_NAMES) of this call."""
    Pq = _f32c(Pq, "Pq")
    if Pq.dim() != 3:
        raise CflNativeError("score_topk_monomer_source: Pq must be [Q,K,d]")
    Q, K, d = Pq.shape
    A, lda, W = _monomer_source_catalog(A, W, "score_topk_monomer_source")
    N = A.shape[0]
    if A.shape[1] != d or W.shape[1] != K:
        raise CflNativeError(f"score_topk_monomer_source: A {tuple(A.shape)}, W {tuple(W.shape)} do not match "
                             f"Pq {tuple(Pq.shape)}")
    if A.device != Pq.device or W.device != Pq.device:
        raise CflNativeError("score_topk_monomer_source: Pq, A and W must be on the same device")
    P2, ldq = _rows(Pq.reshape(Q, K * d), "Pq")
    dev = Pq.device
    top_val = torch.empty(Q, k, dtype=torch.float32, device=dev)
    top_idx = torch.empty(Q, k, dtype=torch.int64, device=dev)
    stats = torch.zeros(SCORE_NSTATS, dtype=torch.int64, device=dev) if want_stats else None
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    ws = _ws.get(lib().cfl_score_topk_monomer_source_workspace_bytes(Q, K, d, N, k), dev)
    _check(lib().cfl_score_topk_monomer_source(_ptr(P2), ldq, Q, K, d, _ptr(image), _ptr(A), lda, _ptr(W), N, _ptr(mu),
                                               int(k), int(idx_base), _ptr(top_val), _ptr(top_idx), _ptr(stats),
                                               _ptr(ws), ws.numel(), _stream()), "cfl_score_topk_monomer_source")
    return (top_val, top_idx, stats) if want_stats else (top_val, top_idx)


def topk_merge(vals, idx):
    """vals/idx: [R,Q,k] sorted per (r,q) -> merged [Q,k]."""
    vals = _f32c(vals, "vals").contiguous()
    idx = idx.contiguous()
    if idx.dtype != torch.int64:
        raise CflNativeError("topk_merge: idx must be int64")
    R, Q, k = vals.shape
    tv = torch.empty(Q, k, dtype=torch.float32, device=vals.device)
    ti = torch.empty(Q, k, dtype=torch.int64, device=vals.device)
    _check(lib().cfl_topk_merge(_ptr(vals), _ptr(idx), R, Q, k, _ptr(tv), _ptr(ti), _stream()),
           "cfl_topk_merge")
    return tv, ti


def topk_record_bytes(Q, k):
    return int(lib().cfl_topk_record_bytes(Q, k))


def topk_pack_records(vals, idx, rec):
    """[Q,k] lists of this rank -> its exchange record (uint8 buffer of topk_record_bytes(Q,k))."""
    Q, k = vals.shape
    _check(lib().cfl_topk_pack_records(_ptr(vals), _ptr(idx), Q, k, _ptr(rec), _stream()), "cfl_topk_pack_records")
    return rec


def topk_merge_records(recs, R, Q, k):
    """Gathered records of R ranks (uint8, R * topk_record_bytes(Q,k)) -> merged (dist [Q,k], index [Q,k])."""
    tv = torch.empty(Q, k, dtype=torch.float32, device=recs.device)
    ti = torch.empty(Q, k, dtype=torch.int64, device=recs.device)
    _check(lib().cfl_topk_merge_records(_ptr(recs), R, Q, k, _ptr(tv), _ptr(ti), _stream()), "cfl_topk_merge_records")
    return tv, ti


def _rank_operands(mode, query, catalog, w):
    """(Pq2, Q, K, d, ldq, w, E2, N, lde) for cfl_pair_dist_rows / cfl_rank_counts.

    pcd / siamese: query [Q,K,d] (or [Q,d]) prototypes, catalog [N,d] embeddings; monomer: query [Q,d] = a, w [Q,K]
    its gate, catalog [N,K,d] prototypes.  The source modes swap the roles: pcd_source: query [Q,d] = the targets'
    e0, catalog [N,K,d] = the sources' prototypes; monomer_source: query [Q,K,d] = the targets' prototypes, catalog
    [N,d] = the sources' a, w [N,K] = the sources' gate."""
    if mode == "pcd_source":
        if catalog.dim() != 3 or w is not None:
            raise CflNativeError("rank counts (pcd_source): catalog must be [N,K,d] source prototypes, no gate")
        N, K, d = catalog.shape
        q2, ldq = _rows(query, "query")
        E2, lde = _rows(_f32c(catalog, "catalog").reshape(N, K * d), "catalog")
        if q2.shape[1] != d:
            raise CflNativeError(f"rank counts (pcd_source): query has d={q2.shape[1]} but the catalog is "
                                 f"{tuple(catalog.shape)}")
        return q2, q2.shape[0], K, d, ldq, None, E2, N, lde
    if mode == "monomer_source":
        query = _f32c(query, "query")
        if query.dim() != 3 or w is None:
            raise CflNativeError("rank counts (monomer_source): query must be [Q,K,d] target prototypes and w the "
                                 "sources' [N,K] gate")
        Q, K, d = query.shape
        q2, ldq = _rows(query.reshape(Q, K * d), "query")
        E2, lde = _rows(catalog, "catalog")
        w = _f32c(w, "w").contiguous()
        if E2.shape[1] != d or tuple(w.shape) != (E2.shape[0], K):
            raise CflNativeError("rank counts (monomer_source): catalog/gate shapes do not match the queries")
        return q2, Q, K, d, ldq, w, E2, E2.shape[0], lde
    if mode == "monomer":
        if catalog.dim() != 3 or w is None:
            raise CflNativeError("rank counts (monomer): catalog must be [N,K,d] prototypes and w the [Q,K] gate")
        N, K, d = catalog.shape
        q2, ldq = _rows(query, "query")
        E2, lde = _rows(_f32c(catalog, "catalog").reshape(N, K * d), "catalog")
        w = _f32c(w, "w").contiguous()
        if q2.shape[1] != d or tuple(w.shape) != (q2.shape[0], K):
            raise CflNativeError("rank counts (monomer): query/gate shapes do not match the catalog")
        return q2, q2.shape[0], K, d, ldq, w, E2, N, lde
    query = _f32c(query, "query")
    if query.dim() == 2:
        query = query[:, None, :]
    Q, K, d = query.shape
    q2, ldq = _rows(query.reshape(Q, K * d), "query")
    E2, lde = _rows(catalog, "catalog")
    if E2.shape[1] != d:
        raise CflNativeError(f"rank counts: query has d={d} but the catalog is {tuple(E2.shape)}")
    return q2, Q, K, d, ldq, None, E2, E2.shape[0], lde


def pair_dist_rows(mode, query, catalog, pos_idx, w=None):
    """dist(q, catalog[pos_idx[q,j]]) -> [Q,J] float32; NaN where pos_idx is outside this shard."""
    q2, Q, K, d, ldq, w, E2, N, lde = _rank_operands(mode, query, catalog, w)
    pos_idx = pos_idx.contiguous()
    if pos_idx.dtype != torch.int64 or pos_idx.dim() != 2 or pos_idx.shape[0] != Q or not pos_idx.is_cuda:
        raise CflNativeError("pair_dist_rows: pos_idx must be a CUDA int64 [Q,J] tensor")
    J = pos_idx.shape[1]
    out = torch.empty(Q, J, dtype=torch.float32, device=E2.device)
    _check(lib().cfl_pair_dist_rows(MODES[mode], _ptr(q2), Q, K, d, ldq, _ptr(w), _ptr(E2), N, lde, _ptr(pos_idx), J,
                                    _ptr(out), _stream()), "cfl_pair_dist_rows")
    return out


def rank_counts(mode, query, catalog, pos_dist, w=None):
    """-> int64 [Q,J,2]: (#{c: dist(q,c) < pos_dist[q,j]}, #{c: dist(q,c) == pos_dist[q,j]}) over this shard."""
    q2, Q, K, d, ldq, w, E2, N, lde = _rank_operands(mode, query, catalog, w)
    pos_dist = _f32c(pos_dist, "pos_dist").contiguous()
    if pos_dist.dim() != 2 or pos_dist.shape[0] != Q:
        raise CflNativeError("rank_counts: pos_dist must be [Q,J]")
    J = pos_dist.shape[1]
    out = torch.empty(Q, J, 2, dtype=torch.int64, device=E2.device)
    _check(lib().cfl_rank_counts(MODES[mode], _ptr(q2), Q, K, d, ldq, _ptr(w), _ptr(E2), N, lde, _ptr(pos_dist), J,
                                 _ptr(out), _stream()), "cfl_rank_counts")
    return out


def rank_counts_packed(query, catalog, image, mu, pos_dist, want_stats=False, mode=None):
    """``rank_counts("pcd", ...)`` on the tensor cores: the counts are taken inside the fused scoring kernel's epilogue
    over the packed catalog ``image`` (``catalog_pack`` of the same catalog / ``mu``), near-ties re-evaluated in the
    direct form -> the same int64 [Q,J,2] as ``rank_counts``.  want_stats: also a dict of the call's statistics.
    Query batches beyond 65536 go through the C entry point in chunks (one call holds at most 4096 scoring CTAs).
    ``mode``: None = pcd (siamese at K = 1) as ``rank_counts("pcd", ...)``; "pcd_source" = ``rank_counts("pcd_source",
    ...)`` with ``image = source_catalog_pack(catalog, mu)``."""
    src = mode == "pcd_source"
    if mode not in (None, "pcd_source"):
        raise CflNativeError(f"rank_counts_packed: mode {mode!r} has no tensor-core count (None or 'pcd_source')")
    q2, Q, K, d, ldq, _, E2, N, lde = _rank_operands("pcd_source" if src else "pcd", query, catalog, None)
    pos_dist = _f32c(pos_dist, "pos_dist").contiguous()
    if pos_dist.dim() != 2 or pos_dist.shape[0] != Q:
        raise CflNativeError("rank_counts_packed: pos_dist must be [Q,J]")
    J = pos_dist.shape[1]
    out = torch.empty(Q, J, 2, dtype=torch.int64, device=E2.device)
    mode = MODES["pcd_source"] if src else MODES["siamese"] if K == 1 else MODES["pcd"]
    ws_bytes = lib().cfl_rank_counts_packed_source_workspace_bytes if src else lib().cfl_rank_counts_packed_workspace_bytes
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    chunk = 65536
    tot = dict(records=0, worst_ratio=0.0, beyond_half_band=0, recounted_queries=0)
    for lo in range(0, max(Q, 1), chunk):
        hi = min(Q, lo + chunk)
        need = ws_bytes(hi - lo, K, d, N)
        ws = _ws.get(need, E2.device)
        _check(lib().cfl_rank_counts_packed(mode, _ptr(q2[lo:hi]), hi - lo, K, d, ldq, _ptr(E2), _ptr(image), N, lde,
                                            _ptr(mu), _ptr(pos_dist[lo:hi]), J, _ptr(out[lo:hi]), _ptr(ws), ws.numel(),
                                            _stream()), "cfl_rank_counts_packed")
        if want_stats:
            raw = (C.c_int64 * 4)()
            _check(lib().cfl_rank_counts_packed_stats(hi - lo, K, d, N, _ptr(ws), ws.numel(), raw, _stream()),
                   "cfl_rank_counts_packed_stats")
            tot["records"] += int(raw[0]); tot["worst_ratio"] = max(tot["worst_ratio"], raw[1] / 1048576.0)
            tot["beyond_half_band"] += int(raw[2]); tot["recounted_queries"] += int(raw[3])
    return (out, tot) if want_stats else out


def dense_rank_counts(dense, pos_dist):
    """Counts of ``rank_counts`` over a dense [Q,N] distance matrix (score_topk's want_dense output)."""
    dense, ldn = _rows(dense, "dense")
    pos_dist = _f32c(pos_dist, "pos_dist").contiguous()
    Q, N = dense.shape
    if pos_dist.dim() != 2 or pos_dist.shape[0] != Q:
        raise CflNativeError("dense_rank_counts: pos_dist must be [Q,J]")
    J = pos_dist.shape[1]
    out = torch.empty(Q, J, 2, dtype=torch.int64, device=dense.device)
    _check(lib().cfl_dense_rank_counts(_ptr(dense), Q, N, ldn, _ptr(pos_dist), J, _ptr(out), _stream()),
           "cfl_dense_rank_counts")
    return out


WITHIN_MAX_RESULTS = 1 << 28          # rows of one range query result: 3 GB of int64 index + fp32 distance
WITHIN_STAT_NAMES = ("records", "worst_ratio", "beyond_half_band", "reemitted_queries", "count_mismatch_queries")


def within_radius(radius, Q, device):
    """A scalar or a [Q] radius -> contiguous float32 [Q] on ``device``."""
    r = torch.as_tensor(radius, dtype=torch.float32, device=device)
    if r.dim() == 0:
        r = r.expand(Q)
    if tuple(r.shape) != (Q,):
        raise CflNativeError(f"radius must be a scalar or [{Q}], got {tuple(r.shape)}")
    return r.contiguous()


def within_counts(mode, query, catalog, radius, w=None, image=None, mu=None):
    """Result size of every query of ``score_within``: #{c : dist(q, c) < radius[q]} -> int64 [Q] (device).  The
    counting pass of ``rank_counts_packed`` (image given: pcd, pcd_source) or ``rank_counts`` with J = 1."""
    if image is not None and catalog.shape[0] > 0:
        c = rank_counts_packed(query, catalog, image, mu, radius[:, None],
                               mode="pcd_source" if mode == "pcd_source" else None)
    else:
        c = rank_counts(mode, query, catalog, radius[:, None], w=w)
    return c[:, 0, 0]


def score_within(mode, query, catalog, radius, w=None, image=None, mu=None, idx_base=0,
                 max_results=WITHIN_MAX_RESULTS, want_stats=False, counts=None):
    """Every catalog row closer than the radius: ``{c : dist(q, c) < radius[q]}`` (strict), exact, as CSR lists
    ``(offsets [Q+1] int64, index [T] int64 = idx_base + row, dist [T] float32)`` ordered by (distance, index) within
    each query.  The distances are the direct-form values of ``pair_dist_rows``, bit for bit; NaN selects nothing.

    ``radius``: a scalar or [Q].  Operands as ``rank_counts``.  ``image`` (= ``catalog_pack(catalog, K, mu)``, pcd;
    ``source_catalog_pack(catalog, mu)``, pcd_source) emits the rows from the tensor-core scoring epilogue; without it
    (monomer, monomer_source, shapes without a tcgen05 tiling) the CUDA cores evaluate every pair in the direct form.  ``counts`` = ``within_counts`` of the same call when the caller
    has them already.

    The result size is data-dependent, so the call reads T = offsets[Q] back to the host once to size the outputs
    (it waits for the counting pass).  T > ``max_results`` raises CflNativeError before the outputs are allocated.
    want_stats: also a dict of the call's counters (WITHIN_STAT_NAMES; ``count_mismatch_queries`` must be 0)."""
    q2, Q, K, d, ldq, w, E2, N, lde = _rank_operands(mode, query, catalog, w)
    dev = E2.device
    r = within_radius(radius, Q, dev)
    mu = None if mu is None else _f32c(mu, "mu").contiguous()
    if N == 0:
        image = None
    if counts is None:
        counts = within_counts(mode, query, catalog, r, w=w, image=image, mu=mu)
    offsets = torch.zeros(Q + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=offsets[1:])
    T = int(offsets[-1])
    if T > max_results:
        raise CflNativeError(f"score_within: the result has {T} rows, more than max_results = {max_results}")
    out_idx = torch.empty(T, dtype=torch.int64, device=dev)
    out_dist = torch.empty(T, dtype=torch.float32, device=dev)
    tot = dict.fromkeys(WITHIN_STAT_NAMES, 0)
    if T == 0:                                                 # nothing to emit (empty outputs have no storage)
        return (offsets, out_idx, out_dist, tot) if want_stats else (offsets, out_idx, out_dist)
    chunk = 65536                                              # one call holds at most 4096 scoring CTAs
    for lo in range(0, Q, chunk):
        hi = min(Q, lo + chunk)
        ws = _ws.get(lib().cfl_score_within_workspace_bytes(MODES[mode], hi - lo, K, d, N), dev)
        _check(lib().cfl_score_within(MODES[mode], _ptr(q2[lo:hi]), hi - lo, K, d, ldq,
                                      None if w is None else _ptr(w if mode == "monomer_source" else w[lo:hi]),
                                      _ptr(E2), _ptr(image), N, lde, _ptr(mu),
                                      _ptr(r[lo:hi]), _ptr(offsets[lo:hi + 1]), int(idx_base), _ptr(out_idx),
                                      _ptr(out_dist), _ptr(ws), ws.numel(), _stream()), "cfl_score_within")
        if want_stats and hi > lo:
            raw = (C.c_int64 * 5)()
            _check(lib().cfl_score_within_stats(_ptr(ws), ws.numel(), raw, _stream()), "cfl_score_within_stats")
            for i, n in enumerate(WITHIN_STAT_NAMES):
                tot[n] = max(tot[n], raw[i] / 1048576.0) if n == "worst_ratio" else tot[n] + int(raw[i])
    return (offsets, out_idx, out_dist, tot) if want_stats else (offsets, out_idx, out_dist)


def within_merge(offsets, idx, dist, out_offsets):
    """Sharded range-query result: rank r's CSR lists (global indices) in row r of ``idx`` / ``dist`` [R, ld] with
    ``offsets`` [R, Q+1] -> the merged (index [T], dist [T]) under ``out_offsets`` [Q+1], ordered by (distance, index)."""
    R, Q1 = offsets.shape
    ld = idx.shape[1]
    T = int(out_offsets[-1])
    out_idx = torch.empty(T, dtype=torch.int64, device=idx.device)
    out_dist = torch.empty(T, dtype=torch.float32, device=idx.device)
    _check(lib().cfl_within_merge(_ptr(offsets.contiguous()), _ptr(idx.contiguous()), _ptr(_f32c(dist, "dist").contiguous()),
                                  ld, R, Q1 - 1, _ptr(out_offsets.contiguous()), _ptr(out_idx), _ptr(out_dist), _stream()),
           "cfl_within_merge")
    return out_idx, out_dist


def auc_counts(pos_scores, neg_scores):
    """-> int64[4] device tensor: twoU, n_pos, n_neg, correct@0 (cfl/utils.py:247-268)."""
    pos = _f32c(pos_scores, "pos_scores").reshape(-1).contiguous()
    neg = _f32c(neg_scores, "neg_scores").reshape(-1).contiguous()
    out = torch.empty(4, dtype=torch.int64, device=pos.device)
    ws = _ws.get(lib().cfl_auc_workspace_bytes(pos.numel(), neg.numel()), pos.device)
    _check(lib().cfl_auc(_ptr(pos), pos.numel(), _ptr(neg), neg.numel(), _ptr(out), _ptr(ws),
                         ws.numel(), _stream()), "cfl_auc")
    return out


def adam_step(p, g, m, v, step, lr, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0):
    for t, n in ((p, "p"), (g, "g"), (m, "m"), (v, "v")):
        _f32c(t, n)
        if not t.is_contiguous():
            raise CflNativeError(f"adam_step: {n} must be contiguous")
    _check(lib().cfl_adam_step(_ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), int(step), float(lr),
                               float(beta1), float(beta2), float(eps), float(grad_scale), _stream()),
           "cfl_adam_step")


def adam_step_dev(p, g, m, v, step_dev, lr, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0):
    """adam_step with the step count read from a device int32 tensor when the kernel runs (CUDA graphs)."""
    for t, n in ((p, "p"), (g, "g"), (m, "m"), (v, "v")):
        _f32c(t, n)
        if not t.is_contiguous():
            raise CflNativeError(f"adam_step_dev: {n} must be contiguous")
    if step_dev.dtype != torch.int32 or not step_dev.is_cuda:
        raise CflNativeError("adam_step_dev: step_dev must be a CUDA int32 tensor")
    _check(lib().cfl_adam_step_dev(_ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), _ptr(step_dev), float(lr),
                                   float(beta1), float(beta2), float(eps), float(grad_scale), _stream()),
           "cfl_adam_step_dev")


def set_kernel_timer(start_event=None, stop_event=None):
    """Records the two torch.cuda.Event objects around the dominant scoring kernel of every
    following score_topk call on this thread (bench.py's roofline timing); None clears."""
    if start_event is None or stop_event is None:
        _check(lib().cfl_set_kernel_timer(None, None), "cfl_set_kernel_timer")
        return
    for ev in (start_event, stop_event):
        ev.record()                      # forces creation of the underlying cudaEvent_t
    _check(lib().cfl_set_kernel_timer(C.c_void_p(start_event.cuda_event), C.c_void_p(stop_event.cuda_event)),
           "cfl_set_kernel_timer")


def selftest_umma_f16(A, Bm):
    """D[128,N] = fp16(A)[128,Kd] @ fp16(Bm)[N,Kd]^T with ONE kind::f16 MMA per 16 dimensions (test only)."""
    A = _f32c(A, "A").contiguous()
    Bm = _f32c(Bm, "Bm").contiguous()
    N, Kd = Bm.shape
    D = torch.empty(128, N, dtype=torch.float32, device=A.device)
    _check(lib().cfl_selftest_umma_f16(_ptr(A), _ptr(Bm), _ptr(D), N, Kd, _stream()), "cfl_selftest_umma_f16")
    return D


def selftest_umma(A, Bm):
    """D[128,N] = A[128,Kd] @ Bm[N,Kd]^T through the tcgen05 3xTF32 core (test only)."""
    A = _f32c(A, "A").contiguous()
    Bm = _f32c(Bm, "Bm").contiguous()
    N, Kd = Bm.shape
    D = torch.empty(128, N, dtype=torch.float32, device=A.device)
    _check(lib().cfl_selftest_umma(_ptr(A), _ptr(Bm), _ptr(D), N, Kd, _stream()), "cfl_selftest_umma")
    return D
