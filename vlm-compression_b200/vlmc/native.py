"""ctypes binding of libvlmc.so (include/vlmc.h) for torch tensors.

PyTorch is plumbing here: it owns device memory and streams; every statistic, selection and
update runs in the hand-written sm_100a kernels behind the C ABI.  There is no CPU path and no
fallback: a missing library or a non-CUDA tensor raises.
"""
import ctypes
import os
import threading

import torch

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libvlmc.so")

F32, F16, BF16 = 0, 1, 2
_DTYPES = {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16}

(OP_SQNORM, OP_DSNOT_STATS, OP_WANDA_SELECT, OP_LORA_MERGE, OP_HESSIAN, OP_CHOL, OP_OBS, OP_DSNOT_REFINE,
 OP_SPARSE24_LINEAR) = range(9)
WS_COUNTER_BYTES = 4096
NOT_POSDEF = 1


class VlmcError(RuntimeError):
    def __init__(self, fn, status, detail=""):
        self.status = status
        super().__init__(f"{fn} failed: status {status} ({detail})")


_lib = None
_lock = threading.Lock()

_vp, _i, _i64, _d, _f, _sz = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double,
                              ctypes.c_float, ctypes.c_size_t)

# name -> (restype, argtypes); must list every symbol include/vlmc.h declares
SIGNATURES = {
    "vlmc_version": (_i, []),
    "vlmc_status_string": (ctypes.c_char_p, [_i]),
    "vlmc_last_cuda_error": (_i, []),
    "vlmc_workspace_bytes": (_sz, [_i, _i64, _i64, _i64]),
    "vlmc_sqnorm_accum": (_i, [_vp, _i, _i64, _i, _i64, _vp, _d, _d, _vp, _sz, _vp]),
    "vlmc_sqnorm_accum_batch_workspace_bytes": (_sz, [_vp, _i, _i]),
    "vlmc_sqnorm_accum_batch": (_i, [_vp, _i, _i, _vp, _sz, _vp]),
    "vlmc_dsnot_stats_batch_workspace_bytes": (_sz, [_vp, _i, _i]),
    "vlmc_dsnot_stats_batch": (_i, [_vp, _i, _i, _vp, _sz, _vp]),
    "vlmc_dsnot_stats": (_i, [_vp, _i, _i64, _i64, _i, _i64, _vp, _vp, _vp, _vp, _d, _d, _d, _vp, _sz, _vp]),
    "vlmc_wanda_rowselect": (_i, [_vp, _i, _i, _i, _i64, _vp, _i, _i, _vp, _i64, _vp, _vp, _sz, _vp]),
    "vlmc_wanda_nm": (_i, [_vp, _i, _i, _i, _i64, _vp, _i, _i, _i, _vp, _i64, _vp, _vp, _sz, _vp]),
    "vlmc_wanda_nm_batch_workspace_bytes": (_sz, [_vp, _i, _i, _i]),
    "vlmc_wanda_nm_batch": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "vlmc_wanda_rowselect_batch_workspace_bytes": (_sz, [_vp, _i]),
    "vlmc_wanda_rowselect_batch": (_i, [_vp, _vp, _i, _i, _i, _vp, _sz, _vp]),
    "vlmc_wanda_threshold": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _i, _vp, _i64, _vp, _vp, _sz, _vp]),
    "vlmc_mask_pack": (_i, [_vp, _i, _i, _i64, _vp, _i64, _vp]),
    "vlmc_mask_apply_packed": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _i, _i64, _vp, _i64, _i, _vp]),
    "vlmc_mask_pack_batch": (_i, [_vp, _i, _vp]),
    "vlmc_mask_apply_packed_batch": (_i, [_vp, _i, _i, _i, _vp]),
    "vlmc_sparselora_merge": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp, _i, _f, _vp, _i64, _i, _vp]),
    "vlmc_sparselora_merge_batch": (_i, [_vp, _i, _i, _i, _vp]),
    "vlmc_sparselora_effective_weight": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp, _i, _f, _vp, _i64, _i, _vp, _i64, _vp]),
    "vlmc_sparselora_linear_forward": (_i, [_vp, _i, _i64, _i, _i64, _vp, _i, _i64, _vp, _vp, _i, _f, _vp, _i64, _i, _vp, _vp, _i64, _vp]),
    "vlmc_sparselora_lora_grads_workspace_bytes": (_sz, [_i, _i, _i]),
    "vlmc_sparselora_lora_grads": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _i, _vp, _vp, _i, _f, _vp, _vp, _vp, _sz, _vp]),
    "vlmc_sparse24_compress": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _vp, _i64, _vp, _vp]),
    "vlmc_sparse24_decompress": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _vp, _i64, _vp]),
    "vlmc_sparse24_linear_forward": (_i, [_vp, _i, _i64, _i, _i64, _vp, _i64, _vp, _i64, _i, _vp, _vp, _i64, _vp, _sz, _vp]),
    "vlmc_sparse24_linear_sp_forward": (_i, [_vp, _i, _i64, _i, _i64, _vp, _i64, _vp, _i64, _i, _vp, _vp, _i64, _vp]),
    "vlmc_sparse24_compress_masked": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp]),
    "vlmc_sparse24_lora_effective_weight": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _vp, _vp, _i, _f, _i, _vp, _i64, _vp]),
    "vlmc_sparse24_lora_grads": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _i, _vp, _vp, _i, _f, _vp, _vp, _vp, _sz, _vp]),
    "vlmc_sparse24_lora_merge": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _vp, _vp, _i, _f, _vp]),
    "vlmc_count_nonzero_batch": (_i, [_vp, _i, _i, _vp, _vp]),
    "vlmc_scores_workspace_bytes": (_sz, [_vp, _i, _i]),
    "vlmc_scores_kth": (_i, [_vp, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "vlmc_scores_protect": (_i, [_vp, _i, _i, _vp, _vp]),
    "vlmc_scores_mask": (_i, [_vp, _i, _i, _vp, _vp]),
    "vlmc_scores_sum": (_i, [_vp, _i, _vp, _vp, _sz, _vp]),
    "vlmc_importance_accum": (_i, [_vp, _i, _i, _vp]),
    "vlmc_importance_finalize": (_i, [_vp, _i, _i, _d, _vp]),
    "vlmc_hessian_prepare": (_i, [_vp, _i, _i64, _f, _vp, _vp, _vp]),
    "vlmc_hessian_add_damp": (_i, [_vp, _i, _i64, _vp, _vp]),
    "vlmc_chol_inv_upper": (_i, [_vp, _i, _i64, _vp, _i64, _vp, _vp, _sz, _vp]),
    "vlmc_chol_set_lookahead": (_i, [_i]),
    "vlmc_gram_upper": (_i, [_vp, _i, _i64, _vp, _i64, _vp]),
    "vlmc_chol_upper": (_i, [_vp, _i, _i64, _vp, _i64, _vp, _vp, _sz, _vp]),
    "vlmc_matrix_nonfinite_count": (_i, [_vp, _i, _i, _i64, _vp, _vp]),
    "vlmc_matrix_replace_inf": (_i, [_vp, _i, _i, _i64, _f, _i, _vp]),
    "vlmc_diag_abs_mean": (_i, [_vp, _i, _i64, _f, _vp, _vp]),
    "vlmc_gemm_tf32x3": (_i, [_i, _i, _i, _i, _f, _vp, _i64, _vp, _i64, _f, _vp, _i64, _i, _i, _vp]),
    "vlmc_obs_sweep": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _vp, _d, _i, _i, _i, _vp, _i64, _vp, _vp, _sz, _vp]),
    "vlmc_obs_sweep_guarded": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _vp, _d, _i, _i, _i, _vp, _i64, _vp, _vp, _vp, _sz,
                                    _vp]),
    "vlmc_hessian_accum": (_i, [_vp, _i, _i64, _i, _i64, _vp, _i64, _d, _d, _i, _i64, _vp]),
    "vlmc_obs_begin": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "vlmc_obs_block_hist": (_i, [_i, _i, _vp, _i64, _i, _i, _i64, _d, _vp, _vp, _sz, _vp]),
    "vlmc_obs_block_finish": (_i, [_vp, _i, _i, _i, _i64, _vp, _i64, _i, _i64, _d, _i, _i, _vp, _i64, _vp, _vp, _sz,
                                   _vp]),
    "vlmc_dsnot_refine_walk": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp, _vp, _i, _i, _i, _f, _i, _f, _i, _i, _i, _vp, _vp,
                                    _sz, _vp]),
    "vlmc_dsnot_refine_apply": (_i, [_vp, _i, _i, _i, _i64, _vp, _i, _i, _i, _i, _vp, _i, _i, _vp, _i64, _vp, _sz, _vp]),
    "vlmc_dsnot_refine": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp, _vp, _i, _i, _i, _f, _i, _f, _i, _i, _i, _i, _i, _vp,
                               _i64, _vp, _vp, _sz, _vp]),
}


def lib_path():
    return _LIB_PATH


def load():
    """Loads the CUDA extension; fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(_LIB_PATH):
            raise ImportError(
                f"{_LIB_PATH} not found: build it with `python vlm-compression_b200/build.py` "
                "(there is no CPU or PyTorch fallback for this path)")
        lib = ctypes.CDLL(_LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name, None)
            if fn is None:
                continue  # reported by tests/test_abi.py; calling it raises AttributeError
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _check(fn, status):
    if status < 0:
        lib = load()
        detail = lib.vlmc_status_string(status).decode()
        if status == -5:
            detail += f", cudaError {lib.vlmc_last_cuda_error()}"
        raise VlmcError(fn, status, detail)
    return status


def _dtype(t):
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"vlmc kernels take float32/float16/bfloat16, got {t.dtype}") from None


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("vlmc has no CPU path: tensors must live on a CUDA device "
                               f"(got device {t.device})")


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


# one zero-initialised workspace per (device, stream); kernels leave the ticket area zero
_workspaces = {}


def workspace(ref, nbytes):
    key = (ref.device.index, _stream(ref))
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.zeros(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=ref.device)
        _workspaces[key] = ws
    return ws


def _rows2d(x):
    """View activations as [T, C] rows without copying when possible (reference: inp.reshape(-1, C))."""
    x2 = x.reshape(-1, x.shape[-1])
    if x2.stride(-1) != 1:
        x2 = x2.contiguous()
    return x2


def sqnorm_accum(x, scaler_row, n_before, b):
    """K1: scaler_row <- scaler_row*n/(n+b) + sum_t x[t,:]^2/(n+b)   (wanda_pruner.py:77-81)."""
    _require_cuda(x, scaler_row)
    lib = load()
    x2 = _rows2d(x)
    T, C = x2.shape
    need = lib.vlmc_workspace_bytes(OP_SQNORM, T, C, 0)
    ws = workspace(x2, need)
    with torch.cuda.device(x2.device):
        st = lib.vlmc_sqnorm_accum(x2.data_ptr(), _dtype(x2), T, C, x2.stride(0), scaler_row.data_ptr(),
                                   float(n_before), float(b), ws.data_ptr(), ws.numel(), _stream(x2))
    _check("vlmc_sqnorm_accum", st)


class StatsItem(ctypes.Structure):
    _fields_ = [("x", _vp), ("T", _i64), ("C", _i), ("ldx", _i64), ("scaler_row", _vp), ("n_before", _d), ("b", _d)]


def sqnorm_accum_batch(xs, scaler_rows, n_before, b):
    """K1 for several linears in ONE launch (vlmc_sqnorm_accum_batch): xs[i] -> scaler_rows[i], the same n_before / b for
    all (the linears of a block see the same calibration samples).  Same results as sqnorm_accum per item."""
    xs = [_rows2d(x) for x in xs]
    _require_cuda(*xs, *scaler_rows)
    lib = load()
    out = None
    by_dtype = {}
    for i, x in enumerate(xs):
        by_dtype.setdefault(_dtype(x), []).append(i)
    for dt, idx in by_dtype.items():
        for c0 in range(0, len(idx), 16):
            chunk = idx[c0:c0 + 16]
            items = (StatsItem * len(chunk))()
            for j, i in enumerate(chunk):
                x = xs[i]
                items[j] = StatsItem(x.data_ptr(), x.shape[0], x.shape[1], x.stride(0), scaler_rows[i].data_ptr(),
                                     float(n_before), float(b))
            need = lib.vlmc_sqnorm_accum_batch_workspace_bytes(items, len(chunk), dt)
            ws = workspace(xs[chunk[0]], need)
            with torch.cuda.device(xs[chunk[0]].device):
                _check("vlmc_sqnorm_accum_batch", lib.vlmc_sqnorm_accum_batch(items, len(chunk), dt, ws.data_ptr(), ws.numel(),
                                                                              _stream(xs[chunk[0]])))
    return out


class DsnotStatsItem(ctypes.Structure):
    _fields_ = [("x", _vp), ("nseg", _i64), ("S", _i64), ("C", _i), ("ldx", _i64), ("scaler_row", _vp), ("sum_row", _vp),
                ("mean", _vp), ("var", _vp), ("n_before", _d), ("b_per_seg", _d), ("ntok_before", _d)]


def dsnot_stats_batch(xs, states, n_before, b_per_seg, ntok_before, nseg=1):
    """K2 for several linears in ONE launch (vlmc_dsnot_stats_batch).  states[i] = (scaler_row, sum_row, mean, var); the
    same n_before / b_per_seg / nseg for all (the linears of a block see the same calibration calls); ntok_before may be
    a list (per item).  Same results as dsnot_stats per item, bit for bit."""
    xs = [_rows2d(x) for x in xs]
    _require_cuda(*xs, *[t for st in states for t in st])
    lib = load()
    if not isinstance(ntok_before, (list, tuple)):
        ntok_before = [ntok_before] * len(xs)
    by_dtype = {}
    for i, x in enumerate(xs):
        if x.shape[0] % nseg:
            raise ValueError("rows must divide evenly into segments")
        by_dtype.setdefault(_dtype(x), []).append(i)
    for dt, idx in by_dtype.items():
        for c0 in range(0, len(idx), 16):
            chunk = idx[c0:c0 + 16]
            items = (DsnotStatsItem * len(chunk))()
            for j, i in enumerate(chunk):
                x, st = xs[i], states[i]
                items[j] = DsnotStatsItem(x.data_ptr(), int(nseg), x.shape[0] // nseg, x.shape[1], x.stride(0),
                                          st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), st[3].data_ptr(),
                                          float(n_before), float(b_per_seg), float(ntok_before[i]))
            need = lib.vlmc_dsnot_stats_batch_workspace_bytes(items, len(chunk), dt)
            ws = workspace(xs[chunk[0]], need)
            with torch.cuda.device(xs[chunk[0]].device):
                _check("vlmc_dsnot_stats_batch", lib.vlmc_dsnot_stats_batch(items, len(chunk), dt, ws.data_ptr(), ws.numel(),
                                                                            _stream(xs[chunk[0]])))


def dsnot_stats(x, scaler_row, sum_row, mean, var, n_before, b_per_seg, ntok_before, nseg=1):
    """K2: DSnoT statistics (dsnot_pruner.py:79-101); x = nseg consecutive calls of equal length."""
    _require_cuda(x, scaler_row, sum_row, mean, var)
    lib = load()
    x2 = _rows2d(x)
    T, C = x2.shape
    if T % nseg:
        raise ValueError("rows must divide evenly into segments")
    need = lib.vlmc_workspace_bytes(OP_DSNOT_STATS, T, C, nseg)
    ws = workspace(x2, need)
    with torch.cuda.device(x2.device):
        st = lib.vlmc_dsnot_stats(x2.data_ptr(), _dtype(x2), nseg, T // nseg, C, x2.stride(0),
                                  scaler_row.data_ptr(), sum_row.data_ptr(), mean.data_ptr(), var.data_ptr(),
                                  float(n_before), float(b_per_seg), float(ntok_before),
                                  ws.data_ptr(), ws.numel(), _stream(x2))
    _check("vlmc_dsnot_stats", st)


def _select_common(W, scaler_row, keep_mask):
    _require_cuda(W, scaler_row, keep_mask)
    if W.dim() != 2 or W.stride(1) != 1:
        raise ValueError("W must be a 2-D row-major weight")
    R, C = W.shape
    if keep_mask is None:
        keep_mask = torch.empty((R, C), dtype=torch.bool, device=W.device)
    if keep_mask.dtype != torch.bool or keep_mask.shape != W.shape or keep_mask.stride(1) != 1:
        raise ValueError("keep_mask must be a bool tensor shaped like W")
    lib = load()
    ws = workspace(W, lib.vlmc_workspace_bytes(OP_WANDA_SELECT, R, C, 0))
    score_mean = torch.empty(1, dtype=torch.float32, device=W.device)
    return lib, R, C, keep_mask, ws, score_mean


def wanda_rowselect(W, scaler_row, k, zero_w=True, keep_mask=None, score_mean=None):
    """K4+K5 (wanda_pruner.py:318-341).  Returns (keep_mask bool [R,C], score_mean 1-elem tensor).  keep_mask / score_mean
    may be passed in (callers that launch on a side stream allocate them on the caller's stream)."""
    lib, R, C, keep_mask, ws, own_mean = _select_common(W, scaler_row, keep_mask)
    if score_mean is None:
        score_mean = own_mean
    elif not score_mean.is_cuda or score_mean.dtype != torch.float32 or score_mean.numel() != 1:
        raise ValueError("score_mean must be a 1-element float32 CUDA tensor")
    with torch.cuda.device(W.device):
        st = lib.vlmc_wanda_rowselect(W.data_ptr(), _dtype(W), R, C, W.stride(0), scaler_row.data_ptr(), int(k),
                                      int(bool(zero_w)), keep_mask.data_ptr(), keep_mask.stride(0),
                                      score_mean.data_ptr(), ws.data_ptr(), ws.numel(), _stream(W))
    _check("vlmc_wanda_rowselect", st)
    return keep_mask, score_mean


def wanda_nm(W, scaler_row, n, m, zero_w=True, keep_mask=None):
    """K4+K6 (wanda_pruner.py:323-329)."""
    lib, R, C, keep_mask, ws, score_mean = _select_common(W, scaler_row, keep_mask)
    with torch.cuda.device(W.device):
        st = lib.vlmc_wanda_nm(W.data_ptr(), _dtype(W), R, C, W.stride(0), scaler_row.data_ptr(), int(n), int(m),
                               int(bool(zero_w)), keep_mask.data_ptr(), keep_mask.stride(0),
                               score_mean.data_ptr(), ws.data_ptr(), ws.numel(), _stream(W))
    _check("vlmc_wanda_nm", st)
    return keep_mask, score_mean


class SelectItem(ctypes.Structure):
    """vlmc_select_item (include/vlmc.h)."""
    _fields_ = [("W", _vp), ("ldw", _i64), ("R", _i), ("C", _i), ("scaler_row", _vp), ("keep_mask", _vp),
                ("ldm", _i64), ("score_mean", _vp)]


def wanda_nm_batch(Ws, scaler_rows, n, m, zero_w=True, keep_masks=None):
    """K4+K6 for all linears of a block in ONE launch (vlmc_wanda_nm_batch).  Ws: list of 2-D weights of one dtype on
    one device; scaler_rows: matching [C] fp32 tensors.  Returns ([keep_mask], score_means [len(Ws)] device tensor);
    same masks and weights as len(Ws) calls of wanda_nm."""
    if not Ws:
        return [], None
    dev, dt = Ws[0].device, Ws[0].dtype
    _require_cuda(*Ws, *scaler_rows)
    if keep_masks is None:
        keep_masks = [torch.empty(W.shape, dtype=torch.bool, device=dev) for W in Ws]
    means = torch.empty(len(Ws), dtype=torch.float32, device=dev)
    items = (SelectItem * len(Ws))()
    for i, (W, s, k) in enumerate(zip(Ws, scaler_rows, keep_masks)):
        if W.dim() != 2 or W.stride(1) != 1 or W.dtype != dt or W.device != dev:
            raise ValueError("weights must be 2-D row-major tensors of one dtype on one device")
        if k.dtype != torch.bool or k.shape != W.shape or k.stride(1) != 1:
            raise ValueError("keep_mask must be a bool tensor shaped like W")
        if s.dtype != torch.float32 or s.numel() != W.shape[1]:
            raise ValueError("scaler_row must be float32 [C]")
        items[i] = SelectItem(W.data_ptr(), W.stride(0), W.shape[0], W.shape[1], s.data_ptr(), k.data_ptr(), k.stride(0),
                              means[i:i + 1].data_ptr())
    lib = load()
    ws = workspace(Ws[0], lib.vlmc_wanda_nm_batch_workspace_bytes(items, len(Ws), _DTYPES[dt], int(m)))
    with torch.cuda.device(dev):
        st = lib.vlmc_wanda_nm_batch(items, len(Ws), _dtype(Ws[0]), int(n), int(m), int(bool(zero_w)), ws.data_ptr(),
                                     ws.numel(), _stream(Ws[0]))
    _check("vlmc_wanda_nm_batch", st)
    return keep_masks, means


def wanda_rowselect_batch(Ws, scaler_rows, ks, zero_w=True, keep_masks=None):
    """K4+K5 for several linears in ONE call (vlmc_wanda_rowselect_batch: one launch per distinct row length).  Ws: list of
    2-D weights (or row shards) of one dtype on one device; ks: rows' prune count per linear.  Returns ([keep_mask],
    score_means [len(Ws)] device tensor); same masks, weights and means as len(Ws) calls of wanda_rowselect."""
    if not Ws:
        return [], None
    dev, dt = Ws[0].device, Ws[0].dtype
    _require_cuda(*Ws, *scaler_rows)
    if keep_masks is None:
        keep_masks = [torch.empty(W.shape, dtype=torch.bool, device=dev) for W in Ws]
    out_masks, means_all = list(keep_masks), torch.empty(len(Ws), dtype=torch.float32, device=dev)
    lib = load()
    for c0 in range(0, len(Ws), 16):
        sl = slice(c0, min(c0 + 16, len(Ws)))
        n = sl.stop - sl.start
        items = (SelectItem * n)()
        karr = (ctypes.c_int * n)(*[int(k) for k in ks[sl]])
        for i, (W, s, k) in enumerate(zip(Ws[sl], scaler_rows[sl], keep_masks[sl])):
            if W.dim() != 2 or W.stride(1) != 1 or W.dtype != dt or W.device != dev:
                raise ValueError("weights must be 2-D row-major tensors of one dtype on one device")
            if k.dtype != torch.bool or k.shape != W.shape or k.stride(1) != 1:
                raise ValueError("keep_mask must be a bool tensor shaped like W")
            if s.dtype != torch.float32 or s.numel() != W.shape[1]:
                raise ValueError("scaler_row must be float32 [C]")
            items[i] = SelectItem(W.data_ptr(), W.stride(0), W.shape[0], W.shape[1], s.data_ptr(), k.data_ptr(), k.stride(0),
                                  means_all[c0 + i:c0 + i + 1].data_ptr())
        ws = workspace(Ws[0], lib.vlmc_wanda_rowselect_batch_workspace_bytes(items, n))
        with torch.cuda.device(dev):
            st = lib.vlmc_wanda_rowselect_batch(items, karr, n, _dtype(Ws[0]), int(bool(zero_w)), ws.data_ptr(), ws.numel(),
                                                _stream(Ws[0]))
        _check("vlmc_wanda_rowselect_batch", st)
    return out_masks, means_all


def wanda_threshold(W, scaler_row, k_global, zero_w=True, keep_mask=None):
    """K4+K7 (wanda_pruner.py:682-683)."""
    lib, R, C, keep_mask, ws, score_mean = _select_common(W, scaler_row, keep_mask)
    with torch.cuda.device(W.device):
        st = lib.vlmc_wanda_threshold(W.data_ptr(), _dtype(W), R, C, W.stride(0), scaler_row.data_ptr(),
                                      int(k_global), int(bool(zero_w)), keep_mask.data_ptr(),
                                      keep_mask.stride(0), score_mean.data_ptr(), ws.data_ptr(), ws.numel(),
                                      _stream(W))
    _check("vlmc_wanda_threshold", st)
    return keep_mask, score_mean


def mask_pack(keep_mask, bits=None):
    """keep_mask [R, C] bool/uint8 -> bits [R, C // 8] uint8 (bit e of byte j = column 8 j + e)."""
    _require_cuda(keep_mask, bits)
    R, C = keep_mask.shape
    if bits is None:
        bits = torch.empty((R, C // 8), dtype=torch.uint8, device=keep_mask.device)
    with torch.cuda.device(keep_mask.device):
        st = load().vlmc_mask_pack(keep_mask.data_ptr(), R, C, keep_mask.stride(0), bits.data_ptr(), bits.stride(0),
                                   _stream(keep_mask))
    _check("vlmc_mask_pack", st)
    return bits


def mask_apply_packed(W, bits, keep_mask=None, zero_w=True, rows_per_seg=0, seg_stride=0):
    """bits -> keep_mask bytes (optional) and zeroed weights (in place on W [R, C]).  bits is [R, C // 8], or, with
    rows_per_seg > 0, a flat uint8 buffer in which the rows [g * rows_per_seg, (g + 1) * rows_per_seg) start at byte
    g * seg_stride (the [rank][row shard] layout of one all-gather)."""
    _require_cuda(W, bits, keep_mask)
    R, C = W.shape
    ldb = bits.stride(0) if bits.dim() == 2 else C // 8
    with torch.cuda.device(W.device):
        st = load().vlmc_mask_apply_packed(W.data_ptr(), _dtype(W), R, C, W.stride(0), bits.data_ptr(), ldb,
                                           int(rows_per_seg), int(seg_stride), keep_mask.data_ptr() if keep_mask is not None else None,
                                           keep_mask.stride(0) if keep_mask is not None else 0, int(zero_w), _stream(W))
    _check("vlmc_mask_apply_packed", st)
    return keep_mask


class PackItem(ctypes.Structure):
    """vlmc_pack_item (include/vlmc.h)."""
    _fields_ = [("keep_mask", _vp), ("R", _i), ("C", _i), ("ldm", _i64), ("bits", _vp), ("ldb", _i64)]


class ApplyItem(ctypes.Structure):
    """vlmc_apply_item (include/vlmc.h)."""
    _fields_ = [("W", _vp), ("R", _i), ("C", _i), ("ldw", _i64), ("bits", _vp), ("ldb", _i64), ("rows_per_seg", _i),
                ("seg_stride", _i64), ("keep_mask", _vp), ("ldm", _i64)]


def mask_pack_batch(keep_masks, bits_list):
    """mask_pack for up to 16 (keep_mask [R, C], bits [R, C // 8]) pairs per launch; same bits."""
    _require_cuda(*keep_masks, *bits_list)
    lib = load()
    for c0 in range(0, len(keep_masks), 16):
        ks, bs = keep_masks[c0:c0 + 16], bits_list[c0:c0 + 16]
        items = (PackItem * len(ks))()
        for i, (k, b) in enumerate(zip(ks, bs)):
            items[i] = PackItem(k.data_ptr(), k.shape[0], k.shape[1], k.stride(0), b.data_ptr(), b.stride(0))
        with torch.cuda.device(ks[0].device):
            st = lib.vlmc_mask_pack_batch(items, len(ks), _stream(ks[0]))
        _check("vlmc_mask_pack_batch", st)
    return bits_list


def mask_apply_packed_batch(Ws, bits_list, keep_masks, zero_w=True, rows_per_seg=None, seg_stride=0):
    """mask_apply_packed for up to 16 matrices of one dtype per launch.  bits_list[i] is the flat uint8 buffer (or view) that
    holds matrix i's bits in the [segment][row shard] layout; rows_per_seg[i] rows per segment, seg_stride bytes apart."""
    _require_cuda(*Ws, *bits_list, *keep_masks)
    lib = load()
    for c0 in range(0, len(Ws), 16):
        ws_, bs, ks = Ws[c0:c0 + 16], bits_list[c0:c0 + 16], keep_masks[c0:c0 + 16]
        items = (ApplyItem * len(ws_))()
        for i, (W, b, k) in enumerate(zip(ws_, bs, ks)):
            R, C = W.shape
            rps = int(rows_per_seg[c0 + i]) if rows_per_seg is not None else 0
            items[i] = ApplyItem(W.data_ptr(), R, C, W.stride(0), b.data_ptr(), b.stride(0) if b.dim() == 2 else C // 8, rps,
                                 int(seg_stride), k.data_ptr() if k is not None else None, k.stride(0) if k is not None else 0)
        with torch.cuda.device(ws_[0].device):
            st = lib.vlmc_mask_apply_packed_batch(items, len(ws_), _dtype(ws_[0]), int(bool(zero_w)), _stream(ws_[0]))
        _check("vlmc_mask_apply_packed_batch", st)
    return keep_masks


def sparselora_merge(W, A, B, scaling, keep_mask, remask=True):
    """K14 (lora.py:384-387 + train.py:634-637), in place on W."""
    _require_cuda(W, A, B, keep_mask)
    if W.dim() != 2 or W.stride(1) != 1:
        raise ValueError("W must be a 2-D row-major weight")
    if A.dtype != torch.float32 or B.dtype != torch.float32:
        raise TypeError("lora_A / lora_B must be float32")
    A = A.contiguous()
    B = B.contiguous()
    R, C = W.shape
    rank = A.shape[0]
    if A.shape != (rank, C) or B.shape != (R, rank):
        raise ValueError("lora_A must be [r, C] and lora_B [R, r]")
    if keep_mask.dtype != torch.bool or keep_mask.shape != W.shape or keep_mask.stride(1) != 1:
        raise ValueError("mask must be a bool tensor shaped like W")
    lib = load()
    with torch.cuda.device(W.device):
        st = lib.vlmc_sparselora_merge(W.data_ptr(), _dtype(W), R, C, W.stride(0), A.data_ptr(), B.data_ptr(),
                                       rank, float(scaling), keep_mask.data_ptr(), keep_mask.stride(0),
                                       int(bool(remask)), _stream(W))
    _check("vlmc_sparselora_merge", st)
    return W


class MergeItem(ctypes.Structure):
    """vlmc_merge_item (include/vlmc.h)."""
    _fields_ = [("W", _vp), ("ldw", _i64), ("R", _i), ("C", _i), ("A", _vp), ("B", _vp), ("rank", _i), ("scaling", _f),
                ("keep_mask", _vp), ("ldm", _i64)]


def sparselora_merge_batch(Ws, As, Bs, scalings, keep_masks, remask=True):
    """K14 for several LoRA linears of one dtype in one launch per 16 (train.py:626-637 merges module by module).
    Same results as sparselora_merge per linear; ranks above 8 fall back to the per-linear kernel."""
    keep = []
    todo = []
    for W, A, B, s, M in zip(Ws, As, Bs, scalings, keep_masks):
        R, C, rank, A, B = _lora_common(W, A, B, M)
        if rank > 8:
            sparselora_merge(W, A, B, s, M, remask=remask)
            continue
        keep += [A, B]
        todo.append(MergeItem(W.data_ptr(), W.stride(0), R, C, A.data_ptr(), B.data_ptr(), rank, float(s), M.data_ptr(),
                              M.stride(0)))
    if not todo:
        return
    lib = load()
    dt, ref = _dtype(Ws[0]), Ws[0]
    if any(_dtype(W) != dt for W in Ws):
        raise TypeError("all weights of one call must share a dtype")
    with torch.cuda.device(ref.device):
        for c0 in range(0, len(todo), 16):
            chunk = todo[c0:c0 + 16]
            items = (MergeItem * len(chunk))(*chunk)
            _check("vlmc_sparselora_merge_batch",
                   lib.vlmc_sparselora_merge_batch(items, len(chunk), dt, int(bool(remask)), _stream(ref)))


class TensorItem(ctypes.Structure):
    """vlmc_tensor_item (include/vlmc.h)."""
    _fields_ = [("ptr", _vp), ("numel", _i64)]


def count_nonzero(tensors):
    """K17: number of non-zero elements of every tensor (evaluate_old.py:331-334), as one int64 device tensor
    [len(tensors)] in the order given.  Tensors of one device; float32 / float16 / bfloat16; non-contiguous ones are
    copied.  64 tensors of one dtype per launch."""
    tensors = list(tensors)
    if not tensors:
        return torch.zeros(0, dtype=torch.int64)
    _require_cuda(*tensors)
    dev = tensors[0].device
    out = torch.zeros(len(tensors), dtype=torch.int64, device=dev)
    lib = load()
    by_dtype = {}
    for i, t in enumerate(tensors):
        by_dtype.setdefault(_dtype(t), []).append(i)
    keep = []                                              # contiguous copies must outlive the launches
    with torch.cuda.device(dev):
        for dt, idx in by_dtype.items():
            for c0 in range(0, len(idx), 64):
                chunk = idx[c0:c0 + 64]
                items = (TensorItem * len(chunk))()
                for j, i in enumerate(chunk):
                    t = tensors[i] if tensors[i].is_contiguous() else tensors[i].contiguous()
                    keep.append(t)
                    items[j] = TensorItem(t.data_ptr() if t.numel() else None, t.numel())
                part = torch.empty(len(chunk), dtype=torch.int64, device=dev)
                _check("vlmc_count_nonzero_batch",
                       lib.vlmc_count_nonzero_batch(items, len(chunk), dt, part.data_ptr(), _stream(part)))
                out[torch.tensor(chunk, device=dev)] = part
    return out


# ---- SURVEY 8f-4: global sparsity allocation on fp32 importance scores (K18-K22) -------------------------------------
class ScoreItem(ctypes.Structure):
    _fields_ = [("scores", _vp), ("numel", _i64), ("segment", _i), ("aux_dtype", _i), ("aux", _vp), ("out", _vp)]


def _score_items(scores, segments=None, aux=None, outs=None):
    """Host array of vlmc_score_item for fp32 CUDA score tensors (used in place, so they must be contiguous)."""
    scores = list(scores)
    if not scores:
        raise ValueError("no score tensors given")
    _require_cuda(*scores)
    dev = scores[0].device
    items = (ScoreItem * len(scores))()
    for i, t in enumerate(scores):
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev:
            raise TypeError("importance scores must be contiguous float32 tensors on one CUDA device")
        a = aux[i] if aux is not None else None
        o = outs[i] if outs is not None else None
        adt = 0
        if a is not None:
            _require_cuda(a)
            if a.numel() != t.numel() or not a.is_contiguous() or a.device != dev:
                raise ValueError("parameter / gradient tensors must be contiguous and sized like their scores")
            adt = _dtype(a)
        if o is not None:
            _require_cuda(o)
            if o.dtype != torch.float32 or o.numel() != t.numel() or not o.is_contiguous() or o.device != dev:
                raise ValueError("outputs must be contiguous float32 tensors sized like their scores")
        n = t.numel()
        items[i] = ScoreItem(t.data_ptr() if n else None, n, int(segments[i]) if segments is not None else 0, adt,
                             a.data_ptr() if (a is not None and n) else None,
                             o.data_ptr() if (o is not None and n) else None)
    return items, dev, scores[0]


def scores_kth(scores, segments, k):
    """K18: exact k-th smallest score (1-based) per segment, torch.topk order (layer_single_base_pruner.py:157-158,
    :168-170).  scores: fp32 CUDA tensors; segments[i]: segment of scores[i]; k: one rank per segment.  Returns a float32
    device tensor [nseg]; nothing is synchronised."""
    k = [int(x) for x in k]
    nseg = len(k)
    sizes = [0] * nseg
    for t, sg in zip(scores, segments):
        sizes[sg] += t.numel()
    for ks, n in zip(k, sizes):
        if ks < 1 or ks > n:
            # topk(k=0)[0][-1] on the reference side
            raise IndexError(f"rank {ks} is outside a segment of {n} scores")
    items, dev, ref = _score_items(scores, segments)
    lib = load()
    with torch.cuda.device(dev):
        # ranks go up through pinned memory: a pageable host-to-device copy would make the call wait for the stream
        kd = torch.tensor(k, dtype=torch.int64).pin_memory().to(dev, non_blocking=True)
        out = torch.empty(nseg, dtype=torch.float32, device=dev)
        nbytes = lib.vlmc_scores_workspace_bytes(items, len(items), nseg)
        ws = workspace(ref, nbytes)
        _check("vlmc_scores_kth", lib.vlmc_scores_kth(items, len(items), nseg, kd.data_ptr(), out.data_ptr(),
                                                      ws.data_ptr(), ws.numel(), _stream(ref)))
    return out


def scores_protect(scores, segments, thr):
    """K19: scores[v >= thr[segment]] = finfo(float32).max in place (layer_single_base_pruner.py:160)."""
    items, dev, ref = _score_items(scores, segments)
    _require_cuda(thr)
    with torch.cuda.device(dev):
        _check("vlmc_scores_protect", load().vlmc_scores_protect(items, len(items), thr.numel(), thr.data_ptr(),
                                                                 _stream(ref)))


def scores_mask(scores, segments, thr, outs=None, params=None):
    """K20: outs[i] = (scores[i] > thr[segment]) as float32 (layer_single_base_pruner.py:174) and, when params is given,
    params[i] *= that mask in the parameter's dtype (:223-225)."""
    items, dev, ref = _score_items(scores, segments, aux=params, outs=outs)
    _require_cuda(thr)
    with torch.cuda.device(dev):
        _check("vlmc_scores_mask", load().vlmc_scores_mask(items, len(items), thr.numel(), thr.data_ptr(), _stream(ref)))


def scores_sum(scores):
    """K21: per-tensor sums as a float64 device tensor (layer_single_base_pruner.py:296), fixed summation order."""
    items, dev, ref = _score_items(scores)
    lib = load()
    with torch.cuda.device(dev):
        out = torch.empty(len(items), dtype=torch.float64, device=dev)
        nbytes = lib.vlmc_scores_workspace_bytes(items, len(items), 1)
        ws = workspace(ref, nbytes)
        _check("vlmc_scores_sum", lib.vlmc_scores_sum(items, len(items), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                                      _stream(ref)))
    return out


IMPORTANCE_MODES = {"obd": 0, "abs": 1, "gradient": 2}


def importance_accum(accs, grads, mode):
    """K22a: accs[i] += grads[i].float() ** 2 ("obd") or .abs() ("abs") (layer_single_base_pruner.py:455-458)."""
    items, dev, ref = _score_items(accs, aux=list(grads))
    with torch.cuda.device(dev):
        _check("vlmc_importance_accum", load().vlmc_importance_accum(items, len(items), IMPORTANCE_MODES[mode],
                                                                     _stream(ref)))


def importance_finalize(accs, params, outs, mode, num_batches):
    """K22b: outs[i] = params[i].float() ** 2 * (accs[i] / num_batches) ("obd"), |w| * |acc / n| ("abs") or |acc / n|
    ("gradient") (layer_single_base_pruner.py:460-473)."""
    m = IMPORTANCE_MODES[mode]
    items, dev, ref = _score_items(accs, aux=None if m == 2 else list(params), outs=list(outs))
    with torch.cuda.device(dev):
        _check("vlmc_importance_finalize", load().vlmc_importance_finalize(items, len(items), m, float(num_batches),
                                                                           _stream(ref)))


def _lora_common(W, A, B, keep_mask):
    _require_cuda(W, A, B, keep_mask)
    if W.dim() != 2 or W.stride(1) != 1:
        raise ValueError("W must be a 2-D row-major tensor")
    if A.dtype != torch.float32 or B.dtype != torch.float32:
        raise TypeError("lora_A / lora_B must be float32")
    R, C = W.shape
    rank = A.shape[0]
    if A.shape != (rank, C) or B.shape != (R, rank):
        raise ValueError("lora_A must be [r, C] and lora_B [R, r]")
    if keep_mask is not None and (keep_mask.dtype != torch.bool or keep_mask.shape != W.shape or keep_mask.stride(1) != 1):
        raise ValueError("mask must be a bool tensor shaped like W")
    return R, C, rank, A.contiguous(), B.contiguous()


def sparselora_effective_weight(W, A, B, scaling, keep_mask, sparse=True, out=None):
    """K15 (lora.py:364-375): the weight of the masked training forward, (W + s*BA) * M or W * M + s*BA, in W's dtype.
    W is left untouched; returns `out` [R, C]."""
    R, C, rank, A, B = _lora_common(W, A, B, keep_mask)
    if out is None:
        out = torch.empty((R, C), dtype=W.dtype, device=W.device)
    _require_cuda(out)
    with torch.cuda.device(W.device):
        st = load().vlmc_sparselora_effective_weight(W.data_ptr(), _dtype(W), R, C, W.stride(0), A.data_ptr(), B.data_ptr(),
                                                     rank, float(scaling), keep_mask.data_ptr(), keep_mask.stride(0),
                                                     int(bool(sparse)), out.data_ptr(), out.stride(0), _stream(W))
    _check("vlmc_sparselora_effective_weight", st)
    return out


def sparselora_linear_forward_supported(x, W, keep_mask, rank):
    """True when K23 takes the call: 16-bit layer dtype, x in that dtype, TMA-compatible pitches."""
    R, C = W.shape
    return (W.dtype in (torch.float16, torch.bfloat16) and x.dtype == W.dtype and W.is_cuda and 1 <= rank <= 16 and
            C % 8 == 0 and R % 8 == 0 and W.stride(1) == 1 and W.stride(0) % 8 == 0 and keep_mask.stride(1) == 1 and
            keep_mask.stride(0) % 16 == 0 and W.data_ptr() % 16 == 0 and keep_mask.data_ptr() % 16 == 0)


def sparselora_linear_forward(x, W, A, B, scaling, keep_mask, sparse=True, bias=None, out=None):
    """K23 (lora.py:359-382): y = F.linear(x, W_eff, bias) with W_eff = (W + s*BA) * M or W * M + s*BA built on chip
    (never written to HBM).  x [..., C] and W [R, C] in fp16 / bf16; returns y [..., R] in that dtype."""
    R, C, rank, A, B = _lora_common(W, A, B, keep_mask)
    _require_cuda(x)
    if x.dtype != W.dtype or x.shape[-1] != C:
        raise ValueError("x must be [..., C] in the layer's dtype")
    x2 = x.reshape(-1, C)
    if x2.stride(1) != 1 or x2.stride(0) % 8 != 0 or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    Tn = x2.shape[0]
    if bias is not None:
        bias = bias.to(W.dtype).contiguous()
    y = out if out is not None else torch.empty((Tn, R), dtype=W.dtype, device=W.device)
    _require_cuda(y)
    if Tn == 0:
        return y.reshape(*x.shape[:-1], R)
    with torch.cuda.device(W.device):
        st = load().vlmc_sparselora_linear_forward(x2.data_ptr(), _dtype(W), Tn, C, x2.stride(0), W.data_ptr(), R, W.stride(0),
                                                   A.data_ptr(), B.data_ptr(), rank, float(scaling), keep_mask.data_ptr(),
                                                   keep_mask.stride(0), int(bool(sparse)),
                                                   bias.data_ptr() if bias is not None else None, y.data_ptr(), y.stride(0),
                                                   _stream(W))
    _check("vlmc_sparselora_linear_forward", st)
    return y.reshape(*x.shape[:-1], R)


def sparselora_lora_grads(G, A, B, scaling, keep_mask, sparse=True):
    """K16: (dA [r, C], dB [R, r]) fp32 from G = dL/dW_eff [R, C] (W's dtype): the autograd of K15's expression."""
    R, C, rank, A, B = _lora_common(G, A, B, keep_mask if sparse else None)
    lib = load()
    dA = torch.empty((rank, C), dtype=torch.float32, device=G.device)
    dB = torch.empty((R, rank), dtype=torch.float32, device=G.device)
    ws = workspace(G, lib.vlmc_sparselora_lora_grads_workspace_bytes(R, C, rank))
    with torch.cuda.device(G.device):
        st = lib.vlmc_sparselora_lora_grads(G.data_ptr(), _dtype(G), R, C, G.stride(0),
                                            keep_mask.data_ptr() if sparse else None, keep_mask.stride(0) if sparse else 0,
                                            int(bool(sparse)), A.data_ptr(), B.data_ptr(), rank, float(scaling),
                                            dA.data_ptr(), dB.data_ptr(), ws.data_ptr(), ws.numel(), _stream(G))
    _check("vlmc_sparselora_lora_grads", st)
    return dA, dB


NOT_2OF4 = 8                     # status bit of vlmc_sparse24_compress (include/vlmc.h)


def _sparse24_weight_dtype(t):
    if t.dtype not in (torch.float16, torch.bfloat16):
        raise TypeError(f"compressed 2:4 weights are float16 / bfloat16, got {t.dtype}")
    return _dtype(t)


def _sparse24_operands(values, meta, C):
    """Checks a (values [R, C/2], meta [R, C/16] int16) pair; meta holds the format's uint16 words bit for bit."""
    _require_cuda(values, meta)
    _sparse24_weight_dtype(values)
    C = int(C)
    if C < 16 or C % 16:
        raise ValueError(f"compressed 2:4 weights need C % 16 == 0, got C = {C}")
    if values.dim() != 2 or values.shape[1] != C // 2 or values.stride(1) != 1:
        raise ValueError("values must be a row-major [R, C/2] tensor")
    R = values.shape[0]
    if meta.dtype != torch.int16 or meta.shape != (R, C // 16) or meta.stride(1) != 1:
        raise ValueError("meta must be a row-major int16 [R, C/16] tensor")
    return R, C


def sparse24_compress(W):
    """K24: a 2:4-sparse fp16 / bf16 weight [R, C] -> (values [R, C/2] in W's dtype, meta [R, C/16] int16 holding the
    uint16 words of include/vlmc.h).  Raises ValueError, leaving W untouched, when a group of 4 columns holds more than
    two non-zeros (synchronises on the status word)."""
    _require_cuda(W)
    dt = _sparse24_weight_dtype(W)
    if W.dim() != 2 or W.stride(1) != 1:
        raise ValueError("W must be a 2-D row-major weight")
    R, C = W.shape
    if C % 16:
        raise ValueError(f"compressed 2:4 weights need C % 16 == 0, got C = {C}")
    values = torch.empty((R, C // 2), dtype=W.dtype, device=W.device)
    meta = torch.empty((R, C // 16), dtype=torch.int16, device=W.device)
    status = torch.empty(1, dtype=torch.int32, device=W.device)
    with torch.cuda.device(W.device):
        st = load().vlmc_sparse24_compress(W.data_ptr(), dt, R, C, W.stride(0), values.data_ptr(), values.stride(0),
                                           meta.data_ptr(), meta.stride(0), status.data_ptr(), _stream(W))
    _check("vlmc_sparse24_compress", st)
    if int(status.item()) & NOT_2OF4:
        raise ValueError("weight is not 2:4 sparse: a group of 4 columns holds more than two non-zeros")
    return values, meta


def sparse24_decompress(values, meta, C, out=None):
    """K25: the dense weight [R, C] of a compressed pair (+0 at pruned positions), into `out` (any row pitch) if given."""
    R, C = _sparse24_operands(values, meta, C)
    if out is None:
        out = torch.empty((R, C), dtype=values.dtype, device=values.device)
    _require_cuda(out)
    if out.dtype != values.dtype or out.shape != (R, C) or out.stride(1) != 1:
        raise ValueError("out must be a row-major [R, C] tensor of the values' dtype")
    with torch.cuda.device(values.device):
        st = load().vlmc_sparse24_decompress(values.data_ptr(), _dtype(values), R, C, values.stride(0), meta.data_ptr(),
                                             meta.stride(0), out.data_ptr(), out.stride(0), _stream(values))
    _check("vlmc_sparse24_decompress", st)
    return out


def _sparse24_linear_operands(x, values, meta, C, bias, out):
    """Checks the operands of K26 / K31 and copies those whose row pitch or base TMA cannot take (meta pitch padded to 16
    bytes).  Returns (R, C, x2 [T, C], values, meta, bias, y [T, R])."""
    R, C = _sparse24_operands(values, meta, C)
    _require_cuda(x)
    if x.dtype != values.dtype or x.shape[-1] != C:
        raise ValueError("x must be [..., C] in the layer's dtype")
    x2 = x.reshape(-1, C)
    if x2.stride(1) != 1 or x2.stride(0) % 8 != 0 or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    if values.stride(0) % 8 != 0 or values.data_ptr() % 16 != 0:
        values = values.contiguous()
    if meta.stride(0) % 8 != 0 or meta.data_ptr() % 16 != 0:
        padded = torch.zeros((R, (C // 16 + 7) // 8 * 8), dtype=torch.int16, device=meta.device)
        padded[:, :C // 16] = meta
        meta = padded[:, :C // 16]
    if bias is not None:
        _require_cuda(bias)
        bias = bias.to(values.dtype).contiguous()
        if bias.shape != (R,):
            raise ValueError("bias must be [R]")
    Tn = x2.shape[0]
    y = out if out is not None else torch.empty((Tn, R), dtype=values.dtype, device=values.device)
    _require_cuda(y)
    if y.dtype != values.dtype or y.shape != (Tn, R) or y.stride(1) != 1:
        raise ValueError("out must be a row-major [T, R] tensor of the values' dtype")
    return R, C, x2, values, meta, bias, y


def sparse24_linear_supported(x, values, meta, C):
    """True when K26 takes the call: CUDA tensors, x in the values' fp16 / bf16 dtype, C % 16 == 0, matching shapes."""
    return (values.is_cuda and meta.is_cuda and x.is_cuda and values.dtype in (torch.float16, torch.bfloat16) and
            x.dtype == values.dtype and C >= 16 and C % 16 == 0 and x.shape[-1] == C and values.dim() == 2 and
            values.shape[1] == C // 2 and meta.dtype == torch.int16 and meta.shape == (values.shape[0], C // 16))


def sparse24_linear(x, values, meta, C, bias=None, out=None):
    """K26: y = F.linear(x, decompress(values, meta), bias) read from the compressed weight.  x [..., C] in the values'
    dtype; returns y [..., R].  Operands whose row pitch TMA cannot take are copied (meta pitch padded to 16 bytes)."""
    R, C, x2, values, meta, bias, y = _sparse24_linear_operands(x, values, meta, C, bias, out)
    Tn = x2.shape[0]
    if Tn == 0:
        return y.reshape(*x.shape[:-1], R)
    lib = load()
    ws = workspace(x2, lib.vlmc_workspace_bytes(OP_SPARSE24_LINEAR, Tn, R, C))
    with torch.cuda.device(values.device):
        st = lib.vlmc_sparse24_linear_forward(x2.data_ptr(), _dtype(values), Tn, C, x2.stride(0), values.data_ptr(),
                                              values.stride(0), meta.data_ptr(), meta.stride(0), R,
                                              bias.data_ptr() if bias is not None else None, y.data_ptr(), y.stride(0),
                                              ws.data_ptr(), ws.numel(), _stream(values))
    _check("vlmc_sparse24_linear_forward", st)
    return y.reshape(*x.shape[:-1], R)


def sparse24_linear_sp_supported(x, values, meta, C):
    """True when K31 takes the call: sparse24_linear_supported and C % 32 == 0 (whole K = 32 sparse MMAs)."""
    return sparse24_linear_supported(x, values, meta, C) and C % 32 == 0


def sparse24_linear_sp(x, values, meta, C, bias=None, out=None):
    """K31: y = x . decompress(values, meta)^T (+ bias) on the sparse tensor cores, which multiply only the two positions
    meta names in each group of four (an inf / NaN of x at an unnamed position does not reach y; include/vlmc.h).  x
    [..., C] in the values' dtype, C % 32 == 0; returns y [..., R].  Operands whose row pitch TMA cannot take are
    copied (meta pitch padded to 16 bytes)."""
    if int(C) % 32:
        raise ValueError(f"the sparse tensor-core linear needs C % 32 == 0, got C = {C}")
    R, C, x2, values, meta, bias, y = _sparse24_linear_operands(x, values, meta, C, bias, out)
    Tn = x2.shape[0]
    if Tn == 0:
        return y.reshape(*x.shape[:-1], R)
    with torch.cuda.device(values.device):
        st = load().vlmc_sparse24_linear_sp_forward(x2.data_ptr(), _dtype(values), Tn, C, x2.stride(0),
                                                    values.data_ptr(), values.stride(0), meta.data_ptr(),
                                                    meta.stride(0), R, bias.data_ptr() if bias is not None else None,
                                                    y.data_ptr(), y.stride(0), _stream(values))
    _check("vlmc_sparse24_linear_sp_forward", st)
    return y.reshape(*x.shape[:-1], R)


def hessian_accum(x, H, n_before, b, kc=0, slab_tokens=0):
    """K3: H <- H*n/(n+b) + 2/(n+b) * X^T X   (sparsegpt_pruner.py:76-79), tcgen05 SYRK."""
    _require_cuda(x, H)
    lib = load()
    x2 = _rows2d(x)
    T, C = x2.shape
    if H.dtype != torch.float32 or H.shape != (C, C) or H.stride(1) != 1:
        raise ValueError("H must be a float32 [C, C] row-major matrix")
    with torch.cuda.device(x2.device):
        st = lib.vlmc_hessian_accum(x2.data_ptr(), _dtype(x2), T, C, x2.stride(0), H.data_ptr(), H.stride(0),
                                    float(n_before), float(b), int(kc), int(slab_tokens), _stream(x2))
    _check("vlmc_hessian_accum", st)


def hessian_prepare(H, percdamp, damp=None, dead=None):
    """sparsegpt_pruner.py:95-96,111: fix dead channels in place; returns (damp 1-elem tensor, dead uint8 [C]).
    damp / dead may be passed in (callers that run on a side stream allocate them on the main one)."""
    _require_cuda(H)
    lib = load()
    C = H.shape[0]
    damp = torch.empty(1, dtype=torch.float32, device=H.device) if damp is None else damp
    dead = torch.empty(C, dtype=torch.uint8, device=H.device) if dead is None else dead
    with torch.cuda.device(H.device):
        st = lib.vlmc_hessian_prepare(H.data_ptr(), C, H.stride(0), float(percdamp), damp.data_ptr(), dead.data_ptr(),
                                      _stream(H))
    _check("vlmc_hessian_prepare", st)
    return damp, dead


def hessian_add_damp(H, damp):
    _require_cuda(H, damp)
    lib = load()
    with torch.cuda.device(H.device):
        st = lib.vlmc_hessian_add_damp(H.data_ptr(), H.shape[0], H.stride(0), damp.data_ptr(), _stream(H))
    _check("vlmc_hessian_add_damp", st)


class chol_lookahead:
    """with chol_lookahead(False): ...  Host-side schedule switch of vlmc_chol_inv_upper (include/vlmc.h): callers that
    enqueue several factorisation chains concurrently turn the look-ahead off for the duration."""

    def __init__(self, on):
        self.mode = 1 if on else 0

    def __enter__(self):
        prev = load().vlmc_chol_set_lookahead(self.mode)
        self.prev = -1 if prev == 2 else prev
        return self

    def __exit__(self, *exc):
        load().vlmc_chol_set_lookahead(self.prev)
        return False


def chol_inv_upper(H, U=None, status=None):
    """K10: returns (U, status tensor).  status.item() == NOT_POSDEF means: damp and retry."""
    _require_cuda(H)
    lib = load()
    C = H.shape[0]
    if H.dtype != torch.float32 or H.shape != (C, C) or H.stride(1) != 1:
        raise ValueError("H must be a float32 [C, C] row-major matrix")
    if U is None:
        U = torch.empty((C, C), dtype=torch.float32, device=H.device)
    if status is None:       # the kernel clears it first
        status = torch.empty(1, dtype=torch.int32, device=H.device)
    ws = workspace(H, lib.vlmc_workspace_bytes(OP_CHOL, C, 0, 0))
    with torch.cuda.device(H.device):
        st = lib.vlmc_chol_inv_upper(H.data_ptr(), C, H.stride(0), U.data_ptr(), U.stride(0), status.data_ptr(),
                                     ws.data_ptr(), ws.numel(), _stream(H))
    _check("vlmc_chol_inv_upper", st)
    return U, status


NOT_POSDEF, NONFINITE, HUGE_FACTOR = 1, 2, 4          # bits of the factorisation status word (include/vlmc.h)


def _square_f32(A):
    C = A.shape[0]
    if A.dtype != torch.float32 or A.shape != (C, C) or A.stride(1) != 1:
        raise ValueError("expected a float32 [C, C] row-major matrix")
    return C


def gram_upper(U, out=None):
    """Hinv = U^T U (the value of torch.cholesky_inverse(cholesky(H)) for U = chol_inv_upper(H), sparsegpt_pruner.py:131)."""
    _require_cuda(U)
    C = _square_f32(U)
    out = torch.empty((C, C), dtype=torch.float32, device=U.device) if out is None else out
    with torch.cuda.device(U.device):
        _check("vlmc_gram_upper", load().vlmc_gram_upper(U.data_ptr(), C, U.stride(0), out.data_ptr(), out.stride(0),
                                                         _stream(U)))
    return out


def chol_upper(A, U=None, status=None):
    """U = cholesky(A, upper=True) (sparsegpt_pruner.py:146).  Returns (U, status tensor) like chol_inv_upper."""
    _require_cuda(A)
    lib = load()
    C = _square_f32(A)
    U = torch.empty((C, C), dtype=torch.float32, device=A.device) if U is None else U
    status = torch.empty(1, dtype=torch.int32, device=A.device) if status is None else status
    ws = workspace(A, lib.vlmc_workspace_bytes(OP_CHOL, C, 0, 0))
    with torch.cuda.device(A.device):
        _check("vlmc_chol_upper", lib.vlmc_chol_upper(A.data_ptr(), C, A.stride(0), U.data_ptr(), U.stride(0),
                                                      status.data_ptr(), ws.data_ptr(), ws.numel(), _stream(A)))
    return U, status


def matrix_nonfinite_count(A):
    """(number of +inf, -inf, NaN entries) of a 2-D float32 matrix; synchronises (the caller branches on it)."""
    _require_cuda(A)
    out = torch.empty(3, dtype=torch.int64, device=A.device)
    with torch.cuda.device(A.device):
        _check("vlmc_matrix_nonfinite_count", load().vlmc_matrix_nonfinite_count(
            A.data_ptr(), A.shape[0], A.shape[1], A.stride(0), out.data_ptr(), _stream(A)))
    return tuple(int(v) for v in out.tolist())


def matrix_replace_inf(A, value, negative):
    _require_cuda(A)
    with torch.cuda.device(A.device):
        _check("vlmc_matrix_replace_inf", load().vlmc_matrix_replace_inf(
            A.data_ptr(), A.shape[0], A.shape[1], A.stride(0), float(value), int(bool(negative)), _stream(A)))


def diag_abs_mean(A, scale, out=None):
    """scale * mean(|diag(A)|) as a 1-element device tensor (sparsegpt_pruner.py:143)."""
    _require_cuda(A)
    C = _square_f32(A)
    out = torch.empty(1, dtype=torch.float32, device=A.device) if out is None else out
    with torch.cuda.device(A.device):
        _check("vlmc_diag_abs_mean", load().vlmc_diag_abs_mean(A.data_ptr(), C, A.stride(0), float(scale), out.data_ptr(),
                                                               _stream(A)))
    return out


def matrix_quantile(A, q):
    """torch.quantile(A, q) (interpolation "linear") of a contiguous float32 matrix without sorting it and without torch's
    16 M element limit: the two neighbouring order statistics come from the exact radix select (vlmc_scores_kth) and are
    combined with torch's own float32 rank arithmetic (ATen quantile_compute: rank = q * (n - 1) in float32, lerp).
    Returns a python float (synchronises).  NaN entries sort last here; the caller rejects matrices that hold NaN."""
    import numpy as np
    if not A.is_contiguous():
        raise ValueError("matrix_quantile needs a contiguous matrix")
    n = A.numel()
    rank = np.float32(q) * np.float32(n - 1)
    below = int(np.floor(rank))
    above = int(np.ceil(rank))
    w = np.float32(rank - np.float32(below))
    flat = A.reshape(-1)
    vals = scores_kth([flat, flat], [0, 1], [below + 1, above + 1]).tolist()
    a, b = np.float32(vals[0]), np.float32(vals[1])
    with np.errstate(all="ignore"):
        res = a + w * (b - a) if w < np.float32(0.5) else b - (b - a) * (np.float32(1) - w)      # at::lerp
    return float(res)


def gemm_tf32x3(A, B, C=None, alpha=1.0, beta=0.0, b_nk=False, tri=False, kc=0):
    """C = beta * C + alpha * A @ (B.T if b_nk else B) in fp32 on the tensor cores (3xTF32 split, gemm3x.cu).
    A, B, C may be views with a row stride (last dim contiguous)."""
    _require_cuda(A, B, C)
    M, K = A.shape
    N = B.shape[0] if b_nk else B.shape[1]
    assert (B.shape[1] if b_nk else B.shape[0]) == K
    if C is None:
        C = torch.empty(M, N, device=A.device, dtype=torch.float32)
    for t in (A, B, C):
        assert t.dtype == torch.float32 and t.stride(-1) == 1
    _check("vlmc_gemm_tf32x3", load().vlmc_gemm_tf32x3(
        int(b_nk), M, N, K, float(alpha), A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), float(beta),
        C.data_ptr(), C.stride(0), int(tri), int(kc), _stream(A)))
    return C


def obs_sweep(W, U, sparsity, prune_n=0, prune_m=0, dead=None, blocksize=128, want_mask=False, score=None, keep=None,
              fail_flag=None):
    """K11-K13 (sparsegpt_pruner.py:160-215), in place on W.  Returns (keep_mask or None, importance 1-elem tensor).
    score / keep may be passed in (pre-allocated outputs).  fail_flag: the int32 status word of chol_inv_upper; when it
    is non-zero at run time W and keep are left untouched (vlmc_obs_sweep_guarded)."""
    _require_cuda(W, U, dead)
    if W.dim() != 2 or W.stride(1) != 1:
        raise ValueError("W must be a 2-D row-major weight")
    lib = load()
    R, C = W.shape
    if keep is None and want_mask:
        keep = torch.empty((R, C), dtype=torch.bool, device=W.device)
    if score is None:
        score = torch.empty(1, dtype=torch.float32, device=W.device)
    ws = workspace(W, lib.vlmc_workspace_bytes(OP_OBS, R, C, blocksize))
    with torch.cuda.device(W.device):
        st = lib.vlmc_obs_sweep_guarded(W.data_ptr(), _dtype(W), R, C, W.stride(0), U.data_ptr(), U.stride(0),
                                        dead.data_ptr() if dead is not None else None, float(sparsity), int(prune_n),
                                        int(prune_m), int(blocksize), keep.data_ptr() if keep is not None else None,
                                        keep.stride(0) if keep is not None else 0, score.data_ptr(),
                                        fail_flag.data_ptr() if fail_flag is not None else None, ws.data_ptr(), ws.numel(),
                                        _stream(W))
    _check("vlmc_obs_sweep_guarded", st)
    return keep, score


def obs_sweep_row_shard(W, U, sparsity, rows_total, reduce_sum, prune_n=0, prune_m=0, dead=None, want_mask=False):
    """K11-K13 on this rank's row shard of one linear (in place on W, a [R_local, C] view).

    reduce_sum(tensor): in-place SUM all-reduce over the ranks that hold the other rows; called on the three 8 KB
    block histograms (unstructured only) and once on the importance-score sum.  Returns (keep or None, importance
    score 1-elem tensor = mean over all rows_total rows)."""
    _require_cuda(W, U, dead)
    if W.dim() != 2 or W.stride(1) != 1:
        raise ValueError("W must be a 2-D row-major weight")
    lib = load()
    R, C = W.shape
    nblk = (C + 127) // 128
    keep = torch.empty((R, C), dtype=torch.bool, device=W.device) if want_mask else None
    score = torch.zeros(1, dtype=torch.float32, device=W.device)
    ws = workspace(W, lib.vlmc_workspace_bytes(OP_OBS, R, C, 128))
    hist = torch.zeros((nblk, 3, 2048), dtype=torch.int32, device=W.device) if prune_n == 0 else None
    st = _stream(W)
    args_u = (U.data_ptr(), U.stride(0))
    with torch.cuda.device(W.device):
        _check("vlmc_obs_begin", lib.vlmc_obs_begin(W.data_ptr(), _dtype(W), R, C, W.stride(0), *args_u,
                                                    dead.data_ptr() if dead is not None else None, score.data_ptr(),
                                                    ws.data_ptr(), ws.numel(), st))
        reduce_sum(score)
        for blk in range(nblk):
            if prune_n == 0:
                for ps in range(3):
                    _check("vlmc_obs_block_hist",
                           lib.vlmc_obs_block_hist(R, C, *args_u, blk, ps, int(rows_total), float(sparsity),
                                                   hist.data_ptr(), ws.data_ptr(), ws.numel(), st))
                    reduce_sum(hist[blk, ps])
            _check("vlmc_obs_block_finish",
                   lib.vlmc_obs_block_finish(W.data_ptr(), _dtype(W), R, C, W.stride(0), *args_u, blk, int(rows_total),
                                             float(sparsity), int(prune_n), int(prune_m),
                                             keep.data_ptr() if keep is not None else None,
                                             keep.stride(0) if keep is not None else 0,
                                             hist.data_ptr() if hist is not None else None, ws.data_ptr(), ws.numel(),
                                             st))
    return keep, score / float(rows_total * C)


def dsnot_refine(W, scaler_row, sum_metric_row, var, k, prune_n=0, prune_m=0, pow_of_var=1.0, max_cycle_time=100,
                 update_threshold=0.1, without_same_sign=True, initial_method="wanda", argmin_rule=1, ref_fixup=True,
                 zero_w=True, keep_mask=None, reduce_ncycles=None):
    """K8+K9 (dsnot_pruner.py:359-755), in place on W.  Returns (keep_mask bool [R,C], ncycles 1-elem int tensor).

    reduce_ncycles: optional callable(tensor) run between the two passes - the MAX all-reduce of the executed cycle
    count when the rows of one linear are sharded across ranks."""
    _require_cuda(W, scaler_row, sum_metric_row, var, keep_mask)
    if W.dim() != 2 or W.stride(1) != 1:
        raise ValueError("W must be a 2-D row-major weight")
    if initial_method not in ("wanda", "magnitude"):
        raise NotImplementedError("initial_method must be 'wanda' or 'magnitude' (the reference's 'sparsegpt' "
                                  "branch is dead code: no Hessian is ever accumulated, SURVEY F11)")
    R, C = W.shape
    if keep_mask is None:
        keep_mask = torch.empty((R, C), dtype=torch.bool, device=W.device)
    if keep_mask.dtype != torch.bool or keep_mask.shape != W.shape or keep_mask.stride(1) != 1:
        raise ValueError("keep_mask must be a bool tensor shaped like W")
    lib = load()
    mc = int(max_cycle_time)
    ws = workspace(W, lib.vlmc_workspace_bytes(OP_DSNOT_REFINE, R, C, mc))
    ncyc = torch.zeros(1, dtype=torch.int32, device=W.device)
    var = var.reshape(-1)
    common = (int(prune_n), int(prune_m))
    with torch.cuda.device(W.device):
        st = lib.vlmc_dsnot_refine_walk(W.data_ptr(), _dtype(W), R, C, W.stride(0), scaler_row.data_ptr(),
                                        sum_metric_row.data_ptr(), var.data_ptr(), int(k), *common,
                                        float(pow_of_var or 0.0), mc, float(update_threshold),
                                        int(bool(without_same_sign)), int(initial_method == "magnitude"),
                                        int(argmin_rule), ncyc.data_ptr(), ws.data_ptr(), ws.numel(), _stream(W))
        _check("vlmc_dsnot_refine_walk", st)
        if reduce_ncycles is not None:
            reduce_ncycles(ncyc)
        st = lib.vlmc_dsnot_refine_apply(W.data_ptr(), _dtype(W), R, C, W.stride(0), scaler_row.data_ptr(), *common,
                                         int(initial_method == "magnitude"), mc, ncyc.data_ptr(), int(bool(ref_fixup)),
                                         int(bool(zero_w)), keep_mask.data_ptr(), keep_mask.stride(0), ws.data_ptr(),
                                         ws.numel(), _stream(W))
        _check("vlmc_dsnot_refine_apply", st)
    return keep_mask, ncyc


def sparse24_compress_masked(W, keep_mask):
    """K27: (W [R, C] fp16 / bf16, keep_mask [R, C] bool) -> (values [R, C/2], meta [R, C/16] int16) with the kept set
    read from the mask, not from W's non-zeros: the values keep W's bits at exactly the mask's positions.  Raises
    ValueError unless every group of 4 columns keeps exactly two (synchronises on the status word).  W is not modified."""
    _require_cuda(W, keep_mask)
    dt = _sparse24_weight_dtype(W)
    if W.dim() != 2 or W.stride(1) != 1:
        raise ValueError("W must be a 2-D row-major weight")
    R, C = W.shape
    if C < 16 or C % 16:
        raise ValueError(f"compressed 2:4 weights need C % 16 == 0, got C = {C}")
    if keep_mask.dtype != torch.bool or keep_mask.shape != W.shape or keep_mask.stride(1) != 1:
        raise ValueError("mask must be a row-major bool tensor shaped like W")
    values = torch.empty((R, C // 2), dtype=W.dtype, device=W.device)
    meta = torch.empty((R, C // 16), dtype=torch.int16, device=W.device)
    status = torch.empty(1, dtype=torch.int32, device=W.device)
    with torch.cuda.device(W.device):
        st = load().vlmc_sparse24_compress_masked(W.data_ptr(), dt, R, C, W.stride(0), keep_mask.data_ptr(),
                                                  keep_mask.stride(0), values.data_ptr(), values.stride(0), meta.data_ptr(),
                                                  meta.stride(0), status.data_ptr(), _stream(W))
    _check("vlmc_sparse24_compress_masked", st)
    if int(status.item()) & NOT_2OF4:
        raise ValueError("mask is not 2:4: a group of 4 columns does not keep exactly two elements")
    return values, meta


def _sparse24_lora_common(values, meta, C, A, B):
    R, C = _sparse24_operands(values, meta, C)
    _require_cuda(A, B)
    if A.dtype != torch.float32 or B.dtype != torch.float32:
        raise TypeError("lora_A / lora_B must be float32")
    rank = A.shape[0]
    if A.dim() != 2 or A.shape != (rank, C) or B.shape != (R, rank):
        raise ValueError("lora_A must be [r, C] and lora_B [R, r]")
    if values.stride(0) % 4 or values.data_ptr() % 8:
        raise ValueError("values rows must be 8-byte aligned")
    return R, C, rank, A.contiguous(), B.contiguous()


def sparse24_lora_effective_weight(values, meta, C, A, B, scaling, sparse=True, out=None):
    """K28 (lora.py:364-375) on a mask-driven compressed weight: (W + s*BA) * M or W * M + s*BA with W = decompress(values,
    meta) and M the kept set of meta, in the values' dtype.  Bit-identical to sparselora_effective_weight on (W, M).
    Returns `out` [R, C] (any row pitch that keeps 16-byte rows)."""
    R, C, rank, A, B = _sparse24_lora_common(values, meta, C, A, B)
    if out is None:
        out = torch.empty((R, C), dtype=values.dtype, device=values.device)
    _require_cuda(out)
    if out.dtype != values.dtype or out.shape != (R, C) or out.stride(1) != 1:
        raise ValueError("out must be a row-major [R, C] tensor of the values' dtype")
    with torch.cuda.device(values.device):
        st = load().vlmc_sparse24_lora_effective_weight(values.data_ptr(), _dtype(values), R, C, values.stride(0),
                                                        meta.data_ptr(), meta.stride(0), A.data_ptr(), B.data_ptr(), rank,
                                                        float(scaling), int(bool(sparse)), out.data_ptr(), out.stride(0),
                                                        _stream(values))
    _check("vlmc_sparse24_lora_effective_weight", st)
    return out


def sparse24_lora_grads(G, meta, A, B, scaling, sparse=True):
    """K29: sparselora_lora_grads with the mask taken from meta.  G [R, C] (the values' dtype) -> (dA [r, C], dB [R, r])
    fp32, bit-identical to K16 on (G, M)."""
    _require_cuda(G, meta, A, B)
    _sparse24_weight_dtype(G)
    if G.dim() != 2 or G.stride(1) != 1:
        raise ValueError("G must be a 2-D row-major tensor")
    R, C = G.shape
    if C < 16 or C % 16:
        raise ValueError(f"compressed 2:4 weights need C % 16 == 0, got C = {C}")
    if meta.dtype != torch.int16 or meta.shape != (R, C // 16) or meta.stride(1) != 1:
        raise ValueError("meta must be a row-major int16 [R, C/16] tensor")
    if A.dtype != torch.float32 or B.dtype != torch.float32:
        raise TypeError("lora_A / lora_B must be float32")
    rank = A.shape[0]
    if A.shape != (rank, C) or B.shape != (R, rank):
        raise ValueError("lora_A must be [r, C] and lora_B [R, r]")
    A, B = A.contiguous(), B.contiguous()
    lib = load()
    dA = torch.empty((rank, C), dtype=torch.float32, device=G.device)
    dB = torch.empty((R, rank), dtype=torch.float32, device=G.device)
    ws = workspace(G, lib.vlmc_sparselora_lora_grads_workspace_bytes(R, C, rank))
    with torch.cuda.device(G.device):
        st = lib.vlmc_sparse24_lora_grads(G.data_ptr(), _dtype(G), R, C, G.stride(0), meta.data_ptr(), meta.stride(0),
                                          int(bool(sparse)), A.data_ptr(), B.data_ptr(), rank, float(scaling),
                                          dA.data_ptr(), dB.data_ptr(), ws.data_ptr(), ws.numel(), _stream(G))
    _check("vlmc_sparse24_lora_grads", st)
    return dA, dB


def sparse24_lora_merge(values, meta, C, A, B, scaling):
    """K30 (lora.py:384-394 + train.py:634-637), in place on values: every stored slot becomes
    round(v + s * (B A)[slot]) with K14's arithmetic; decompress() of the result equals sparselora_merge(W, A, B, s, M,
    remask=True) on the dense pair."""
    R, C, rank, A, B = _sparse24_lora_common(values, meta, C, A, B)
    with torch.cuda.device(values.device):
        st = load().vlmc_sparse24_lora_merge(values.data_ptr(), _dtype(values), R, C, values.stride(0), meta.data_ptr(),
                                             meta.stride(0), A.data_ptr(), B.data_ptr(), rank, float(scaling),
                                             _stream(values))
    _check("vlmc_sparse24_lora_merge", st)
    return values
