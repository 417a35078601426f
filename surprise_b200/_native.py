"""ctypes binding of libsurprise_b200.so (the C-ABI declared in include/surprise_b200.h).

PyTorch is used for exactly three things: device memory (torch tensors own every device buffer the
kernels read or write), the current CUDA stream, and torch.distributed for multi-GPU plumbing.  There
is no CPU fallback: if the shared library is missing, or no CUDA device is usable, every compute entry
point raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsurprise_b200.so")

OK, ERR_CUDA, ERR_INVALID, ERR_ZERO_DIVISION, ERR_DUPLICATE, ERR_UNSUPPORTED = range(6)
SIM_KINDS = {"cosine": 0, "msd": 1, "pearson": 2, "pearson_baseline": 3}

_i64, _i32, _int, _dbl, _vp = C.c_int64, C.c_int32, C.c_int, C.c_double, C.c_void_p


class SgdParams(C.Structure):
    _fields_ = [("n_factors", C.c_int32), ("n_epochs", C.c_int32), ("biased", C.c_int32), ("reserved", C.c_int32),
                ("global_mean", _dbl), ("lr_bu", _dbl), ("lr_bi", _dbl), ("lr_pu", _dbl), ("lr_qi", _dbl),
                ("lr_yj", _dbl), ("reg_bu", _dbl), ("reg_bi", _dbl), ("reg_pu", _dbl), ("reg_qi", _dbl),
                ("reg_yj", _dbl)]


class NmfParams(C.Structure):
    _fields_ = [("n_factors", C.c_int32), ("n_epochs", C.c_int32), ("biased", C.c_int32), ("reserved", C.c_int32),
                ("global_mean", _dbl), ("reg_pu", _dbl), ("reg_qi", _dbl), ("reg_bu", _dbl), ("reg_bi", _dbl),
                ("lr_bu", _dbl), ("lr_bi", _dbl)]


# name -> (restype, argtypes); every symbol of include/surprise_b200.h
SIGNATURES = {
    "sb2_last_error": (C.c_char_p, []),
    "sb2_version": (_int, []),
    "sb2_device_info": (_int, [_vp, _vp, _vp, _vp]),
    "sb2_launch_count": (_i64, []),
    "sb2_reset_launch_count": (None, []),
    "sb2_sim_build_dev": (_int, [_int, _i64, _i64, _vp, _vp, _vp, _i64, _int, _int, _dbl, _vp, _vp, _dbl, _i64, _i64,
                                 _vp, _vp]),
    "sb2_sim_build_upper_dev": (_int, [_int, _i64, _i64, _vp, _vp, _vp, _i64, _int, _int, _dbl, _vp, _vp, _dbl, _i64, _i64,
                                 _vp, _vp]),
    "sb2_sim_build": (_int, [_int, _i64, _i64, _vp, _vp, _vp, _i64, _int, _int, _dbl, _vp, _vp, _dbl, _i64, _i64,
                             _vp]),
    "sb2_gemm_u8_selftest_dev": (_int, [_int, _i64, _i64, _i64, _vp, _vp, _vp, _vp]),
    "sb2_baseline_als_dev": (_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _dbl, _int, _dbl, _dbl, _vp, _vp, _vp]),
    "sb2_baseline_als": (_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _dbl, _int, _dbl, _dbl, _vp, _vp]),
    "sb2_baseline_als_pass_dev": (_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _dbl, _dbl, _vp, _vp]),
    "sb2_baseline_sgd_dev": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _dbl, _int, _dbl, _dbl, _vp, _vp, _vp]),
    "sb2_baseline_sgd": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _dbl, _int, _dbl, _dbl, _vp, _vp]),
    "sb2_svd_fit_dev": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_svd_fit": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_svd_plan_create": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _int, _vp]),
    "sb2_svd_plan_reset": (_int, [_vp, _vp, _vp, _vp]),
    "sb2_svd_plan_create_dev": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp, _vp]),
    "sb2_svd_plan_reset_dev": (_int, [_vp, _vp, _vp, _vp, _vp]),
    "sb2_svd_plan_read_dev": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_svd_plan_run": (_int, [_vp, _int, _vp]),
    "sb2_svd_plan_read": (_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_svd_plan_destroy": (None, [_vp]),
    "sb2_svd_plan_bytes_per_update": (_i64, [_vp]),
    "sb2_svd_plan_grid": (_int, [_vp, _vp, _vp]),
    "sb2_svd_plan_layout": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_svd_plan_status": (_int, [_vp, _vp]),
    "sb2_svd_ring_create_dev": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _int, _vp, _vp, _int, _int, _vp, _vp]),
    "sb2_svd_ring_ipc_handle": (_int, [_vp, _vp]),
    "sb2_svd_ring_connect_ipc": (_int, [_vp, _vp, _vp]),
    "sb2_svd_ring_connect_local": (_int, [_vp, _vp, _vp]),
    "sb2_svd_ring_epoch_dev": (_int, [_vp, _int, _vp, _vp]),
    "sb2_svd_ring_run_local": (_int, [_vp, _int, _int, _vp]),
    "sb2_svd_ring_epoch_local": (_int, [_vp, _int, _vp, _vp]),
    "sb2_svd_ring_info": (_int, [_vp, _vp, _vp, _vp, _vp]),
    "sb2_svd_plan_profile": (_int, [_vp, _vp]),
    "sb2_svdpp_fit_dev": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_svdpp_fit": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_nmf_fit_dev": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_nmf_fit": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_nmf_plan_create_dev": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _int, _vp, _vp]),
    "sb2_nmf_plan_epoch_dev": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp]),
    "sb2_nmf_plan_status": (_int, [_vp, _vp]),
    "sb2_nmf_plan_destroy": (None, [_vp]),
    "sb2_mf_predict_dev": (_int, [_i64, _vp, _vp, _int, _int, _dbl, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                  _vp]),
    "sb2_mf_predict": (_int, [_i64, _vp, _vp, _i64, _i64, _int, _int, _dbl, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                              _vp]),
    "sb2_knn_predict_dev": (_int, [_i64, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _int, _int, _int, _dbl, _vp, _vp,
                                   _vp, _vp, _vp, _vp]),
    "sb2_knn_predict": (_int, [_i64, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _int, _int, _int, _dbl, _vp, _vp, _vp,
                               _vp, _vp]),
    "sb2_knn_predict_rows_dev": (_int, [_i64, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _int, _int, _int, _dbl,
                                        _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_slope_one_fit_dev": (_int, [_i64, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "sb2_slope_one_fit": (_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "sb2_rating_denominator_dev": (_int, [_vp, _i64, _vp, _vp]),
    "sb2_sim_build_rows_dev": (_int, [_int, _i64, _i64, _vp, _vp, _vp, _i64, _int, _int, _dbl, _vp, _vp, _dbl, _vp,
                                      _i64, _vp, _i64, _vp]),
    "sb2_get_neighbors_dev": (_int, [_i64, _vp, _i64, _i64, _vp, _int, _vp, _vp]),
    "sb2_slope_one_predict_dev": (_int, [_i64, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_coclustering_fit_dev": (_int, [_i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _dbl, _int, _int,
                                        _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_coclustering_fit": (_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _dbl, _int, _int, _int, _vp,
                                    _vp, _vp, _vp, _vp]),
    "sb2_coclustering_predict_dev": (_int, [_i64, _vp, _vp, _i64, _i64, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                            _dbl, _vp, _vp]),
    "sb2_mf_score_block_dev": (_int, [_i64, _vp, _i64, _int, _int, _dbl, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                      _i64, _vp]),
    "sb2_top_n_select_dev": (_int, [_i64, _vp, _i64, _vp, _i64, _vp, _dbl, _dbl, _dbl, _dbl, _vp, _vp, _int, _vp,
                                    _vp, _vp, _vp]),
    "sb2_top_n_hits_dev": (_int, [_i64, _vp, _i64, _vp, _int, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sb2_top_n_lists_dev": (_int, [_i64, _vp, _i64, _vp, _vp, _int, _int, _dbl, _i64, _vp, _vp, _vp, _vp, _vp, _vp,
                                   _vp]),
    "sb2_top_n_ranks_dev": (_int, [_i64, _vp, _i64, _vp, _i64, _vp, _dbl, _dbl, _dbl, _dbl, _vp, _vp, _vp, _vp, _i64,
                                   _vp, _vp, _vp, _vp, _vp]),
    "sb2_fcp_counts_dev": (_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "sb2_precision_at_k_counts_dev": (_int, [_i64, _i64, _vp, _vp, _vp, _vp, _dbl, _vp, _vp]),
}

_lib = None


def lib():
    """Load the shared library; fail loudly (no fallback) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("surprise_b200: %s is missing -- build it with `python -c 'import "
                               "__graft_entry__ as g; g.build()'` (there is no CPU fallback)" % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


class NativeError(RuntimeError):
    pass


def check(rc):
    if rc == OK:
        return
    msg = lib().sb2_last_error().decode("utf-8", "replace")
    if rc == ERR_ZERO_DIVISION:
        raise ZeroDivisionError(msg)
    if rc in (ERR_INVALID, ERR_DUPLICATE, ERR_UNSUPPORTED):
        raise ValueError(msg)
    raise NativeError(msg)


def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        raise NativeError("surprise_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


def device():
    torch = torch_cuda()
    return torch.device("cuda", torch.cuda.current_device())


def to_dev(a, dtype):
    """numpy array (or torch tensor) -> contiguous CUDA tensor of the given numpy dtype."""
    torch = torch_cuda()
    if isinstance(a, torch.Tensor):
        t = a.to(device=device(), dtype=getattr(torch, np.dtype(dtype).name)).contiguous()
        return t
    arr = np.ascontiguousarray(a, dtype=dtype)
    return torch.from_numpy(arr).to(device(), non_blocking=False)


def empty_dev(shape, dtype):
    torch = torch_cuda()
    return torch.empty(shape, dtype=getattr(torch, np.dtype(dtype).name), device=device())


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def hptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def stream():
    torch = torch_cuda()
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
