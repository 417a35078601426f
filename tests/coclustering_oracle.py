"""TEST INFRASTRUCTURE -- NOT PRODUCT CODE.

ctypes front-end of ``tests/coclustering_oracle.c``, the plain-C sequential restatement of the reference's
CoClustering (fit, compute_averages, estimate).  The library is compiled on first use with
gcc -O2 -ffp-contract=off (strict IEEE fp64, like the reference's Cython build) into a temporary directory keyed by
the source's hash, so the source tree is never written.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "coclustering_oracle.c")
OK, NOMEM, OVERFLOW = 0, 2, 3

_lib = None


def lib():
    global _lib
    if _lib is None:
        with open(_SRC, "rb") as fh:
            digest = hashlib.sha256(fh.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "sb2_coclustering_oracle_%d_%s.so" % (os.getuid(), digest))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", tmp, _SRC])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _check(rc):
    if rc == OVERFLOW:
        raise OverflowError("value too large to convert to int")
    if rc != OK:
        raise MemoryError("coclustering oracle rc=%d" % rc)


def fit(n_users, n_items, u_csr, i_csr, user_mean, item_mean, global_mean, n_cltr_u, n_cltr_i, n_epochs, cltr_u,
        cltr_i):
    """u_csr / i_csr: (ptr, idx, r) of trainset.ur / trainset.ir; cltr_u / cltr_i: the rng draw (copied).
    Returns (cltr_u, cltr_i, avg_cltr_u, avg_cltr_i, avg_cocltr) with int64 clusters."""
    up, ui, ur = (np.ascontiguousarray(a, dtype=t) for a, t in zip(u_csr, (np.int64, np.int32, np.float64)))
    ip, iu, ir = (np.ascontiguousarray(a, dtype=t) for a, t in zip(i_csr, (np.int64, np.int32, np.float64)))
    um, im = np.ascontiguousarray(user_mean, dtype=np.float64), np.ascontiguousarray(item_mean, dtype=np.float64)
    cu, ci = np.array(cltr_u, dtype=np.int64), np.array(cltr_i, dtype=np.int64)
    au, ai, ac = np.empty(n_cltr_u), np.empty(n_cltr_i), np.empty((n_cltr_u, n_cltr_i))
    _check(lib().orc_coclustering_fit(C.c_int64(n_users), C.c_int64(n_items), _p(up, C.c_int64), _p(ui, C.c_int32),
                                      _p(ur, C.c_double), _p(ip, C.c_int64), _p(iu, C.c_int32), _p(ir, C.c_double),
                                      _p(um, C.c_double), _p(im, C.c_double), C.c_double(global_mean),
                                      C.c_int(n_cltr_u), C.c_int(n_cltr_i), C.c_int(n_epochs), _p(cu, C.c_int64),
                                      _p(ci, C.c_int64), _p(au, C.c_double), _p(ai, C.c_double), _p(ac, C.c_double)))
    return cu, ci, au, ai, ac


def estimate(u, i, cltr_u, cltr_i, user_mean, item_mean, avg_cltr_u, avg_cltr_i, avg_cocltr, global_mean):
    """u / i: inner ids, -1 = unknown (-> global_mean)."""
    u, i = np.ascontiguousarray(u, dtype=np.int32), np.ascontiguousarray(i, dtype=np.int32)
    cu, ci = np.ascontiguousarray(cltr_u, dtype=np.int64), np.ascontiguousarray(cltr_i, dtype=np.int64)
    um, im, au, ai, ac = (np.ascontiguousarray(a, dtype=np.float64)
                          for a in (user_mean, item_mean, avg_cltr_u, avg_cltr_i, avg_cocltr))
    est = np.empty(len(u))
    _check(lib().orc_coclustering_estimate(C.c_int64(len(u)), _p(u, C.c_int32), _p(i, C.c_int32),
                                           C.c_int(ac.shape[1]), _p(cu, C.c_int64), _p(ci, C.c_int64),
                                           _p(um, C.c_double), _p(im, C.c_double), _p(au, C.c_double),
                                           _p(ai, C.c_double), _p(ac, C.c_double), C.c_double(global_mean),
                                           _p(est, C.c_double)))
    return est
