"""TEST INFRASTRUCTURE -- NOT PRODUCT CODE.

ctypes front-end of ``oracle/surprise_oracle.c``, the plain-C CPU restatement of the reference's
fit-time hot path (see that file's header for the reference file:line each function follows and
for how the restatement is pinned against the compiled reference).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import this package.  ``surprise_b200`` never does.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")
_SRC = os.path.join(_HERE, "surprise_oracle.c")

OK, ZERO_DIVISION, NOMEM = 0, 1, 2
KINDS = {"cosine": 0, "msd": 1, "pearson": 2, "pearson_baseline": 3}


def build(force=False):
    """gcc -O2 -ffp-contract=off: strict IEEE fp64 like the reference's Cython build."""
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", _SO, _SRC, "-lm"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def _p(a, t):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


class ZeroDivision(ZeroDivisionError):
    pass


def _check(rc):
    if rc == ZERO_DIVISION:
        raise ZeroDivision("float division")
    if rc != OK:
        raise MemoryError("oracle rc=%d" % rc)


def flatten_yr(yr, n_y=None):
    """dict {y: [(x, r), ...]} -> CSR in dict-iteration order (what iteritems(yr) visits).

    Keys need not be 0..n_y-1 (tests/test_similarities.py uses an arbitrary dict); for
    pearson_baseline the key itself indexes y_biases, so slot = key when n_y is given."""
    keys = list(yr.keys())
    if n_y is None:
        n_y = len(keys)
        slots = range(len(keys))
    else:
        slots = keys
        assert keys == sorted(keys), "keyed layout needs ascending keys to preserve iteration order"
    ptr = np.zeros(n_y + 1, dtype=np.int64)
    for s, k in zip(slots, keys):
        ptr[s + 1] = len(yr[k])
    np.cumsum(ptr, out=ptr)
    xs = np.empty(ptr[-1], dtype=np.int32)
    rs = np.empty(ptr[-1], dtype=np.float64)
    for s, k in zip(slots, keys):
        o = ptr[s]
        for t, (x, r) in enumerate(yr[k]):
            xs[o + t] = x
            rs[o + t] = r
    return ptr, xs, rs


def similarity(kind, n_x, y_ptr, x_idx, r, min_support, global_mean=0.0, x_biases=None, y_biases=None,
               shrinkage=100.0):
    y_ptr, x_idx, r = _i64(y_ptr), _i32(x_idx), _f64(r)
    xb, yb = _f64(x_biases), _f64(y_biases)
    sim = np.empty((n_x, n_x), dtype=np.float64)
    rc = lib().orc_similarity(C.c_int(KINDS[kind]), C.c_int64(n_x), C.c_int64(len(y_ptr) - 1),
                              _p(y_ptr, C.c_int64), _p(x_idx, C.c_int32), _p(r, C.c_double),
                              C.c_int(int(min_support)), C.c_double(global_mean), _p(xb, C.c_double),
                              _p(yb, C.c_double), C.c_double(shrinkage), _p(sim, C.c_double))
    _check(rc)
    return sim


def similarity_pairs(kind, pi, pj, x_ptr, y_idx, r, min_support, global_mean=0.0, x_biases=None,
                     y_biases=None, shrinkage=100.0):
    pi, pj, x_ptr, y_idx, r = _i32(pi), _i32(pj), _i64(x_ptr), _i32(y_idx), _f64(r)
    xb, yb = _f64(x_biases), _f64(y_biases)
    out = np.empty(len(pi), dtype=np.float64)
    rc = lib().orc_similarity_pairs(C.c_int(KINDS[kind]), C.c_int64(len(pi)), _p(pi, C.c_int32),
                                    _p(pj, C.c_int32), _p(x_ptr, C.c_int64), _p(y_idx, C.c_int32),
                                    _p(r, C.c_double), C.c_int(int(min_support)), C.c_double(global_mean),
                                    _p(xb, C.c_double), _p(yb, C.c_double), C.c_double(shrinkage),
                                    _p(out, C.c_double))
    _check(rc)
    return out


def baseline_als(n_users, n_items, u_ptr, ui_idx, u_r, i_ptr, iu_idx, i_r, global_mean, n_epochs=10,
                 reg_u=15.0, reg_i=10.0):
    bu = np.zeros(n_users)
    bi = np.zeros(n_items)
    u_ptr, ui_idx, u_r = _i64(u_ptr), _i32(ui_idx), _f64(u_r)
    i_ptr, iu_idx, i_r = _i64(i_ptr), _i32(iu_idx), _f64(i_r)
    rc = lib().orc_baseline_als(C.c_int64(n_users), C.c_int64(n_items), _p(u_ptr, C.c_int64),
                                _p(ui_idx, C.c_int32), _p(u_r, C.c_double), _p(i_ptr, C.c_int64),
                                _p(iu_idx, C.c_int32), _p(i_r, C.c_double), C.c_double(global_mean),
                                C.c_int(n_epochs), C.c_double(reg_u), C.c_double(reg_i),
                                _p(bu, C.c_double), _p(bi, C.c_double))
    _check(rc)
    return bu, bi


def baseline_sgd(n_users, n_items, u, i, r, global_mean, n_epochs=20, reg=0.02, lr=0.005):
    bu = np.zeros(n_users)
    bi = np.zeros(n_items)
    u, i, r = _i32(u), _i32(i), _f64(r)
    rc = lib().orc_baseline_sgd(C.c_int64(n_users), C.c_int64(n_items), C.c_int64(len(u)),
                                _p(u, C.c_int32), _p(i, C.c_int32), _p(r, C.c_double),
                                C.c_double(global_mean), C.c_int(n_epochs), C.c_double(reg), C.c_double(lr),
                                _p(bu, C.c_double), _p(bi, C.c_double))
    _check(rc)
    return bu, bi


def svd_sgd(u, i, r, pu, qi, n_epochs, biased, global_mean, lr_bu, lr_bi, lr_pu, lr_qi, reg_bu, reg_bi,
            reg_pu, reg_qi):
    """pu, qi: the rng.normal init (copied); returns (pu, qi, bu, bi)."""
    u, i, r = _i32(u), _i32(i), _f64(r)
    pu, qi = np.array(pu, dtype=np.float64, order="C"), np.array(qi, dtype=np.float64, order="C")
    bu, bi = np.zeros(pu.shape[0]), np.zeros(qi.shape[0])
    d = C.c_double
    rc = lib().orc_svd_sgd(C.c_int64(len(u)), C.c_int(pu.shape[1]), _p(u, C.c_int32), _p(i, C.c_int32),
                           _p(r, C.c_double), C.c_int(n_epochs), C.c_int(int(bool(biased))),
                           d(global_mean if biased else 0.0), d(lr_bu), d(lr_bi), d(lr_pu), d(lr_qi),
                           d(reg_bu), d(reg_bi), d(reg_pu), d(reg_qi), _p(pu, C.c_double),
                           _p(qi, C.c_double), _p(bu, C.c_double), _p(bi, C.c_double))
    _check(rc)
    return pu, qi, bu, bi


def svdpp_sgd(u, i, r, u_ptr, ui_idx, pu, qi, yj, n_epochs, global_mean, lr_bu, lr_bi, lr_pu, lr_qi, lr_yj,
              reg_bu, reg_bi, reg_pu, reg_qi, reg_yj):
    u, i, r = _i32(u), _i32(i), _f64(r)
    u_ptr, ui_idx = _i64(u_ptr), _i32(ui_idx)
    pu, qi, yj = (np.array(a, dtype=np.float64, order="C") for a in (pu, qi, yj))
    bu, bi = np.zeros(pu.shape[0]), np.zeros(qi.shape[0])
    d = C.c_double
    rc = lib().orc_svdpp_sgd(C.c_int64(len(u)), C.c_int(pu.shape[1]), _p(u, C.c_int32), _p(i, C.c_int32),
                             _p(r, C.c_double), _p(u_ptr, C.c_int64), _p(ui_idx, C.c_int32),
                             C.c_int(n_epochs), d(global_mean), d(lr_bu), d(lr_bi), d(lr_pu), d(lr_qi),
                             d(lr_yj), d(reg_bu), d(reg_bi), d(reg_pu), d(reg_qi), d(reg_yj),
                             _p(pu, C.c_double), _p(qi, C.c_double), _p(yj, C.c_double),
                             _p(bu, C.c_double), _p(bi, C.c_double))
    _check(rc)
    return pu, qi, yj, bu, bi


# variant bits of svdpp_relaxed_sgd: deliberate deviations from the relaxation, for the mutation tests
PP_Y_FROZEN, PP_NO_DECAY, PP_ISQ_INV_N, PP_Z_FROZEN, PP_C_RATERS, PP_G_KEPT = 1, 2, 4, 8, 16, 32


def svdpp_relaxed_sgd(u, i, r, u_ptr, ui_idx, stratum, order, bounds, pu, qi, yj, n_epochs, global_mean, lr_bu,
                      lr_bi, lr_pu, lr_qi, lr_yj, reg_bu, reg_bi, reg_pu, reg_qi, reg_yj, variant=0):
    """NOT the reference: the stratified kernel's SVD++ relaxation in fp64 (see orc_svdpp_relaxed_sgd).
    stratum: per rating (indexed like u); order: the ratings in the sequence they are applied; bounds: the chunks'
    strata, chunk c = [bounds[c], bounds[c + 1]).  Returns (pu, qi, yj, bu, bi)."""
    u, i, r = _i32(u), _i32(i), _f64(r)
    u_ptr, ui_idx, stratum, order, bounds = _i64(u_ptr), _i32(ui_idx), _i32(stratum), _i64(order), _i32(bounds)
    assert len(u_ptr) == len(pu) + 1 and len(stratum) == len(u) and len(bounds) >= 2
    pu, qi, yj = (np.array(a, dtype=np.float64, order="C") for a in (pu, qi, yj))
    bu, bi = np.zeros(pu.shape[0]), np.zeros(qi.shape[0])
    d = C.c_double
    rc = lib().orc_svdpp_relaxed_sgd(C.c_int64(pu.shape[0]), C.c_int64(qi.shape[0]), C.c_int64(len(u)),
                                     C.c_int(pu.shape[1]), _p(u, C.c_int32), _p(i, C.c_int32), _p(r, C.c_double),
                                     _p(u_ptr, C.c_int64), _p(ui_idx, C.c_int32), _p(stratum, C.c_int32),
                                     C.c_int64(len(order)), _p(order, C.c_int64), C.c_int(len(bounds) - 1),
                                     _p(bounds, C.c_int32), C.c_int(n_epochs), d(global_mean), d(lr_bu), d(lr_bi),
                                     d(lr_pu), d(lr_qi), d(lr_yj), d(reg_bu), d(reg_bi), d(reg_pu), d(reg_qi),
                                     d(reg_yj), C.c_int(variant), _p(pu, C.c_double), _p(qi, C.c_double),
                                     _p(yj, C.c_double), _p(bu, C.c_double), _p(bi, C.c_double))
    _check(rc)
    return pu, qi, yj, bu, bi


def nmf_sgd(n_users, n_items, u, i, r, n_ur, n_ir, pu, qi, n_epochs, biased, global_mean, reg_pu, reg_qi,
            reg_bu, reg_bi, lr_bu, lr_bi):
    u, i, r = _i32(u), _i32(i), _f64(r)
    n_ur, n_ir = _i64(n_ur), _i64(n_ir)
    pu, qi = np.array(pu, dtype=np.float64, order="C"), np.array(qi, dtype=np.float64, order="C")
    bu, bi = np.zeros(n_users), np.zeros(n_items)
    d = C.c_double
    rc = lib().orc_nmf_sgd(C.c_int64(n_users), C.c_int64(n_items), C.c_int64(len(u)), C.c_int(pu.shape[1]),
                           _p(u, C.c_int32), _p(i, C.c_int32), _p(r, C.c_double), _p(n_ur, C.c_int64),
                           _p(n_ir, C.c_int64), C.c_int(n_epochs), C.c_int(int(bool(biased))),
                           d(global_mean if biased else 0.0), d(reg_pu), d(reg_qi), d(reg_bu), d(reg_bi),
                           d(lr_bu), d(lr_bi), _p(pu, C.c_double), _p(qi, C.c_double), _p(bu, C.c_double),
                           _p(bi, C.c_double))
    _check(rc)
    return pu, qi, bu, bi


def mf_estimate(u, i, biased, global_mean, pu, qi, bu, bi, yj=None, u_ptr=None, ui_idx=None):
    u, i = _i32(u), _i32(i)
    pu, qi, bu, bi, yj = _f64(pu), _f64(qi), _f64(bu), _f64(bi), _f64(yj)
    if yj is not None:
        u_ptr, ui_idx = _i64(u_ptr), _i32(ui_idx)
    est = np.empty(len(u))
    imp = np.empty(len(u), dtype=np.uint8)
    rc = lib().orc_mf_estimate(C.c_int64(len(u)), _p(u, C.c_int32), _p(i, C.c_int32), C.c_int(pu.shape[1]),
                               C.c_int(int(bool(biased))), C.c_double(global_mean), _p(pu, C.c_double),
                               _p(qi, C.c_double), _p(bu, C.c_double), _p(bi, C.c_double),
                               _p(yj, C.c_double), _p(u_ptr, C.c_int64) if yj is not None else None,
                               _p(ui_idx, C.c_int32) if yj is not None else None, _p(est, C.c_double),
                               _p(imp, C.c_uint8))
    _check(rc)
    return est, imp


def knn_estimate(x, y, sim, y_ptr, x_idx, r, k, min_k, baseline=0, global_mean=0.0, bx=None, by=None):
    """baseline: 0 = KNNBasic, 1 / 2 = KNNBaseline with x = user / item, 3 = KNNWithMeans (bx = means),
    4 = KNNWithZScore (bx = means, by = sigmas, both per x)."""
    x, y = _i32(x), _i32(y)
    sim = _f64(sim)
    y_ptr, x_idx, r = _i64(y_ptr), _i32(x_idx), _f64(r)
    bx, by = _f64(bx), _f64(by)
    est = np.empty(len(x))
    ak = np.empty(len(x), dtype=np.int32)
    imp = np.empty(len(x), dtype=np.uint8)
    rc = lib().orc_knn_estimate(C.c_int64(len(x)), _p(x, C.c_int32), _p(y, C.c_int32),
                                C.c_int64(sim.shape[0]), _p(sim, C.c_double), _p(y_ptr, C.c_int64),
                                _p(x_idx, C.c_int32), _p(r, C.c_double), C.c_int(k), C.c_int(min_k),
                                C.c_int(baseline), C.c_double(global_mean), _p(bx, C.c_double),
                                _p(by, C.c_double), _p(est, C.c_double), _p(ak, C.c_int32),
                                _p(imp, C.c_uint8))
    _check(rc)
    return est, ak, imp


def slope_one_fit(n_items, u_ptr, i_idx, r):
    u_ptr, i_idx, r = _i64(u_ptr), _i32(i_idx), _f64(r)
    freq = np.empty((n_items, n_items), dtype=np.int64)
    dev = np.empty((n_items, n_items), dtype=np.float64)
    rc = lib().orc_slope_one_fit(C.c_int64(n_items), C.c_int64(len(u_ptr) - 1), _p(u_ptr, C.c_int64),
                                 _p(i_idx, C.c_int32), _p(r, C.c_double), _p(freq, C.c_int64), _p(dev, C.c_double))
    _check(rc)
    return freq, dev


def slope_one_estimate(u, i, freq, dev, u_ptr, i_idx, user_mean):
    u, i = _i32(u), _i32(i)
    freq = np.ascontiguousarray(freq, dtype=np.int64)
    dev, user_mean = _f64(dev), _f64(user_mean)
    u_ptr, i_idx = _i64(u_ptr), _i32(i_idx)
    est = np.empty(len(u))
    imp = np.empty(len(u), dtype=np.uint8)
    rc = lib().orc_slope_one_estimate(C.c_int64(len(u)), _p(u, C.c_int32), _p(i, C.c_int32),
                                      C.c_int64(freq.shape[0]), _p(freq, C.c_int64), _p(dev, C.c_double),
                                      _p(u_ptr, C.c_int64), _p(i_idx, C.c_int32), _p(user_mean, C.c_double),
                                      _p(est, C.c_double), _p(imp, C.c_uint8))
    _check(rc)
    return est, imp


def reference_path():
    """Directory holding the compiled reference package (oracle/_ref), or None."""
    p = os.path.join(_HERE, "_ref")
    return p if os.path.isdir(os.path.join(p, "surprise")) else None


def import_reference():
    """Import the compiled, unmodified reference as module ``surprise`` (from oracle/_ref)."""
    p = reference_path()
    if p is None:
        raise ImportError("oracle/_ref is not built (run oracle/build_ref.sh where /root/reference exists)")
    if p not in sys.path:
        sys.path.insert(0, p)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import surprise  # noqa
    return surprise
