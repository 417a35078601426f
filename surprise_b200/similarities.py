"""Drop-in for the reference's surprise/similarities.pyx: cosine, msd, pearson, pearson_baseline.

Same call signatures and return contract (float64 ndarray n_x x n_x, symmetric, unit diagonal, caller
owns it): similarities.pyx:28, :100, :169, :261.  The work is done by sb2_sim_build_dev
(include/surprise_b200.h): dense masked contractions on the int8 tensor cores + an fp64 finalize kernel.

``yr`` may be the reference's dict ``{y: [(x, r), ...]}`` or an already flat CSR triple
``(y_ptr, x_idx, r)`` (what the array-backed Trainset hands over, skipping 10^7 Python tuples).
"""
import numpy as np

from . import _native as nat

_DENOMS = (1, 2, 4, 5, 10, 20, 100, 1000)


def _flatten(yr, n_y_hint=None):
    if isinstance(yr, tuple):
        ptr, idx, val = yr
        return (np.ascontiguousarray(ptr, dtype=np.int64), np.ascontiguousarray(idx, dtype=np.int32),
                np.ascontiguousarray(val, dtype=np.float64))
    keys = list(yr.keys())
    n_y = (max(keys) + 1) if keys else 0
    if n_y_hint is not None:
        n_y = max(n_y, n_y_hint)
    ptr = np.zeros(n_y + 1, dtype=np.int64)
    for k in keys:
        ptr[k + 1] = len(yr[k])
    np.cumsum(ptr, out=ptr)
    idx = np.empty(ptr[-1], dtype=np.int32)
    val = np.empty(ptr[-1], dtype=np.float64)
    for k in keys:
        o = ptr[k]
        for t, (x, r) in enumerate(yr[k]):
            idx[o + t] = x
            val[o + t] = r
    return ptr, idx, val


def rating_denominator(r):
    """Smallest supported d with r*d integral for every rating (1 for stars, 2 for half-stars, 100 for
    Jester's two decimals).  Raises ValueError when the ratings are not on such a grid."""
    r = np.asarray(r, dtype=np.float64)
    if r.size == 0:
        return 1
    for d in _DENOMS:
        q = r * d
        if np.all(np.abs(q - np.rint(q)) <= 1e-9 * np.maximum(1.0, np.abs(q))):
            if q.min() < 0 or q.max() > 65535:
                break
            return d
    raise ValueError("similarity kernels need non-negative ratings on a 1/d grid, d in %s, with r*d <= 65535"
                     % (_DENOMS,))


def upload_inputs(kind, n_x, yr, x_biases=None, y_biases=None):
    """Host-side preparation shared by every build on the same ratings: flatten yr, find the rating grid, copy the CSR
    (and the baselines) to the device.  Returns a dict consumed by build_device(..., inputs=...)."""
    import ctypes as C
    n_x = int(n_x)
    ptr, idx, val = _flatten(yr, None if y_biases is None else len(y_biases))
    n_y = len(ptr) - 1
    d_idx, d_val = nat.to_dev(idx, np.int32), nat.to_dev(val, np.float64)
    # the checks that need a pass over the ratings run on the device copy (0.4 s of numpy at 20M ratings otherwise)
    if len(val) and (int(d_idx.min()) < 0 or int(d_idx.max()) >= n_x):
        raise IndexError("x index out of range for n_x=%d" % n_x)
    # denom = 0: the ratings lie on none of the supported 1/d grids (or are negative): sb2_sim_build_dev then takes the
    # general fp64 path (csrc/sim_general.cu: the reference's own summation order on the CUDA cores)
    denom = C.c_int(1)
    nat.check(nat.lib().sb2_rating_denominator_dev(nat.ptr(d_val), len(val), C.byref(denom), nat.stream()))
    inp = dict(n_x=n_x, n_y=n_y, nnz=len(val), denom=denom.value, ptr=nat.to_dev(ptr, np.int64), idx=d_idx, val=d_val,
               bx=None, by=None)
    if kind == "pearson_baseline":
        bx = np.ascontiguousarray(x_biases, dtype=np.float64)
        by = np.ascontiguousarray(y_biases, dtype=np.float64)
        if len(bx) < n_x or len(by) < n_y:
            raise IndexError("bias arrays are shorter than n_x / n_y")
        inp["bx"], inp["by"] = nat.to_dev(bx, np.float64), nat.to_dev(by, np.float64)
    return inp


def build_device(kind, n_x, yr, min_support, global_mean=0.0, x_biases=None, y_biases=None, shrinkage=100,
                 row_begin=0, row_end=None, upper=False, inputs=None):
    """Returns the (row_end-row_begin) x n_x similarity block as a CUDA float64 torch tensor.  upper=True: only the
    columns >= row_begin are computed (shard of a symmetric multi-rank build), the others are zero.
    inputs: the result of upload_inputs() for the same (kind, n_x, yr, biases), to skip the host-side preparation."""
    inp = inputs if inputs is not None else upload_inputs(kind, n_x, yr, x_biases, y_biases)
    n_x = inp["n_x"]
    row_end = n_x if row_end is None else int(row_end)
    out = nat.empty_dev((row_end - row_begin, n_x), np.float64)
    if upper:
        out.zero_()
    fn = nat.lib().sb2_sim_build_upper_dev if upper else nat.lib().sb2_sim_build_dev
    rc = fn(nat.SIM_KINDS[kind], n_x, inp["n_y"], nat.ptr(inp["ptr"]), nat.ptr(inp["idx"]), nat.ptr(inp["val"]),
            inp["nnz"], inp["denom"], int(min_support), float(global_mean), nat.ptr(inp["bx"]), nat.ptr(inp["by"]),
            float(shrinkage), int(row_begin), row_end, nat.ptr(out), nat.stream())
    nat.check(rc)
    return out


def build_rows_device(kind, inputs, rows, out, min_support, global_mean=0.0, shrinkage=100):
    """Rows ``rows`` (CUDA int32 tensor, any order, repeats allowed) of the similarity matrix of ``inputs`` (the
    result of upload_inputs()) into the first len(rows) rows of ``out`` (CUDA float64, n_x columns, contiguous): the
    bits of the same rows of build_device()."""
    n_x = inputs["n_x"]
    rows = nat.to_dev(rows, np.int32)
    if (str(out.dtype) != "torch.float64" or out.dim() != 2 or out.shape[1] != n_x or out.shape[0] < len(rows)
            or not out.is_contiguous()):
        raise ValueError("out must be a contiguous (>= %d) x %d float64 tensor" % (len(rows), n_x))
    rc = nat.lib().sb2_sim_build_rows_dev(nat.SIM_KINDS[kind], n_x, inputs["n_y"], nat.ptr(inputs["ptr"]),
                                          nat.ptr(inputs["idx"]), nat.ptr(inputs["val"]), inputs["nnz"],
                                          inputs["denom"], int(min_support), float(global_mean),
                                          nat.ptr(inputs["bx"]), nat.ptr(inputs["by"]), float(shrinkage),
                                          nat.ptr(rows), len(rows), nat.ptr(out), n_x, nat.stream())
    nat.check(rc)
    return out


def _host(t):
    return t.cpu().numpy()


def cosine(n_x, yr, min_support):
    """similarities.pyx:28-97."""
    return _host(build_device("cosine", n_x, yr, min_support))


def msd(n_x, yr, min_support):
    """similarities.pyx:100-166."""
    return _host(build_device("msd", n_x, yr, min_support))


def pearson(n_x, yr, min_support):
    """similarities.pyx:169-258."""
    return _host(build_device("pearson", n_x, yr, min_support))


def pearson_baseline(n_x, yr, min_support, global_mean, x_biases, y_biases, shrinkage=100):
    """similarities.pyx:261-361 (min_support is clamped to >= 2 there, :334)."""
    return _host(build_device("pearson_baseline", n_x, yr, min_support, global_mean, x_biases, y_biases, shrinkage))
