"""k-NN algorithms (reference: prediction_algorithms/knns.py:20-403): KNNBasic, KNNWithMeans, KNNBaseline,
KNNWithZScore.

fit() builds the similarity matrix on the device (tensor-core contractions) and keeps it there;
test() ships all known (x, y) pairs to the warp-select kernel (sb2_knn_predict_dev) which reproduces
heapq.nlargest + the ordered weighted sum bit-for-bit.  ``.sim`` is materialised to numpy lazily.

When the dense n_x x n_x matrix would take more than _DENSE_SIM_FRACTION of the device's memory (user-based models
at the ml-20M, ml-25M and Netflix shapes), fit() does not build it: every predict-time call builds the rows its pairs
read, one band at a time (sb2_sim_build_rows_dev, then sb2_knn_predict_rows_dev), with the dense route's bits.
"""
import ctypes

import numpy as np

from .. import _native as nat
from .. import similarities as sims
from .algo_base import AlgoBase
from .predictions import PredictionImpossible

# fit() keeps the dense similarity matrix when its 8 n_x^2 bytes take at most this share of the device's memory;
# otherwise the model streams its similarity rows
_DENSE_SIM_FRACTION = 0.5
# bytes of similarity rows a streamed model holds on the device at a time (None: an eighth of the device's memory)
_STREAM_BAND_BYTES = None


def streams_similarities(n_x, device_bytes):
    """True when a k-NN model over n_x users / items does not keep the dense matrix on a device of this size."""
    return 8 * int(n_x) * int(n_x) > _DENSE_SIM_FRACTION * device_bytes


def band_rows(n_x, device_bytes):
    """Similarity rows per band of a streamed model: the band budget over the 8 n_x bytes of a row, at least 1."""
    budget = _STREAM_BAND_BYTES if _STREAM_BAND_BYTES is not None else device_bytes // 8
    return max(1, int(budget) // (8 * int(n_x)))


def plan_bands(x, rows_per_band):
    """Plan of a streamed k-NN call over the pairs whose x ids are the int32 tensor ``x`` (< 0: unknown), on x's
    device.  The pairs are grouped by x (stable sort, unknown x first) and the distinct known x are cut into bands of
    ``rows_per_band``.  Returns (order, inv, rows, slot, bands):
      order  int64: the grouped pairs are x[order];
      inv    int64: the inverse permutation, the grouped position of every input pair (grouped[inv] is in input order);
      rows   int32: the distinct known x, ascending; band b builds rows[b * rows_per_band:(b + 1) * rows_per_band];
      slot   int32: for every grouped pair, the row of its x within its band (0 for unknown x, whose pairs read none);
      bands  list of (pair_begin, pair_end, row_begin, row_end) over the grouped pairs and ``rows``, in order; the
             unknown x belong to the first band.  No band when there are no pairs."""
    import torch
    dev = x.device
    n = int(x.numel())
    if n == 0:
        empty = torch.zeros(0, dtype=torch.int64, device=dev)
        return empty, empty, empty.int(), empty.int(), []
    xs, order = torch.sort(x, stable=True)
    n_unk = int(torch.count_nonzero(xs < 0))
    rows, counts = torch.unique_consecutive(xs[n_unk:], return_counts=True)
    n_rows = len(rows)
    rank = torch.repeat_interleave(torch.arange(n_rows, device=dev), counts)
    slot = torch.zeros(n, dtype=torch.int32, device=dev)
    slot[n_unk:] = (rank % rows_per_band).to(torch.int32)
    inv = torch.empty_like(order)
    inv[order] = torch.arange(n, device=dev)
    if n_rows == 0:
        return order, inv, rows.int(), slot, [(0, n, 0, 0)]
    last = torch.tensor(list(range(rows_per_band, n_rows, rows_per_band)) + [n_rows], device=dev) - 1
    bands, p0 = [], 0
    for b, p1 in enumerate((n_unk + torch.cumsum(counts, 0)[last]).tolist()):
        bands.append((p0, p1, b * rows_per_band, min((b + 1) * rows_per_band, n_rows)))
        p0 = p1
    return order, inv, rows.int(), slot, bands


def _device_bytes():
    torch = nat.torch_cuda()
    return torch.cuda.get_device_properties(nat.device()).total_memory


class SymmetricAlgo(AlgoBase):
    """user_based <-> item_based symmetry helper (knns.py:20-52): x is the entity similarities are
    computed between, y the other one."""
    _streamed = False     # no dense matrix: similarity rows are built by the calls that read them
    _sim_inputs = None    # streamed: upload_inputs() of the similarity, kept on the device

    def __init__(self, sim_options={}, **kwargs):
        AlgoBase.__init__(self, sim_options=sim_options, **kwargs)

    def fit(self, trainset):
        AlgoBase.fit(self, trainset)
        ub = self.sim_options["user_based"]
        self.n_x = trainset.n_users if ub else trainset.n_items
        self.n_y = trainset.n_items if ub else trainset.n_users
        self._sim_dev = None
        self._sim_host = None
        self._yr_dev = None
        self._streamed = False
        self._sim_inputs = None
        return self

    def _fit_similarities(self):
        """The dense matrix on the device, or -- when it would take more than _DENSE_SIM_FRACTION of the device's
        memory -- the streamed route: the similarity's inputs are uploaded once and rows are built at predict time.
        A streamed fit raises what the dense build raises.  The only build error that depends on the ratings is
        ZeroDivisionError (msd with min_support <= 0 and a pair without common ratings; pearson_baseline with a
        shrinkage of -(n - 1)); only in those cases is every row built once, band by band, to find out."""
        if not streams_similarities(self.n_x, _device_bytes()):
            self._sim_dev = self.compute_similarities_device()
            return
        name, n_x, yr, kw = self._sim_args()
        self._streamed = True
        self._sim_kind = (name, kw["min_support"], kw.get("global_mean", 0.0), kw.get("shrinkage", 100))
        self._sim_inputs = sims.upload_inputs(name, n_x, yr, kw.get("x_biases"), kw.get("y_biases"))
        shrinkage = float(self._sim_kind[3])
        if ((name == "msd" and int(kw["min_support"]) <= 0)
                or (name == "pearson_baseline" and shrinkage <= -1 and shrinkage.is_integer())):
            torch = nat.torch_cuda()
            for _ in self._sim_bands(torch.arange(n_x, dtype=torch.int32, device=nat.device())):
                pass

    def _stream_inputs(self):
        if self._sim_inputs is None:   # after unpickling
            name, n_x, yr, kw = self._sim_args()
            self._sim_inputs = sims.upload_inputs(name, n_x, yr, kw.get("x_biases"), kw.get("y_biases"))
        return self._sim_inputs

    def _sim_bands(self, rows):
        """Yields (r0, r1, block) for consecutive bands of the device int32 ``rows``: block[:r1 - r0] holds
        sim[rows[r0:r1]] (one device buffer, reused for every band)."""
        inp = self._stream_inputs()
        name, min_support, global_mean, shrinkage = self._sim_kind
        per = band_rows(self.n_x, _device_bytes())
        block = nat.empty_dev((max(1, min(per, len(rows))), self.n_x), np.float64)
        for r0 in range(0, len(rows), per):
            r1 = min(r0 + per, len(rows))
            sims.build_rows_device(name, inp, rows[r0:r1], block, min_support, global_mean, shrinkage)
            yield r0, r1, block

    @property
    def xr(self):
        return self.trainset.ur if self.sim_options["user_based"] else self.trainset.ir

    @property
    def yr(self):
        return self.trainset.ir if self.sim_options["user_based"] else self.trainset.ur

    def switch(self, u_stuff, i_stuff):
        if self.sim_options["user_based"]:
            return u_stuff, i_stuff
        return i_stuff, u_stuff

    # the similarity matrix: device-resident, numpy view on demand (5.8 GB at ml-20M scale); a streamed model
    # builds it band by band into one host array (numpy's MemoryError when the host cannot hold it)
    @property
    def sim(self):
        if self._sim_host is None and self._sim_dev is not None:
            self._sim_host = self._sim_dev.cpu().numpy()
        elif self._sim_host is None and self._streamed:
            torch = nat.torch_cuda()
            out = np.empty((self.n_x, self.n_x))
            for r0, r1, block in self._sim_bands(torch.arange(self.n_x, dtype=torch.int32, device=nat.device())):
                out[r0:r1] = block[:r1 - r0].cpu().numpy()
            self._sim_host = out
        return self._sim_host

    @sim.setter
    def sim(self, value):
        self._sim_host = None if value is None else np.ascontiguousarray(value, dtype=np.float64)
        self._sim_dev = None
        self._streamed = False        # an assigned matrix is used as the dense one
        self._sim_inputs = None

    def _sim_device(self):
        if self._sim_dev is None:
            self._sim_dev = nat.to_dev(self._sim_host, np.float64)
        return self._sim_dev

    def _yr_device(self):
        if self._yr_dev is None and self._streamed:
            inp = self._stream_inputs()   # the similarity's yr CSR is the one the estimates read
            self._yr_dev = (inp["ptr"], inp["idx"], inp["val"])
        if self._yr_dev is None:
            ts = self.trainset
            ptr, idx, val = ts.item_csr() if self.sim_options["user_based"] else ts.user_csr()
            self._yr_dev = (nat.to_dev(ptr, np.int64), nat.to_dev(idx, np.int32), nat.to_dev(val, np.float64))
        return self._yr_dev

    def __getstate__(self):
        state = dict(self.__dict__)
        # materialise before dropping device handles; a streamed model stores no matrix and rebuilds its rows
        state["_sim_host"] = None if self._streamed else self.sim
        state["_sim_dev"] = None
        state["_yr_dev"] = None
        state["_sim_inputs"] = None
        return state

    def _knn_dev(self, d_u, d_i, mode, bx=None, by=None):
        """(est, actual_k, impossible) device tensors for the device pairs (d_u, d_i)."""
        d_x, d_y = self.switch(d_u, d_i)
        n = len(d_x)
        ptr, idx, val = self._yr_device()
        est = nat.empty_dev((max(n, 1),), np.float64)
        ak = nat.empty_dev((max(n, 1),), np.int32)
        imp = nat.empty_dev((max(n, 1),), np.uint8)
        d_bx = nat.to_dev(bx, np.float64) if bx is not None else None
        d_by = nat.to_dev(by, np.float64) if by is not None else None
        if self._streamed:
            self._knn_streamed(d_x, d_y, mode, d_bx, d_by, est, ak, imp)
            return est, ak, imp
        sim = self._sim_device()
        rc = nat.lib().sb2_knn_predict_dev(n, nat.ptr(d_x), nat.ptr(d_y), self.n_x, nat.ptr(sim), self.n_x,
                                           nat.ptr(ptr), nat.ptr(idx), nat.ptr(val), int(self.k), int(self.min_k),
                                           mode, float(self.trainset.global_mean), nat.ptr(d_bx), nat.ptr(d_by),
                                           nat.ptr(est), nat.ptr(ak), nat.ptr(imp), nat.stream())
        nat.check(rc)
        return est, ak, imp

    def _knn_streamed(self, d_x, d_y, mode, d_bx, d_by, est, ak, imp):
        """_knn_dev without the dense matrix: the pairs are grouped by x, each band of distinct x is built by
        sb2_sim_build_rows_dev and its pairs estimated by sb2_knn_predict_rows_dev from the band's rows, and the
        results go back to input order."""
        n = len(d_x)
        if n == 0:
            return
        ptr, idx, val = self._yr_device()
        order, inv, rows, slot, bands = plan_bands(d_x, band_rows(self.n_x, _device_bytes()))
        xs, ys = d_x[order], d_y[order]
        e_s, a_s, i_s = (nat.empty_dev((n,), t) for t in (np.float64, np.int32, np.uint8))
        built = self._sim_bands(rows)
        lib, stream = nat.lib(), nat.stream()
        for p0, p1, r0, r1 in bands:
            block = next(built)[2] if r1 > r0 else None   # a band of unknown x only reads no row
            nat.check(lib.sb2_knn_predict_rows_dev(p1 - p0, nat.ptr(xs[p0:]), nat.ptr(ys[p0:]), self.n_x,
                                                   nat.ptr(block), self.n_x, nat.ptr(slot[p0:]), nat.ptr(ptr),
                                                   nat.ptr(idx), nat.ptr(val), int(self.k), int(self.min_k), mode,
                                                   float(self.trainset.global_mean), nat.ptr(d_bx), nat.ptr(d_by),
                                                   nat.ptr(e_s[p0:]), nat.ptr(a_s[p0:]), nat.ptr(i_s[p0:]), stream))
        est[:n] = e_s[inv]
        ak[:n] = a_s[inv]
        imp[:n] = i_s[inv]

    def get_neighbors(self, iid, k):
        """AlgoBase.get_neighbors; a streamed model builds the one row and selects on it."""
        if not self._streamed:
            return AlgoBase.get_neighbors(self, iid, k)
        n = self.n_x
        k = max(0, min(int(k), n - 1))
        if k == 0 or not 0 <= int(iid) < n:   # the dense kernel pads a row outside [0, n) with -1
            return []
        rows = nat.to_dev(np.array([int(iid)], dtype=np.int32), np.int32)
        row = next(self._sim_bands(rows))[2]
        out = nat.empty_dev((1, k), np.int32)
        # sb2_get_neighbors_dev reads row iid at sim + iid * n: point that address at the one built row
        base = ctypes.c_void_p(row.data_ptr() - int(iid) * n * 8)
        nat.check(nat.lib().sb2_get_neighbors_dev(n, base, n, 1, nat.ptr(rows), k, nat.ptr(out), nat.stream()))
        return [int(j) for j in out.cpu().numpy()[0] if j >= 0]

    def _knn_batch(self, iu, ii, mode, bx=None, by=None):
        n = len(iu)
        est, ak, imp = self._knn_dev(nat.to_dev(iu, np.int32), nat.to_dev(ii, np.int32), mode, bx, by)
        return est.cpu().numpy()[:n], ak.cpu().numpy()[:n], imp.cpu().numpy()[:n]

    def _estimate_dev(self, d_u, d_i):
        """(est, impossible) device tensors for the device pairs (d_u, d_i)."""
        est, _, imp = self._knn_dev(d_u, d_i, *self._knn_args())
        return est, imp


def _as_inner(v):
    return int(v) if isinstance(v, (int, np.integer)) else -1


class KNNBasic(SymmetricAlgo):
    """knns.py:55-123.  est = sum(sim * r) / sum(sim) over the k most similar neighbours with sim > 0."""

    def __init__(self, k=40, min_k=1, sim_options={}, **kwargs):
        SymmetricAlgo.__init__(self, sim_options=sim_options, **kwargs)
        self.k = k
        self.min_k = min_k

    def fit(self, trainset):
        SymmetricAlgo.fit(self, trainset)
        self._fit_similarities()
        return self

    def _knn_args(self):
        return (0,)

    def _estimate_batch(self, iu, ii):
        est, ak, imp = self._knn_batch(iu, ii, 0)
        details = []
        for k in range(len(est)):
            if imp[k] == 2:
                raise ZeroDivisionError("division by zero")  # min_k <= 0 and no positive neighbour
            if imp[k]:
                reason = ("User and/or item is unkown." if (iu[k] < 0 or ii[k] < 0) else "Not enough neighbors.")
                details.append({"was_impossible": True, "reason": reason})
            else:
                details.append({"actual_k": int(ak[k]), "was_impossible": False})
        return est, details

    def estimate(self, u, i):
        est, details = self._estimate_batch(np.array([_as_inner(u)], dtype=np.int32),
                                            np.array([_as_inner(i)], dtype=np.int32))
        d = details[0]
        if d["was_impossible"]:
            raise PredictionImpossible(d["reason"])
        return est[0], {"actual_k": d["actual_k"]}

    _batch_estimate_of = estimate


class KNNBaseline(SymmetricAlgo):
    """knns.py:211-309.  est = b_ui + sum(sim * (r - b_vi)) / sum(sim)."""

    def __init__(self, k=40, min_k=1, sim_options={}, bsl_options={}):
        SymmetricAlgo.__init__(self, sim_options=sim_options, bsl_options=bsl_options)
        self.k = k
        self.min_k = min_k

    def fit(self, trainset):
        SymmetricAlgo.fit(self, trainset)
        self.bu, self.bi = self.compute_baselines()
        self.bx, self.by = self.switch(self.bu, self.bi)
        self._fit_similarities()
        return self

    def _knn_args(self):
        return (1 if self.sim_options["user_based"] else 2), self.bx, self.by

    def _estimate_batch(self, iu, ii):
        est, ak, _ = self._knn_batch(iu, ii, *self._knn_args())
        details = [({"actual_k": int(ak[k]), "was_impossible": False} if ak[k] >= 0 else {"was_impossible": False})
                   for k in range(len(est))]
        return est, details

    def estimate(self, u, i):
        est, details = self._estimate_batch(np.array([_as_inner(u)], dtype=np.int32),
                                            np.array([_as_inner(i)], dtype=np.int32))
        if "actual_k" in details[0]:
            return est[0], {"actual_k": details[0]["actual_k"]}
        return est[0]

    _batch_estimate_of = estimate


def _row_stats(trainset, user_based, with_sigma):
    """means[x] (and sigmas[x]) over xr[x] in list order, with the bits np.mean / np.std give per row (knns.py:168-170,
    :362-366).  Rows of equal length are stacked and reduced along the contiguous last axis in one call: numpy runs
    the same pairwise summation over each row of a C-contiguous 2-D array as over the 1-D row itself, so the results
    are identical to the reference's per-row loop (tests/test_host.py::test_row_stats_match_per_row_numpy) at one
    numpy call per distinct row length instead of one per row."""
    ptr, _, val = trainset.user_csr() if user_based else trainset.item_csr()
    n_x = len(ptr) - 1
    means = np.zeros(n_x)
    sigmas = np.zeros(n_x) if with_sigma else None
    lens = np.diff(ptr)
    order = np.argsort(lens, kind="stable")
    sorted_lens = lens[order]
    starts = np.nonzero(np.diff(np.concatenate(([-1], sorted_lens))))[0]
    ends = np.concatenate((starts[1:], [n_x]))
    for a, b in zip(starts.tolist(), ends.tolist()):
        length = int(sorted_lens[a])
        rows = order[a:b]
        if length == 0:
            means[rows] = np.nan      # np.mean([]) (with numpy's warning in the reference); cannot occur for a trainset
            if with_sigma:
                sigmas[rows] = np.nan
            continue
        block = val[ptr[rows][:, None] + np.arange(length)[None, :]]   # (rows, length), C-contiguous
        means[rows] = np.mean(block, axis=1)
        if with_sigma:
            sigmas[rows] = np.std(block, axis=1)
    return means, sigmas


class _MeanCenteredKNN(SymmetricAlgo):
    _mode = 3

    def __init__(self, k=40, min_k=1, sim_options={}, **kwargs):
        SymmetricAlgo.__init__(self, sim_options=sim_options, **kwargs)
        self.k = k
        self.min_k = min_k

    def _knn_args(self):
        return self._mode, self.means, getattr(self, "sigmas", None)

    def _estimate_batch(self, iu, ii):
        est, ak, imp = self._knn_batch(iu, ii, *self._knn_args())
        details = [({"was_impossible": True, "reason": "User and/or item is unkown."} if imp[k]
                    else {"actual_k": int(ak[k]), "was_impossible": False}) for k in range(len(est))]
        return est, details

    def estimate(self, u, i):
        est, details = self._estimate_batch(np.array([_as_inner(u)], dtype=np.int32),
                                            np.array([_as_inner(i)], dtype=np.int32))
        if details[0]["was_impossible"]:
            raise PredictionImpossible(details[0]["reason"])
        return est[0], {"actual_k": details[0]["actual_k"]}


class KNNWithMeans(_MeanCenteredKNN):
    """knns.py:126-208.  est = mu_x + sum(sim * (r - mu_nb)) / sum(sim)."""
    _mode = 3

    def fit(self, trainset):
        SymmetricAlgo.fit(self, trainset)
        self._fit_similarities()
        self.means, _ = _row_stats(trainset, self.sim_options["user_based"], False)
        return self

    estimate = _MeanCenteredKNN.estimate
    _batch_estimate_of = estimate


class KNNWithZScore(_MeanCenteredKNN):
    """knns.py:312-403.  est = mu_x + sigma_x * sum(sim * (r - mu_nb) / sigma_nb) / sum(sim)."""
    _mode = 4

    def fit(self, trainset):
        SymmetricAlgo.fit(self, trainset)
        self.means, sigmas = _row_stats(trainset, self.sim_options["user_based"], True)
        self.overall_sigma = np.std(trainset.user_csr()[2])  # all_ratings() order, knns.py:359-360
        self.sigmas = np.where(sigmas == 0.0, self.overall_sigma, sigmas)
        self._fit_similarities()
        return self

    estimate = _MeanCenteredKNN.estimate
    _batch_estimate_of = estimate
