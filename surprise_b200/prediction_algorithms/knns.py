"""k-NN algorithms (reference: prediction_algorithms/knns.py:20-403): KNNBasic, KNNWithMeans, KNNBaseline,
KNNWithZScore.

fit() builds the similarity matrix on the device (tensor-core contractions) and keeps it there;
test() ships all known (x, y) pairs to the warp-select kernel (sb2_knn_predict_dev) which reproduces
heapq.nlargest + the ordered weighted sum bit-for-bit.  ``.sim`` is materialised to numpy lazily.
"""
import numpy as np

from .. import _native as nat
from .algo_base import AlgoBase
from .predictions import PredictionImpossible


class SymmetricAlgo(AlgoBase):
    """user_based <-> item_based symmetry helper (knns.py:20-52): x is the entity similarities are
    computed between, y the other one."""

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
        return self

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

    # the similarity matrix: device-resident, numpy view on demand (5.8 GB at ml-20M scale)
    @property
    def sim(self):
        if self._sim_host is None and self._sim_dev is not None:
            self._sim_host = self._sim_dev.cpu().numpy()
        return self._sim_host

    @sim.setter
    def sim(self, value):
        self._sim_host = None if value is None else np.ascontiguousarray(value, dtype=np.float64)
        self._sim_dev = None

    def _sim_device(self):
        if self._sim_dev is None:
            self._sim_dev = nat.to_dev(self._sim_host, np.float64)
        return self._sim_dev

    def _yr_device(self):
        if self._yr_dev is None:
            ts = self.trainset
            ptr, idx, val = ts.item_csr() if self.sim_options["user_based"] else ts.user_csr()
            self._yr_dev = (nat.to_dev(ptr, np.int64), nat.to_dev(idx, np.int32), nat.to_dev(val, np.float64))
        return self._yr_dev

    def __getstate__(self):
        state = dict(self.__dict__)
        state["_sim_host"] = self.sim  # materialise before dropping device handles
        state["_sim_dev"] = None
        state["_yr_dev"] = None
        return state

    def _knn_dev(self, d_u, d_i, mode, bx=None, by=None):
        """(est, actual_k, impossible) device tensors for the device pairs (d_u, d_i)."""
        d_x, d_y = self.switch(d_u, d_i)
        n = len(d_x)
        ptr, idx, val = self._yr_device()
        sim = self._sim_device()
        est = nat.empty_dev((max(n, 1),), np.float64)
        ak = nat.empty_dev((max(n, 1),), np.int32)
        imp = nat.empty_dev((max(n, 1),), np.uint8)
        d_bx = nat.to_dev(bx, np.float64) if bx is not None else None
        d_by = nat.to_dev(by, np.float64) if by is not None else None
        rc = nat.lib().sb2_knn_predict_dev(n, nat.ptr(d_x), nat.ptr(d_y), self.n_x, nat.ptr(sim), self.n_x,
                                           nat.ptr(ptr), nat.ptr(idx), nat.ptr(val), int(self.k), int(self.min_k),
                                           mode, float(self.trainset.global_mean), nat.ptr(d_bx), nat.ptr(d_by),
                                           nat.ptr(est), nat.ptr(ak), nat.ptr(imp), nat.stream())
        nat.check(rc)
        return est, ak, imp

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
        self._sim_dev = self.compute_similarities_device()
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
        self._sim_dev = self.compute_similarities_device()
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
        self._sim_dev = self.compute_similarities_device()
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
        self._sim_dev = self.compute_similarities_device()
        return self

    estimate = _MeanCenteredKNN.estimate
    _batch_estimate_of = estimate
