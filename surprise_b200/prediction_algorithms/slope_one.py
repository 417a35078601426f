"""SlopeOne (reference: prediction_algorithms/slope_one.pyx:16-97).

fit(): ``freq`` and ``dev`` are by-products of the similarity contractions (freq = M M^T, the rating sums
R M^T) and come from the same tensor-core path (sb2_slope_one_fit_dev); they stay on the device and are
materialised to numpy lazily.  test() sends all known pairs to the warp-per-pair kernel
(sb2_slope_one_predict_dev), which reproduces ``sum(dev[i, j] for j in Ri) / len(Ri)`` in ur[u] order.
"""
import numpy as np

from .. import _native as nat
from .algo_base import AlgoBase, list_means
from .predictions import PredictionImpossible


def _as_inner(v):
    return int(v) if isinstance(v, (int, np.integer)) else -1


class SlopeOne(AlgoBase):

    def __init__(self):
        AlgoBase.__init__(self)

    def fit(self, trainset):
        AlgoBase.fit(self, trainset)
        ts = trainset
        ptr, idx, val = ts.user_csr()
        self._ur_dev = (nat.to_dev(ptr, np.int64), nat.to_dev(idx, np.int32), nat.to_dev(val, np.float64))
        n = ts.n_items
        self._freq_dev = nat.empty_dev((n, n), np.int64)
        self._dev_dev = nat.empty_dev((n, n), np.float64)
        self._freq_host = self._dev_host = None
        nat.check(nat.lib().sb2_slope_one_fit_dev(n, ts.n_users, nat.ptr(self._ur_dev[0]), nat.ptr(self._ur_dev[1]),
                                                  nat.ptr(self._ur_dev[2]), len(val), nat.ptr(self._freq_dev),
                                                  nat.ptr(self._dev_dev), nat.stream()))
        # mean ratings of all users (slope_one.pyx:76-77): np.mean over each ur[u] list
        self.user_mean = list(list_means(ptr, val))
        self._mean_dev = nat.to_dev(np.asarray(self.user_mean, dtype=np.float64), np.float64)
        return self

    # n_items x n_items arrays: device-resident, numpy on demand
    @property
    def freq(self):
        if self._freq_host is None and self._freq_dev is not None:
            self._freq_host = self._freq_dev.cpu().numpy()
        return self._freq_host

    @property
    def dev(self):
        if self._dev_host is None and self._dev_dev is not None:
            self._dev_host = self._dev_dev.cpu().numpy()
        return self._dev_host

    def __getstate__(self):
        state = dict(self.__dict__)
        state["_freq_host"], state["_dev_host"] = self.freq, self.dev
        for k in ("_freq_dev", "_dev_dev", "_ur_dev", "_mean_dev"):
            state[k] = None
        return state

    def _device_state(self):
        if self._freq_dev is None:  # unpickled
            ptr, idx, val = self.trainset.user_csr()
            self._ur_dev = (nat.to_dev(ptr, np.int64), nat.to_dev(idx, np.int32), nat.to_dev(val, np.float64))
            self._freq_dev = nat.to_dev(self._freq_host, np.int64)
            self._dev_dev = nat.to_dev(self._dev_host, np.float64)
            self._mean_dev = nat.to_dev(np.asarray(self.user_mean, dtype=np.float64), np.float64)
        return self._freq_dev, self._dev_dev, self._ur_dev, self._mean_dev

    def _estimate_dev(self, d_u, d_i):
        """(est, impossible) device tensors for the device pairs (d_u, d_i)."""
        n = len(d_u)
        freq, dev, ur, mean = self._device_state()
        est = nat.empty_dev((max(n, 1),), np.float64)
        imp = nat.empty_dev((max(n, 1),), np.uint8)
        nat.check(nat.lib().sb2_slope_one_predict_dev(n, nat.ptr(d_u), nat.ptr(d_i), self.trainset.n_items,
                                                      nat.ptr(freq), nat.ptr(dev), nat.ptr(ur[0]), nat.ptr(ur[1]),
                                                      nat.ptr(mean), nat.ptr(est), nat.ptr(imp), nat.stream()))
        return est, imp

    def _estimate_batch(self, iu, ii):
        n = len(iu)
        est, imp = self._estimate_dev(nat.to_dev(iu, np.int32), nat.to_dev(ii, np.int32))
        est, imp = est.cpu().numpy()[:n], imp.cpu().numpy()[:n]
        details = [{"was_impossible": True, "reason": "User and/or item is unkown."} if imp[k]
                   else {"was_impossible": False} for k in range(n)]
        return est, details

    def estimate(self, u, i):
        est, details = self._estimate_batch(np.array([_as_inner(u)], dtype=np.int32),
                                            np.array([_as_inner(i)], dtype=np.int32))
        if details[0]["was_impossible"]:
            raise PredictionImpossible(details[0]["reason"])
        return est[0]

    _batch_estimate_of = estimate
