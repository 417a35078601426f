"""BaselineOnly (reference: prediction_algorithms/baseline_only.py:10-46): est = mu + b_u + b_i, each bias only
when the id is known.

fit() computes the baselines on the device (sb2_baseline_als / sb2_baseline_sgd through
AlgoBase.compute_baselines); test() is batched: all pairs go through the factor-model estimate kernel with zero
factors (sb2_mf_predict_dev, n_factors = 0), whose biased branch performs exactly the reference's additions
((mu + b_u) + b_i, unknown ids skipped), so the estimates carry the same bits.
"""
import numpy as np

from .. import _native as nat
from .algo_base import AlgoBase


class BaselineOnly(AlgoBase):

    def __init__(self, bsl_options={}):
        AlgoBase.__init__(self, bsl_options=bsl_options)
        self._bias_dev = None

    def fit(self, trainset):
        AlgoBase.fit(self, trainset)
        self._bias_dev = None
        self.bu, self.bi = self.compute_baselines()
        return self

    def __setattr__(self, name, value):
        # the reference's estimate() reads bu / bi live: assigning them after fit must drop the device copies
        if name in ("bu", "bi", "trainset") and "_bias_dev" in self.__dict__:
            self.__dict__["_bias_dev"] = None
        object.__setattr__(self, name, value)

    def __getstate__(self):
        state = dict(self.__dict__)
        state["_bias_dev"] = None
        return state

    def _biases_dev(self):
        if getattr(self, "_bias_dev", None) is None:
            self._bias_dev = (nat.to_dev(self.bu, np.float64), nat.to_dev(self.bi, np.float64))
        return self._bias_dev

    def _estimate_dev(self, d_u, d_i):
        """(est, impossible) device tensors for the device pairs (d_u, d_i)."""
        n = len(d_u)
        d_bu, d_bi = self._biases_dev()
        est = nat.empty_dev((max(n, 1),), np.float64)
        imp = nat.empty_dev((max(n, 1),), np.uint8)
        nat.check(nat.lib().sb2_mf_predict_dev(n, nat.ptr(d_u), nat.ptr(d_i), 0, 1, float(self.trainset.global_mean), None,
                                               None, nat.ptr(d_bu), nat.ptr(d_bi), None, None, None, nat.ptr(est),
                                               nat.ptr(imp), nat.stream()))
        return est, imp

    def _estimate_batch(self, iu, ii):
        n = len(iu)
        est, _ = self._estimate_dev(nat.to_dev(iu, np.int32), nat.to_dev(ii, np.int32))
        return est.cpu().numpy()[:n], [{"was_impossible": False} for _ in range(n)]

    def _top_n_scorer(self):
        d_bu, d_bi = self._biases_dev()
        return dict(f=0, biased=1, pu=None, qi=None, bu=d_bu, bi=d_bi)

    def estimate(self, u, i):
        as_inner = lambda v: int(v) if isinstance(v, (int, np.integer)) else -1
        est, _ = self._estimate_batch(np.array([as_inner(u)], dtype=np.int32), np.array([as_inner(i)], dtype=np.int32))
        return est[0]

    _batch_estimate_of = estimate
