"""CoClustering (reference: prediction_algorithms/co_clustering.pyx:68-237 fit / compute_averages, then estimate).

fit(): the initial clusters are drawn on the host with numpy (``rng.randint``, users first), so seeds agree with
the reference; the user / item means are np.mean of every ur[u] / ir[i] list (the shared ``list_means``).  The
epoch loop runs on the device in one call (sb2_coclustering_fit_dev) and is bit-identical to the reference.
test() sends all pairs to the one-thread-per-pair estimate kernel (sb2_coclustering_predict_dev); an unknown user
or item gets the global mean as a normal estimate, as in the reference.
"""
import numpy as np

from .. import _native as nat
from ..utils import get_rng
from .algo_base import AlgoBase, list_means


def _as_inner(v):
    return int(v) if isinstance(v, (int, np.integer)) else -1


class CoClustering(AlgoBase):

    def __init__(self, n_cltr_u=3, n_cltr_i=3, n_epochs=20, random_state=None, verbose=False):
        AlgoBase.__init__(self)
        self.n_cltr_u = n_cltr_u
        self.n_cltr_i = n_cltr_i
        self.n_epochs = n_epochs
        self.random_state = random_state
        self.verbose = verbose
        self._dev = None

    def fit(self, trainset):
        AlgoBase.fit(self, trainset)
        ts = trainset
        rng = get_rng(self.random_state)
        cltr_u = rng.randint(self.n_cltr_u, size=ts.n_users)
        cltr_i = rng.randint(self.n_cltr_i, size=ts.n_items)
        up, ui, ur = ts.user_csr()
        ip, iu, ir = ts.item_csr()
        self.user_mean = list_means(up, ur)
        self.item_mean = list_means(ip, ir)
        n_cu, n_ci = int(self.n_cltr_u), int(self.n_cltr_i)
        d_cu, d_ci = nat.to_dev(cltr_u, np.int32), nat.to_dev(cltr_i, np.int32)
        d_um, d_im = nat.to_dev(self.user_mean, np.float64), nat.to_dev(self.item_mean, np.float64)
        d_au, d_ai, d_ac = nat.empty_dev((n_cu,), np.float64), nat.empty_dev((n_ci,), np.float64), \
            nat.empty_dev((n_cu, n_ci), np.float64)
        d_u = (nat.to_dev(up, np.int64), nat.to_dev(ui, np.int32), nat.to_dev(ur, np.float64))
        d_i = (nat.to_dev(ip, np.int64), nat.to_dev(iu, np.int32), nat.to_dev(ir, np.float64))
        if self.verbose:
            for epoch in range(self.n_epochs):
                print("Processing epoch {}".format(epoch))
        rc = nat.lib().sb2_coclustering_fit_dev(
            ts.n_users, ts.n_items, len(ur), *map(nat.ptr, d_u), *map(nat.ptr, d_i), nat.ptr(d_um), nat.ptr(d_im),
            float(ts.global_mean), n_cu, n_ci, int(self.n_epochs), nat.ptr(d_cu), nat.ptr(d_ci), nat.ptr(d_au),
            nat.ptr(d_ai), nat.ptr(d_ac), nat.stream())
        if rc == nat.ERR_INVALID:
            # the cluster counts were accepted by randint, so this is a rating outside the C int range, which the
            # reference's `cdef int r` rejects with OverflowError
            raise OverflowError(nat.lib().sb2_last_error().decode("utf-8", "replace"))
        nat.check(rc)
        self.cltr_u = d_cu.cpu().numpy().astype(np.int64)
        self.cltr_i = d_ci.cpu().numpy().astype(np.int64)
        self.avg_cltr_u, self.avg_cltr_i, self.avg_cocltr = d_au.cpu().numpy(), d_ai.cpu().numpy(), d_ac.cpu().numpy()
        self._dev = (d_cu, d_ci, d_um, d_im, d_au, d_ai, d_ac)
        return self

    def __getstate__(self):
        state = dict(self.__dict__)
        state["_dev"] = None
        return state

    def _device_state(self):
        if self._dev is None:  # unpickled
            self._dev = (nat.to_dev(self.cltr_u, np.int32), nat.to_dev(self.cltr_i, np.int32),
                         nat.to_dev(self.user_mean, np.float64), nat.to_dev(self.item_mean, np.float64),
                         nat.to_dev(self.avg_cltr_u, np.float64), nat.to_dev(self.avg_cltr_i, np.float64),
                         nat.to_dev(self.avg_cocltr, np.float64))
        return self._dev

    def _estimate_dev(self, d_u, d_i):
        """(est, None) for the device pairs (d_u, d_i): CoClustering has no impossible pairs."""
        n = len(d_u)
        ts = self.trainset
        cu, ci, um, im, au, ai, ac = self._device_state()
        est = nat.empty_dev((max(n, 1),), np.float64)
        nat.check(nat.lib().sb2_coclustering_predict_dev(n, nat.ptr(d_u), nat.ptr(d_i), ts.n_users, ts.n_items,
                                                         int(self.n_cltr_i), nat.ptr(cu), nat.ptr(ci), nat.ptr(um),
                                                         nat.ptr(im), nat.ptr(au), nat.ptr(ai), nat.ptr(ac),
                                                         float(ts.global_mean), nat.ptr(est), nat.stream()))
        return est, None

    def _estimate_batch(self, iu, ii):
        n = len(iu)
        est, _ = self._estimate_dev(nat.to_dev(iu, np.int32), nat.to_dev(ii, np.int32))
        return est.cpu().numpy()[:n], [{"was_impossible": False} for _ in range(n)]

    def estimate(self, u, i):
        est, _ = self._estimate_batch(np.array([_as_inner(u)], dtype=np.int32), np.array([_as_inner(i)], dtype=np.int32))
        return est[0]

    _batch_estimate_of = estimate
