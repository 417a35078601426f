"""AlgoBase -- the drop-in boundary (reference: prediction_algorithms/algo_base.py:21-334).

fit / predict / test / compute_baselines / compute_similarities / get_neighbors keep the reference's
semantics (raw -> inner id mapping, 'UKN__' ids, PredictionImpossible -> default_prediction, offset and
clipping, the train()/fit() compatibility shim).  The one structural change: ``test()`` is the batching
point -- algorithms that provide ``_estimate_batch`` get all (u, i) pairs of the testset in one device
call instead of one Python ``estimate`` call per pair (algo_base.py:213-217).
"""
import warnings

import numpy as np

from .. import similarities as sims
from .optimize_baselines import baseline_als, baseline_sgd
from .predictions import Prediction, PredictionImpossible


def _func(m):
    return getattr(m, "__func__", m)


def list_means(ptr, val):
    """np.mean of every list of a flattened yr CSR (``np.mean([r for (_, r) in ur[u]])`` for all u), as a float64
    array.  Quarter-step ratings take an exact fast path: every partial sum is exact, so any summation order gives
    np.mean's bits; other ratings run np.mean list by list."""
    n = len(ptr) - 1
    cnt = np.diff(ptr)
    if len(val) and np.array_equal(val * 4, np.rint(val * 4)) and np.abs(val).max() < 2 ** 20 and cnt.min() > 0:
        sums = np.bincount(np.repeat(np.arange(n), cnt), weights=val, minlength=n)
        return sums / cnt
    return np.array([np.mean(val[ptr[k]:ptr[k + 1]].tolist()) for k in range(n)], dtype=np.float64)


class AlgoBase(object):
    # set by device-backed subclasses to the estimate() their _estimate_batch is equivalent to
    _batch_estimate_of = None

    def __init__(self, **kwargs):
        self.bsl_options = kwargs.get("bsl_options", {})
        self.sim_options = kwargs.get("sim_options", {})
        if "user_based" not in self.sim_options:
            self.sim_options["user_based"] = True
        self.skip_train = False
        cls = self.__class__
        if _func(cls.fit) is _func(AlgoBase.fit) and _func(cls.train) is not _func(AlgoBase.train):
            warnings.warn("It looks like this algorithm (" + str(cls) + ") implements train() instead of fit(): "
                          "train() is deprecated, please use fit() instead.", UserWarning)

    def train(self, trainset):
        """Deprecated alias of fit() (algo_base.py:49-58)."""
        warnings.warn("train() is deprecated. Use fit() instead", UserWarning)
        self.skip_train = True
        self.fit(trainset)
        return self

    def fit(self, trainset):
        # old-style algorithms override train(); route fit() through it once (algo_base.py:88-92)
        if _func(self.__class__.train) is not _func(AlgoBase.train) and not self.skip_train:
            self.train(trainset)
            return
        self.skip_train = False
        self.trainset = trainset
        self.bu = self.bi = None
        return self

    # -- prediction ----------------------------------------------------------------------------------
    def _inner_ids(self, uid, iid):
        try:
            iuid = self.trainset.to_inner_uid(uid)
        except ValueError:
            iuid = "UKN__" + str(uid)
        try:
            iiid = self.trainset.to_inner_iid(iid)
        except ValueError:
            iiid = "UKN__" + str(iid)
        return iuid, iiid

    def _finish(self, uid, iid, r_ui, est, details, clip, verbose):
        est -= self.trainset.offset
        if clip:
            low, high = self.trainset.rating_scale
            est = min(high, est)
            est = max(low, est)
        pred = Prediction(uid, iid, r_ui, est, details)
        if verbose:
            print(pred)
        return pred

    def predict(self, uid, iid, r_ui=None, clip=True, verbose=False):
        iuid, iiid = self._inner_ids(uid, iid)
        details = {}
        try:
            est = self.estimate(iuid, iiid)
            if isinstance(est, tuple):
                est, details = est
            details["was_impossible"] = False
        except PredictionImpossible as e:
            est = self.default_prediction()
            details["was_impossible"] = True
            details["reason"] = str(e)
        return self._finish(uid, iid, r_ui, est, details, clip, verbose)

    def default_prediction(self):
        return self.trainset.global_mean

    def _batched(self):
        cls = type(self)
        return cls._batch_estimate_of is not None and _func(cls.estimate) is _func(cls._batch_estimate_of)

    def test(self, testset, verbose=False):
        """algo_base.py:191-218.  Device-backed algorithms get the whole testset in ONE estimate call: raw -> inner ids
        through a table lookup (no per-pair exception handling), offset / clipping as array operations; only the
        Prediction tuples the reference returns are built one by one."""
        rows = testset.tolist() if isinstance(testset, np.ndarray) else testset
        off = self.trainset.offset
        if not self._batched():
            return [self.predict(uid, iid, r - off, verbose=verbose) for (uid, iid, r) in rows]
        rows = list(rows)
        n = len(rows)
        ts = self.trainset
        uids = [row[0] for row in rows]
        iids = [row[1] for row in rows]
        iu, ii = ts.to_inner_uids(uids), ts.to_inner_iids(iids)
        est, details = self._estimate_batch(iu, ii)
        est = np.asarray(est, dtype=np.float64).copy()
        imp = np.fromiter((bool(d.get("was_impossible")) for d in details), dtype=bool, count=n)
        if imp.any():
            est[imp] = self.default_prediction()
        est -= off
        low, high = ts.rating_scale
        est = np.maximum(low, np.minimum(high, est))      # est = min(high, est); est = max(low, est)
        r_ui = (np.fromiter((row[2] for row in rows), dtype=np.float64, count=n) - off).tolist()
        out = [Prediction(uid, iid, r, e, d) for uid, iid, r, e, d in zip(uids, iids, r_ui, est.tolist(), details)]
        if verbose:
            for pred in out:
                print(pred)
        return out

    # -- shared fit-time helpers ----------------------------------------------------------------------
    def compute_baselines(self):
        """(bu, bi), computed once per fit (algo_base.py:220-254)."""
        if self.bu is not None:
            return self.bu, self.bi
        methods = {"als": baseline_als, "sgd": baseline_sgd}
        name = self.bsl_options.get("method", "als")
        if name not in methods:
            raise ValueError("Invalid method " + name + " for baseline computation. Available methods are als and "
                             "sgd.")
        self.bu, self.bi = methods[name](self)
        return self.bu, self.bi

    def _sim_args(self):
        ts = self.trainset
        if self.sim_options["user_based"]:
            n_x, yr = ts.n_users, ts.item_csr()
        else:
            n_x, yr = ts.n_items, ts.user_csr()
        name = self.sim_options.get("name", "msd").lower()
        if name not in sims.nat.SIM_KINDS:
            raise NameError("Wrong sim name " + name + ". Allowed values are " + ", ".join(sims.nat.SIM_KINDS) + ".")
        kw = dict(min_support=self.sim_options.get("min_support", 1))
        if name == "pearson_baseline":
            bu, bi = self.compute_baselines()
            bx, by = (bu, bi) if self.sim_options["user_based"] else (bi, bu)
            kw.update(global_mean=ts.global_mean, x_biases=bx, y_biases=by,
                      shrinkage=self.sim_options.get("shrinkage", 100))
        return name, n_x, yr, kw

    def compute_similarities_device(self):
        """The similarity matrix as a CUDA float64 tensor (stays in HBM for the k-NN predict kernel)."""
        name, n_x, yr, kw = self._sim_args()
        return sims.build_device(name, n_x, yr, **kw)

    def compute_similarities(self):
        """The similarity matrix as a float64 ndarray (algo_base.py:256-301)."""
        return self.compute_similarities_device().cpu().numpy()

    def get_neighbors(self, iid, k):
        """Inner ids of the k most similar users / items (algo_base.py:303-334): stable sort of the sim
        row in descending order, self excluded.  Runs on the device-resident matrix when the algorithm keeps
        one (the k-NN family); a user-assigned host ``sim`` is uploaded once by ``_sim_device``."""
        from .. import _native as nat
        n = self.trainset.n_users if self.sim_options["user_based"] else self.trainset.n_items
        sim = self._sim_device() if hasattr(self, "_sim_device") else nat.to_dev(np.asarray(self.sim), np.float64)
        k = max(0, min(int(k), n - 1))
        if k == 0:
            return []
        rows = nat.to_dev(np.array([int(iid)], dtype=np.int32), np.int32)
        out = nat.empty_dev((1, k), np.int32)
        nat.check(nat.lib().sb2_get_neighbors_dev(n, nat.ptr(sim), n, 1, nat.ptr(rows), k, nat.ptr(out), nat.stream()))
        return [int(j) for j in out.cpu().numpy()[0] if j >= 0]
