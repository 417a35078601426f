"""cross_validate: the caller of the hot path (reference: model_selection/validation.py:29-142,
fit_and_score :683-769), single process -- fit/test run on the GPU, fold-level joblib fan-out would
only multiply CUDA contexts.

fit_and_score scores a device-batched algorithm from arrays: the fold's pairs are mapped to inner ids once
(``Fold``), the estimates come from the algorithm's device estimate and the measures from
``accuracy._of_arrays``, which gives the bits ``accuracy.<m>(algo.test(testset))`` gives without building a
Prediction per pair.  Any other algorithm or measure takes the tuple route.
"""
import time

import numpy as np

from .. import accuracy
from .split import get_cv


class _Pairs(object):
    """Prediction pairs as arrays: inner ids (-1 unknown), r_ui minus the offset, and the users fcp groups by."""

    def __init__(self, iu, ii, r_ui, uids=None, users=None):
        self.iu, self.ii, self.r_ui = iu, ii, r_ui
        self._uids, self._users, self._dev = uids, users, None

    def device_ids(self):
        if self._dev is None:
            from .. import _native as nat
            self._dev = nat.to_dev(self.iu, np.int32), nat.to_dev(self.ii, np.int32)
        return self._dev

    def users(self):
        """(code, n_users): users numbered in first appearance order, equal raw uids merged (as accuracy.fcp)."""
        if self._users is None:
            codes = {}
            setd = codes.setdefault
            code = np.array([setd(u, len(codes)) for u in self._uids], dtype=np.int64)
            self._users = code, len(codes)
        return self._users


class Fold(object):
    """One (trainset, testset) split, with the arrays its predictions are scored from built on first use and kept
    for every algorithm scored on it."""

    def __init__(self, trainset, testset):
        self.trainset, self.testset = trainset, testset
        self._test = self._train = None

    def test_pairs(self):
        if self._test is None:
            ts = self.trainset
            rows = self.testset.tolist() if isinstance(self.testset, np.ndarray) else list(self.testset)
            uids = [row[0] for row in rows]
            iu, ii = ts.to_inner_uids(uids), ts.to_inner_iids([row[1] for row in rows])
            r_ui = np.fromiter((row[2] for row in rows), dtype=np.float64, count=len(rows)) - ts.offset
            self._test = _Pairs(iu, ii, r_ui, uids=uids)
        return self._test

    def train_pairs(self):
        """The pairs of ``trainset.build_testset()``: all_ratings() order, so users appear in inner id order."""
        if self._train is None:
            ts = self.trainset
            u, i, r = ts.coo()
            rated = np.diff(ts.user_csr()[0]) > 0
            code = (np.cumsum(rated) - 1)[u]
            self._train = _Pairs(u, i, r - ts.offset, users=(code, int(rated.sum())))
        return self._train


def _estimates(algo, pairs):
    """What ``algo.test`` gives as est for the pairs, as a float64 array."""
    n = len(pairs.r_ui)
    if not n:
        accuracy._need(())
    est, code = algo._estimate_dev(*pairs.device_ids())
    return algo._final_estimates(est.cpu().numpy()[:n], None if code is None else code.cpu().numpy()[:n])


def fit_and_score(algo, trainset, testset, measures, return_train_measures=False):
    return _fit_and_score(algo, Fold(trainset, testset), measures, return_train_measures)


def _fit_and_score(algo, fold, measures, return_train_measures):
    t0 = time.time()
    algo.fit(fold.trainset)
    fit_time = time.time() - t0
    if algo._batched() and all(m.lower() in accuracy.ARRAY_MEASURES for m in measures):
        t0 = time.time()
        test = fold.test_pairs()
        est = _estimates(algo, test)
        test_time = time.time() - t0
        test_m = {m: accuracy._of_arrays(m.lower(), test.r_ui, est, test.users) for m in measures}
        train_m = {}
        if return_train_measures:
            train = fold.train_pairs()
            est = _estimates(algo, train)
            train_m = {m: accuracy._of_arrays(m.lower(), train.r_ui, est, train.users) for m in measures}
        return test_m, train_m, fit_time, test_time
    t0 = time.time()
    predictions = algo.test(fold.testset)
    test_time = time.time() - t0
    train_predictions = algo.test(fold.trainset.build_testset()) if return_train_measures else None
    test_m, train_m = {}, {}
    for m in measures:
        f = getattr(accuracy, m.lower())
        test_m[m] = f(predictions, verbose=0)
        if return_train_measures:
            train_m[m] = f(train_predictions, verbose=0)
    return test_m, train_m, fit_time, test_time


def cross_validate(algo, data, measures=["rmse", "mae"], cv=None, return_train_measures=False, n_jobs=1,
                   pre_dispatch="2*n_jobs", verbose=False):
    measures = [m.lower() for m in measures]
    cv = get_cv(cv)
    outs = [fit_and_score(algo, tr, te, measures, return_train_measures) for tr, te in cv.split(data)]
    ret = {}
    for m in measures:
        ret["test_" + m] = np.array([o[0][m] for o in outs])
        if return_train_measures:
            ret["train_" + m] = np.array([o[1][m] for o in outs])
    ret["fit_time"] = tuple(o[2] for o in outs)
    ret["test_time"] = tuple(o[3] for o in outs)
    if verbose:
        for k, v in ret.items():
            print(k, v)
    return ret
