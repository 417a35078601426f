"""cross_validate: the caller of the hot path (reference: model_selection/validation.py:29-142,
fit_and_score :683-769), single process -- fit/test run on the GPU, fold-level joblib fan-out would
only multiply CUDA contexts.

fit_and_score scores a device-batched algorithm from arrays: the fold's pairs are mapped to inner ids once
(``Fold``), the estimates come from the algorithm's device estimate and the measures from
``accuracy._of_arrays``, which gives the bits ``accuracy.<m>(algo.test(testset))`` gives without building a
Prediction per pair.  Any other algorithm or rating measure takes the tuple route.  The top-N measures hr@N,
arhr@N, precision@N, recall@N and ndcg@N (threshold None) and the list measures user_coverage@N, catalog_coverage@N,
novelty@N and diversity@N (over the same evaluated users) and the rank measures auc, mrr and mpr over the full ranking
come from one ``algo._top_n_fold`` pass per fold.
"""
import time

import numpy as np

from .. import accuracy
from .split import get_cv


class _Pairs(object):
    """Prediction pairs as arrays: inner ids (-1 unknown), r_ui minus the offset, and the users fcp groups by."""

    def __init__(self, iu, ii, r_ui, uids=None, users=None, iids=None):
        self.iu, self.ii, self.r_ui = iu, ii, r_ui
        self._uids, self._users, self._dev, self._iids = uids, users, None, iids

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

    def relevant(self, threshold, n_items):
        """The held-out relevant items of accuracy.top_n_measures: (iu, n_rel, rel_ptr, rel_idx).  iu (int32) is the
        inner uid (-1 unknown) of each evaluated user -- a user with at least one row whose r_ui (minus the offset) is
        >= threshold, or with any row for threshold None -- in first-appearance order among those rows, equal raw uids
        merged; n_rel (int64) their |R_u|, distinct raw iids counted, unknown items included.  rel_ptr (int64) /
        rel_idx (int32) is the CSR, over the evaluated users the trainset knows, in that order, of their distinct
        known relevant inner iids, ascending.  No evaluated user raises ValueError."""
        n = len(self.r_ui)
        if threshold is None:
            rows = np.arange(n)
        else:
            rows = np.flatnonzero(np.fromiter((x >= threshold for x in self.r_ui.tolist()), dtype=bool, count=n))
        if not len(rows):
            raise ValueError("top-N measures need at least one relevant rating in the testset")
        code = self.users()[0][rows]
        _, first, inv = np.unique(code, return_index=True, return_inverse=True)
        rank = np.empty(len(first), dtype=np.int64)
        rank[np.argsort(first, kind="stable")] = np.arange(len(first))
        star = rank[inv.reshape(-1)]                   # evaluated user of each relevant row
        n_star = len(first)
        iu = np.empty(n_star, dtype=np.int32)
        iu[star] = self.iu[rows]                      # equal raw uids have one inner id
        item = self.ii[rows].astype(np.int64)
        unknown = np.flatnonzero(item < 0)
        if len(unknown):                              # unknown items: numbered past n_items by raw iid
            codes = {}
            setd = codes.setdefault
            item[unknown] = n_items + np.fromiter((setd(self._iids[k], len(codes)) for k in rows[unknown].tolist()),
                                                  dtype=np.int64, count=len(unknown))
        base = int(item.max()) + 1
        k_user, k_item = np.divmod(np.unique(star * base + item), base)     # distinct (user, item), by user then item
        n_rel = np.bincount(k_user, minlength=n_star)
        known = iu >= 0
        keep = known[k_user] & (k_item < n_items)
        slot = np.cumsum(known) - 1                   # position of a known user among the known ones
        rel_ptr = np.zeros(int(known.sum()) + 1, dtype=np.int64)
        np.cumsum(np.bincount(slot[k_user[keep]], minlength=len(rel_ptr) - 1), out=rel_ptr[1:])
        return iu, n_rel, rel_ptr, k_item[keep].astype(np.int32)


class Fold(object):
    """One (trainset, testset) split, with the arrays its predictions are scored from built on first use and kept
    for every algorithm scored on it."""

    def __init__(self, trainset, testset):
        self.trainset, self.testset = trainset, testset
        self._test = self._train = self._cosine = None

    def item_cosine(self):
        """The item-item cosine similarity of the trainset (min_support 1), a CUDA float64 tensor: diversity@N's
        similarity, built on first use.  ValueError when its 8 n_items^2 bytes exceed half the device's memory."""
        if self._cosine is None:
            from .. import similarities as sims
            from ..prediction_algorithms.knns import _device_bytes, streams_similarities
            ts = self.trainset
            if streams_similarities(ts.n_items, _device_bytes()):
                raise ValueError("diversity@N needs the %d x %d item-item cosine matrix, which takes more than half "
                                 "the device's memory" % (ts.n_items, ts.n_items))
            self._cosine = sims.build_device("cosine", ts.n_items, ts.user_csr(), min_support=1)
        return self._cosine

    def test_pairs(self):
        if self._test is None:
            ts = self.trainset
            rows = self.testset.tolist() if isinstance(self.testset, np.ndarray) else list(self.testset)
            uids = [row[0] for row in rows]
            iids = [row[1] for row in rows]
            iu, ii = ts.to_inner_uids(uids), ts.to_inner_iids(iids)
            r_ui = np.fromiter((row[2] for row in rows), dtype=np.float64, count=len(rows)) - ts.offset
            self._test = _Pairs(iu, ii, r_ui, uids=uids, iids=iids)
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
    top_n = {m: accuracy._top_n_measure(m) for m in measures}
    top_n = {m: v for m, v in top_n.items() if v is not None}
    lists = {m: accuracy._top_n_list_measure(m) for m in measures}
    lists = {m: v for m, v in lists.items() if v is not None}
    ranks = {m: accuracy._rank_measure(m) for m in measures}
    ranks = {m: v for m, v in ranks.items() if v is not None}
    if (top_n or lists or ranks) and return_train_measures:
        raise ValueError("return_train_measures cannot be used with top-N measures (%s): trainset items are never "
                         "recommended, so they would be 0" % ", ".join(list(top_n) + list(lists) + list(ranks)))
    t0 = time.time()
    algo.fit(fold.trainset)
    fit_time = time.time() - t0
    rating = [m for m in measures if m not in top_n and m not in lists and m not in ranks]
    test_m, train_m, test_time = _score_ratings(algo, fold, rating, return_train_measures) if rating else ({}, {}, 0.0)
    if top_n or lists or ranks:
        t0 = time.time()
        hit_ns = sorted(set(n for _, n in top_n.values()))
        list_ns = sorted(set(n for _, n in lists.values()))
        sim = fold.item_cosine() if any(key == "diversity" for key, _ in lists.values()) else None
        hit_res, list_res, rank_res = algo._top_n_fold(fold, hit_ns, list_ns, sim, rank=bool(ranks))
        test_time += time.time() - t0
        by_n, by_list_n = dict(zip(hit_ns, hit_res)), dict(zip(list_ns, list_res))
        test_m.update((m, by_n[n][key]) for m, (key, n) in top_n.items())
        test_m.update((m, by_list_n[n][key]) for m, (key, n) in lists.items())
        test_m.update((m, rank_res[key]) for m, key in ranks.items())
        test_m = {m: test_m[m] for m in measures}
    return test_m, train_m, fit_time, test_time


def _score_ratings(algo, fold, measures, return_train_measures):
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
        return test_m, train_m, test_time
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
    return test_m, train_m, test_time


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
