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


# scores of one user block of top_n_inner: near the B200's 126 MB L2
_TOP_N_BLOCK_BYTES = 96 << 20
# rows sb2_mf_score_block_dev accepts per call (65535 blocks of 16 rows); tiny catalogues would otherwise exceed it
_TOP_N_MAX_SCORER_ROWS = 65535 * 16


def _check_top_n(n):
    if isinstance(n, bool) or not isinstance(n, (int, np.integer)) or n < 1:
        raise ValueError("n must be an int >= 1 (got %r)" % (n,))
    return min(int(n), 2 ** 31 - 1)


def rank_top_n(est, items):
    """Order of the entries (est[k], items[k]) in the top-N ranking: est descending with -0.0 == 0.0 and NaN last,
    ties by ascending item -- a stable sort(reverse=True) of a list in ascending item order."""
    est = np.asarray(est, dtype=np.float64)
    nan = np.isnan(est)
    return np.lexsort((np.asarray(items), -np.where(nan, 0.0, est), nan))


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

    def _final_estimates(self, est, code):
        """The values test() gives a batch of raw estimates: ``default_prediction()`` where ``code`` is 1 (impossible),
        ZeroDivisionError if any code is 2 (KNNBasic with min_k <= 0 and no positive neighbour), then minus the offset
        and clipped to the rating scale as predict() clips one estimate.  ``code`` may be None (nothing impossible)."""
        est = np.array(est, dtype=np.float64)
        if code is not None:
            code = np.asarray(code)
            if (code == 2).any():
                raise ZeroDivisionError("division by zero")
            imp = code == 1
            if imp.any():
                est[imp] = self.default_prediction()
        est -= self.trainset.offset
        low, high = self.trainset.rating_scale
        return np.maximum(low, np.minimum(high, est))      # est = min(high, est); est = max(low, est)

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
        imp = np.fromiter((bool(d.get("was_impossible")) for d in details), dtype=np.uint8, count=n)
        est = self._final_estimates(est, imp)
        r_ui = (np.fromiter((row[2] for row in rows), dtype=np.float64, count=n) - off).tolist()
        out = [Prediction(uid, iid, r, e, d) for uid, iid, r, e, d in zip(uids, iids, r_ui, est.tolist(), details)]
        if verbose:
            for pred in out:
                print(pred)
        return out

    # -- top-N recommendations -------------------------------------------------------------------------
    def get_top_n(self, n=10, uids=None):
        """The n best items each user has not rated, as the reference FAQ computes them:

            get_top_n(algo.test(trainset.build_anti_testset()), n)

        i.e. {raw uid: [(raw iid, est), ...]} with every est the bits ``test()`` gives the pair, sorted by est
        descending, ties in ascending inner item id (Python's stable sort(reverse=True) of the anti-testset).  -0.0
        ranks equal to 0.0; NaN (diverged factors, where the FAQ's order is undefined) ranks after every number.
        Users who rated every item get no entry.  ``uids`` (raw ids) restricts the output to those users, keys in
        the given order; an unknown uid raises ValueError.  Device-batched algorithms score and rank on the GPU
        (see ``top_n_inner``); any other algorithm goes through ``test()`` on the requested users' anti-testset."""
        n = _check_top_n(n)
        ts = self.trainset
        if uids is None:
            users = np.arange(ts.n_users, dtype=np.int32)
            raw_u = [ts.to_raw_uid(u) for u in range(ts.n_users)]
        else:
            raw_u = list(uids)
            users = np.array([ts.to_inner_uid(x) for x in raw_u], dtype=np.int32)
        items, est, count = self.top_n_inner(n, users)
        raw_i = np.empty(ts.n_items, dtype=object)
        raw_i[:] = [ts.to_raw_iid(i) for i in range(ts.n_items)]
        out = {}
        for k in np.flatnonzero(count).tolist():
            c = int(count[k])
            out[raw_u[k]] = list(zip(raw_i[items[k, :c]].tolist(), est[k, :c].tolist()))
        return out

    def top_n_inner(self, n=10, users=None, _block_rows=None, _events=None):
        """``get_top_n`` on inner ids: (items int32 [U, w], est float64 [U, w], count int32 [U]) for the users
        ``users`` (inner ids, default all), w = min(n, n_items).  Row k holds the count[k] best items of users[k],
        padded with -1 / NaN.  ``_block_rows`` overrides the number of users scored per device block (the output
        does not depend on it).  ``_events``, a list, receives three recorded CUDA events per block (before the
        scoring, between scoring and selection, after the selection) for timing."""
        n = _check_top_n(n)
        ts = self.trainset
        if users is None:
            users = np.arange(ts.n_users, dtype=np.int32)
        else:
            users = np.asarray(users).reshape(-1)
            if users.size and (users.dtype.kind not in "iu" or users.min() < 0 or users.max() >= ts.n_users):
                raise ValueError("users must be inner user ids in [0, %d)" % ts.n_users)
            users = users.astype(np.int32)
        width = min(n, ts.n_items)
        if not self._batched():
            return self._top_n_by_test(width, users)
        items, est, count = self._top_n_dev(width, users, _block_rows, _events)
        n_u = len(users)
        return items.cpu().numpy()[:n_u], est.cpu().numpy()[:n_u], count.cpu().numpy()[:n_u]

    def _top_n_dev(self, width, users, _block_rows=None, _events=None, on_block=None, on_scores=None, select=True,
                   d_csr=None):
        """top_n_inner's device block loop: (items, est, count) as device arrays of max(len(users), 1) rows.
        ``on_scores(b0, nr, d_rows, scores, impossible)``, if given, is called with each block's scores (row k of the
        block at scores + k * n_items) and impossible codes (None when there are none) before its selection.
        ``on_block(b0, nr, items, est, count)``, if given, is called after each block's selection, when rows
        b0 .. b0 + nr of the device arrays are final.  With ``select`` False nothing is selected and (None, None, None)
        is returned.  ``d_csr`` is the trainset's user CSR (ptr, idx) on the device, uploaded here when None."""
        from .. import _native as nat
        torch = nat.torch_cuda()
        ts = self.trainset
        n_u, n_i = len(users), ts.n_items
        items = est = count = None
        if select:
            items = nat.empty_dev((max(n_u, 1), width), np.int32)
            est = nat.empty_dev((max(n_u, 1), width), np.float64)
            count = nat.empty_dev((max(n_u, 1),), np.int32)
        d_up, d_ui = self._user_csr_dev() if d_csr is None else d_csr
        d_users = nat.to_dev(users, np.int32)
        scorer = self._top_n_scorer()
        rows = int(_block_rows) if _block_rows else max(1, _TOP_N_BLOCK_BYTES // (8 * n_i))
        rows = min(rows, max(n_u, 1), _TOP_N_MAX_SCORER_ROWS)
        low, high = ts.rating_scale
        scores = nat.empty_dev((rows * n_i,), np.float64) if scorer is not None else None
        lib, stream = nat.lib(), nat.stream()
        for b0 in range(0, n_u, rows):
            d_rows = d_users[b0:b0 + rows]
            nr = len(d_rows)
            imp = None
            ev = None
            if _events is not None:
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                _events.append(ev)
                ev[0].record()
            if scorer is not None:
                nat.check(lib.sb2_mf_score_block_dev(nr, nat.ptr(d_rows), n_i, scorer["f"], scorer["biased"],
                                                     float(ts.global_mean), nat.ptr(scorer["pu"]),
                                                     nat.ptr(scorer["qi"]), nat.ptr(scorer["bu"]),
                                                     nat.ptr(scorer["bi"]), nat.ptr(scorer.get("yj")),
                                                     nat.ptr(scorer.get("up")), nat.ptr(scorer.get("ui")),
                                                     nat.ptr(scores), n_i, stream))
                sc = scores
            else:
                d_u = d_rows.repeat_interleave(n_i)
                d_i = torch.arange(n_i, dtype=torch.int32, device=d_rows.device).repeat(nr)
                sc, imp = self._estimate_dev(d_u, d_i)
            if ev:
                ev[1].record()
            if on_scores is not None:
                on_scores(b0, nr, d_rows, sc, imp)
            if select:
                nat.check(lib.sb2_top_n_select_dev(nr, nat.ptr(d_rows), n_i, nat.ptr(sc), n_i, nat.ptr(imp),
                                                   float(self.default_prediction()), float(ts.offset), float(low),
                                                   float(high), nat.ptr(d_up), nat.ptr(d_ui), width,
                                                   nat.ptr(items[b0:]), nat.ptr(est[b0:]), nat.ptr(count[b0:]),
                                                   stream))
            if ev:
                ev[2].record()
            if select and on_block is not None:
                on_block(b0, nr, items, est, count)
        return items, est, count

    def _user_csr_dev(self):
        from .. import _native as nat
        ptr, idx, _ = self.trainset.user_csr()
        return nat.to_dev(ptr, np.int64), nat.to_dev(idx, np.int32)

    # -- top-N measures against held-out ratings -------------------------------------------------------
    def top_n_measures(self, testset, n=10, threshold=None):
        """Hit rate, ARHR, precision@n, recall@n and nDCG@n of this algorithm's top-n lists against the held-out rows
        ``(raw uid, raw iid, r_ui)`` of ``testset``: bit for bit ``accuracy.top_n_measures(self.get_top_n(n), testset,
        n, threshold, offset=self.trainset.offset, verbose=False)``, without building get_top_n's dict or any
        Prediction.  Only the evaluated users the trainset knows are ranked; a device-batched algorithm scores their
        lists against the relevant items on the device (sb2_top_n_hits_dev), any other one through get_top_n."""
        from ..model_selection.validation import Fold
        return self._top_n_measures(Fold(self.trainset, testset), [n], threshold)[0]

    # -- where held-out items land in the full ranking ---------------------------------------------------
    def rank_measures(self, testset, threshold=None, _block_rows=None):
        """AUC, MRR and mean percentile rank of the held-out rows ``(raw uid, raw iid, r_ui)`` of ``testset`` over each
        user's full ranking of the items they did not rate: bit for bit ``accuracy.rank_measures(self.get_top_n(
        self.trainset.n_items), testset, self.trainset, threshold, verbose=False)``, without building get_top_n's dict.
        A device-batched algorithm scores the evaluated users the trainset knows one block at a time and counts where
        their relevant items rank in each block's scores on the device (sb2_top_n_ranks_dev); nothing is selected.
        Any other algorithm goes through the definition over get_top_n for those users.  ``_block_rows`` overrides the
        number of users scored per device block (the result does not depend on it)."""
        from ..model_selection.validation import Fold
        return self._top_n_fold(Fold(self.trainset, testset), [], [], None, threshold, _block_rows, rank=True)[2]

    def _top_n_measures(self, fold, ns, threshold, _block_rows=None):
        """top_n_measures for each cutoff of ``ns`` on the testset of ``fold`` (a validation.Fold of this trainset): the
        lists are ranked once at the largest cutoff, whose first N entries are the top-N lists (the ranking is a total
        order), and the hits are counted once per cutoff."""
        return self._top_n_fold(fold, ns, [], None, threshold, _block_rows)[0]

    def _top_n_fold(self, fold, hit_ns, list_ns, sim, threshold=None, _block_rows=None, rank=False):
        """(top_n_measures at each cutoff of ``hit_ns``, top_n_list_measures at each cutoff of ``list_ns``,
        rank_measures when ``rank`` else None) on the testset of ``fold``, from one scoring pass, with a selection at
        the largest cutoff when there is one.  The list measures are taken over the evaluated users U* of
        ``threshold`` (users unknown to the trainset have no list) with no est threshold; ``sim`` (a CUDA float64
        item-item matrix, or None) gives diversity."""
        from .. import accuracy
        hit_ns = [_check_top_n(n) for n in hit_ns]
        list_ns = [_check_top_n(n) for n in list_ns]
        ts = self.trainset
        pairs = fold.test_pairs()
        iu, n_rel, rel_ptr, rel_idx = pairs.relevant(threshold, ts.n_items)
        known = iu >= 0
        top = max(hit_ns + list_ns + ([ts.n_items] if rank and not self._batched() else []), default=0)
        if not self._batched():
            lists = self.get_top_n(top, uids=[ts.to_raw_uid(u) for u in iu[known].tolist()])
            hits = [accuracy.top_n_measures({u: l_u[:n] for u, l_u in lists.items()}, fold.testset, n, threshold,
                                            ts.offset, verbose=False) for n in hit_ns]
            star = list(dict.fromkeys(u for u, r in zip(pairs._uids, pairs.r_ui.tolist())
                                      if threshold is None or r >= threshold))
            sim_h = None if sim is None else sim.cpu().numpy()
            return hits, [accuracy.top_n_list_measures(lists, ts, n, star, None, sim_h, verbose=False)
                          for n in list_ns], \
                accuracy.rank_measures(lists, fold.testset, ts, threshold, verbose=False) if rank else None
        from .. import _native as nat
        width = min(top, ts.n_items)
        n_k = int(known.sum())
        lib, stream = nat.lib(), nat.stream()
        hooks, outs = [], []
        if hit_ns:
            d_ptr, d_idx = nat.to_dev(rel_ptr, np.int64), nat.to_dev(rel_idx, np.int32)
            inv, disc, idcg = accuracy._rank_tables(min(max(hit_ns), max(width, int(n_rel.max()))))
            d_inv, d_disc = nat.to_dev(inv, np.float64), nat.to_dev(disc, np.float64)
            outs = [tuple(nat.empty_dev((max(n_k, 1),), t) for t in (np.int32, np.float64, np.float64))
                    for _ in hit_ns]

            def count_hits(b0, nr, items, est, count):
                for n, (hits, rr, dcg) in zip(hit_ns, outs):
                    nat.check(lib.sb2_top_n_hits_dev(nr, nat.ptr(items[b0:]), width, nat.ptr(count[b0:]),
                                                     min(n, width), nat.ptr(d_ptr[b0:]), nat.ptr(d_idx), len(rel_idx),
                                                     nat.ptr(d_inv), nat.ptr(d_disc), nat.ptr(hits[b0:]),
                                                     nat.ptr(rr[b0:]), nat.ptr(dcg[b0:]), stream))
            hooks.append(count_hits)
        if list_ns:
            count_lists, finish_lists = self._list_counter(list_ns, width, n_k, None, sim)
            hooks.append(count_lists)

        d_csr = self._user_csr_dev() if n_k else None
        count_ranks, finish_ranks = self._rank_counter(n_k, rel_ptr, rel_idx, d_csr) if rank else (None, None)

        def on_block(*blk):
            for hook in hooks:
                hook(*blk)

        count = None
        if n_k:
            count = self._top_n_dev(width, iu[known], _block_rows, on_block=on_block, on_scores=count_ranks,
                                    select=bool(hit_ns or list_ns), d_csr=d_csr)[2]
        res = []
        for n, out in zip(hit_ns, outs):
            hits, rr, dcg = np.zeros(len(iu), dtype=np.int64), np.zeros(len(iu)), np.zeros(len(iu))
            for host, dev in zip((hits, rr, dcg), out):
                host[known] = dev.cpu().numpy()[:n_k]
            res.append(accuracy._top_n_of_counts(hits, rr, dcg, n_rel, n, idcg, False))
        rank_res = None
        if rank:
            c, k, s = (np.zeros(len(iu), dtype=np.int64) for _ in range(3))
            f = np.full(len(iu), -1, dtype=np.int64)
            if n_k:
                for host, dev in zip((c, k, s, f), finish_ranks()):
                    host[known] = dev
            rank_res = accuracy._rank_of_counts(c, k, s, f, n_rel, False)
        return res, (finish_lists(known, count) if list_ns else []), rank_res

    def _rank_counter(self, n_rows, rel_ptr, rel_idx, d_csr):
        """(on_scores, finish) counting where the relevant items rank over one _top_n_dev pass of n_rows users:
        on_scores is the pass's score hook (sb2_top_n_ranks_dev on each block, against the relevant CSR rel_ptr /
        rel_idx of those users, with d_csr the trainset's user CSR on the device); finish() returns the (c, k, s, f)
        counts of the n_rows users as host int64 arrays."""
        from .. import _native as nat
        ts = self.trainset
        low, high = ts.rating_scale
        d_ptr, d_idx = nat.to_dev(rel_ptr, np.int64), nat.to_dev(rel_idx, np.int32)
        outs = [nat.empty_dev((max(n_rows, 1),), t) for t in (np.int32, np.int32, np.int64, np.int32)]
        lib, stream = nat.lib(), nat.stream()

        def count_ranks(b0, nr, d_rows, sc, imp):
            nat.check(lib.sb2_top_n_ranks_dev(nr, nat.ptr(d_rows), ts.n_items, nat.ptr(sc), ts.n_items, nat.ptr(imp),
                                              float(self.default_prediction()), float(ts.offset), float(low),
                                              float(high), nat.ptr(d_csr[0]), nat.ptr(d_csr[1]), nat.ptr(d_ptr[b0:]),
                                              nat.ptr(d_idx), len(rel_idx), *(nat.ptr(o[b0:]) for o in outs), stream))

        def finish():
            return [o.cpu().numpy()[:n_rows].astype(np.int64) for o in outs]

        return count_ranks, finish

    # -- coverage, novelty and diversity of the top-N lists --------------------------------------------
    def top_n_list_measures(self, n=10, uids=None, threshold=None, sim=None, _block_rows=None):
        """User coverage, catalog coverage, novelty and (with ``sim``) diversity of this algorithm's top-n lists for the
        users ``uids`` (raw ids; default every user): bit for bit ``accuracy.top_n_list_measures(self.get_top_n(n,
        uids), self.trainset, n, uids, threshold, sim_array, verbose=False)``, without building get_top_n's dict.

        An unknown uid raises ValueError, as get_top_n does.  ``sim`` is an (n_items, n_items) array indexed by this
        trainset's inner item ids, uploaded once, or a fitted item-based k-NN model whose trainset is this one, whose
        device matrix is read in place; a streamed or user-based model, or one fitted on another trainset, raises
        ValueError.  A device-batched algorithm counts the lists on the device (sb2_top_n_lists_dev) when ``threshold``
        is None or a real number float64 holds exactly; otherwise the definition runs over get_top_n."""
        from .. import accuracy
        n = _check_top_n(n)
        ts = self.trainset
        if uids is None:
            raw_u, users = None, np.arange(ts.n_users, dtype=np.int32)
        else:
            raw_u = list(dict.fromkeys(uids))
            users = np.array([ts.to_inner_uid(x) for x in raw_u], dtype=np.int32)
        if not len(users):
            raise ValueError("top-N list measures need at least one user")
        model = self._list_sim_model(sim)
        if not self._batched() or not (threshold is None or accuracy._exact_reals([threshold])):
            arr = model.sim if model is not None else sim
            return accuracy.top_n_list_measures(self.get_top_n(n, raw_u), ts, n, raw_u, threshold, arr, verbose=False)
        from .. import _native as nat
        if model is not None:
            d_sim = model._sim_device()
        else:
            d_sim = None if sim is None else nat.to_dev(accuracy._check_list_sim(sim, ts.n_items), np.float64)
        width = min(n, ts.n_items)
        count_lists, finish_lists = self._list_counter([n], width, len(users), threshold, d_sim)
        count = self._top_n_dev(width, users, _block_rows, on_block=count_lists)[2]
        return finish_lists(np.ones(len(users), dtype=bool), count)[0]

    def _list_sim_model(self, sim):
        """``sim`` when it is a k-NN model top_n_list_measures can read the matrix of; None for an array or None."""
        from .knns import SymmetricAlgo
        if not isinstance(sim, SymmetricAlgo):
            return None
        if sim.sim_options["user_based"]:
            raise ValueError("sim must be an item-based k-NN model (user_based=False)")
        if getattr(sim, "trainset", None) is not self.trainset:
            raise ValueError("sim must be a k-NN model fitted on this algorithm's trainset")
        if sim._streamed:
            raise ValueError("sim is a streamed k-NN model, which keeps no similarity matrix; pass the matrix instead")
        return sim

    def _list_counter(self, ns, width, n_rows, threshold, sim):
        """(on_block, finish) computing top_n_list_measures at each cutoff of ``ns`` over the rows of one _top_n_dev
        pass of n_rows users at ``width``: on_block is the pass's block hook (sb2_top_n_lists_dev once per cutoff);
        finish(known, count) returns the results for the users U, where ``known`` (bool per user of U) marks the users
        that had a row, in order, and ``count`` is the pass's count array (the others have no list)."""
        from .. import _native as nat
        from .. import accuracy
        torch = nat.torch_cuda()
        ts = self.trainset
        d_info = nat.to_dev(accuracy._novelty_table(ts), np.float64)
        rows = max(n_rows, 1)
        outs = [(nat.empty_dev((rows,), np.int32), nat.empty_dev((rows,), np.float64),
                 nat.empty_dev((rows,), np.float64) if sim is not None else None,
                 torch.zeros(ts.n_items, dtype=torch.uint8, device=nat.device())) for _ in ns]
        has_t = threshold is not None
        lib, stream = nat.lib(), nat.stream()

        def count_lists(b0, nr, items, est, count):
            for n, (cov, nov, ils, seen) in zip(ns, outs):
                nat.check(lib.sb2_top_n_lists_dev(nr, nat.ptr(items[b0:]), width, nat.ptr(est[b0:]),
                                                  nat.ptr(count[b0:]), min(n, width), int(has_t),
                                                  float(threshold) if has_t else 0.0, ts.n_items, nat.ptr(d_info),
                                                  nat.ptr(sim), nat.ptr(cov[b0:]), nat.ptr(nov[b0:]),
                                                  None if ils is None else nat.ptr(ils[b0:]), nat.ptr(seen), stream))

        def finish(known, count):
            c_u = np.zeros(len(known), dtype=np.int64)
            if n_rows:
                c_u[known] = count.cpu().numpy()[:n_rows]
            res = []
            for n, (cov, nov, ils, seen) in zip(ns, outs):
                h_cov, h_nov, h_ils = np.zeros(len(known), dtype=bool), np.zeros(len(known)), np.zeros(len(known))
                if n_rows:
                    h_cov[known] = cov.cpu().numpy()[:n_rows] != 0
                    h_nov[known] = nov.cpu().numpy()[:n_rows]
                    if ils is not None:
                        h_ils[known] = ils.cpu().numpy()[:n_rows]
                res.append(accuracy._top_n_lists_of_counts(h_cov, h_nov, None if ils is None else h_ils,
                                                           np.minimum(c_u, n), int(seen.sum()), ts.n_items, n, False))
            return res

        return count_lists, finish

    def _top_n_scorer(self):
        """Device arrays for sb2_mf_score_block_dev (dict: f, biased, pu, qi, bu, bi[, yj, up, ui]), or None when
        the algorithm is scored pair by pair through ``_estimate_dev``."""
        return None

    def _top_n_by_test(self, width, users):
        """top_n_inner through ``test()``: for algorithms whose estimate() is not the device batch."""
        ts = self.trainset
        ptr, idx, _ = ts.user_csr()
        fill = ts.global_mean
        items = np.full((len(users), width), -1, dtype=np.int32)
        est = np.full((len(users), width), np.nan)
        count = np.zeros(len(users), dtype=np.int32)
        all_i = np.arange(ts.n_items)
        for k, u in enumerate(users.tolist()):
            cand = np.setdiff1d(all_i, idx[ptr[u]:ptr[u + 1]])
            if not len(cand):
                continue
            ru = ts.to_raw_uid(u)
            preds = self.test([(ru, ts.to_raw_iid(i), fill) for i in cand.tolist()])
            e = np.array([p.est for p in preds], dtype=np.float64)
            order = rank_top_n(e, cand)[:width]
            c = len(order)
            items[k, :c], est[k, :c], count[k] = cand[order], e[order], c
        return items, est, count

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
