"""rmse / mse / mae / fcp over a list of Prediction tuples (reference: surprise/accuracy.py:22-143), the FAQ's
precision_recall_at_k, top_n_measures: hit rate, ARHR, precision@N, recall@N and nDCG@N of get_top_n output against
held-out ratings, top_n_list_measures: user and catalog coverage, novelty and diversity of the lists themselves, and
rank_measures: AUC, MRR and mean percentile rank of held-out items over each user's full candidate ranking.

fcp and precision_recall_at_k reduce to integer counts per user.  Where a CUDA device is usable and every r_ui and est
is a real number that float64 holds exactly, the counts come from the device (csrc/rank_metrics.cu, DESIGN.md section
3.7); otherwise from the Python loops below, which are the metrics' definition (and what the tests compare against).
The arithmetic on the counts runs on the host either way, so both routes return the same values.
"""
import re
from collections import defaultdict
from operator import index, itemgetter

import numpy as np

__all__ = ["rmse", "mse", "mae", "fcp", "precision_recall_at_k", "top_n_measures", "top_n_list_measures",
           "rank_measures"]


def _need(predictions):
    if not predictions:
        raise ValueError("Prediction list is empty.")


def rmse(predictions, verbose=True):
    out = np.sqrt(mse(predictions, verbose=False))
    if verbose:
        print("RMSE: {0:1.4f}".format(out))
    return out


def mse(predictions, verbose=True):
    _need(predictions)
    out = np.mean([float((true_r - est) ** 2) for (_, _, true_r, est, _) in predictions])
    if verbose:
        print("MSE: {0:1.4f}".format(out))
    return out


def mae(predictions, verbose=True):
    _need(predictions)
    out = np.mean([float(abs(true_r - est)) for (_, _, true_r, est, _) in predictions])
    if verbose:
        print("MAE:  {0:1.4f}".format(out))
    return out


def fcp(predictions, verbose=True):
    _need(predictions)
    return _fcp_of_counts(*_fcp_counts(predictions), verbose)


def _fcp_of_counts(nc, nd, verbose):
    c_mean = np.mean(list(nc.values())) if nc else 0
    d_mean = np.mean(list(nd.values())) if nd else 0
    try:
        out = c_mean / (c_mean + d_mean)
    except ZeroDivisionError:
        raise ValueError("cannot compute fcp on this list of prediction. Does every user have at least two "
                         "predictions?")
    if verbose:
        print("FCP:  {0:1.4f}".format(out))
    return out


def precision_recall_at_k(predictions, k=10, threshold=3.5):
    """Precision and recall at k per user, as the Surprise FAQ's recipe computes them: each user's predictions sorted
    by est descending (a stable sort), the first k of them recommended where est >= threshold, relevant where
    r_ui >= threshold.  Returns (precisions, recalls), two dicts keyed by uid in first-appearance order.

    precisions[uid] = n_rel_and_rec_k / n_rec_k and recalls[uid] = n_rel_and_rec_k / n_rel, each the int 0 where its
    denominator is 0 (the current FAQ; releases before it gave 1).  k follows list slicing: None means all, a negative
    k counts from the end, and a k that is not an index raises TypeError (only when there is at least one user).

    The counts come from the device when it is usable and threshold and every r_ui and est is a float, a bool, an int
    with |x| <= 2**53 or a numpy float64, bool or integer scalar.  A user with a NaN est (for which the stable sort has
    no defined order) gets the recipe itself, on the host; so does a user with numpy scalars when threshold is a Python
    number, because which of the recipe's sums become numpy integers then depends on which entries are in the top k.
    With a numpy threshold every compare is a numpy bool, so every non-empty sum is a numpy integer."""
    if _device_usable() and _exact_reals([threshold]):
        predictions = predictions if isinstance(predictions, (list, tuple)) else list(predictions)
        cols = _exact_columns(predictions)
        if cols is not None:
            return _precision_recall_dev(*cols, k, threshold)
    user_est_true = defaultdict(list)
    for uid, _, true_r, est, _ in predictions:
        user_est_true[uid].append((est, true_r))
    precisions = dict()
    recalls = dict()
    for uid, user_ratings in user_est_true.items():
        precisions[uid], recalls[uid] = _precision_recall_user(user_ratings, k, threshold)
    return precisions, recalls


def _precision_recall_user(user_ratings, k, threshold):
    user_ratings.sort(key=lambda x: x[0], reverse=True)
    n_rel = sum((true_r >= threshold) for (_, true_r) in user_ratings)
    n_rec_k = sum((est >= threshold) for (est, _) in user_ratings[:k])
    n_rel_and_rec_k = sum(((true_r >= threshold) and (est >= threshold)) for (est, true_r) in user_ratings[:k])
    return (n_rel_and_rec_k / n_rec_k if n_rec_k != 0 else 0,
            n_rel_and_rec_k / n_rel if n_rel != 0 else 0)


def _fcp_counts(predictions):
    """nc, nd: {uid: count} in first-appearance order."""
    if _device_usable():
        predictions = predictions if isinstance(predictions, (list, tuple)) else list(predictions)
        cols = _exact_columns(predictions)
        if cols is not None:
            return _fcp_counts_dev(*cols)
    per_user = defaultdict(list)
    for u0, _, r0, est, _ in predictions:
        per_user[u0].append((est, r0))
    nc, nd = {}, {}
    for u0, prefs in per_user.items():
        c = d = 0
        for esi, ri in prefs:
            for esj, rj in prefs:
                if esi > esj and ri > rj:
                    c += 1
                if esi >= esj and ri < rj:
                    d += 1
        nc[u0], nd[u0] = c, d
    return nc, nd


def top_n_measures(top_n, testset, n, threshold=None, offset=0, verbose=True):
    """Top-N measures of ``top_n`` (get_top_n output, ``{raw uid: [(raw iid, est), ...]}``) against the held-out rows
    ``(raw uid, raw iid, r_ui)`` of ``testset``, as a dict of floats with keys hr, arhr, precision, recall, ndcg.

    This plain-Python function is what the measures mean: AlgoBase.top_n_measures computes them on the device and the
    tests compare it against this function.

    * A row is relevant when ``threshold`` is None or ``r_ui - offset >= threshold`` (``r_ui - offset`` is the value
      ``test()`` reports: a float64 subtraction, then a Python compare).
    * The evaluated users U* are the uids with at least one relevant row, in first-appearance order, equal uids merged
      as dict keys merge them.  No such user raises ValueError.
    * R_u is the set of u's relevant raw iids (duplicates collapse; items the trainset does not know count).  L_u is
      the first n raw iids of ``top_n.get(u, [])``, and H_u the positions p (0-based, ascending) with L_u[p] in R_u.
      A user absent from ``top_n`` (unknown to the trainset, or who rated every item) has no hits but is evaluated.
    * With the host tables inv[p] = 1.0 / (p + 1), disc[p] = 1.0 / np.log2(p + 2) and idcg[m] the left-to-right sum of
      disc[:m]: hits_u = |H_u|, rr_u and dcg_u the left-to-right sums from 0.0 of inv[p] and disc[p] over H_u,
      prec_u = hits_u / n, rec_u = hits_u / |R_u|, ndcg_u = dcg_u / idcg[min(|R_u|, n)].
    * hr = sum(hits_u) / sum(|R_u|), arhr = float(np.sum(rr)) / sum(|R_u|); precision, recall and ndcg are
      float(np.mean(...)) of the per-user values in U* order.

    With one held-out rating per user (LeaveOneOut) and threshold None, hr is the leave-one-out hit rate and arhr the
    average reciprocal hit rank.  ``n`` must be an int >= 1."""
    from .prediction_algorithms.algo_base import _check_top_n
    n = _check_top_n(n)
    relevant = {}
    for uid, iid, r_ui in testset:
        if threshold is None or float(r_ui) - offset >= threshold:
            relevant.setdefault(uid, set()).add(iid)
    if not relevant:
        raise ValueError("top-N measures need at least one relevant rating in the testset")
    lists = [[iid for iid, _ in top_n.get(u, [])][:n] for u in relevant]
    inv, disc, idcg = _rank_tables(min(n, max(max(map(len, lists)), max(map(len, relevant.values())))))
    inv, disc = inv.tolist(), disc.tolist()
    hits, rr, dcg = [], [], []
    for r_u, l_u in zip(relevant.values(), lists):
        h, a, d = 0, 0.0, 0.0
        for p, iid in enumerate(l_u):
            if iid in r_u:
                h += 1
                a += inv[p]
                d += disc[p]
        hits.append(h)
        rr.append(a)
        dcg.append(d)
    return _top_n_of_counts(hits, rr, dcg, [len(r_u) for r_u in relevant.values()], n, idcg, verbose)


def _rank_tables(m):
    """inv[p] = 1.0 / (p + 1) and disc[p] = 1.0 / np.log2(p + 2) for p < m (float64 arrays; an entry does not depend
    on m), and idcg[k] = the left-to-right sum of disc[:k] for k <= m."""
    p = np.arange(m, dtype=np.float64)
    inv, disc = 1.0 / (p + 1), 1.0 / np.log2(p + 2)
    idcg = [0.0]
    for d in disc.tolist():
        idcg.append(idcg[-1] + d)
    return inv, disc, np.array(idcg)


_TOP_N_LABELS = {"hr": "HR", "arhr": "ARHR", "precision": "Precision", "recall": "Recall", "ndcg": "nDCG"}


def _top_n_of_counts(hits, rr, dcg, n_rel, n, idcg, verbose):
    """top_n_measures' result from the per-user hits, rr, dcg and |R_u| in U* order (both routes end here)."""
    hits, n_rel = np.asarray(hits, dtype=np.int64), np.asarray(n_rel, dtype=np.int64)
    rr, dcg = np.asarray(rr, dtype=np.float64), np.asarray(dcg, dtype=np.float64)
    total = int(n_rel.sum())
    out = {"hr": int(hits.sum()) / total,
           "arhr": float(np.sum(rr)) / total,
           "precision": float(np.mean(hits / n)),
           "recall": float(np.mean(hits / n_rel)),
           "ndcg": float(np.mean(dcg / idcg[np.minimum(n_rel, n)]))}
    if verbose:
        for key, label in _TOP_N_LABELS.items():
            print("{0}@{1}:  {2:1.4f}".format(label, n, out[key]))
    return out


def _top_n_measure(name):
    """(key, N) for a measure name key@N with key in hr, arhr, precision, recall, ndcg (any case) and N an int >= 1;
    None for any other name.  A top-N key with a malformed N raises ValueError."""
    key, at, num = name.lower().partition("@")
    if not at or key not in _TOP_N_LABELS:
        return None
    if not re.fullmatch("[0-9]+", num) or int(num) < 1:
        raise ValueError("%s: N in %s@N must be an int >= 1" % (name, key))
    return key, int(num)


def top_n_list_measures(top_n, trainset, n, uids=None, threshold=None, sim=None, verbose=True):
    """Coverage, novelty and diversity of ``top_n`` (get_top_n output, ``{raw uid: [(raw iid, est), ...]}``) over the
    users ``uids`` of ``trainset``, as a dict of floats with keys user_coverage, catalog_coverage and novelty, plus
    diversity when ``sim`` is given.

    This plain-Python function is what the measures mean: AlgoBase.top_n_list_measures computes them on the device and
    the tests compare it against this function.

    * U is the distinct raw uids of ``uids`` in first-appearance order (equal uids merged as dict keys merge them), or
      every trainset user in inner-id order when ``uids`` is None.  An empty U raises ValueError.  L_u is the first n
      entries of ``top_n.get(u, [])`` and c_u = |L_u|: a uid absent from ``top_n`` (unknown to the trainset, or who
      rated every item) has c_u = 0.  ``n`` must be an int >= 1.
    * user_coverage = |{u in U : some entry of L_u has est >= threshold}| / |U|, a Python compare (a NaN est never
      counts); with threshold None, a user counts when c_u > 0.
    * catalog_coverage = |union over U of the iids of L_u| / trainset.n_items.
    * novelty is the mean self-information of the recommended entries.  With the host table
      ``info = np.log2(trainset.n_users / cnt)``, cnt the int64 np.diff of the item CSR's ptr (len(ir[i]); duplicate
      ratings count), nov_u is the left-to-right sum from 0.0 of info[inner(iid)] over L_u, and
      novelty = float(np.sum(nov)) over U in order, divided by sum(c_u); nan when sum(c_u) = 0.
    * diversity = 1 - intra-list similarity, only when ``sim`` is given: a float64 (n_items, n_items) array indexed
      by this trainset's inner item ids (any other shape raises ValueError).  ils_u is the sum from 0.0 of
      float(sim[inner(L_u[p]), inner(L_u[q])]) over p < q, p ascending and q ascending inside it, and
      diversity = 1.0 - float(np.sum(ils)) / sum(c_u (c_u - 1) / 2); nan when there are no pairs.

    With ``verbose``, one line per key is printed."""
    from .prediction_algorithms.algo_base import _check_top_n
    n = _check_top_n(n)
    if uids is None:
        users = [trainset.to_raw_uid(u) for u in range(trainset.n_users)]
    else:
        users = list(dict.fromkeys(uids))
    if not users:
        raise ValueError("top-N list measures need at least one user")
    if sim is not None:
        sim = _check_list_sim(sim, trainset.n_items)
    info = _novelty_table(trainset).tolist()
    covered, nov, ils, count, seen = [], [], [], [], set()
    for u in users:
        l_u = top_n.get(u, [])[:n]
        inner = [trainset.to_inner_iid(iid) for iid, _ in l_u]
        covered.append(len(l_u) > 0 if threshold is None else any(est >= threshold for _, est in l_u))
        count.append(len(l_u))
        seen.update(inner)
        s = 0.0
        for i in inner:
            s += info[i]
        nov.append(s)
        if sim is not None:
            t = 0.0
            for p in range(len(inner)):
                for q in range(p + 1, len(inner)):
                    t += float(sim[inner[p], inner[q]])
            ils.append(t)
    return _top_n_lists_of_counts(covered, nov, ils if sim is not None else None, count, len(seen), trainset.n_items,
                                  n, verbose)


def _check_list_sim(sim, n_items):
    sim = np.asarray(sim, dtype=np.float64)
    if sim.shape != (n_items, n_items):
        raise ValueError("sim must be an (n_items, n_items) = (%d, %d) array indexed by inner item ids (got shape %s)"
                         % (n_items, n_items, sim.shape))
    return sim


def _novelty_table(trainset):
    """info[i] = np.log2(n_users / cnt[i]) (float64), cnt the number of ratings of inner item i (duplicates count)."""
    cnt = np.diff(trainset.item_csr()[0]).astype(np.int64)
    with np.errstate(divide="ignore"):
        return np.log2(trainset.n_users / cnt)


_LIST_LABELS = {"user_coverage": "User coverage", "catalog_coverage": "Catalog coverage", "novelty": "Novelty",
                "diversity": "Diversity"}


def _top_n_lists_of_counts(covered, nov, ils, count, n_seen, n_items, n, verbose):
    """top_n_list_measures' result from the per-user covered flags, nov, ils (None without sim) and c_u in U order and
    the number of distinct recommended items (both routes end here)."""
    count = np.asarray(count, dtype=np.int64)
    total = int(count.sum())
    pairs = int((count * (count - 1) // 2).sum())
    out = {"user_coverage": int(np.count_nonzero(covered)) / len(count),
           "catalog_coverage": n_seen / n_items,
           "novelty": float(np.sum(np.asarray(nov, dtype=np.float64))) / total if total else float("nan")}
    if ils is not None:
        ils_sum = float(np.sum(np.asarray(ils, dtype=np.float64)))
        out["diversity"] = 1.0 - ils_sum / pairs if pairs else float("nan")
    if verbose:
        for key in out:
            print("{0}@{1}:  {2:1.4f}".format(_LIST_LABELS[key], n, out[key]))
    return out


def _top_n_list_measure(name):
    """(key, N) for a measure name key@N with key in user_coverage, catalog_coverage, novelty, diversity (any case)
    and N an int >= 1; None for any other name.  A list-measure key with a malformed N raises ValueError."""
    key, at, num = name.lower().partition("@")
    if not at or key not in _LIST_LABELS:
        return None
    if not re.fullmatch("[0-9]+", num) or int(num) < 1:
        raise ValueError("%s: N in %s@N must be an int >= 1" % (name, key))
    return key, int(num)


def rank_measures(top_n, testset, trainset, threshold=None, verbose=True):
    """AUC, MRR and mean percentile rank (MPR) of the held-out rows ``(raw uid, raw iid, r_ui)`` of ``testset`` over
    each user's full ranking ``top_n`` (get_top_n output at n = trainset.n_items), as a dict of floats with keys auc,
    mrr and mpr.  Higher AUC and MRR are better; lower MPR is better.

    This plain-Python function is what the measures mean: AlgoBase.rank_measures computes them on the device and the
    tests compare it against this function.

    * Users and relevance are those of top_n_measures: a row is relevant when ``threshold`` is None or
      ``float(r_ui) - trainset.offset >= threshold``; U* is the uids with a relevant row, in first-appearance order,
      equal uids merged as dict keys merge them; R_u is u's set of relevant raw iids (unknown items count) and
      n_rel_u = |R_u|.  No relevant row raises ValueError.
    * F_u = ``top_n.get(u, [])`` must be u's complete ranking: every item u did not rate in ``trainset``, in get_top_n
      order, so len(F_u) = n_items - |distinct items of ur[u]| for a user the trainset knows and 0 for any other;
      otherwise ValueError (pass ``get_top_n(n=trainset.n_items)``).
    * c_u = len(F_u); K_u is the ascending list of 0-based positions p with F_u[p][0] in R_u, k_u = len(K_u),
      s_u = sum(K_u) and f_u = K_u[0] when k_u > 0.  A relevant item not in F_u (unknown to the trainset, or rated by
      u in it) is unranked.
    * Per user, in integers until the divisions (each a float64 division): rr_u = 1.0 / (f_u + 1) if k_u else 0.0.
      With neg_u = c_u - k_u negatives, when neg_u > 0, correct_u = k_u (c_u - 1) - s_u - k_u (k_u - 1) // 2 is the
      number of (relevant, negative) pairs ordered correctly (an unranked relevant item makes none) and
      auc_u = correct_u / (n_rel_u neg_u); a user with neg_u = 0 (an unknown user, or every candidate relevant) has no
      AUC.  mpr_u = (s_u / (c_u - 1) if c_u > 1 else 0.0) + (n_rel_u - k_u): an unranked relevant item counts as
      percentile 1.0, the bottom.
    * mrr = float(np.mean(rr)) over U*; auc = float(np.mean(auc_u)) over the users that have one, nan when none does;
      mpr = float(np.sum(mpr_u)) over U* divided by sum(n_rel_u).

    The AUC is taken per user and then averaged over users (what some libraries call GAUC), never pooled over the
    pairs of all users: the estimates of different users are not on a common scale.  With ``verbose``, one line per
    measure is printed."""
    relevant = {}
    for uid, iid, r_ui in testset:
        if threshold is None or float(r_ui) - trainset.offset >= threshold:
            relevant.setdefault(uid, set()).add(iid)
    if not relevant:
        raise ValueError("rank measures need at least one relevant rating in the testset")
    users = list(relevant)
    inner = trainset.to_inner_uids(users)
    ptr, idx, _ = trainset.user_csr()
    c, k, s, f = [], [], [], []
    for u, iu, r_u in zip(users, inner.tolist(), relevant.values()):
        f_u = top_n.get(u, [])
        want = trainset.n_items - len(np.unique(idx[ptr[iu]:ptr[iu + 1]])) if iu >= 0 else 0
        if len(f_u) != want:
            raise ValueError("rank measures need each user's complete ranking, %d items for user %r (got %d): pass "
                             "get_top_n(n=trainset.n_items)" % (want, u, len(f_u)))
        k_u = [p for p, (iid, _) in enumerate(f_u) if iid in r_u]
        c.append(len(f_u))
        k.append(len(k_u))
        s.append(sum(k_u))
        f.append(k_u[0] if k_u else -1)
    return _rank_of_counts(c, k, s, f, [len(r_u) for r_u in relevant.values()], verbose)


_RANK_LABELS = {"auc": "AUC", "mrr": "MRR", "mpr": "MPR"}


def _rank_of_counts(c, k, s, f, n_rel, verbose):
    """rank_measures' result from the per-user c_u, k_u, s_u, f_u (-1 when k_u = 0) and n_rel_u in U* order (both
    routes end here)."""
    c, k, s, f, n_rel = (np.asarray(x, dtype=np.int64) for x in (c, k, s, f, n_rel))
    neg = c - k
    has = neg > 0
    correct = k * (c - 1) - s - k * (k - 1) // 2
    auc_u = correct[has] / (n_rel[has] * neg[has])
    with np.errstate(divide="ignore", invalid="ignore"):    # the branches np.where drops
        rr = np.where(k > 0, 1.0 / (f + 1), 0.0)
        pct = np.where(c > 1, s / (c - 1), 0.0)
    out = {"auc": float(np.mean(auc_u)) if len(auc_u) else float("nan"),
           "mrr": float(np.mean(rr)),
           "mpr": float(np.sum(pct + (n_rel - k))) / int(n_rel.sum())}
    if verbose:
        for key, label in _RANK_LABELS.items():
            print("{0}:  {1:1.4f}".format(label, out[key]))
    return out


def _rank_measure(name):
    """The key of a rank measure name (auc, mrr or mpr, any case), or None for any other name."""
    key = name.lower()
    return key if key in _RANK_LABELS else None


# -- device route ----------------------------------------------------------------------------------------------------
_EXACT_INT = 2 ** 53


def _device_usable():
    """A CUDA device the library's sm_100a kernels run on (compute capability 10.0)."""
    import torch
    return torch.cuda.is_available() and torch.cuda.get_device_capability() == (10, 0)


def _exact_reals(values):
    """True when every value is a float, a bool, an int with |x| <= 2**53, or a numpy float64, bool or integer scalar
    with |x| <= 2**53: float64 holds these exactly, and Python and numpy compare them with each other exactly.  (numpy
    compares a float32 with a Python float in float32, so float32 and other float widths are left out.)"""
    for t in set(map(type, values)):
        if t is float or t is bool or t is np.float64 or t is np.bool_:
            continue
        if not (t is int or issubclass(t, np.integer)):
            return False
        if not all(-_EXACT_INT <= int(x) <= _EXACT_INT for x in values if type(x) is t):
            return False
    return True


def _exact_columns(predictions):
    """(keys, code, r_ui, est, has_numpy), or None when the Python route must run.  The columns are read as
    `for uid, _, r_ui, est, _ in predictions` reads them (an item that does not unpack raises the same exception);
    keys are the distinct uids as defaultdict(list) keeps them (first appearance, equal uids merged into the first), code
    the position of each prediction's uid in keys."""
    if not predictions:
        return None
    kinds = set(map(type, predictions))
    if all(t is list or (issubclass(t, tuple) and t.__iter__ is tuple.__iter__ and t.__getitem__ is tuple.__getitem__)
           for t in kinds) and set(map(len, predictions)) == {5}:
        uid, r_ui, est = (list(map(itemgetter(c), predictions)) for c in (0, 2, 3))
    else:
        uid, r_ui, est = map(list, zip(*[(u, r, e) for u, _, r, e, _ in predictions]))
    if not (_exact_reals(r_ui) and _exact_reals(est)):
        return None
    has_numpy = any(issubclass(t, np.generic) for t in set(map(type, r_ui)) | set(map(type, est)))
    codes = {}
    setd = codes.setdefault
    code = np.array([setd(u, len(codes)) for u in uid], dtype=np.int64)
    return list(codes), code, r_ui, est, has_numpy


def _segments(code, n_seg, r_ui, est):
    """Device segment CSR: seg_ptr (int64) and r, est (float64) grouped by code, prediction order kept in a group."""
    from . import _native as nat
    torch = nat.torch_cuda()
    d_code = nat.to_dev(code, np.int64)
    order = torch.sort(d_code, stable=True).indices
    seg_ptr = torch.zeros(n_seg + 1, dtype=torch.int64, device=d_code.device)
    seg_ptr[1:] = torch.cumsum(torch.bincount(d_code, minlength=n_seg), 0)
    r = nat.to_dev(np.array(r_ui, dtype=np.float64), np.float64)[order]
    e = nat.to_dev(np.array(est, dtype=np.float64), np.float64)[order]
    return seg_ptr, r, e


def _fcp_counts_dev(keys, code, r_ui, est, has_numpy):
    from . import _native as nat
    seg_ptr, r, e = _segments(code, len(keys), r_ui, est)
    counts = nat.empty_dev((len(keys), 2), np.int64)
    nat.check(nat.lib().sb2_fcp_counts_dev(len(keys), len(code), nat.ptr(seg_ptr), nat.ptr(r), nat.ptr(e),
                                           nat.ptr(counts), nat.stream()))
    nc, nd = counts.cpu().numpy().T.tolist()
    return dict(zip(keys, nc)), dict(zip(keys, nd))


def _precision_recall_dev(keys, code, r_ui, est, has_numpy, k, threshold):
    from . import _native as nat
    [][:k]                                      # a k that is not an index raises here, as the recipe's slice does
    n_seg = len(keys)
    m = np.bincount(code, minlength=n_seg)
    if k is None:
        k_eff = m
    else:
        kk = max(min(index(k), 1 << 62), -(1 << 62))
        k_eff = np.minimum(m, kk) if kk >= 0 else np.maximum(m + kk, 0)
    seg_ptr, r, e = _segments(code, n_seg, r_ui, est)
    d_k_eff = nat.to_dev(k_eff, np.int64)
    counts = nat.empty_dev((n_seg, 3), np.int64)
    nat.check(nat.lib().sb2_precision_at_k_counts_dev(n_seg, len(code), nat.ptr(seg_ptr), nat.ptr(r), nat.ptr(e),
                                                      nat.ptr(d_k_eff), float(threshold), nat.ptr(counts),
                                                      nat.stream()))
    n_rel, n_rec_k, n_rel_and_rec_k = counts.cpu().numpy().T.tolist()
    numpy_threshold = isinstance(threshold, np.generic)
    if numpy_threshold:
        # the recipe's sums over numpy bools: a numpy integer, or the int 0 when the top k is empty
        num = type(sum([threshold >= threshold]))
        top = k_eff.tolist()
        n_rel = [num(a) for a in n_rel]
        n_rec_k = [num(b) if t else 0 for b, t in zip(n_rec_k, top)]
        n_rel_and_rec_k = [num(c) if t else 0 for c, t in zip(n_rel_and_rec_k, top)]
    precisions = dict()
    recalls = dict()
    for uid, a, b, c in zip(keys, n_rel, n_rec_k, n_rel_and_rec_k):
        precisions[uid] = c / b if b != 0 else 0
        recalls[uid] = c / a if a != 0 else 0
    # users the recipe itself must run for: a NaN est, or numpy scalars compared with a Python threshold
    on_host_rows = np.isnan(np.array(est, dtype=np.float64))
    if has_numpy and not numpy_threshold:
        on_host_rows |= np.fromiter((isinstance(x, np.generic) or isinstance(y, np.generic)
                                     for x, y in zip(r_ui, est)), dtype=bool, count=len(code))
    if on_host_rows.any():
        rows = np.nonzero(np.isin(code, np.unique(code[on_host_rows])))[0]
        user_est_true = defaultdict(list)
        for j in rows.tolist():
            user_est_true[int(code[j])].append((est[j], r_ui[j]))
        for u, user_ratings in user_est_true.items():
            precisions[keys[u]], recalls[keys[u]] = _precision_recall_user(user_ratings, k, threshold)
    return precisions, recalls


# -- measures of predictions held in arrays (model_selection's array route) ------------------------------------------
ARRAY_MEASURES = ("rmse", "mse", "mae", "fcp")


def _of_arrays(measure, r_ui, est, users):
    """``measure(predictions, verbose=False)`` with the same bits, for predictions given as float64 arrays r_ui and est
    (measure one of ARRAY_MEASURES).  ``users()`` returns (code, n_users): each prediction's user numbered in first
    appearance order, equal uids merged, as fcp groups them; it is only called for fcp.

    The squares are Python's ``d ** 2``, which calls libm's pow as the tuple route does: ``d * d`` and np.square
    round differently from glibc's pow for some d.  The sums are np.mean's pairwise sum over the same sequence."""
    if not len(r_ui):
        _need(())
    d = r_ui - est
    if measure == "mae":
        return np.mean(np.abs(d))
    if measure in ("mse", "rmse"):
        out = np.mean([x ** 2 for x in d.tolist()])
        return out if measure == "mse" else np.sqrt(out)
    code, n_users = users()
    if _device_usable():
        nc, nd = _fcp_counts_dev(range(n_users), code, r_ui, est, False)
    else:
        n = len(code)
        nc, nd = _fcp_counts(list(zip(code.tolist(), [None] * n, r_ui.tolist(), est.tolist(), [None] * n)))
    return _fcp_of_counts(nc, nd, False)
