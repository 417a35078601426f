"""The oracle's k-NN estimate for user-based pairs at shapes where no dense similarity matrix fits anywhere: the
entries each pair reads come from orc_similarity_pairs, and the k-NN step of orc_knn_estimate is restated over them.
Shared by tests/test_gpu_knn_stream.py and tools/bench_knn_stream.py."""
import numpy as np

import oracle


def knn_restated(x, y, sims_of, y_ptr, x_idx, r, k, mode, mu=0.0, bx=None, by=None):
    """orc_knn_estimate's k-NN step (mode 0: KNNBasic, 1: KNNBaseline with x = user) over the similarities each pair
    reads (sims_of[p] = sim[x[p], x_idx[y_ptr[y[p]]:y_ptr[y[p] + 1]]]): descending by similarity (NaN last), ties in
    list order, the first k; the positive similarities summed in that order.  Returns (est, actual_k); est of
    KNNBasic is 0 where the estimate is impossible."""
    est = np.empty(len(x))
    ak = np.full(len(x), -1, dtype=np.int32)
    for p in range(len(x)):
        e = 0.0
        if mode == 1:
            e = mu
            if x[p] >= 0:
                e += bx[x[p]]
            if y[p] >= 0:
                e += by[y[p]]
        if x[p] < 0 or y[p] < 0:
            est[p] = e
            continue
        b = y_ptr[y[p]]
        s = sims_of[p]
        key = np.where(np.isnan(s), -np.inf, s)
        top = np.lexsort((np.arange(len(s)), -key))[:k]
        sum_sim = sum_r = 0.0
        n = 0
        for a in top.tolist():
            sa = float(s[a])
            if sa > 0:
                sum_sim += sa
                rr = float(r[b + a])
                if mode == 1:
                    sum_r += sa * (rr - (mu + bx[x_idx[b + a]] + by[y[p]]))
                else:
                    sum_r += sa * rr
                n += 1
        ak[p] = n
        if mode == 1:
            if n > 0:
                e += sum_r / sum_sim
        elif n > 0:
            e = sum_r / sum_sim
        est[p] = e
    return est, ak


def user_based(kind, mode, ts, u, i, r, pu, pi, k, bu=None, bi=None):
    """(est, actual_k) of the user-based pairs (pu[p], pi[p]) (inner ids, < 0 unknown) of a trainset built from the
    COO (u, i, r): similarities of kind ``kind`` with min_support 1 (shrinkage 100, baselines bu / bi for
    pearson_baseline)."""
    y_ptr, x_idx, r_y = ts.item_csr()
    o = np.lexsort((i, u))
    x_ptr = np.concatenate(([0], np.cumsum(np.bincount(u, minlength=ts.n_users)))).astype(np.int64)
    known = (pu >= 0) & (pi >= 0)
    lens = np.where(known, y_ptr[np.maximum(pi, 0) + 1] - y_ptr[np.maximum(pi, 0)], 0)
    qi = np.repeat(np.where(known, pu, 0), lens).astype(np.int32)
    qj = np.concatenate([x_idx[y_ptr[y]:y_ptr[y + 1]] for y, kn in zip(pi.tolist(), known.tolist()) if kn] + [[]])
    s_all = oracle.similarity_pairs(kind, qi, qj.astype(np.int32), x_ptr, i[o], r[o], 1, float(ts.global_mean),
                                    bu if mode else None, bi if mode else None, 100.0)
    kw = dict(mu=float(ts.global_mean), bx=bu, by=bi) if mode else {}
    return knn_restated(pu, pi, np.split(s_all, np.cumsum(lens)[:-1]), y_ptr, x_idx, r_y, k, mode, **kw)
