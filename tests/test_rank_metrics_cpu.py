"""fcp and precision_recall_at_k without a GPU: the reference's fcp loop and the Surprise FAQ's precision_recall_at_k
(both transcribed literally) against a numpy restatement of the per-user count rules, and accuracy.fcp /
accuracy.precision_recall_at_k against the transcriptions: the same dict keys in the same order, the same values and
the same value types, the same warnings and exceptions."""
import math
import warnings
from collections import defaultdict

import numpy as np
import pytest

from surprise_b200 import accuracy
from surprise_b200.prediction_algorithms.predictions import Prediction


def reference_fcp(predictions, verbose=True):
    """accuracy.fcp as this project transcribed it from the reference (accuracy.py:91-143), before the device route."""
    if not predictions:
        raise ValueError("Prediction list is empty.")
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


def faq_precision_recall_at_k(predictions, k=10, threshold=3.5):
    """The Surprise FAQ's precision_recall_at_k (current version: 0 where a value is undefined), as written there."""
    user_est_true = defaultdict(list)
    for uid, _, true_r, est, _ in predictions:
        user_est_true[uid].append((est, true_r))
    precisions = dict()
    recalls = dict()
    for uid, user_ratings in user_est_true.items():
        user_ratings.sort(key=lambda x: x[0], reverse=True)
        n_rel = sum((true_r >= threshold) for (_, true_r) in user_ratings)
        n_rec_k = sum((est >= threshold) for (est, _) in user_ratings[:k])
        n_rel_and_rec_k = sum(((true_r >= threshold) and (est >= threshold))
                              for (est, true_r) in user_ratings[:k])
        precisions[uid] = n_rel_and_rec_k / n_rec_k if n_rec_k != 0 else 0
        recalls[uid] = n_rel_and_rec_k / n_rel if n_rel != 0 else 0
    return precisions, recalls


# -- the count rules, restated with numpy ------------------------------------------------------------------------------
def group(predictions):
    """(keys, seg_ptr, r, est): defaultdict(list) grouping (first appearance, equal uids merged into the first) as a
    segment CSR over float64 columns, prediction order kept inside a user."""
    codes, r, est = {}, [], []
    for uid, _, true_r, e, _ in predictions:
        codes.setdefault(uid, len(codes))
    code = np.array([codes[p[0]] for p in predictions], dtype=np.int64)
    order = np.argsort(code, kind="stable")
    r = np.array([p[2] for p in predictions], dtype=np.float64)[order]
    est = np.array([p[3] for p in predictions], dtype=np.float64)[order]
    seg_ptr = np.concatenate(([0], np.cumsum(np.bincount(code, minlength=len(codes))))).astype(np.int64)
    return list(codes), seg_ptr, r, est


def k_eff(k, m):
    return len(range(m)[:k])


def count_oracle(seg_ptr, r, est, k_effs=None, threshold=None, chunk=2048):
    """Per segment: (nc, nd) when k_effs is None, else (n_rel, n_rec_k, n_rel_and_rec_k) with rank_j = #{i : e_i > e_j}
    + #{i < j : e_i == e_j} and top = rank < k_eff.  Rows are compared in chunks so that long segments fit."""
    out = np.zeros((len(seg_ptr) - 1, 2 if k_effs is None else 3), dtype=np.int64)
    for s in range(len(seg_ptr) - 1):
        rs, es = r[seg_ptr[s]:seg_ptr[s + 1]], est[seg_ptr[s]:seg_ptr[s + 1]]
        m = len(rs)
        if k_effs is not None:
            top = np.zeros(m, dtype=bool)
        for a in range(0, m, chunk):
            e, rr = es[a:a + chunk, None], rs[a:a + chunk, None]
            if k_effs is None:
                out[s, 0] += np.count_nonzero((e > es) & (rr > rs))
                out[s, 1] += np.count_nonzero((e >= es) & (rr < rs))
            else:
                pos = np.arange(a, min(a + chunk, m))[:, None]
                rank = np.count_nonzero(es > e, axis=1) + np.count_nonzero((es == e) & (np.arange(m) < pos), axis=1)
                top[a:a + chunk] = rank < k_effs[s]
        if k_effs is not None:
            rec = top & (es >= threshold)
            out[s] = (np.count_nonzero(rs >= threshold), np.count_nonzero(rec),
                      np.count_nonzero(rec & (rs >= threshold)))
    return out


# -- cases -------------------------------------------------------------------------------------------------------------
NAN, INF = float("nan"), float("inf")


def preds_of(rows):
    return [Prediction(u, "i%d" % n, r, e, {}) for n, (u, r, e) in enumerate(rows)]


def interleave(table):
    """{uid: [(r, est), ...]} -> rows taking one entry of each user in turn, so users interleave."""
    rows, lists = [], {u: list(v) for u, v in table.items()}
    while any(lists.values()):
        for u, v in lists.items():
            if v:
                rows.append((u, *v.pop(0)))
    return rows


def random_grid(seed, n_users=30, step=0.5):
    rng = np.random.RandomState(seed)
    rows = []
    for _ in range(600):
        u = int(rng.randint(n_users) ** 2 % n_users)
        rows.append(("u%d" % u, float(rng.randint(2, 11) * step), float(rng.randint(2, 11) * step)))
    return rows


CASES = {
    "ties": interleave({"a": [(4.0, 3.5), (3.0, 3.5), (4.0, 4.0), (2.0, 2.0), (5.0, 3.5), (4.0, 4.0)],
                        "b": [(1.0, 1.0), (2.0, 1.0), (2.0, 1.0)]}),
    "zeros_inf": interleave({"z": [(0.0, -0.0), (-0.0, 0.0), (INF, INF), (-INF, -INF), (1.0, 0.0), (-1.0, -0.0),
                                   (0.0, 0.0)],
                             "y": [(INF, 1.0), (INF, INF), (-INF, INF), (0.0, -INF)]}),
    "nan": interleave({"n": [(NAN, 2.0), (3.0, NAN), (4.0, 3.0), (5.0, 1.0), (2.0, NAN)],
                       "m": [(NAN, 1.0), (4.0, 2.0), (NAN, 3.0), (3.5, 3.0)],
                       "o": [(4.0, 4.0), (3.0, 2.0)]}),
    "singles_equal": interleave({"s1": [(4.0, 3.0)], "s2": [(1.0, 5.0)], "eq": [(1.0, 2.5), (5.0, 2.5), (3.0, 2.5),
                                                                                 (4.0, 2.5), (3.5, 2.5)]}),
    "merge": [(1, 4.0, 3.0), (1.0, 2.0, 4.0), (True, 5.0, 5.0), (2, 3.0, 3.0), ("x", 1.0, 1.0), (2.0, 4.0, 1.0),
              (1, 3.0, 3.0)],
    "ints_bools": [("a", 4, 3), ("a", 5, True), ("a", 3, 4), ("b", True, 4), ("b", 4, 4), ("a", 2, 2 ** 53),
                   ("b", False, -(2 ** 53))],
    "numpy": [("a", np.float64(4.0), 3.5), ("a", 3.0, np.float64(4.0)), ("a", np.int64(5), 4), ("b", 4.0, 3.0),
              ("b", 2.0, 4.5), ("c", np.bool_(True), np.float64(1.0)), ("c", 4.0, 3.0)],
    "grid": random_grid(0),
}


def k_values(rows):
    m = max(sum(1 for u, _, _ in rows if u == v) for v, _, _ in rows)
    return [None, 0, 1, -1, -m, m, m + 5, 2 ** 40, True]


THRESHOLDS = [3.5, 4, 3.0, 0.0]
NUMPY_THRESHOLDS = [np.float64(3.5), np.int64(4), np.bool_(True), np.float64(-0.0), np.float64("nan")]


def same_value(a, b):
    return type(a) is type(b) and (a == b or (a != a and b != b)) and math.copysign(1, a) == math.copysign(1, b)


def assert_same_dict(got, want):
    assert list(got) == list(want)
    assert [type(u) for u in got] == [type(u) for u in want]
    for u in want:
        assert same_value(got[u], want[u]), (u, got[u], want[u])


def call(f, *args, **kw):
    """(result, warning categories) of f; an exception is returned as (type, message)."""
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        try:
            out = f(*args, **kw)
        except Exception as e:  # noqa: BLE001
            out = (type(e), str(e))
    return out, sorted({x.category.__name__ for x in w})


def assert_same_fcp(preds):
    got, want = call(accuracy.fcp, preds, verbose=False), call(reference_fcp, preds, verbose=False)
    assert got[1] == want[1]
    if isinstance(want[0], tuple):
        assert got[0] == want[0]
    else:
        assert same_value(got[0], want[0]), (got[0], want[0])
    return want[0]


def assert_same_precision_recall(preds, k, threshold):
    got = call(accuracy.precision_recall_at_k, preds, k=k, threshold=threshold)
    want = call(faq_precision_recall_at_k, preds, k=k, threshold=threshold)
    assert got[1] == want[1]
    if isinstance(want[0][0], type):
        assert got[0] == want[0]
        return
    assert_same_dict(got[0][0], want[0][0])
    assert_same_dict(got[0][1], want[0][1])


# -- the transcriptions against the count rules ------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(CASES))
def test_fcp_counts_rule(case):
    preds = preds_of(CASES[case])
    keys, seg_ptr, r, est = group(preds)
    counts = count_oracle(seg_ptr, r, est)
    want_c, want_d = np.mean(counts[:, 0]), np.mean(counts[:, 1])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = want_c / (want_c + want_d)
    got = call(reference_fcp, preds, verbose=False)[0]
    assert same_value(got, want), (got, want)


@pytest.mark.parametrize("case", sorted(CASES))
def test_precision_recall_counts_rule(case):
    preds = preds_of(CASES[case])
    keys, seg_ptr, r, est = group(preds)
    nan_users = {keys[s] for s in range(len(keys)) if np.isnan(est[seg_ptr[s]:seg_ptr[s + 1]]).any()}
    for k in k_values(CASES[case]):
        for t in THRESHOLDS:
            ks = np.array([k_eff(k, int(m)) for m in np.diff(seg_ptr)])
            counts = count_oracle(seg_ptr, r, est, ks, t)
            prec, rec = faq_precision_recall_at_k(preds, k, t)
            assert list(prec) == keys
            for s, u in enumerate(keys):
                if u in nan_users or case == "numpy":
                    continue
                n_rel, n_rec, n_rr = (int(x) for x in counts[s])
                assert same_value(prec[u], n_rr / n_rec if n_rec != 0 else 0), (u, k, t)
                assert same_value(rec[u], n_rr / n_rel if n_rel != 0 else 0), (u, k, t)


def test_nan_estimates_have_no_sorted_order():
    # why a user with a NaN est gets the recipe itself: timsort leaves this list as it is
    xs = [(2.0, 0), (NAN, 1), (3.0, 2), (1.0, 3)]
    xs.sort(key=lambda x: x[0], reverse=True)
    assert [i for _, i in xs] == [0, 1, 2, 3]


# -- accuracy against the transcriptions -------------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(CASES))
def test_fcp_matches_reference(case):
    assert_same_fcp(preds_of(CASES[case]))


@pytest.mark.parametrize("case", sorted(CASES))
def test_precision_recall_matches_faq(case):
    preds = preds_of(CASES[case])
    for k in k_values(CASES[case]):
        for t in THRESHOLDS:
            assert_same_precision_recall(preds, k, t)


@pytest.mark.parametrize("case", sorted(CASES))
def test_precision_recall_numpy_threshold_matches_faq(case):
    preds = preds_of(CASES[case])
    for k in k_values(CASES[case]):
        for t in NUMPY_THRESHOLDS:
            assert_same_precision_recall(preds, k, t)


def test_fcp_all_zero_counts_is_nan_with_warning():
    preds = preds_of([("a", 4.0, 3.0), ("b", 3.0, 2.0), ("c", 1.0, 1.0)])
    out = assert_same_fcp(preds)
    assert np.isnan(out)
    assert call(accuracy.fcp, preds, verbose=False)[1] == ["RuntimeWarning"]


def test_odd_inputs_behave_as_the_python_code():
    good = CASES["ties"]
    for rows in ([("a", None, 3.0), ("a", 4.0, 2.0)],                       # r_ui = None: TypeError
                 [("a", 4.0, "3.5"), ("a", 3.0, "2.0")],                    # string estimates (compare as strings)
                 [("a", 4.0, "3.5"), ("a", 3.0, 2.0)],                      # mixed: TypeError
                 [("a", 4.0, 2 ** 60), ("a", 3.0, 2 ** 60 + 1)],            # ints float64 does not hold
                 [("a", 4.0, np.float32(0.1)), ("a", 3.0, 0.1)],            # float32 against a Python float
                 good):
        preds = preds_of(rows)
        assert_same_fcp(preds)
        for k in (1, None):
            for t in (3.5, 4):
                assert_same_precision_recall(preds, k, t)
    assert_same_precision_recall(preds_of(good), 1.5, 3.5)                  # TypeError from the slice
    assert_same_precision_recall([], 1.5, 3.5)                              # no user: k is not looked at
    assert_same_precision_recall(preds_of(good), 2, np.float64(3.5))
    assert_same_fcp([])
    assert_same_fcp([("a", "i", 1.0, 2.0)])                                 # an item that does not unpack
    assert_same_precision_recall([("a", "i", 1.0, 2.0, {}, 0)], 2, 3.5)


def test_generator_input():
    rows = CASES["grid"]
    assert accuracy.fcp(iter(preds_of(rows)), verbose=False) == reference_fcp(preds_of(rows), verbose=False)
    got = accuracy.precision_recall_at_k(iter(preds_of(rows)), 3, 3.5)
    want = faq_precision_recall_at_k(preds_of(rows), 3, 3.5)
    assert_same_dict(got[0], want[0])
    assert_same_dict(got[1], want[1])


def test_public_surface():
    assert "precision_recall_at_k" in accuracy.__all__
    import surprise_b200 as sb
    assert sb.accuracy.precision_recall_at_k is accuracy.precision_recall_at_k
