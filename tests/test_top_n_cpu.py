"""Top-N recommendations without a GPU: the reference FAQ's get_top_n (transcribed literally) against a numpy
restatement of the ordering rule, argument validation, and AlgoBase.get_top_n through test() for an algorithm with
its own Python estimate()."""
import struct
from collections import defaultdict

import numpy as np
import pytest

import surprise_b200 as sb
from surprise_b200.prediction_algorithms.algo_base import rank_top_n
from surprise_b200.prediction_algorithms.predictions import Prediction, PredictionImpossible


def faq_get_top_n(predictions, n=10):
    """The reference FAQ's get_top_n (examples/top_n_recommendations.py), as written there."""
    top_n = defaultdict(list)
    for uid, iid, true_r, est, _ in predictions:
        top_n[uid].append((iid, est))
    for uid, user_ratings in top_n.items():
        user_ratings.sort(key=lambda x: x[1], reverse=True)
        top_n[uid] = user_ratings[:n]
    return top_n


def numpy_top_n(uids, iids, est, n):
    """The ordering rule restated: per user (first-appearance order), a stable lexsort on score descending then
    position ascending; the first n."""
    out = {}
    uids, est = list(uids), np.asarray(est, dtype=np.float64)
    pos = np.arange(len(uids))
    for u in dict.fromkeys(uids):
        sel = pos[[x == u for x in uids]]
        order = sel[np.lexsort((sel, -est[sel]))][:n]
        out[u] = [(iids[k], float(est[k])) for k in order]
    return out


def bits(top):
    return {u: [(i, struct.pack("<d", e)) for i, e in v] for u, v in top.items()}


def assert_same_top_n(got, want):
    assert list(got.keys()) == list(want.keys())
    assert bits(got) == bits(want)


def clipped(est, offset, low, high):
    e = np.asarray(est, dtype=np.float64) - offset
    return np.maximum(low, np.minimum(high, e))


HAND_MADE = [
    # (raw scores per (user, item), offset, rating scale)
    ({"a": [5.2, 5.0, 4.9, 5.7, 1.0, 0.3], "b": [0.9, 0.5, 1.0, 3.0, 3.0]}, 0, (1, 5)),         # ties at high / low
    ({"a": [11.0, 11.0, 10.5, 11.5, 0.0]}, 11, (-10, 10)),                                     # offset scale
    ({"a": [-0.0, 0.0, -0.0, 0.0, 0.5, -0.5]}, 0, (-1, 1)),                                   # signed zeros
    ({"a": [3.0, 2.0], "b": [], "c": [1.0]}, 0, (1, 5)),                                       # a user with no candidates
]


@pytest.mark.parametrize("case", range(len(HAND_MADE)))
@pytest.mark.parametrize("n", [1, 2, 3, 10])
def test_faq_matches_numpy_rule(case, n):
    table, offset, (low, high) = HAND_MADE[case]
    uids, iids, est = [], [], []
    for u, row in table.items():
        for k, s in enumerate(row):
            uids.append(u)
            iids.append("i%d" % k)
            est.append(s)
    est = clipped(est, offset, low, high)
    preds = [Prediction(u, i, None, e, {}) for u, i, e in zip(uids, iids, est.tolist())]
    want = numpy_top_n(uids, iids, est, n)
    assert_same_top_n(faq_get_top_n(preds, n), want)
    assert "b" not in faq_get_top_n(preds, n) or table.get("b")


def test_rank_top_n_rule():
    est = np.array([1.0, np.nan, 2.0, -0.0, 0.0, 2.0, np.nan, -np.inf])
    items = np.arange(len(est))
    assert rank_top_n(est, items).tolist() == [2, 5, 0, 3, 4, 7, 1, 6]


class TableAlgo(sb.AlgoBase):
    """A Python estimate() from a table (not device-batched): get_top_n goes through test()."""

    def __init__(self, table, impossible=()):
        sb.AlgoBase.__init__(self)
        self.table, self.impossible = table, set(impossible)

    def estimate(self, u, i):
        if (u, i) in self.impossible:
            raise PredictionImpossible("no")
        return self.table[u, i]


def table_trainset(rating_scale=(1, 5), offset=0, seed=0):
    rng = np.random.RandomState(seed)
    n_u, n_i = 7, 9
    pairs = [(u, i) for u in range(n_u) for i in range(n_i) if rng.rand() < 0.3 or i == u]
    pairs += [(6, i) for i in range(n_i) if (6, i) not in pairs]          # user 6 rated every item
    u, i = (np.array(x, dtype=np.int32) for x in zip(*pairs))
    r = rng.randint(1, 6, len(u)).astype(np.float64) + offset
    raw_u = ["u%d" % k for k in range(n_u)]
    raw_i = ["i%d" % k for k in range(n_i)]
    return sb.Trainset.from_coo(u, i, r, n_u, n_i, rating_scale, offset, raw_u, raw_i)


@pytest.mark.parametrize("scale,offset", [((1, 5), 0), ((-10, 10), 11)])
def test_get_top_n_through_test(scale, offset):
    ts = table_trainset(scale, offset)
    rng = np.random.RandomState(1)
    table = np.round(rng.uniform(-3, 20, (ts.n_users, ts.n_items)) * 2) / 2     # many ties, many clipped
    table[0, :4] = -0.0
    algo = TableAlgo(table, impossible=[(1, 2), (3, 3)])
    algo.fit(ts)
    preds = algo.test(ts.build_anti_testset())
    for n in (1, 3, ts.n_items + 5):
        got = algo.get_top_n(n)
        assert_same_top_n(got, faq_get_top_n(preds, n))
        assert "u6" not in got
    items, est, count = algo.top_n_inner(4)
    assert items.shape == est.shape == (ts.n_users, 4) and count[6] == 0
    assert (items[6] == -1).all() and np.isnan(est[6]).all()
    uids = ["u4", "u0", "u2"]
    sub = [p for u in uids for p in preds if p.uid == u]
    assert_same_top_n(algo.get_top_n(3, uids=uids), faq_get_top_n(sub, 3))
    with pytest.raises(ValueError):
        algo.get_top_n(3, uids=["nobody"])


@pytest.mark.parametrize("bad", [0, -1, 2.0, "3", None, True])
def test_n_is_validated_before_any_device_call(bad):
    ts = table_trainset()
    algo = sb.SVD()
    sb.AlgoBase.fit(algo, ts)          # a trainset, no factors and no device state
    with pytest.raises(ValueError):
        algo.get_top_n(bad)
    with pytest.raises(ValueError):
        algo.top_n_inner(bad)


def test_users_are_validated():
    ts = table_trainset()
    algo = TableAlgo(np.zeros((ts.n_users, ts.n_items)))
    algo.fit(ts)
    for bad in ([ts.n_users], [-1], [0.5]):
        with pytest.raises(ValueError):
            algo.top_n_inner(2, bad)
