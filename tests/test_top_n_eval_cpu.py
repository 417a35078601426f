"""Top-N measures against held-out ratings and LeaveOneOut, without a GPU: accuracy.top_n_measures on hand-built cases
with known answers, LeaveOneOut against upstream Surprise 1.1's algorithm (restated below, and the compiled reference
when oracle/_ref is built), list- and array-backed datasets splitting alike, the host side of the device route
(_Pairs.relevant), the route for algorithms that are not device-batched, and the measure names of cross_validate and
the searches."""
from collections import defaultdict
from math import log2

import numpy as np
import pytest

import surprise_b200 as sb
from surprise_b200 import accuracy
from surprise_b200.model_selection import GridSearchCV, KFold, LeaveOneOut, cross_validate, fit_and_score
from surprise_b200.model_selection.validation import Fold
from surprise_b200.utils import get_rng


def bits(x):
    return np.float64(x).tobytes()


def same_result(a, b):
    return list(a) == list(b) and all(bits(a[k]) == bits(b[k]) for k in a)


# -- the definition on hand-built cases ------------------------------------------------------------------------------
def lists(**users):
    return {u: [(i, 5.0 - k * 0.1) for k, i in enumerate(items)] for u, items in users.items()}


def test_hits_at_given_positions():
    top = lists(a=["i0", "i1", "i2", "i3", "i4"], b=["i9", "i8"])
    test = [("a", "i1", 4.0), ("a", "i3", 2.0), ("a", "zz", 5.0), ("b", "i7", 1.0)]
    got = accuracy.top_n_measures(top, test, 5, verbose=False)
    rr_a = 0.0 + 1.0 / 2 + 1.0 / 4
    dcg_a = 0.0 + 1.0 / np.log2(3.0) + 1.0 / np.log2(5.0)
    idcg = [0.0]
    for p in range(5):
        idcg.append(idcg[-1] + 1.0 / np.log2(p + 2.0))
    want = {"hr": 2 / 4, "arhr": float(np.sum([rr_a, 0.0])) / 4, "precision": float(np.mean([2 / 5, 0 / 5])),
            "recall": float(np.mean([2 / 3, 0 / 1])), "ndcg": float(np.mean([dcg_a / idcg[3], 0.0 / idcg[1]]))}
    assert same_result(got, want)
    assert got["hr"] == 0.5 and got["arhr"] == 0.75 / 4
    # only the first n entries of a list count
    got = accuracy.top_n_measures(top, test, 2, verbose=False)
    assert got["hr"] == 1 / 4 and got["arhr"] == 0.5 / 4 and got["precision"] == np.mean([0.5, 0.0])


def test_duplicates_unknown_users_and_items():
    top = lists(a=["x", "y", "z"], b=["y"])
    # a: x twice (one relevant item), an unknown item; b rated nothing relevant in the lists; c is unknown
    test = [("a", "x", 3.0), ("c", "x", 3.0), ("a", "x", 1.0), ("a", "new", 4.0), ("b", "q", 2.0)]
    got = accuracy.top_n_measures(top, test, 3, verbose=False)
    # U* = a, c, b; |R| = 2, 1, 1
    assert got["hr"] == 1 / 4
    assert got["recall"] == float(np.mean([1 / 2, 0.0, 0.0]))
    assert got["precision"] == float(np.mean([1 / 3, 0.0, 0.0]))
    assert got["ndcg"] == float(np.mean([1.0 / (1.0 + 1.0 / log2(3)), 0.0, 0.0]))


def test_equal_uids_merge_as_dict_keys():
    top = {1: [("p", 4.0), ("q", 3.0)]}
    got = accuracy.top_n_measures(top, [(1, "q", 4.0), (1.0, "p", 4.0), (True, "q", 1.0)], 2, verbose=False)
    assert got["hr"] == 1.0 and got["recall"] == 1.0 and got["precision"] == 1.0


def test_threshold_on_an_offset_dataset(capsys):
    reader = sb.Reader(rating_scale=(-10, 10))
    assert reader.offset == 11
    rows = [("u%d" % (k % 4), "i%d" % (k % 7), float((k * 7) % 21 - 10), None) for k in range(40)]
    data = sb.Dataset.load_from_arrays(np.array([r[0] for r in rows]), np.array([r[1] for r in rows]),
                                       np.array([r[2] for r in rows]), reader)
    testset = data.construct_testset(data._take(np.arange(40)))
    assert all(r == raw[2] + 11 for (_, _, r), raw in zip(testset, rows))
    top = lists(u0=["i0", "i1", "i2"], u1=["i3", "i4"], u2=["i5"], u3=["i6", "i0"])
    for threshold in (-3, 0.5, 4):
        relevant = defaultdict(set)
        for u, i, r, _ in rows:
            if r >= threshold:
                relevant[u].add(i)
        got = accuracy.top_n_measures(top, testset, 3, threshold=threshold, offset=11, verbose=False)
        hits = [sum(i in relevant[u] for i, _ in top[u][:3]) for u in relevant]
        assert got["hr"] == sum(hits) / sum(map(len, relevant.values())), threshold
    with pytest.raises(ValueError):
        accuracy.top_n_measures(top, testset, 3, threshold=11, offset=11, verbose=False)
    accuracy.top_n_measures(top, testset, 3, threshold=0.5, offset=11)
    out = capsys.readouterr().out.splitlines()
    assert [line.split(":")[0] for line in out] == ["HR@3", "ARHR@3", "Precision@3", "Recall@3", "nDCG@3"]


def test_n_larger_than_lists_and_bad_n():
    top = lists(a=["x", "y"])
    got = accuracy.top_n_measures(top, [("a", "y", 1.0)], 10 ** 12, verbose=False)
    assert got["hr"] == 1.0 and got["arhr"] == 0.5 and got["precision"] == 1 / (2 ** 31 - 1)
    assert got["ndcg"] == 1.0 / log2(3)
    for bad in (0, -1, True, 2.5, "3", None):
        with pytest.raises(ValueError):
            accuracy.top_n_measures(top, [("a", "y", 1.0)], bad, verbose=False)
    with pytest.raises(ValueError):
        accuracy.top_n_measures(top, [], 3, verbose=False)


def test_rank_table_entries_do_not_depend_on_length():
    inv, disc, idcg = accuracy._rank_tables(5000)
    for m in (1, 2, 31, 32, 33, 1000):
        i2, d2, g2 = accuracy._rank_tables(m)
        assert inv[:m].tobytes() == i2.tobytes() and disc[:m].tobytes() == d2.tobytes()
        assert idcg[:m + 1].tobytes() == g2.tobytes()
    assert [disc[p] for p in (0, 2, 6)] == [1.0, 0.5, 1.0 / 3]


# -- LeaveOneOut -----------------------------------------------------------------------------------------------------
def upstream_leave_one_out(raw_ratings, n_splits, random_state, min_n_ratings):
    """Upstream Surprise 1.1's LeaveOneOut.split, restated."""
    user_ratings = defaultdict(list)
    for uid, iid, r_ui, _ in raw_ratings:
        user_ratings[uid].append((uid, iid, r_ui, None))
    rng = get_rng(random_state)
    for _ in range(n_splits):
        raw_trainset, raw_testset = [], []
        for uid, ratings in user_ratings.items():
            if len(ratings) > min_n_ratings:
                i = rng.randint(0, len(ratings))
                raw_testset.append(ratings[i])
                raw_trainset += [rating for (j, rating) in enumerate(ratings) if j != i]
        if not raw_trainset:
            raise ValueError("Could not build any trainset. Maybe min_n_ratings is too high?")
        yield raw_trainset, raw_testset


def small_data(seed=0, n=600):
    rng = np.random.RandomState(seed)
    uids = rng.zipf(1.5, n) % 53 + 100
    iids = rng.randint(0, 80, n) * 3
    rs = rng.randint(1, 6, n).astype(np.float64)
    arrays = sb.Dataset.load_from_arrays(uids, iids, rs, sb.Reader(rating_scale=(1, 5)))
    listed = sb.Dataset.load_from_arrays(uids, iids, rs, sb.Reader(rating_scale=(1, 5)))
    listed._arrays, listed.raw_ratings = None, [(int(u), int(i), float(r), None) for u, i, r in zip(uids, iids, rs)]
    return arrays, listed


def trainset_rows(ts):
    return [(ts.to_raw_uid(u), ts.to_raw_iid(i), r) for u, i, r in ts.all_ratings()]


@pytest.mark.parametrize("seed", [0, 1, 7, 123])
def test_leave_one_out_matches_upstream(seed):
    arrays, listed = small_data(seed)
    for min_n in (0, 1, 4, 9):
        ref = list(upstream_leave_one_out(listed.raw_ratings, 4, seed, min_n))
        for data in (listed, arrays):
            got = list(LeaveOneOut(n_splits=4, random_state=seed, min_n_ratings=min_n).split(data))
            assert len(got) == 4
            for (trs, tes), (rtr, rte) in zip(got, ref):
                assert tes == [(u, i, r) for u, i, r, _ in rte]
                # the trainset is built from the user-grouped rows, in that order
                want = listed.construct_trainset(rtr)
                assert trs.n_users == want.n_users and trs.n_items == want.n_items
                assert trainset_rows(trs) == trainset_rows(want)
                for a, b in zip(trs.user_csr() + trs.item_csr(), want.user_csr() + want.item_csr()):
                    assert np.array_equal(a, b)
        # the splits share one RNG: they differ from one another
        assert len({tuple(te) for _, te in ref}) > 1


def test_leave_one_out_list_and_array_backed_agree():
    arrays, listed = small_data(3)
    for (ta, ea), (tl, el) in zip(LeaveOneOut(3, random_state=5).split(arrays),
                                  LeaveOneOut(3, random_state=5).split(listed)):
        assert ea == el
        assert trainset_rows(ta) == trainset_rows(tl)
        assert [ta.to_raw_uid(u) for u in range(ta.n_users)] == [tl.to_raw_uid(u) for u in range(tl.n_users)]
        assert [ta.to_raw_iid(i) for i in range(ta.n_items)] == [tl.to_raw_iid(i) for i in range(tl.n_items)]
        for a, b in zip(ta.user_csr() + ta.item_csr(), tl.user_csr() + tl.item_csr()):
            assert np.array_equal(a, b)


def test_leave_one_out_options():
    arrays, listed = small_data(2)
    assert LeaveOneOut(n_splits=7).get_n_folds() == 7
    lengths = np.bincount(np.unique(arrays._arrays[0], return_inverse=True)[1].reshape(-1))
    for min_n in (0, 3, int(lengths.max()) - 1):
        tr, te = next(LeaveOneOut(1, random_state=0, min_n_ratings=min_n).split(arrays))
        assert len(te) == int((lengths > min_n).sum())
        assert tr.n_ratings == int(lengths[lengths > min_n].sum()) - len(te)
    for data in (arrays, listed):
        with pytest.raises(ValueError, match="min_n_ratings is too high"):
            next(LeaveOneOut(min_n_ratings=int(lengths.max())).split(data))
    # one rating per user: every trainset is empty
    one = sb.Dataset.load_from_arrays(np.arange(5), np.arange(5), np.ones(5), sb.Reader(rating_scale=(1, 5)))
    with pytest.raises(ValueError, match="Could not build any trainset"):
        next(LeaveOneOut().split(one))
    # random_state=None draws from numpy's global state, as upstream does
    np.random.seed(11)
    a = [te for _, te in LeaveOneOut(2).split(listed)]
    np.random.seed(11)
    assert a == [[(u, i, r) for u, i, r, _ in te] for _, te in upstream_leave_one_out(listed.raw_ratings, 2, None, 0)]


def test_vectorised_draws_consume_the_scalar_stream():
    """LeaveOneOut draws a split's per-user indices with one randint(0, lengths) call; upstream makes one scalar call
    per user.  Both leave the RandomState in the same state with the same values, including lengths past 2**31."""
    rng = np.random.RandomState(4)
    high = rng.randint(1, 3000, 5000)
    high[::9] = 1
    high[::13] = 2 ** 31 + 7
    for seed in range(5):
        a, b = np.random.RandomState(seed), np.random.RandomState(seed)
        assert [a.randint(0, h) for h in high.tolist()] == b.randint(0, high).tolist()
        assert a.randint(0, 10 ** 9) == b.randint(0, 10 ** 9)


def test_leave_one_out_matches_compiled_reference():
    try:
        import oracle
        ref = oracle.import_reference()
    except ImportError:
        pytest.skip("oracle/_ref is not built")
    import pandas as pd
    from surprise.model_selection import LeaveOneOut as RefLeaveOneOut
    arrays, listed = small_data(9)
    df = pd.DataFrame([r[:3] for r in listed.raw_ratings], columns=["u", "i", "r"])
    rdata = ref.Dataset.load_from_df(df, ref.Reader(rating_scale=(1, 5)))
    for min_n in (0, 5):
        got = list(LeaveOneOut(3, random_state=2, min_n_ratings=min_n).split(arrays))
        want = list(RefLeaveOneOut(3, random_state=2, min_n_ratings=min_n).split(rdata))
        for (trs, tes), (rtr, rte) in zip(got, want):
            assert [(int(u), int(i), float(r)) for u, i, r in rte] == tes
            assert [(rtr.to_raw_uid(u), rtr.to_raw_iid(i), r) for u, i, r in rtr.all_ratings()] == trainset_rows(trs)


# -- the host side of the device route -------------------------------------------------------------------------------
def test_relevant_items_match_the_definition():
    arrays, _ = small_data(5)
    trs, tes = next(KFold(3, random_state=0).split(arrays))
    tes = tes + [(100, 10 ** 6, 5.0), (10 ** 6, 3, 5.0), (10 ** 6, 10 ** 6, 5.0), (100, 10 ** 6, 4.0), (100.0, 3, 2.0)]
    for threshold in (None, 3.5, 4, 6):
        relevant = {}
        for u, i, r in tes:
            if threshold is None or r - trs.offset >= threshold:
                relevant.setdefault(u, set()).add(i)
        if not relevant:
            with pytest.raises(ValueError):
                Fold(trs, tes).test_pairs().relevant(threshold, trs.n_items)
            continue
        iu, n_rel, rel_ptr, rel_idx = Fold(trs, tes).test_pairs().relevant(threshold, trs.n_items)
        assert iu.tolist() == trs.to_inner_uids(list(relevant)).tolist()
        assert n_rel.tolist() == [len(s) for s in relevant.values()]
        known = [u for u in relevant if trs.to_inner_uids([u])[0] >= 0]
        assert len(rel_ptr) == len(known) + 1
        for k, u in enumerate(known):
            want = sorted(int(trs.to_inner_iid(i)) for i in relevant[u] if trs.to_inner_iids([i])[0] >= 0)
            assert rel_idx[rel_ptr[k]:rel_ptr[k + 1]].tolist() == want


class PyAlgo(sb.AlgoBase):
    """An algorithm with a Python estimate (not device-batched), with ties and a prediction it cannot make."""

    def estimate(self, u, i):
        if not (self.trainset.knows_user(u) and self.trainset.knows_item(i)):
            raise sb.PredictionImpossible("unknown")
        return float((u * 7 + i * 3) % 5) + 0.5


def test_non_batched_route_equals_the_definition():
    arrays, _ = small_data(6, n=300)
    for trs, tes in LeaveOneOut(2, random_state=1).split(arrays):
        algo = PyAlgo().fit(trs)
        assert not algo._batched()
        for n in (1, 3, trs.n_items + 5):
            for threshold in (None, 3.5, 4):
                got = algo.top_n_measures(tes, n, threshold)
                want = accuracy.top_n_measures(algo.get_top_n(n), tes, n, threshold, offset=trs.offset,
                                               verbose=False)
                assert same_result(got, want), (n, threshold)


# -- cross_validate / searches ---------------------------------------------------------------------------------------
def test_measure_names():
    parse = accuracy._top_n_measure
    assert parse("HR@10") == ("hr", 10) and parse("nDCG@1") == ("ndcg", 1) and parse("Recall@007") == ("recall", 7)
    assert parse("arhr@3") == ("arhr", 3) and parse("precision@100") == ("precision", 100)
    for other in ("rmse", "fcp", "mae", "hr", "foo@3"):
        assert parse(other) is None
    for bad in ("hr@0", "hr@", "hr@-1", "ndcg@1.5", "precision@x", "recall@ 3"):
        with pytest.raises(ValueError):
            parse(bad)


def test_train_measures_are_refused_with_top_n_measures():
    arrays, _ = small_data(1, n=200)
    trs, tes = next(LeaveOneOut(1, random_state=0).split(arrays))
    algo = PyAlgo()
    with pytest.raises(ValueError, match="return_train_measures"):
        fit_and_score(algo, trs, tes, ["rmse", "hr@10"], return_train_measures=True)
    assert not hasattr(algo, "trainset")          # refused before the fit
    with pytest.raises(ValueError):
        cross_validate(algo, arrays, ["ndcg@5"], cv=LeaveOneOut(2), return_train_measures=True)


def test_cross_validate_and_search_with_top_n_measures():
    arrays, _ = small_data(4, n=300)
    measures = ["HR@3", "ndcg@3", "rmse", "precision@10"]
    got = cross_validate(PyAlgo(), arrays, measures, cv=LeaveOneOut(2, random_state=3))
    assert list(got)[:4] == ["test_hr@3", "test_ndcg@3", "test_rmse", "test_precision@10"]
    for k, (trs, tes) in enumerate(LeaveOneOut(2, random_state=3).split(arrays)):
        algo = PyAlgo().fit(trs)
        m3, m10 = algo.top_n_measures(tes, 3), algo.top_n_measures(tes, 10)
        assert bits(got["test_hr@3"][k]) == bits(m3["hr"]) and bits(got["test_ndcg@3"][k]) == bits(m3["ndcg"])
        assert bits(got["test_precision@10"][k]) == bits(m10["precision"])
        assert bits(got["test_rmse"][k]) == bits(accuracy.rmse(algo.test(tes), verbose=False))

    class Shifted(PyAlgo):
        def __init__(self, shift=0):
            PyAlgo.__init__(self)
            self.shift = shift

        def estimate(self, u, i):
            PyAlgo.estimate(self, u, i)              # raises for unknown ids
            return float((u * 7 + (i + self.shift) * 3) % 5) + 0.5

    gs = GridSearchCV(Shifted, {"shift": [0, 1, 2, 3]}, measures=["hr@10", "rmse"], cv=LeaveOneOut(2, random_state=0))
    gs.fit(arrays)
    mean = gs.cv_results["mean_test_hr@10"]
    assert gs.best_index["hr@10"] == int(np.argmax(mean)) and gs.best_params["hr@10"] == {"shift": int(np.argmax(mean))}
    assert gs.cv_results["rank_test_hr@10"][int(np.argmax(mean))] == 1
