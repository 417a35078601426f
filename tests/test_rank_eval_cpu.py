"""AUC, MRR and mean percentile rank over the full ranking, without a GPU: accuracy.rank_measures on hand-built cases
with known answers, its closed-form pair count against brute force, the rankings and testsets it refuses, the measure
names of cross_validate and the searches, and the route for algorithms that are not device-batched."""
import os
import re

import numpy as np
import pytest

import surprise_b200 as sb
from surprise_b200 import _native as nat
from surprise_b200 import accuracy
from surprise_b200.model_selection import GridSearchCV, KFold, LeaveOneOut, cross_validate, fit_and_score

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bits(x):
    return np.float64(x).tobytes()


def same_result(a, b):
    return list(a) == list(b) and all(bits(a[k]) == bits(b[k]) for k in a)


def toy_trainset(offset_scale=False):
    """Items x, y, z, w.  a rated x, y (candidates z, w); b rated x, y, z (candidate w); c rated x twice and w
    (candidates y, z)."""
    rows = [("a", "x", 4.0), ("a", "y", 2.0), ("b", "x", 5.0), ("b", "y", 3.0), ("b", "z", 1.0), ("c", "x", 1.0),
            ("c", "w", 4.0), ("c", "x", 2.0)]
    u, i, r = (np.array([row[k] for row in rows]) for k in range(3))
    reader = sb.Reader(rating_scale=(-10, 10) if offset_scale else (1, 5))
    return sb.Dataset.load_from_arrays(u, i, r.astype(np.float64), reader).build_full_trainset()


def rank(ts, top, testset, threshold=None):
    return accuracy.rank_measures(top, testset, ts, threshold, verbose=False)


# -- the definition --------------------------------------------------------------------------------------------------
def test_closed_form_pair_count_equals_brute_force():
    rng = np.random.RandomState(0)
    for _ in range(500):
        c = int(rng.randint(0, 40))
        rel = set(rng.choice(c, rng.randint(0, c + 1), replace=False).tolist()) if c else set()
        unranked = int(rng.randint(0, 4))
        k = len(rel)
        s = sum(rel)
        # a relevant item ordered above a negative; unranked relevant items order no pair
        brute = sum(1 for p in rel for q in range(c) if q not in rel and p < q)
        assert k * (c - 1) - s - k * (k - 1) // 2 == brute, (c, rel)
        n_rel = k + unranked
        if c - k > 0 and n_rel:
            f = min(rel) if rel else -1
            got = accuracy._rank_of_counts([c], [k], [s], [f], [n_rel], False)["auc"]
            assert bits(got) == bits(brute / (n_rel * (c - k)))


def test_perfect_and_reversed_rankings():
    ts = toy_trainset()
    tes = [("a", "z", 5.0)]
    got = rank(ts, {"a": [("z", 4.0), ("w", 3.0)]}, tes)
    assert got == {"auc": 1.0, "mrr": 1.0, "mpr": 0.0}
    got = rank(ts, {"a": [("w", 4.0), ("z", 3.0)]}, tes)
    assert got == {"auc": 0.0, "mrr": 0.5, "mpr": 1.0}


def test_unknown_user_and_unranked_items():
    ts = toy_trainset()
    top = {"a": [("w", 4.0), ("z", 3.0)], "b": [("w", 1.0)], "c": [("z", 2.0), ("y", 1.0)]}
    # nobody: unknown user (no AUC, mpr_u = n_rel); a: z at 1 and an unknown item; c: y at 1 and x, which c rated
    tes = [("nobody", "x", 3.0), ("a", "z", 3.0), ("a", "new", 4.0), ("c", "y", 5.0), ("c", "x", 2.0)]
    got = rank(ts, top, tes)
    # a: c=2, k=1, s=1, n_rel=2: correct = 1 - 1 = 0; mpr_u = 1 / 1 + 1.  c: the same
    assert bits(got["auc"]) == bits(0.0)
    assert bits(got["mrr"]) == bits(float(np.mean([0.0, 0.5, 0.5])))
    assert bits(got["mpr"]) == bits((1.0 + 2.0 + 2.0) / 5)
    # a better ranking for a: z first gives correct = 1 of n_rel * neg = 2 pairs
    top["a"] = [("z", 4.0), ("w", 3.0)]
    got = rank(ts, top, tes)
    assert bits(got["auc"]) == bits(float(np.mean([0.5, 0.0])))


def test_every_candidate_relevant_and_single_candidate():
    ts = toy_trainset()
    top = {"a": [("w", 4.0), ("z", 3.0)], "b": [("w", 1.0)], "c": [("z", 2.0), ("y", 1.0)]}
    # a's both candidates are relevant: no negative, no AUC; the only such user gives nan
    got = rank(ts, top, [("a", "z", 3.0), ("a", "w", 3.0)])
    assert np.isnan(got["auc"]) and got["mrr"] == 1.0 and bits(got["mpr"]) == bits(1.0 / 2)
    # b has one candidate (c_u = 1): percentile 0.0, and no negative
    got = rank(ts, top, [("b", "w", 3.0)])
    assert np.isnan(got["auc"]) and got == {"auc": got["auc"], "mrr": 1.0, "mpr": 0.0}
    # b's relevant item y was rated: unranked, one negative (w) ordered above it
    got = rank(ts, top, [("b", "y", 3.0)])
    assert got == {"auc": 0.0, "mrr": 0.0, "mpr": 1.0}
    # users without a negative are left out of the AUC mean, not counted as 0 or 1
    got = rank(ts, top, [("a", "z", 3.0), ("a", "w", 3.0), ("c", "y", 1.0)])
    assert got["auc"] == 0.0


def test_threshold_with_an_offset_dataset(capsys):
    ts = toy_trainset(offset_scale=True)
    off = ts.offset
    assert off != 0
    top = {"a": [("w", 4.0), ("z", 3.0)], "b": [("w", 1.0)], "c": [("z", 2.0), ("y", 1.0)]}
    tes = [("a", "z", off + 2.0), ("a", "w", off + 1.5), ("c", "z", off + 2.5), ("b", "w", off - 3.0)]
    # threshold 2: a's z and c's z are relevant
    got = accuracy.rank_measures(top, tes, ts, 2)
    assert got == {"auc": 0.5, "mrr": 0.75, "mpr": 0.5}
    assert [line.split(":")[0] for line in capsys.readouterr().out.splitlines()] == ["AUC", "MRR", "MPR"]
    assert rank(ts, top, tes, 2.5) == {"auc": 1.0, "mrr": 1.0, "mpr": 0.0}
    with pytest.raises(ValueError, match="relevant"):
        rank(ts, top, tes, 3)
    # threshold None: every row, b included
    assert rank(ts, top, tes)["mrr"] == float(np.mean([1.0, 1.0, 1.0]))


def test_duplicated_rows_and_merged_uids():
    ts = toy_trainset()
    top = {"a": [("w", 4.0), ("z", 3.0)], "b": [("w", 1.0)], "c": [("z", 2.0), ("y", 1.0)]}
    tes = [("c", "y", 4.0), ("a", "z", 4.0), ("c", "y", 2.0), ("a", "z", 5.0), ("c", "z", 1.0)]
    # U* = c, a; R_c = {y, z} (both candidates), R_a = {z}
    got = rank(ts, top, tes)
    assert bits(got["mpr"]) == bits((1.0 / 1 + 1.0 / 1) / 3) and got["auc"] == 0.0
    assert got == rank(ts, top, [("c", "z", 1.0), ("a", "z", 1.0), ("c", "y", 1.0)])
    # equal uids of different types are one user, as dict keys merge them
    tes = [(1, "a", 4.0), (1.0, "b", 4.0), (np.int64(1), "a", 5.0)]
    data = sb.Dataset.load_from_arrays(np.array([1, 1, 2]), np.array(["a", "c", "b"]), np.array([3.0, 3.0, 3.0]),
                                       sb.Reader(rating_scale=(1, 5)))
    ts1 = data.build_full_trainset()
    got = accuracy.rank_measures({1: [("b", 1.0)], 2: [("a", 1.0), ("c", 0.0)]}, tes, ts1, verbose=False)
    # user 1: candidate b only, relevant {a (rated), b}: c=1, k=1, n_rel=2
    assert np.isnan(got["auc"]) and got["mrr"] == 1.0 and got["mpr"] == 0.5


def test_incomplete_rankings_and_empty_testsets_are_refused():
    ts = toy_trainset()
    top = {"a": [("w", 4.0), ("z", 3.0)], "b": [("w", 1.0)], "c": [("z", 2.0), ("y", 1.0)]}
    with pytest.raises(ValueError, match="get_top_n"):
        rank(ts, {"a": [("w", 4.0)]}, [("a", "z", 4.0)])
    with pytest.raises(ValueError, match="get_top_n"):
        rank(ts, {}, [("c", "z", 4.0)])
    with pytest.raises(ValueError, match="get_top_n"):
        rank(ts, dict(top, nobody=[("x", 1.0)]), [("nobody", "z", 4.0)])
    with pytest.raises(ValueError, match="relevant"):
        rank(ts, top, [])
    with pytest.raises(ValueError, match="relevant"):
        rank(ts, top, [("a", "z", 1.0)], 4)


# -- the method's non-batched route ----------------------------------------------------------------------------------
def small_data(seed=0, n=300):
    rng = np.random.RandomState(seed)
    uids = rng.zipf(1.5, n) % 53 + 100
    iids = rng.randint(0, 60, n) * 3
    rs = rng.randint(1, 6, n).astype(np.float64)
    return sb.Dataset.load_from_arrays(uids, iids, rs, sb.Reader(rating_scale=(1, 5)))


class PyAlgo(sb.AlgoBase):
    """An algorithm with a Python estimate (not device-batched), with ties and a prediction it cannot make."""

    def __init__(self, shift=0):
        sb.AlgoBase.__init__(self)
        self.shift = shift

    def estimate(self, u, i):
        if not (self.trainset.knows_user(u) and self.trainset.knows_item(i)):
            raise sb.PredictionImpossible("unknown")
        return float((u * 7 + (i + self.shift) * 3) % (5 + self.shift)) + 0.5


def test_non_batched_route_equals_the_definition():
    data = small_data(1)
    loo = next(LeaveOneOut(1, random_state=0).split(data))
    kf = next(KFold(3, random_state=0).split(data))
    for trs, tes in (loo, kf):
        tes = list(tes) + [(999, 3, 5.0), (tes[0][0], 100000, 4.0), (999, 100000, 2.0)]
        algo = PyAlgo().fit(trs)
        assert not algo._batched()
        top = algo.get_top_n(trs.n_items)
        for threshold in (None, 3.5, 4):
            want = accuracy.rank_measures(top, tes, trs, threshold, verbose=False)
            assert same_result(algo.rank_measures(tes, threshold), want), threshold


# -- cross_validate / searches ---------------------------------------------------------------------------------------
def test_measure_names():
    for name in ("auc", "AUC", "Mrr", "mpr"):
        assert accuracy._rank_measure(name) == name.lower()
        assert accuracy._top_n_measure(name) is None and accuracy._top_n_list_measure(name) is None
    for other in ("rmse", "fcp", "hr@10", "auc@10", "gauc", "mpr@5"):
        assert accuracy._rank_measure(other) is None


def test_train_measures_are_refused_with_rank_measures():
    data = small_data(4)
    trs, tes = next(LeaveOneOut(1, random_state=0).split(data))
    algo = PyAlgo()
    with pytest.raises(ValueError, match="return_train_measures"):
        fit_and_score(algo, trs, tes, ["rmse", "auc"], return_train_measures=True)
    assert not hasattr(algo, "trainset")          # refused before the fit
    for m in ("MRR", "mpr"):
        with pytest.raises(ValueError, match="return_train_measures"):
            cross_validate(algo, data, [m], cv=LeaveOneOut(2), return_train_measures=True)


def test_cross_validate_with_rank_measures():
    data = small_data(5)
    measures = ["hr@3", "AUC", "rmse", "mpr", "Mrr"]
    got = cross_validate(PyAlgo(), data, measures, cv=LeaveOneOut(2, random_state=3))
    assert list(got)[:5] == ["test_" + m.lower() for m in measures]
    for k, (trs, tes) in enumerate(LeaveOneOut(2, random_state=3).split(data)):
        algo = PyAlgo().fit(trs)
        want = accuracy.rank_measures(algo.get_top_n(trs.n_items), tes, trs, verbose=False)
        for key in ("auc", "mpr", "mrr"):
            assert bits(got["test_" + key][k]) == bits(want[key]), (k, key)
        assert bits(got["test_hr@3"][k]) == bits(algo.top_n_measures(tes, 3)["hr"])


def test_search_rank_direction():
    data = small_data(6)
    measures = ["auc", "mrr", "mpr", "rmse"]
    gs = GridSearchCV(PyAlgo, {"shift": [0, 1, 2, 3]}, measures=measures, cv=LeaveOneOut(2, random_state=0))
    gs.fit(data)
    for m, pick in (("auc", np.argmax), ("mrr", np.argmax), ("mpr", np.argmin)):
        mean = gs.cv_results["mean_test_" + m]
        assert len(set(mean.tolist())) == len(mean), m
        best = int(pick(mean))
        assert gs.best_index[m] == best and gs.best_params[m] == {"shift": best}
        order = np.argsort(np.argsort(mean)) + 1
        want = order if m == "mpr" else len(mean) + 1 - order
        assert gs.cv_results["rank_test_" + m].tolist() == want.tolist(), m


def test_header_and_signature():
    hdr = open(os.path.join(ROOT, "include", "surprise_b200.h")).read()
    decl = re.search(r"int sb2_top_n_ranks_dev\((.*?)\);", hdr, re.S).group(1)
    assert len(decl.split(",")) == len(nat.SIGNATURES["sb2_top_n_ranks_dev"][1]) == 20
    assert "int64_t* s" in decl and "const int32_t* rel_idx" in decl
    src = open(os.path.join(ROOT, "surprise_b200", "csrc", "api.cu")).read()
    assert re.search(r"int sb2_top_n_ranks_dev\(", src)
