"""Coverage, novelty and diversity of top-N lists, without a GPU: accuracy.top_n_list_measures on hand-built cases with
known answers, the novelty table, the measure names of cross_validate and the searches, the arguments the method
refuses, the route for algorithms that are not device-batched, and the native entry point's declaration."""
import os
import re
from math import log2

import numpy as np
import pytest

import surprise_b200 as sb
from surprise_b200 import _native as nat
from surprise_b200 import accuracy
from surprise_b200.model_selection import GridSearchCV, LeaveOneOut, cross_validate, fit_and_score

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAN = float("nan")


def bits(x):
    return np.float64(x).tobytes()


def same_result(a, b):
    return list(a) == list(b) and all(bits(a[k]) == bits(b[k]) for k in a)


def toy_trainset(offset_scale=False):
    """Users a, b, c; items x, y, z, w; (c, x) rated twice, so x has 4 ratings and the others 1."""
    rows = [("a", "x", 4.0), ("a", "y", 2.0), ("b", "x", 5.0), ("b", "z", 3.0), ("c", "x", 1.0), ("c", "w", 4.0),
            ("c", "x", 2.0)]
    u, i, r = (np.array([row[k] for row in rows]) for k in range(3))
    reader = sb.Reader(rating_scale=(-10, 10) if offset_scale else (1, 5))
    return sb.Dataset.load_from_arrays(u, i, r.astype(np.float64), reader).build_full_trainset()


def inner_sim(ts):
    """A symmetric sim over inner ids whose entries tell the pairs apart."""
    k = np.arange(ts.n_items, dtype=np.float64)
    return 1.0 / (1.0 + np.add.outer(k, 2 * k) + np.add.outer(2 * k, k))


TOP = {"a": [("z", 4.0), ("w", 3.0)], "b": [("y", NAN), ("w", 3.5)]}


def test_novelty_table_counts_duplicate_ratings():
    ts = toy_trainset()
    cnt = np.array([len(ts.ir[i]) for i in range(ts.n_items)])
    assert cnt[ts.to_inner_iid("x")] == 4 and sorted(cnt.tolist()) == [1, 1, 1, 4]
    assert accuracy._novelty_table(ts).tobytes() == np.log2(3 / cnt.astype(np.int64)).tobytes()


def test_known_values_and_thresholds():
    ts = toy_trainset()
    sim = inner_sim(ts)
    z, w, y = (ts.to_inner_iid(i) for i in "zwy")
    got = accuracy.top_n_list_measures(TOP, ts, 10, sim=sim, verbose=False)
    # U = a, b, c in inner order; c has no list
    assert list(got) == ["user_coverage", "catalog_coverage", "novelty", "diversity"]
    assert got["user_coverage"] == 2 / 3 and got["catalog_coverage"] == 3 / 4
    assert got["novelty"] == float(np.sum([0.0 + log2(3) + log2(3)] * 2)) / 4
    assert got["diversity"] == 1.0 - float(np.sum([0.0 + sim[z, w], 0.0 + sim[y, w]])) / 2
    # a NaN est never passes; 3.5 >= 3.5 does
    for threshold, want in ((3.5, 2 / 3), (4, 1 / 3), (np.float64(4.0), 1 / 3), (4.5, 0.0), (-np.inf, 2 / 3)):
        got_t = accuracy.top_n_list_measures(TOP, ts, 10, threshold=threshold, sim=sim, verbose=False)
        assert got_t["user_coverage"] == want, threshold
        assert same_result({k: v for k, v in got_t.items() if k != "user_coverage"},
                           {k: v for k, v in got.items() if k != "user_coverage"})
    # without sim there is no diversity
    assert list(accuracy.top_n_list_measures(TOP, ts, 10, verbose=False)) == ["user_coverage", "catalog_coverage",
                                                                              "novelty"]


def test_n_one_has_no_pairs_and_large_n_takes_whole_lists():
    ts = toy_trainset()
    sim = inner_sim(ts)
    got = accuracy.top_n_list_measures(TOP, ts, 1, threshold=3.5, sim=sim, verbose=False)
    assert np.isnan(got["diversity"]) and got["user_coverage"] == 1 / 3 and got["catalog_coverage"] == 2 / 4
    assert got["novelty"] == 2 * log2(3) / 2
    assert same_result(accuracy.top_n_list_measures(TOP, ts, 10 ** 12, sim=sim, verbose=False),
                       accuracy.top_n_list_measures(TOP, ts, 2, sim=sim, verbose=False))
    for bad in (0, -1, True, 2.5, "3", None):
        with pytest.raises(ValueError):
            accuracy.top_n_list_measures(TOP, ts, bad, verbose=False)


def test_duplicate_unknown_and_listless_users():
    ts = toy_trainset()
    got = accuracy.top_n_list_measures(TOP, ts, 10, uids=["b", "nobody", "b", "a", "nobody"], verbose=False)
    assert got["user_coverage"] == 2 / 3 and got["catalog_coverage"] == 3 / 4
    # no user with a list: novelty and diversity are nan
    got = accuracy.top_n_list_measures(TOP, ts, 10, uids=["c", "nobody"], sim=inner_sim(ts), verbose=False)
    assert got["user_coverage"] == 0.0 and got["catalog_coverage"] == 0.0
    assert np.isnan(got["novelty"]) and np.isnan(got["diversity"])
    # equal uids merge as dict keys
    top = {1: [("x", 2.0)]}
    ts_int = sb.Dataset.load_from_arrays(np.array([1, 2]), np.array(["x", "y"]), np.array([3.0, 4.0]),
                                         sb.Reader(rating_scale=(1, 5))).build_full_trainset()
    assert accuracy.top_n_list_measures(top, ts_int, 5, uids=[1, 1.0, True], verbose=False)["user_coverage"] == 1.0
    with pytest.raises(ValueError):
        accuracy.top_n_list_measures(TOP, ts, 10, uids=[], verbose=False)


def test_bad_sim_shape():
    ts = toy_trainset()
    for shape in ((3, 3), (4, 5), (16,), (4, 4, 1)):
        with pytest.raises(ValueError, match="sim"):
            accuracy.top_n_list_measures(TOP, ts, 10, sim=np.zeros(shape), verbose=False)


def test_offset_trainset(capsys):
    ts = toy_trainset(offset_scale=True)
    assert ts.offset == 11
    top = {"a": [("z", -6.0), ("w", -7.5)], "b": [("y", -7.0)]}
    for threshold, want in ((None, 2 / 3), (-7.0, 2 / 3), (-6.5, 1 / 3), (np.float64(-6.0), 1 / 3), (0, 0.0)):
        got = accuracy.top_n_list_measures(top, ts, 10, threshold=threshold, verbose=False)
        assert got["user_coverage"] == want, threshold
        assert got["novelty"] == float(np.sum([0.0 + log2(3) + log2(3), 0.0 + log2(3)])) / 3
    accuracy.top_n_list_measures(top, ts, 10, sim=inner_sim(ts))
    out = capsys.readouterr().out.splitlines()
    assert [line.split(":")[0] for line in out] == ["User coverage@10", "Catalog coverage@10", "Novelty@10",
                                                    "Diversity@10"]


# -- the method's arguments and the non-batched route ----------------------------------------------------------------
def small_data(seed=0, n=300):
    rng = np.random.RandomState(seed)
    uids = rng.zipf(1.5, n) % 53 + 100
    iids = rng.randint(0, 60, n) * 3
    rs = rng.randint(1, 6, n).astype(np.float64)
    return sb.Dataset.load_from_arrays(uids, iids, rs, sb.Reader(rating_scale=(1, 5)))


class PyAlgo(sb.AlgoBase):
    """An algorithm with a Python estimate (not device-batched), with ties and a prediction it cannot make."""

    def estimate(self, u, i):
        if not (self.trainset.knows_user(u) and self.trainset.knows_item(i)):
            raise sb.PredictionImpossible("unknown")
        return float((u * 7 + i * 3) % 5) + 0.5


def test_non_batched_route_equals_the_definition():
    ts = small_data(1).build_full_trainset()
    algo = PyAlgo().fit(ts)
    assert not algo._batched()
    sim = inner_sim(ts)
    some = [ts.to_raw_uid(u) for u in (5, 0, 5, 3)]
    for n in (1, 4, ts.n_items + 5):
        for uids in (None, some):
            for threshold in (None, 3.5, 4, np.float64(3.0)):
                got = algo.top_n_list_measures(n, uids, threshold, sim)
                want = accuracy.top_n_list_measures(algo.get_top_n(n, uids), ts, n, uids, threshold, sim,
                                                    verbose=False)
                assert same_result(got, want), (n, uids, threshold)
    with pytest.raises(ValueError):
        algo.top_n_list_measures(5, uids=["nobody"])
    with pytest.raises(ValueError):
        algo.top_n_list_measures(5, uids=[])
    with pytest.raises(ValueError, match="sim"):
        algo.top_n_list_measures(5, sim=np.zeros((ts.n_items, ts.n_items + 1)))


def knn_model(trainset, user_based=False, streamed=False):
    """A k-NN model as fit() leaves it, without building its matrix (which needs the device)."""
    model = sb.KNNBasic(sim_options={"name": "cosine", "user_based": user_based})
    sb.AlgoBase.fit(model, trainset)
    model._streamed, model._sim_host, model._sim_dev = streamed, None, None
    return model


def test_sim_models_that_are_refused():
    ts = small_data(2).build_full_trainset()
    other = small_data(3).build_full_trainset()
    algo = PyAlgo().fit(ts)
    for model, why in ((knn_model(other), "trainset"), (knn_model(ts, user_based=True), "item-based"),
                       (knn_model(ts, streamed=True), "streamed")):
        with pytest.raises(ValueError, match=why):
            algo.top_n_list_measures(5, sim=model)


# -- cross_validate / searches ---------------------------------------------------------------------------------------
def test_measure_names():
    parse = accuracy._top_n_list_measure
    assert parse("Novelty@10") == ("novelty", 10) and parse("USER_COVERAGE@007") == ("user_coverage", 7)
    assert parse("catalog_coverage@1") == ("catalog_coverage", 1) and parse("diversity@100") == ("diversity", 100)
    for other in ("rmse", "fcp", "hr@10", "novelty", "coverage@3", "foo@3", "ndcg@5"):
        assert parse(other) is None
    for bad in ("novelty@0", "diversity@", "catalog_coverage@-1", "user_coverage@1.5", "novelty@x", "diversity@ 3"):
        with pytest.raises(ValueError):
            parse(bad)
    # the hit measures' parser does not take the list names
    for name in ("novelty@3", "diversity@10", "user_coverage@1", "catalog_coverage@5"):
        assert accuracy._top_n_measure(name) is None


def test_train_measures_are_refused_with_list_measures():
    data = small_data(4)
    trs, tes = next(LeaveOneOut(1, random_state=0).split(data))
    algo = PyAlgo()
    with pytest.raises(ValueError, match="return_train_measures"):
        fit_and_score(algo, trs, tes, ["rmse", "novelty@10"], return_train_measures=True)
    assert not hasattr(algo, "trainset")          # refused before the fit
    for m in ("user_coverage@5", "catalog_coverage@5", "diversity@5"):
        with pytest.raises(ValueError):
            cross_validate(algo, data, [m], cv=LeaveOneOut(2), return_train_measures=True)


def test_cross_validate_with_list_measures():
    data = small_data(5)
    measures = ["hr@3", "Novelty@3", "rmse", "catalog_coverage@10", "user_coverage@3"]
    got = cross_validate(PyAlgo(), data, measures, cv=LeaveOneOut(2, random_state=3))
    assert list(got)[:5] == ["test_" + m.lower() for m in measures]
    for k, (trs, tes) in enumerate(LeaveOneOut(2, random_state=3).split(data)):
        algo = PyAlgo().fit(trs)
        star = [u for u, _, _ in tes]              # U*: every test user, unknown ones included
        assert any(trs.to_inner_uids([u])[0] < 0 for u in star)
        for n, names in ((3, ("novelty", "user_coverage")), (10, ("catalog_coverage",))):
            want = accuracy.top_n_list_measures(algo.get_top_n(n), trs, n, star, verbose=False)
            for key in names:
                assert bits(got["test_%s@%d" % (key, n)][k]) == bits(want[key]), (k, key, n)
        assert bits(got["test_hr@3"][k]) == bits(algo.top_n_measures(tes, 3)["hr"])


def test_search_ranks_list_measures_descending():
    data = small_data(6)

    class Shifted(PyAlgo):
        def __init__(self, shift=0):
            PyAlgo.__init__(self)
            self.shift = shift

        def estimate(self, u, i):
            PyAlgo.estimate(self, u, i)              # raises for unknown ids
            return float((u * 7 + (i + self.shift) * 3) % (5 + self.shift)) + 0.5

    measures = ["catalog_coverage@5", "novelty@5", "user_coverage@5", "rmse"]
    gs = GridSearchCV(Shifted, {"shift": [0, 1, 2, 3]}, measures=measures, cv=LeaveOneOut(2, random_state=0))
    gs.fit(data)
    for m in measures[:3]:
        mean = gs.cv_results["mean_test_" + m]
        best = int(np.argmax(mean))
        assert gs.best_index[m] == best and gs.best_params[m] == {"shift": best}
        assert gs.cv_results["rank_test_" + m].tolist() == (len(mean) - np.argsort(np.argsort(mean))).tolist()
    assert len(set(gs.cv_results["mean_test_catalog_coverage@5"].tolist())) > 1


def test_header_and_signature():
    hdr = open(os.path.join(ROOT, "include", "surprise_b200.h")).read()
    decl = re.search(r"int sb2_top_n_lists_dev\((.*?)\);", hdr, re.S).group(1)
    assert "sb2_top_n_lists_dev" in nat.SIGNATURES
    assert len(decl.split(",")) == len(nat.SIGNATURES["sb2_top_n_lists_dev"][1]) == 16
    assert "double threshold" in decl and "uint8_t* seen" in decl
    src = open(os.path.join(ROOT, "surprise_b200", "csrc", "api.cu")).read()
    assert re.search(r"int sb2_top_n_lists_dev\(", src)
