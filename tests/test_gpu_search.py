"""GridSearchCV / RandomizedSearchCV and cross_validate on the device: every score of the array route equals, bit for
bit, accuracy.<m>(algo.test(...)) on the same fitted model, for every device-batched algorithm, with unknown users and
items, train measures, a fold whose k-NN estimates raise ZeroDivisionError, a non-batched subclass and an
ml-1M-shaped fold."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import accuracy, synth  # noqa: E402
from surprise_b200.model_selection import (GridSearchCV, RandomizedSearchCV, ShuffleSplit, cross_validate,  # noqa: E402
                                           fit_and_score)

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MEASURES = ["rmse", "mse", "mae", "fcp"]


class Folds(object):
    """A splitter that yields fixed (trainset, testset) pairs."""

    def __init__(self, pairs):
        self.pairs = pairs

    def split(self, data):
        return iter(self.pairs)


@pytest.fixture(scope="module")
def u1_folds():
    """The u1 fold with unknown users and items appended, and the reverse fold (fit on u1's test file, score 5 000
    rows of its train file, many of them unknown)."""
    reader = sb.Reader("ml-100k")
    data = sb.Dataset.load_from_folds([(os.path.join(GOLDEN, "u1_ml100k_train"),
                                        os.path.join(GOLDEN, "u1_ml100k_test"))], reader)
    raw_train, raw_test = next(data.raw_folds())
    trs = data.construct_trainset(raw_train)
    tes = data.construct_testset(raw_test) + [("nobody", "1", 4.0), ("1", "no-item", 2.0), ("nobody", "x", 1.0)]
    small = data.construct_trainset(raw_test)
    return data, [(trs, tes), (small, data.construct_testset(raw_train[:5000]))]


class Recorder(object):
    """An algo_class that keeps every instance the search makes, in task order."""

    def __init__(self, cls):
        self.cls, self.made = cls, []

    def __call__(self, **params):
        algo = self.cls(**params)
        self.made.append(algo)
        return algo


def assert_search_matches_tuple_route(search, rec, folds):
    n_c = len(search.param_combinations)
    res = search.cv_results
    for k, algo in enumerate(rec.made[:n_c * len(folds)]):
        c, f = divmod(k, len(folds))
        trs, tes = folds[f]
        assert algo.trainset is trs
        for part, preds in (("test", algo.test(tes)), ("train", algo.test(trs.build_testset()))):
            for m in MEASURES:
                want = getattr(accuracy, m)(preds, verbose=False)
                got = res["split%d_%s_%s" % (f, part, m)][c]
                assert np.float64(got).tobytes() == np.float64(want).tobytes(), (type(algo).__name__, c, f, part, m)


CASES = {
    "svd": (sb.SVD, {"n_factors": [10, 30], "n_epochs": [5], "random_state": [0], "lr_all": [0.005, 0.01]}),
    "svdpp": (sb.SVDpp, {"n_factors": [5], "n_epochs": [3, 5], "random_state": [1]}),
    "nmf": (sb.NMF, {"n_factors": [5, 15], "n_epochs": [10], "random_state": [0]}),
    "nmf_biased": (sb.NMF, {"n_factors": [5], "n_epochs": [10], "biased": [True], "random_state": [0, 3]}),
    "baseline_only": (sb.BaselineOnly, {"bsl_options": {"method": ["als", "sgd"], "n_epochs": [5]}}),
    "knn_basic": (sb.KNNBasic, {"k": [10, 40], "sim_options": {"name": ["msd", "cosine"], "user_based": [True]}}),
    "knn_means": (sb.KNNWithMeans, {"k": [20], "min_k": [1, 5], "sim_options": {"name": ["pearson"],
                                                                              "user_based": [False]}}),
    "knn_zscore": (sb.KNNWithZScore, {"k": [20], "sim_options": {"name": ["msd"], "user_based": [True, False]}}),
    "knn_baseline": (sb.KNNBaseline, {"k": [30], "sim_options": {"name": ["pearson_baseline", "msd"],
                                                                "user_based": [False]}}),
    "slope_one": (sb.SlopeOne, {}),
    "coclustering": (sb.CoClustering, {"n_cltr_u": [3, 5], "n_epochs": [5], "random_state": [0]}),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_grid_search_scores_equal_tuple_route(u1_folds, case):
    data, folds = u1_folds
    cls, grid = CASES[case]
    rec = Recorder(cls)
    gs = GridSearchCV(rec, grid, measures=MEASURES, cv=Folds(folds), return_train_measures=True)
    gs.fit(data)
    assert len(rec.made) == len(gs.param_combinations) * len(folds) + len(MEASURES)
    assert_search_matches_tuple_route(gs, rec, folds)


def test_randomized_search_scores_equal_tuple_route(u1_folds):
    from scipy import stats
    data, folds = u1_folds
    rec = Recorder(sb.SVD)
    rs = RandomizedSearchCV(rec, {"lr_all": stats.uniform(0.002, 0.01), "n_factors": [8, 16], "n_epochs": [4],
                                  "random_state": [0]}, n_iter=3, measures=MEASURES, cv=Folds(folds),
                            return_train_measures=True, random_state=5)
    rs.fit(data)
    assert_search_matches_tuple_route(rs, rec, folds)


def test_non_batched_subclass_takes_the_tuple_route(u1_folds):
    data, folds = u1_folds

    class PySVD(sb.SVD):
        def estimate(self, u, i):           # a Python estimate: test() goes pair by pair
            return sb.SVD.estimate(self, u, i) + 0.25

    algo = PySVD(n_factors=5, n_epochs=2, random_state=0)
    assert not algo._batched()
    trs, tes = folds[1]
    test_m = fit_and_score(algo, trs, tes[:500], MEASURES)[0]
    preds = algo.test(tes[:500])
    for m in MEASURES:
        assert np.float64(test_m[m]).tobytes() == np.float64(getattr(accuracy, m)(preds, verbose=False)).tobytes()


def test_zero_division_fold(u1_folds):
    class ZeroSim(sb.KNNBasic):
        def fit(self, trainset):
            sb.KNNBasic.fit(self, trainset)
            self.sim = np.zeros((self.n_x, self.n_x))     # no positive neighbour: 0 / 0 with min_k = 0
            return self

    data, folds = u1_folds
    trs, tes = folds[1]
    algo = ZeroSim(k=5, min_k=0)
    assert algo._batched()
    with pytest.raises(ZeroDivisionError):
        fit_and_score(algo, trs, tes, ["rmse"])
    with pytest.raises(ZeroDivisionError):
        algo.test(tes)
    with pytest.raises(ZeroDivisionError):
        GridSearchCV(ZeroSim, {"min_k": [0]}, cv=Folds(folds)).fit(data)
    # min_k = 1 makes the same pairs impossible instead: default prediction on both routes
    algo = ZeroSim(k=5, min_k=1)
    got = fit_and_score(algo, trs, tes, MEASURES)[0]
    preds = algo.test(tes)
    assert all(p.details["was_impossible"] for p in preds)
    for m in MEASURES:
        assert np.float64(got[m]).tobytes() == np.float64(getattr(accuracy, m)(preds, verbose=False)).tobytes()


def test_cross_validate_on_ml1m_fold():
    d = synth.ratings(*synth.SHAPES["ml-1m"][:3], seed=0, skew=True)
    u, i, r = d["train"]
    data = sb.Dataset.load_from_arrays(u, i, r, sb.Reader(rating_scale=(1, 5)))
    cv = ShuffleSplit(n_splits=1, test_size=0.2, random_state=0)
    for algo in (sb.SVD(n_factors=100, random_state=0), sb.KNNBaseline(sim_options={"name": "pearson_baseline",
                                                                                  "user_based": False})):
        got = cross_validate(algo, data, MEASURES, cv, return_train_measures=True)
        trs, tes = next(cv.split(data))
        # algo is left fitted on the fold; the fold's rows are the same ones
        for part, preds in (("test_", algo.test(tes)), ("train_", algo.test(algo.trainset.build_testset()))):
            for m in MEASURES:
                want = np.array([getattr(accuracy, m)(preds, verbose=False)])
                assert got[part + m].tobytes() == want.tobytes(), (type(algo).__name__, part, m)
