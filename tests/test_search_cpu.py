"""GridSearchCV / RandomizedSearchCV without a GPU: candidates, task order, every cv_results key, ranks with ties,
best_*, refit / predict / test and the ValueErrors, with pure-Python algorithms.  The array scorer of fit_and_score
is checked against algo.test() + accuracy.* on adversarial values (pow-sensitive squares, signed zeros, clipping,
impossible pairs, merged uids), with a CPU stand-in for the device ids."""
import os
from collections import defaultdict

import numpy as np
import pytest
import torch

import surprise_b200 as sb
from surprise_b200 import accuracy
from surprise_b200.model_selection import GridSearchCV, KFold, RandomizedSearchCV, cross_validate, fit_and_score
from surprise_b200.model_selection import validation
from surprise_b200.model_selection.validation import Fold, _fit_and_score
from surprise_b200.prediction_algorithms.predictions import PredictionImpossible

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class Toy(sb.AlgoBase):
    """est = global mean + shift + slope * (inner item id % 3); unknown ids are impossible.  Records every fit."""
    fits = []

    def __init__(self, shift=0.0, slope=0.0, **kwargs):
        sb.AlgoBase.__init__(self, **kwargs)
        self.shift, self.slope = shift, slope

    def fit(self, trainset):
        sb.AlgoBase.fit(self, trainset)
        Toy.fits.append((self.shift, self.slope, trainset))
        return self

    def estimate(self, u, i):
        if not (self.trainset.knows_user(u) and self.trainset.knows_item(i)):
            raise PredictionImpossible("User and/or item is unknown.")
        return self.trainset.global_mean + self.shift + self.slope * (i % 3)


def arrays_data(n=600, seed=0, scale=(1, 5)):
    rng = np.random.RandomState(seed)
    u = rng.randint(0, 40, n)
    i = rng.randint(0, 30, n)
    r = rng.randint(2 * scale[0], 2 * scale[1] + 1, n) / 2.0
    return sb.Dataset.load_from_arrays(u, i, r, sb.Reader(rating_scale=scale))


def file_data(tmp_path, n=300, seed=1):
    """A list-backed dataset with string ids on a scale with an offset."""
    rng = np.random.RandomState(seed)
    path = tmp_path / "ratings.csv"
    path.write_text("".join("u%d,i%d,%d\n" % (rng.randint(25), rng.randint(20), rng.randint(-2, 3)) for _ in range(n)))
    return sb.Dataset.load_from_file(str(path), sb.Reader(line_format="user item rating", sep=",",
                                                           rating_scale=(-2, 2)))


def reference_measures(algo_class, params, folds, measures, train=False):
    """(candidates, folds) arrays of accuracy.<m>(algo.test(...)), fitted one task at a time."""
    out = {m: np.empty((len(params), len(folds))) for m in measures}
    for c, p in enumerate(params):
        for f, (trs, tes) in enumerate(folds):
            algo = algo_class(**p)
            algo.fit(trs)
            preds = algo.test(trs.build_testset() if train else tes)
            for m in measures:
                out[m][c, f] = getattr(accuracy, m)(preds, verbose=False)
    return out


def assert_rank(rank, mean, ascending):
    """Ranks 1..n by mean (ascending, or descending for fcp), ties in the order of mean.argsort(): numpy's default
    sort is not stable on every CPU (its SIMD quicksort), so that order is the definition."""
    n = len(mean)
    assert sorted(rank.tolist()) == list(range(1, n + 1))
    by_rank = mean[np.argsort(rank)]
    assert (np.diff(by_rank) >= 0).all() if ascending else (np.diff(by_rank) <= 0).all()
    order = mean.argsort()
    want = np.empty_like(order)
    want[order] = np.arange(1, n + 1) if ascending else np.arange(n, 0, -1)
    assert rank.tolist() == want.tolist()


# -- candidates --------------------------------------------------------------------------------------------------------
def test_grid_order_and_nested_options():
    grid = {"k": [10, 20], "sim_options": {"name": ["msd", "cosine"], "user_based": [False, True]},
            "bsl_options": {"method": ["als"], "n_epochs": [5, 10]}}
    gs = GridSearchCV(Toy, grid)
    sims = [{"name": n, "user_based": b} for n in ("msd", "cosine") for b in (False, True)]
    bsls = [{"method": "als", "n_epochs": e} for e in (5, 10)]
    want = [{"k": k, "sim_options": s, "bsl_options": b} for k in (10, 20) for s in sims for b in bsls]
    assert gs.param_combinations == want
    assert [list(c) for c in gs.param_combinations] == [["k", "sim_options", "bsl_options"]] * len(want)
    assert grid["sim_options"] == {"name": ["msd", "cosine"], "user_based": [False, True]}   # the caller's dict stays
    assert GridSearchCV(Toy, {"b": [1, 2], "a": [3]}).param_combinations == [{"b": 1, "a": 3}, {"b": 2, "a": 3}]


def test_randomized_lists_draw_distinct_candidates_from_random_state():
    dist = {"shift": [0.0, 0.1, 0.2], "slope": [0.0, 1.0], "sim_options": {"name": ["msd", "cosine"]}}
    grid = GridSearchCV(Toy, dict(dist)).param_combinations
    state = np.random.get_state()
    got = RandomizedSearchCV(Toy, dist, n_iter=7, random_state=3).param_combinations
    assert np.random.get_state()[1].tobytes() == state[1].tobytes()          # numpy's global state untouched
    pick = np.random.RandomState(3).permutation(len(grid))[:7]
    assert got == [grid[k] for k in pick.tolist()]
    assert len({repr(c) for c in got}) == 7
    assert RandomizedSearchCV(Toy, dist, n_iter=7, random_state=3).param_combinations == got
    rs = np.random.RandomState(3)
    assert RandomizedSearchCV(Toy, dist, n_iter=7, random_state=rs).param_combinations == got
    full = RandomizedSearchCV(Toy, dist, n_iter=len(grid), random_state=0).param_combinations
    assert sorted(map(repr, full)) == sorted(map(repr, grid))
    with pytest.raises(ValueError):
        RandomizedSearchCV(Toy, dist, n_iter=len(grid) + 1, random_state=0)


def test_randomized_distributions():
    from scipy import stats
    dist = {"slope": stats.uniform(0, 2), "shift": [0.0, 0.5, 1.0], "bsl_options": {"method": ["als", "sgd"]}}
    got = RandomizedSearchCV(Toy, dist, n_iter=25, random_state=11).param_combinations
    rng = np.random.RandomState(11)
    choices = [{"method": "als"}, {"method": "sgd"}]
    want = []
    for _ in range(25):
        c = {}
        c["bsl_options"] = choices[rng.randint(2)]          # keys in sorted order: bsl_options, shift, slope
        c["shift"] = [0.0, 0.5, 1.0][rng.randint(3)]
        c["slope"] = stats.uniform(0, 2).rvs(random_state=rng)
        want.append(c)
    assert got == want
    assert [list(c) for c in got] == [["bsl_options", "shift", "slope"]] * 25


# -- the search --------------------------------------------------------------------------------------------------------
def test_grid_search_results(tmp_path):
    data = file_data(tmp_path)
    measures = ["RMSE", "mae", "Mse", "fcp"]
    grid = {"shift": [0.5, 0.0, 0.5, -1.0], "slope": [0.0, 0.25]}
    Toy.fits = []
    gs = GridSearchCV(Toy, grid, measures=measures, cv=KFold(3, random_state=0), return_train_measures=True)
    gs.fit(data)
    params = gs.param_combinations
    folds = list(KFold(3, random_state=0).split(data))
    ms = [m.lower() for m in measures]
    assert gs.measures == ms
    # tasks in product(candidates, folds) order, every candidate on the same trainset objects
    assert [(s, p) for s, p, _ in Toy.fits] == [(c["shift"], c["slope"]) for c in params for _ in range(3)]
    assert all(Toy.fits[k][2] is Toy.fits[k % 3][2] for k in range(len(Toy.fits)))
    test = reference_measures(Toy, params, folds, ms)
    train = reference_measures(Toy, params, folds, ms, train=True)
    res = gs.cv_results
    for m in ms:
        for k in range(3):
            assert res["split%d_test_%s" % (k, m)].tobytes() == test[m][:, k].tobytes()
            assert res["split%d_train_%s" % (k, m)].tobytes() == train[m][:, k].tobytes()
        assert res["mean_test_" + m].tobytes() == test[m].mean(axis=1).tobytes()
        assert res["std_test_" + m].tobytes() == test[m].std(axis=1).tobytes()
        assert res["mean_train_" + m].tobytes() == train[m].mean(axis=1).tobytes()
        assert res["std_train_" + m].tobytes() == train[m].std(axis=1).tobytes()
        mean = test[m].mean(axis=1)
        asc = m != "fcp"
        assert_rank(res["rank_test_" + m], mean, asc)
        best = int(np.argmin(mean) if asc else np.argmax(mean))
        assert gs.best_index[m] == best
        assert gs.best_params[m] == params[best]
        assert gs.best_score[m] == mean[best]
        est = gs.best_estimator[m]
        assert isinstance(est, Toy) and (est.shift, est.slope) == (params[best]["shift"], params[best]["slope"])
        assert not hasattr(est, "trainset")
    # the two equal candidates tie in every measure
    assert all(res["mean_test_" + m][0] == res["mean_test_" + m][4] for m in ms)
    for s in ("fit", "test"):
        assert res["mean_%s_time" % s].shape == res["std_%s_time" % s].shape == (len(params),)
    assert res["params"] is params
    assert res["param_shift"] == [c["shift"] for c in params] and res["param_slope"] == [c["slope"] for c in params]
    want_keys = set()
    for m in ms:
        want_keys |= {"split%d_%s_%s" % (k, p, m) for k in range(3) for p in ("test", "train")}
        want_keys |= {"%s_%s_%s" % (a, p, m) for a in ("mean", "std") for p in ("test", "train")} | {"rank_test_" + m}
    want_keys |= {"mean_fit_time", "std_fit_time", "mean_test_time", "std_test_time", "params", "param_shift",
                  "param_slope"}
    assert set(res) == want_keys
    with pytest.raises(ValueError, match="refit is False"):
        gs.predict("u1", "i1")
    with pytest.raises(ValueError, match="refit is False"):
        gs.test([("u1", "i1", 3.0)])


def test_rank_ties_in_candidate_order():
    # constant ratings: rmse = |shift| exactly, so the ties are exact
    u = np.repeat(np.arange(10), 10)
    i = np.tile(np.arange(10), 10)
    data = sb.Dataset.load_from_arrays(u, i, np.full(100, 3.0), sb.Reader(rating_scale=(1, 5)))
    gs = GridSearchCV(Toy, {"shift": [1.0, 1.0, -1.0, 0.0, 0.5]}, measures=["rmse", "mae"], cv=2)
    gs.fit(data)
    assert gs.cv_results["mean_test_rmse"].tolist() == [1.0, 1.0, 1.0, 0.0, 0.5]
    rank = gs.cv_results["rank_test_rmse"]
    assert rank[3] == 1 and rank[4] == 2 and sorted(rank[[0, 1, 2]].tolist()) == [3, 4, 5]
    assert_rank(rank, gs.cv_results["mean_test_rmse"], True)
    assert gs.best_index["rmse"] == 3 and gs.best_params["rmse"] == {"shift": 0.0}


def test_cv_resolution_and_refit():
    data = arrays_data()
    gs = GridSearchCV(Toy, {"shift": [0.0, 0.3]}, cv=None, refit=True)
    gs.fit(data)
    assert len([k for k in gs.cv_results if k.startswith("split") and k.endswith("_test_rmse")]) == 5
    assert gs.refit == "rmse"
    best = gs.best_estimator["rmse"]
    assert best.trainset.n_ratings == 600
    assert gs.predict(3, 4) == best.predict(3, 4)
    te = [(3, 4, 2.0), (99, 4, 1.0)]
    assert gs.test(te) == best.test(te)
    gs = GridSearchCV(Toy, {"shift": [0.0]}, measures=["MAE", "rmse"], cv=4, refit="Mae")
    gs.fit(data)
    assert gs.refit == "mae" and len([k for k in gs.cv_results if k.endswith("_test_mae") and "split" in k]) == 4
    assert gs.best_estimator["mae"].trainset.n_ratings == 600 and not hasattr(gs.best_estimator["rmse"], "trainset")
    assert GridSearchCV(Toy, {"shift": [0.0]}, refit=False).refit is False
    with pytest.raises(ValueError, match="refit"):
        GridSearchCV(Toy, {"shift": [0.0]}, measures=["rmse"], refit="fcp")
    with pytest.raises(ValueError, match="refit"):
        RandomizedSearchCV(Toy, {"shift": [0.0]}, n_iter=1, measures=["rmse"], refit="mae")


def test_refit_refuses_predefined_folds():
    from surprise_b200.model_selection import PredefinedKFold
    data = sb.Dataset.load_from_folds([(os.path.join(GOLDEN, "u1_ml100k_train"),
                                        os.path.join(GOLDEN, "u1_ml100k_test"))], sb.Reader("ml-100k"))
    with pytest.raises(ValueError, match="load_from_folds"):
        GridSearchCV(Toy, {"shift": [0.0]}, cv=PredefinedKFold(), refit=True).fit(data)
    gs = RandomizedSearchCV(Toy, {"shift": [0.0, 0.2]}, n_iter=2, cv=PredefinedKFold(), random_state=0,
                            measures=["rmse"])
    gs.fit(data)
    assert sorted(k for k in gs.cv_results if k.startswith("split")) == ["split0_test_rmse"]


# -- the array route, with CPU tensors standing in for device ids -----------------------------------------------------
class Batched(sb.AlgoBase):
    """A batched algorithm on the host: est from a table (so tests can place differences), code 1 for unknown ids and
    code 2 where ``zero_div`` marks the pair."""

    def __init__(self, table, unknown_est=7.0, zero_div=None):
        sb.AlgoBase.__init__(self)
        self.table, self.unknown_est, self.zero_div = table, unknown_est, zero_div

    def _estimate_dev(self, d_u, d_i):
        u, i = d_u.numpy().astype(np.int64), d_i.numpy().astype(np.int64)
        known = (u >= 0) & (i >= 0)
        est = np.where(known, self.table[np.maximum(u, 0), np.maximum(i, 0)], self.unknown_est)
        code = np.where(known, 0, 1).astype(np.uint8)
        if self.zero_div is not None:
            code[known & self.zero_div[np.maximum(u, 0), np.maximum(i, 0)]] = 2
        return torch.from_numpy(est), torch.from_numpy(code)

    def _estimate_batch(self, iu, ii):
        est, code = self._estimate_dev(torch.from_numpy(np.asarray(iu)), torch.from_numpy(np.asarray(ii)))
        est, code = est.numpy(), code.numpy()
        if (code == 2).any():
            raise ZeroDivisionError("division by zero")
        return est, [{"was_impossible": bool(c)} for c in code]

    def estimate(self, u, i):
        est, details = self._estimate_batch(np.array([u if isinstance(u, int) else -1], dtype=np.int32),
                                            np.array([i if isinstance(i, int) else -1], dtype=np.int32))
        if details[0]["was_impossible"]:
            raise PredictionImpossible("unknown")
        return est[0]

    _batch_estimate_of = estimate


@pytest.fixture
def host_ids(monkeypatch):
    monkeypatch.setattr(validation._Pairs, "device_ids",
                        lambda self: (torch.from_numpy(np.asarray(self.iu, dtype=np.int32)),
                                      torch.from_numpy(np.asarray(self.ii, dtype=np.int32))))


def pow_sensitive(n, seed):
    """Differences d with d * d != d ** 2 (libm pow), plus signed zeros."""
    rng = np.random.RandomState(seed)
    out = []
    while len(out) < n:
        x = float(rng.uniform(-4, 4))
        if x * x != x ** 2:
            out.append(x)
    return out + [0.0, -0.0]


MEASURES = ["rmse", "mse", "mae", "fcp"]


def tuple_route(algo, trainset, testset, measures, train=False):
    preds = algo.test(trainset.build_testset() if train else testset)
    return {m: getattr(accuracy, m)(preds, verbose=False) for m in measures}


def assert_bits(got, want):
    assert list(got) == list(want)
    for m in want:
        assert type(got[m]) is type(want[m]), m
        assert np.float64(got[m]).tobytes() == np.float64(want[m]).tobytes(), (m, got[m], want[m])


def test_square_rule_on_pow_sensitive_differences():
    d = pow_sensitive(3000, 0)
    r = np.round(np.random.RandomState(1).uniform(1, 5, len(d)), 1)
    est = r - np.array(d)
    preds = [sb.Prediction("u%d" % (k % 7), k, rk, ek, {}) for k, (rk, ek) in enumerate(zip(r.tolist(), est.tolist()))]
    assert sum(x * x != x ** 2 for x in (r - est).tolist()) > 2000
    code = np.array([k % 7 for k in range(len(d))], dtype=np.int64)
    for m in MEASURES:
        got = accuracy._of_arrays(m, r, est, lambda: (code, 7))
        want = getattr(accuracy, m)(preds, verbose=False)
        assert np.float64(got).tobytes() == np.float64(want).tobytes(), m
    with pytest.raises(ValueError, match="empty"):
        accuracy._of_arrays("rmse", np.zeros(0), np.zeros(0), None)


def test_mse_printout(capsys):
    preds = [sb.Prediction(0, 0, 3.0, 1.5, {}), sb.Prediction(0, 1, 4.0, 4.0, {})]
    assert accuracy.mse(preds) == 1.125
    assert capsys.readouterr().out == "MSE: 1.1250\n"
    assert accuracy.rmse(preds, verbose=False) == np.sqrt(1.125)
    with pytest.raises(ValueError):
        accuracy.mse([])


@pytest.mark.parametrize("scale", [(1, 5), (-2, 2)])
def test_array_route_matches_tuple_route(host_ids, scale):
    data = arrays_data(n=900, seed=5, scale=scale)
    rng = np.random.RandomState(2)
    for trs, tes in KFold(3, random_state=1).split(data):
        off = trs.offset
        # estimates around the ratings: differences that round differently under d * d, values both sides of the
        # scale, and signed zeros once the offset is taken off
        table = rng.choice(pow_sensitive(50, 3) + [-9.0, 9.0], size=(trs.n_users, trs.n_items)) + 3 + off
        table[0, :] = off + 0.0
        table[1, :] = off - 0.0
        tes = tes + [(123456, 1, 2.0 + off), (0, 98765, 3.0 + off), (4.0, 2, 1.0 + off)]
        fold = Fold(trs, tes)
        for m in (["rmse", "mse", "mae", "fcp"], ["FCP", "Rmse"]):
            algo = Batched(table)
            test_m, train_m, _, _ = _fit_and_score(algo, fold, m, True)
            want = {x: v for x, v in zip(m, tuple_route(algo, trs, tes, [x.lower() for x in m]).values())}
            assert_bits(test_m, want)
            want = {x: v for x, v in zip(m, tuple_route(algo, trs, tes, [x.lower() for x in m], True).values())}
            assert_bits(train_m, want)
        assert fold.test_pairs() is fold.test_pairs() and fold.train_pairs() is fold.train_pairs()


def test_array_route_groups_equal_uids_and_raises_zero_division(host_ids):
    data = arrays_data(n=400, seed=8)
    trs, tes = next(KFold(2, random_state=0).split(data))
    table = np.random.RandomState(0).uniform(0, 6, (trs.n_users, trs.n_items))
    # 1, 1.0 and True are one fcp user, as defaultdict(list) keys them
    tes = [(True if u == 1 else (1.0 if k % 2 else u), i, r) for k, (u, i, r) in enumerate(tes)]
    algo = Batched(table)
    got = _fit_and_score(algo, Fold(trs, tes), MEASURES, False)[0]
    assert_bits(got, tuple_route(algo, trs, tes, MEASURES))
    zero = np.zeros(table.shape, dtype=bool)
    zero[trs.to_inner_uid(tes[5][0]), trs.to_inner_iid(tes[5][1])] = True
    with pytest.raises(ZeroDivisionError):
        Batched(table, zero_div=zero).fit(trs).test(tes)
    with pytest.raises(ZeroDivisionError):
        _fit_and_score(Batched(table, zero_div=zero), Fold(trs, tes), MEASURES, False)
    with pytest.raises(ValueError, match="empty"):
        fit_and_score(Batched(table), trs, [], ["rmse"])


def test_final_estimates_value_rule():
    ts = sb.Trainset.from_coo([0, 1], [0, 1], [4.0, 1.0], rating_scale=(-2, 2), offset=3)
    algo = sb.AlgoBase()
    algo.fit(ts)
    est = np.array([0.5, 5.5, -0.0, 3.0, 7.0, 2.0])
    got = algo._final_estimates(est, np.array([0, 0, 0, 0, 0, 1], dtype=np.uint8))
    assert got.tolist() == [-2.0, 2.0, -2.0, 0.0, 2.0, -0.5]           # default prediction 2.5 - 3
    assert est.tolist()[0] == 0.5                                        # the input is not modified
    assert algo._final_estimates([3.0], None).tolist() == [0.0]
    with pytest.raises(ZeroDivisionError):
        algo._final_estimates(est, np.array([0, 2, 0, 0, 0, 1]))


def test_cross_validate_keeps_its_results(host_ids):
    data = arrays_data(n=500, seed=4)
    trs0, _ = next(KFold(5, random_state=2).split(data))
    table = np.random.RandomState(6).uniform(0, 6, (60, 60))
    got = cross_validate(Batched(table), data, MEASURES, KFold(5, random_state=2), return_train_measures=True)
    want = defaultdict(list)
    for trs, tes in KFold(5, random_state=2).split(data):
        algo = Batched(table)
        algo.fit(trs)
        for part, tr in (("test_", False), ("train_", True)):
            for m, v in tuple_route(algo, trs, tes, MEASURES, tr).items():
                want[part + m].append(v)
    for k, v in want.items():
        assert got[k].tobytes() == np.array(v).tobytes(), k
