"""Coverage, novelty and diversity of top-N lists on the device: AlgoBase.top_n_list_measures equals
accuracy.top_n_list_measures over get_top_n, as float bits (NaN equal to NaN), for every device-batched algorithm on
LeaveOneOut and KFold splits of the u1 fixture; also block sizes, sb2_top_n_lists_dev against numpy, cross_validate and
GridSearchCV with the list measure names, and the sim models the method refuses."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import accuracy  # noqa: E402
from surprise_b200 import similarities as sims  # noqa: E402
from surprise_b200.model_selection import GridSearchCV, KFold, LeaveOneOut, cross_validate  # noqa: E402
from surprise_b200.model_selection.validation import Fold  # noqa: E402
from surprise_b200.prediction_algorithms import knns  # noqa: E402

from test_gpu_top_n_eval import ALGOS  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
THRESHOLDS = (None, 3.5, 4, np.float64(4.0))


def same_result(a, b):
    return list(a) == list(b) and all(np.float64(a[k]).tobytes() == np.float64(b[k]).tobytes() for k in a)


@pytest.fixture(scope="module")
def u1_splits():
    data = sb.Dataset.load_from_file(os.path.join(GOLDEN, "u1_ml100k_train"), sb.Reader("ml-100k"))
    loo = next(LeaveOneOut(1, random_state=0).split(data))
    kf = next(KFold(5, random_state=0).split(data))
    knn = {name: sb.KNNBaseline(sim_options={"user_based": False}).fit(trs) for name, (trs, _) in
           (("loo", loo), ("kfold", kf))}
    return data, {"loo": loo, "kfold": kf}, knn


def user_sets(ts):
    raw = [ts.to_raw_uid(u) for u in range(ts.n_users)]
    subset = raw[::31]
    return {"all": None, "subset": subset, "duplicated": subset[:5] + subset[2:9] + subset[:3]}


@pytest.mark.parametrize("split", ["loo", "kfold"])
@pytest.mark.parametrize("name", sorted(ALGOS))
def test_device_route_equals_definition(u1_splits, name, split):
    trs, _ = u1_splits[1][split]
    knn = u1_splits[2][split]
    algo = ALGOS[name]().fit(trs)
    assert algo._batched()
    groups = user_sets(trs)
    for n in (1, 10, 100, trs.n_items + 5):
        top = algo.get_top_n(n)
        for label, uids in groups.items():
            for threshold in THRESHOLDS:
                got = algo.top_n_list_measures(n, uids, threshold)
                want = accuracy.top_n_list_measures(top, trs, n, uids, threshold, verbose=False)
                assert same_result(got, want), (n, label, threshold)
        # diversity: the Python definition is quadratic in n, so the longest lists are checked on a few users
        uids = groups["subset"] if n <= 100 else groups["subset"][:3]
        want = accuracy.top_n_list_measures(top, trs, n, uids, 3.5, knn.sim, verbose=False)
        assert same_result(algo.top_n_list_measures(n, uids, 3.5, knn.sim), want), n
        assert same_result(algo.top_n_list_measures(n, uids, 3.5, knn), want), n
    top = algo.get_top_n(10)
    want = accuracy.top_n_list_measures(top, trs, 10, None, None, knn.sim, verbose=False)
    assert same_result(algo.top_n_list_measures(10, sim=knn), want)


def test_block_rows_do_not_change_the_result(u1_splits):
    trs, _ = u1_splits[1]["kfold"]
    knn = u1_splits[2]["kfold"]
    algo = sb.SVD(n_factors=20, n_epochs=3, random_state=0).fit(trs)
    for n, threshold in ((10, None), (37, 3.5)):
        want = algo.top_n_list_measures(n, threshold=threshold, sim=knn)
        for rows in (1, 7):
            assert same_result(algo.top_n_list_measures(n, threshold=threshold, sim=knn, _block_rows=rows), want)


def lists_reference(items, est, count, w, threshold, info, sim):
    covered, nov, ils, seen = [], [], [], set()
    for b in range(len(count)):
        c = max(0, min(int(count[b]), w))
        row = items[b, :c].tolist()
        covered.append(int(c > 0 if threshold is None else any(e >= threshold for e in est[b, :c].tolist())))
        s = 0.0
        for i in row:
            s += float(info[i])
        nov.append(s)
        t = 0.0
        for p in range(c):
            for q in range(p + 1, c):
                t += float(sim[row[p], row[q]])
        ils.append(t)
        seen.update(row)
    return covered, nov, ils, seen


def call_lists(items, est, count, w, threshold, info, sim):
    n_rows, n_items = len(count), len(info)
    d = {k: nat.to_dev(v, v.dtype) for k, v in dict(items=items, est=est, count=count, info=info, sim=sim).items()}
    cov, nov, ils = (nat.empty_dev((max(n_rows, 1),), t) for t in (np.int32, np.float64, np.float64))
    seen = nat.to_dev(np.zeros(n_items, dtype=np.uint8), np.uint8)
    nat.check(nat.lib().sb2_top_n_lists_dev(n_rows, nat.ptr(d["items"]), items.shape[1], nat.ptr(d["est"]),
                                            nat.ptr(d["count"]), w, int(threshold is not None),
                                            0.0 if threshold is None else float(threshold), n_items,
                                            nat.ptr(d["info"]), nat.ptr(d["sim"]), nat.ptr(cov), nat.ptr(nov),
                                            nat.ptr(ils), nat.ptr(seen), nat.stream()))
    seen = set(np.flatnonzero(seen.cpu().numpy()).tolist())
    return (cov.cpu().numpy()[:n_rows].tolist(), nov.cpu().numpy()[:n_rows].tolist(),
            ils.cpu().numpy()[:n_rows].tolist(), seen)


def test_lists_kernel_against_numpy():
    rng = np.random.RandomState(0)
    n_rows, ld, n_items = 300, 90, 400
    items = np.full((n_rows, ld), -1, dtype=np.int32)
    est = np.full((n_rows, ld), np.nan)
    count = rng.randint(0, ld + 1, n_rows).astype(np.int32)
    count[:6] = [0, 1, 2, 31, 32, 33]
    for b in range(n_rows):
        items[b, :count[b]] = rng.choice(n_items, count[b], replace=False)
        est[b, :count[b]] = rng.uniform(1, 5, count[b])
    est[3, 5] = est[7, 0] = np.nan
    info = rng.standard_normal(n_items) * 3
    sim = rng.uniform(-1, 1, (n_items, n_items))
    for w in (0, 1, 2, 10, 33, 64, ld):
        for threshold in (None, 3.0, 4.5):
            got = call_lists(items, est, count, w, threshold, info, sim)
            want = lists_reference(items, est, count, w, threshold, info, sim)
            assert got[0] == want[0] and got[3] == want[3], (w, threshold)
            assert np.array(got[1]).tobytes() == np.array(want[1]).tobytes(), (w, threshold)
            assert np.array(got[2]).tobytes() == np.array(want[2]).tobytes(), (w, threshold)
    # a listed item outside [0, n_items) is refused; padding past count is never read
    for value in (n_items, -1, 2 ** 31 - 1):
        bad = items.copy()
        b = int(np.flatnonzero(count >= 3)[0])
        bad[b, 2] = value
        with pytest.raises(ValueError, match="n_items"):
            call_lists(bad, est, count, ld, None, info, sim)
    with pytest.raises(ValueError):
        call_lists(items, est, count, ld + 1, None, info, sim)


def test_cross_validate_equals_method_per_fold(u1_splits):
    data = u1_splits[0]
    cv = LeaveOneOut(2, random_state=4)
    make = lambda: sb.SVD(n_factors=10, n_epochs=3, random_state=0)  # noqa: E731
    got = cross_validate(make(), data, ["hr@10", "novelty@10", "diversity@10", "rmse"], cv)
    for k, (trs, tes) in enumerate(cv.split(data)):
        algo = make().fit(trs)
        # U*: every held-out user, including those whose only rating was held out (no list; the method refuses them)
        star = list(dict.fromkeys(u for u, _, _ in tes))
        known = [u for u in star if trs.to_inner_uids([u])[0] >= 0]
        assert len(known) < len(star)
        cosine = sims.build_device("cosine", trs.n_items, trs.user_csr(), 1).cpu().numpy()
        top = algo.get_top_n(10)
        lists = accuracy.top_n_list_measures(top, trs, 10, star, None, cosine, verbose=False)
        assert same_result(algo.top_n_list_measures(10, known, sim=cosine),
                           accuracy.top_n_list_measures(top, trs, 10, known, None, cosine, verbose=False))
        want = {"hr@10": algo.top_n_measures(tes, 10)["hr"], "novelty@10": lists["novelty"],
                "diversity@10": lists["diversity"], "rmse": accuracy.rmse(algo.test(tes), verbose=False)}
        for name, value in want.items():
            assert np.float64(got["test_" + name][k]).tobytes() == np.float64(value).tobytes(), (k, name)


def test_fold_cosine_is_built_once_and_refused_when_too_large(u1_splits, monkeypatch):
    trs, tes = u1_splits[1]["loo"]
    fold = Fold(trs, tes)
    assert fold.item_cosine() is fold.item_cosine()
    monkeypatch.setattr(knns, "_DENSE_SIM_FRACTION", 0.0)
    with pytest.raises(ValueError, match="cosine"):
        Fold(trs, tes).item_cosine()


def test_grid_search_ranks_diversity_descending(u1_splits):
    data = u1_splits[0]
    gs = GridSearchCV(sb.SVD, {"n_factors": [5, 50], "n_epochs": [1, 10], "random_state": [0]},
                      measures=["diversity@10", "rmse"], cv=LeaveOneOut(2, random_state=0))
    gs.fit(data)
    mean = gs.cv_results["mean_test_diversity@10"]
    assert len(set(mean.tolist())) == len(mean)
    assert gs.best_params["diversity@10"] == gs.param_combinations[int(np.argmax(mean))]
    assert gs.cv_results["rank_test_diversity@10"].tolist() == (len(mean) - np.argsort(np.argsort(mean))).tolist()


def test_wrong_sim_models_are_refused(u1_splits, monkeypatch):
    trs, _ = u1_splits[1]["kfold"]
    algo = sb.SVD(n_factors=5, n_epochs=1, random_state=0).fit(trs)
    with pytest.raises(ValueError, match="item-based"):
        algo.top_n_list_measures(10, sim=sb.KNNBasic(sim_options={"name": "cosine"}).fit(trs))
    with pytest.raises(ValueError, match="trainset"):
        algo.top_n_list_measures(10, sim=u1_splits[2]["loo"])
    monkeypatch.setattr(knns, "_DENSE_SIM_FRACTION", 0.0)
    streamed = sb.KNNBasic(sim_options={"name": "cosine", "user_based": False}).fit(trs)
    assert streamed._streamed
    with pytest.raises(ValueError, match="streamed"):
        algo.top_n_list_measures(10, sim=streamed)
