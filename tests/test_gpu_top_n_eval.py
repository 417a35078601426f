"""Top-N measures on the device: AlgoBase.top_n_measures equals accuracy.top_n_measures over get_top_n, as float bits,
for every device-batched algorithm on LeaveOneOut and KFold splits of the u1 fixture; also a non-batched subclass,
an offset dataset, block boundaries, the prefix property across cutoffs, sb2_top_n_hits_dev against numpy, its launch
count, and cross_validate / GridSearchCV with the top-N measure names."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import accuracy  # noqa: E402
from surprise_b200.model_selection import GridSearchCV, KFold, LeaveOneOut, cross_validate  # noqa: E402
from surprise_b200.model_selection.validation import Fold  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
THRESHOLDS = (None, 3.5, 4)


def same_result(a, b):
    return list(a) == list(b) and all(np.float64(a[k]).tobytes() == np.float64(b[k]).tobytes() for k in a)


def definition(algo, testset, n, threshold, top=None):
    top = algo.get_top_n(n) if top is None else top
    return accuracy.top_n_measures(top, testset, n, threshold, offset=algo.trainset.offset, verbose=False)


@pytest.fixture(scope="module")
def u1_splits():
    data = sb.Dataset.load_from_file(os.path.join(GOLDEN, "u1_ml100k_train"), sb.Reader("ml-100k"))
    loo = next(LeaveOneOut(1, random_state=0).split(data))
    kf = next(KFold(5, random_state=0).split(data))
    # unknown users and items in the held-out rows
    kf = (kf[0], kf[1] + [("nobody", "1", 5.0), ("1", "no-item", 5.0), ("nobody", "x", 4.0)])
    return data, {"loo": loo, "kfold": kf}


ALGOS = {
    "svd": lambda: sb.SVD(n_factors=20, n_epochs=5, random_state=0),
    "svdpp": lambda: sb.SVDpp(n_factors=10, n_epochs=2, random_state=0),
    "nmf": lambda: sb.NMF(n_factors=15, n_epochs=5, random_state=0),
    "baseline_only": lambda: sb.BaselineOnly(),
    "knn_basic": lambda: sb.KNNBasic(sim_options={"name": "msd", "user_based": True}),
    "knn_means": lambda: sb.KNNWithMeans(sim_options={"name": "pearson", "user_based": False}),
    "knn_zscore": lambda: sb.KNNWithZScore(sim_options={"name": "cosine", "user_based": True}),
    "knn_baseline": lambda: sb.KNNBaseline(sim_options={"name": "pearson_baseline", "user_based": False}),
    "slope_one": lambda: sb.SlopeOne(),
    "coclustering": lambda: sb.CoClustering(random_state=0),
}


@pytest.mark.parametrize("split", ["loo", "kfold"])
@pytest.mark.parametrize("name", sorted(ALGOS))
def test_device_route_equals_definition(u1_splits, name, split):
    trs, tes = u1_splits[1][split]
    algo = ALGOS[name]().fit(trs)
    assert algo._batched()
    for n in (1, 10, 100, trs.n_items + 5):
        top = algo.get_top_n(n)
        for threshold in THRESHOLDS:
            got = algo.top_n_measures(tes, n, threshold)
            assert same_result(got, definition(algo, tes, n, threshold, top)), (n, threshold)


def test_non_batched_subclass(u1_splits):
    class PySVD(sb.SVD):
        def estimate(self, u, i):
            return sb.SVD.estimate(self, u, i) + 0.25

    trs, tes = u1_splits[1]["loo"]
    algo = PySVD(n_factors=5, n_epochs=2, random_state=0).fit(trs)
    assert not algo._batched()
    tes = tes[:60]
    for n, threshold in ((10, None), (25, 4)):
        assert same_result(algo.top_n_measures(tes, n, threshold), definition(algo, tes, n, threshold))


def test_offset_dataset(u1_splits):
    raw = u1_splits[0].raw_ratings
    u, i, r = (np.array([row[k] for row in raw]) for k in range(3))
    data = sb.Dataset.load_from_arrays(u, i, r.astype(np.float64) * 4 - 10, sb.Reader(rating_scale=(-10, 10)))
    for trs, tes in LeaveOneOut(2, random_state=3).split(data):
        assert trs.offset == 11
        algo = sb.SVD(n_factors=10, n_epochs=3, random_state=0).fit(trs)
        for threshold in (None, 2, 6.0):
            assert same_result(algo.top_n_measures(tes, 10, threshold), definition(algo, tes, 10, threshold))


def test_block_boundaries_and_prefix_across_cutoffs(u1_splits):
    trs, tes = u1_splits[1]["kfold"]
    for algo in (sb.SVD(n_factors=20, n_epochs=3, random_state=0).fit(trs),
                 sb.KNNBaseline(sim_options={"user_based": False}).fit(trs)):
        fold = Fold(trs, tes)
        ns = [1, 7, 10, 64, 100]
        want = [algo.top_n_measures(tes, n, 3.5) for n in ns]
        for rows in (None, 1, 13, 256):
            got = algo._top_n_measures(fold, ns, 3.5, _block_rows=rows)
            assert all(same_result(g, w) for g, w in zip(got, want)), rows
        # the first N entries of the top-M lists are the top-N lists
        items_m, est_m, count_m = algo.top_n_inner(100)
        for n in (1, 10, 64):
            items, est, count = algo.top_n_inner(n)
            assert np.array_equal(items, items_m[:, :n]) and np.array_equal(count, np.minimum(count_m, n))
            assert est.tobytes() == np.ascontiguousarray(est_m[:, :n]).tobytes()


def hits_reference(items, count, w, rel_ptr, rel_idx, inv, disc):
    out = []
    for b in range(len(count)):
        rel = set(rel_idx[rel_ptr[b]:rel_ptr[b + 1]].tolist())
        h, a, d = 0, 0.0, 0.0
        for p in range(max(0, min(int(count[b]), w))):
            if int(items[b, p]) in rel:
                h, a, d = h + 1, a + float(inv[p]), d + float(disc[p])
        out.append((h, a, d))
    return out


def call_hits(items, count, w, rel_ptr, rel_idx, inv, disc):
    n_rows = len(count)
    d = {k: nat.to_dev(v, v.dtype) for k, v in dict(items=items, count=count, rel_ptr=rel_ptr, rel_idx=rel_idx,
                                                     inv=inv, disc=disc).items()}
    hits, rr, dcg = (nat.empty_dev((max(n_rows, 1),), t) for t in (np.int32, np.float64, np.float64))
    nat.check(nat.lib().sb2_top_n_hits_dev(n_rows, nat.ptr(d["items"]), items.shape[1], nat.ptr(d["count"]), w,
                                           nat.ptr(d["rel_ptr"]), nat.ptr(d["rel_idx"]), len(rel_idx),
                                           nat.ptr(d["inv"]), nat.ptr(d["disc"]), nat.ptr(hits), nat.ptr(rr),
                                           nat.ptr(dcg), nat.stream()))
    return list(zip(hits.cpu().numpy()[:n_rows].tolist(), rr.cpu().numpy()[:n_rows].tolist(),
                    dcg.cpu().numpy()[:n_rows].tolist()))


def test_hits_kernel_against_numpy():
    rng = np.random.RandomState(0)
    n_rows, ld, n_items = 300, 150, 400
    items = np.full((n_rows, ld), -1, dtype=np.int32)
    count = rng.randint(0, ld + 1, n_rows).astype(np.int32)
    count[:5] = [0, 1, 31, 32, 33]
    for b in range(n_rows):
        items[b, :count[b]] = rng.choice(n_items, count[b], replace=False)
    lens = rng.randint(0, 80, n_rows)
    lens[::17] = 0
    rel_ptr = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    rel_idx = np.concatenate([np.sort(rng.choice(n_items + 5, m, replace=False)) for m in lens]).astype(np.int32)
    inv, disc, _ = accuracy._rank_tables(ld)
    for w in (0, 1, 10, 33, 100, ld):
        assert call_hits(items, count, w, rel_ptr, rel_idx, inv, disc) == \
            hits_reference(items, count, w, rel_ptr, rel_idx, inv, disc), w
    # malformed lists and arguments are refused
    bad_idx = rel_idx.copy()
    k = int(np.flatnonzero(lens >= 2)[0])
    bad_idx[rel_ptr[k]], bad_idx[rel_ptr[k] + 1] = bad_idx[rel_ptr[k] + 1], bad_idx[rel_ptr[k]]
    with pytest.raises(ValueError):
        call_hits(items, count, 10, rel_ptr, bad_idx, inv, disc)
    for b, value in ((n_rows, len(rel_idx) + 1), (0, -1), (5, rel_ptr[7] + 1)):
        bad_ptr = rel_ptr.copy()
        bad_ptr[b] = value
        with pytest.raises(ValueError):
            call_hits(items, count, 10, bad_ptr, rel_idx, inv, disc)
    with pytest.raises(ValueError):
        call_hits(items, count, ld + 1, rel_ptr, rel_idx, inv, disc)


def test_launch_count(u1_splits):
    trs, tes = u1_splits[1]["loo"]
    algo = sb.SVD(n_factors=20, n_epochs=3, random_state=0).fit(trs)
    fold = Fold(trs, tes)
    iu = fold.test_pairs().relevant(None, trs.n_items)[0]
    users = iu[iu >= 0]
    lib = nat.lib()
    lib.sb2_reset_launch_count()
    algo.top_n_inner(100, users, _block_rows=100)
    base = lib.sb2_launch_count()
    lib.sb2_reset_launch_count()
    algo._top_n_measures(fold, [10, 100], None, _block_rows=100)
    blocks = -(-len(users) // 100)
    assert lib.sb2_launch_count() == base + 2 * blocks


def test_cross_validate_equals_explicit_loop(u1_splits):
    data = u1_splits[0]
    cv = LeaveOneOut(2, random_state=4)
    got = cross_validate(sb.SVD(n_factors=10, n_epochs=3, random_state=0), data, ["hr@10", "ndcg@10", "rmse"], cv)
    for k, (trs, tes) in enumerate(cv.split(data)):
        algo = sb.SVD(n_factors=10, n_epochs=3, random_state=0).fit(trs)
        m = algo.top_n_measures(tes, 10)
        want = {"hr@10": m["hr"], "ndcg@10": m["ndcg"], "rmse": accuracy.rmse(algo.test(tes), verbose=False)}
        for name, value in want.items():
            assert np.float64(got["test_" + name][k]).tobytes() == np.float64(value).tobytes(), (k, name)


def test_grid_search_picks_the_best_hit_rate(u1_splits):
    data = u1_splits[0]
    gs = GridSearchCV(sb.SVD, {"n_factors": [5, 50], "n_epochs": [1, 10], "random_state": [0]},
                      measures=["hr@10", "rmse"], cv=LeaveOneOut(2, random_state=0))
    gs.fit(data)
    mean = gs.cv_results["mean_test_hr@10"]
    assert gs.best_params["hr@10"] == gs.param_combinations[int(np.argmax(mean))]
    assert gs.best_score["hr@10"] == mean.max()
    assert gs.cv_results["rank_test_hr@10"][int(np.argmax(mean))] == 1
