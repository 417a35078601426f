"""AUC, MRR and MPR over the full ranking on the device: AlgoBase.rank_measures equals accuracy.rank_measures over
get_top_n(n_items), as float bits (NaN equal to NaN), for every device-batched algorithm and a streamed k-NN model on
LeaveOneOut and KFold splits of the u1 fixture with unknown users and items held out; also sb2_top_n_ranks_dev against
numpy (ties, NaN, signed zeros, impossible and clipped values, rows longer than one tile), block sizes,
ZeroDivisionError, malformed relevant lists, and cross_validate / GridSearchCV with the rank measure names."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import accuracy  # noqa: E402
from surprise_b200 import synth  # noqa: E402
from surprise_b200.model_selection import GridSearchCV, KFold, LeaveOneOut, cross_validate  # noqa: E402
from surprise_b200.model_selection.validation import Fold  # noqa: E402
from surprise_b200.prediction_algorithms import knns  # noqa: E402
from surprise_b200.prediction_algorithms.algo_base import rank_top_n  # noqa: E402

from test_gpu_top_n import offset_trainset  # noqa: E402
from test_gpu_top_n_eval import ALGOS  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
THRESHOLDS = (None, 3.5, 4)
UNKNOWN = [("nobody", "1", 5.0), ("1", "no-item", 5.0), ("nobody", "x", 4.0)]


def same_result(a, b):
    return list(a) == list(b) and all(np.float64(a[k]).tobytes() == np.float64(b[k]).tobytes() for k in a)


def definition(algo, testset, threshold, top=None):
    ts = algo.trainset
    top = algo.get_top_n(ts.n_items) if top is None else top
    return accuracy.rank_measures(top, testset, ts, threshold, verbose=False)


@pytest.fixture(scope="module")
def u1_splits():
    data = sb.Dataset.load_from_file(os.path.join(GOLDEN, "u1_ml100k_train"), sb.Reader("ml-100k"))
    loo = next(LeaveOneOut(1, random_state=0).split(data))
    kf = next(KFold(5, random_state=0).split(data))
    return data, {"loo": (loo[0], list(loo[1]) + UNKNOWN), "kfold": (kf[0], list(kf[1]) + UNKNOWN)}


def check_against_definition(algo, tes):
    top = algo.get_top_n(algo.trainset.n_items)
    for threshold in THRESHOLDS:
        got = algo.rank_measures(tes, threshold)
        assert same_result(got, definition(algo, tes, threshold, top)), threshold


@pytest.mark.parametrize("split", ["loo", "kfold"])
@pytest.mark.parametrize("name", sorted(ALGOS))
def test_device_route_equals_definition(u1_splits, name, split):
    trs, tes = u1_splits[1][split]
    algo = ALGOS[name]().fit(trs)
    assert algo._batched()
    check_against_definition(algo, tes)


@pytest.mark.parametrize("split", ["loo", "kfold"])
def test_streamed_knn_equals_definition(u1_splits, split, monkeypatch):
    trs, tes = u1_splits[1][split]
    monkeypatch.setattr(knns, "_DENSE_SIM_FRACTION", 0.0)
    monkeypatch.setattr(knns, "_STREAM_BAND_BYTES", 8 * trs.n_items * 300)
    algo = sb.KNNBaseline(sim_options={"name": "pearson_baseline", "user_based": False}).fit(trs)
    assert algo._streamed
    check_against_definition(algo, tes)


def test_block_rows_do_not_change_the_result(u1_splits):
    trs, tes = u1_splits[1]["kfold"]
    for algo in (sb.SVD(n_factors=20, n_epochs=3, random_state=0).fit(trs), sb.CoClustering(random_state=0).fit(trs)):
        for threshold in (None, 3.5):
            want = algo.rank_measures(tes, threshold)
            for rows in (1, 7, 10 ** 6):
                assert same_result(algo.rank_measures(tes, threshold, _block_rows=rows), want), rows


def test_more_relevant_candidates_than_one_tile():
    d = synth.ratings(40, 6000, 30000, seed=3)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    rated = set(i[u == 0].tolist())
    unrated = [j for j in range(ts.n_items) if j not in rated]
    rng = np.random.RandomState(0)
    picked = rng.choice(unrated, 5000, replace=False).tolist()
    tes = [(ts.to_raw_uid(0), ts.to_raw_iid(j), float(rng.randint(1, 6))) for j in picked]
    tes += [(ts.to_raw_uid(1), ts.to_raw_iid(j), 5.0) for j in range(0, ts.n_items, 7)]
    for algo in (sb.BaselineOnly().fit(ts), sb.SVD(n_factors=10, n_epochs=2, random_state=0).fit(ts)):
        top = algo.get_top_n(ts.n_items)
        for threshold in (None, 3):
            assert same_result(algo.rank_measures(tes, threshold), definition(algo, tes, threshold, top)), threshold


# -- the kernel ------------------------------------------------------------------------------------------------------
def ranks_reference(scores, codes, rows, u_ptr, ui_idx, rel_ptr, rel_idx, n_items, default, offset, low, high):
    out = []
    for b, user in enumerate(rows.tolist()):
        rated = set(ui_idx[u_ptr[user]:u_ptr[user + 1]].tolist())
        cand = np.array([j for j in range(n_items) if j not in rated], dtype=np.int64)
        v = scores[b, cand].copy()
        v[codes[b, cand] == 1] = default
        v = np.maximum(low, np.minimum(high, v - offset))
        order = cand[rank_top_n(v, cand)]
        pos = {int(j): p for p, j in enumerate(order.tolist())}
        ks = sorted(pos[j] for j in rel_idx[rel_ptr[b]:rel_ptr[b + 1]].tolist() if j in pos)
        out.append((len(cand), len(ks), sum(ks), ks[0] if ks else -1))
    return out


def call_ranks(scores, codes, rows, u_ptr, ui_idx, rel_ptr, rel_idx, n_items, default, offset, low, high):
    n_rows = len(rows)
    d = {k: None if v is None else nat.to_dev(np.ascontiguousarray(v), v.dtype)
         for k, v in dict(scores=scores, codes=codes, rows=rows, u_ptr=u_ptr, ui_idx=ui_idx, rel_ptr=rel_ptr,
                          rel_idx=rel_idx).items()}
    outs = [nat.empty_dev((max(n_rows, 1),), t) for t in (np.int32, np.int32, np.int64, np.int32)]
    nat.check(nat.lib().sb2_top_n_ranks_dev(n_rows, nat.ptr(d["rows"]), n_items, nat.ptr(d["scores"]),
                                            scores.shape[1], nat.ptr(d["codes"]), default, offset, low, high,
                                            nat.ptr(d["u_ptr"]), nat.ptr(d["ui_idx"]), nat.ptr(d["rel_ptr"]),
                                            nat.ptr(d["rel_idx"]), len(rel_idx), *(nat.ptr(o) for o in outs),
                                            nat.stream()))
    return list(zip(*(o.cpu().numpy()[:n_rows].tolist() for o in outs)))


def kernel_case(seed=0, n_rows=60, n_items=3000, n_users=25, long_rows=(3, 11)):
    rng = np.random.RandomState(seed)
    ld = n_items + 5
    scores = rng.randint(0, 9, (n_rows, ld)) * 0.75 - 1.0          # many equal values, some outside [low, high]
    scores[rng.rand(n_rows, ld) < 0.02] = np.nan
    scores[rng.rand(n_rows, ld) < 0.05] = -0.0
    scores[rng.rand(n_rows, ld) < 0.05] = 0.0
    codes = (rng.rand(n_rows, ld) < 0.05).astype(np.uint8)
    lens = rng.randint(0, 300, n_users)
    lens[0] = 0
    lens[1] = n_items - 1
    ui_idx = np.concatenate([np.sort(rng.choice(n_items, m, replace=False)) for m in lens]).astype(np.int32)
    u_ptr = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    rows = rng.randint(0, n_users, n_rows).astype(np.int32)
    rows[:3] = [0, 1, 2]
    rel_lens = rng.randint(0, 40, n_rows)
    rel_lens[::9] = 0
    for b in long_rows:
        rel_lens[b] = 2100 + 50 * b           # past one 2048-entry tile, rated items included
    rel_ptr = np.concatenate(([0], np.cumsum(rel_lens))).astype(np.int64)
    rel_idx = np.concatenate([np.sort(rng.choice(n_items, m, replace=False)) for m in rel_lens]).astype(np.int32)
    return scores, codes, rows, u_ptr, ui_idx, rel_ptr, rel_idx, n_items


def test_ranks_kernel_against_numpy():
    case = kernel_case()
    for default, offset, low, high in ((2.5, 0.0, 1.0, 5.0), (-0.0, 1.0, -1.0, 3.0), (0.0, 0.0, -np.inf, np.inf)):
        assert call_ranks(*case, default, offset, low, high) == ranks_reference(*case, default, offset, low, high)
    # no impossible codes
    scores, codes, *rest = case
    assert call_ranks(scores, None, *rest, 3.0, 0.0, 1.0, 5.0) == \
        ranks_reference(scores, np.zeros_like(codes), *rest, 3.0, 0.0, 1.0, 5.0)


def test_ranks_kernel_ties_break_by_item():
    # every candidate scores the same: positions follow the item ids
    n_items = 50
    scores = np.full((1, n_items), 3.0)
    rows = np.zeros(1, dtype=np.int32)
    u_ptr, ui_idx = np.array([0, 2], dtype=np.int64), np.array([4, 9], dtype=np.int32)
    rel_ptr, rel_idx = np.array([0, 3], dtype=np.int64), np.array([3, 9, 20], dtype=np.int32)
    got = call_ranks(scores, None, rows, u_ptr, ui_idx, rel_ptr, rel_idx, n_items, 0.0, 0.0, 1.0, 5.0)
    # candidates 0..49 without 4, 9: item 3 at 3, item 20 at 18, item 9 rated
    assert got == [(48, 2, 21, 3)]


def test_ranks_kernel_refuses_malformed_lists():
    scores, codes, rows, u_ptr, ui_idx, rel_ptr, rel_idx, n_items = kernel_case(1, n_rows=20, long_rows=())
    args = (1.0, 0.0, 1.0, 5.0)
    k = int(np.flatnonzero(np.diff(rel_ptr) >= 2)[0])
    bad_idx = rel_idx.copy()
    bad_idx[rel_ptr[k]], bad_idx[rel_ptr[k] + 1] = bad_idx[rel_ptr[k] + 1], bad_idx[rel_ptr[k]]
    with pytest.raises(ValueError, match="relevant"):
        call_ranks(scores, codes, rows, u_ptr, ui_idx, rel_ptr, bad_idx, n_items, *args)
    for value in (n_items, -1):
        bad_idx = rel_idx.copy()
        bad_idx[rel_ptr[k + 1] - 1] = value
        with pytest.raises(ValueError, match="relevant"):
            call_ranks(scores, codes, rows, u_ptr, ui_idx, rel_ptr, bad_idx, n_items, *args)
    for b, value in ((len(rows), len(rel_idx) + 1), (0, -1), (5, rel_ptr[7] + 1)):
        bad_ptr = rel_ptr.copy()
        bad_ptr[b] = value
        with pytest.raises(ValueError, match="relevant"):
            call_ranks(scores, codes, rows, u_ptr, ui_idx, bad_ptr, rel_idx, n_items, *args)
    with pytest.raises(ValueError):
        call_ranks(scores[:, :n_items - 1], codes, rows, u_ptr, ui_idx, rel_ptr, rel_idx, n_items, *args)


def test_zero_division_is_raised_as_get_top_n_raises():
    ts = offset_trainset(seed=2)
    algo = sb.KNNBasic(k=5, min_k=0).fit(ts)
    algo.sim = np.zeros((ts.n_users, ts.n_users))     # no positive neighbour anywhere: 0 / 0 with min_k = 0
    tes = [(ts.to_raw_uid(3), ts.to_raw_iid(0), 15.0)]
    with pytest.raises(ZeroDivisionError):
        algo.get_top_n(ts.n_items)
    with pytest.raises(ZeroDivisionError):
        algo.rank_measures(tes)


# -- model selection -------------------------------------------------------------------------------------------------
def test_cross_validate_equals_separate_calls(u1_splits):
    data = u1_splits[0]
    cv = LeaveOneOut(2, random_state=4)
    make = lambda: sb.SVD(n_factors=10, n_epochs=3, random_state=0)  # noqa: E731
    got = cross_validate(make(), data, ["hr@10", "AUC", "mpr", "rmse"], cv)
    for k, (trs, tes) in enumerate(cv.split(data)):
        algo = make().fit(trs)
        ranks = algo.rank_measures(tes)
        assert same_result(ranks, definition(algo, tes, None))
        want = {"hr@10": algo.top_n_measures(tes, 10)["hr"], "auc": ranks["auc"], "mpr": ranks["mpr"],
                "rmse": accuracy.rmse(algo.test(tes), verbose=False)}
        for name, value in want.items():
            assert np.float64(got["test_" + name][k]).tobytes() == np.float64(value).tobytes(), (k, name)


def test_rank_only_fold_runs_no_selection(u1_splits, monkeypatch):
    trs, tes = u1_splits[1]["loo"]
    algo = sb.SVD(n_factors=20, n_epochs=3, random_state=0).fit(trs)
    fold = Fold(trs, tes)
    iu = fold.test_pairs().relevant(None, trs.n_items)[0]
    users = iu[iu >= 0]
    blocks = -(-len(users) // 100)
    lib = nat.lib()
    lib.sb2_reset_launch_count()
    algo.top_n_inner(10, users, _block_rows=100)
    base = lib.sb2_launch_count()               # scorer and selection per block
    lib.sb2_reset_launch_count()
    both = algo._top_n_fold(fold, [10], [], None, None, 100, rank=True)
    assert lib.sb2_launch_count() == base + 2 * blocks          # plus the hit and rank kernels
    lib.sb2_reset_launch_count()
    with monkeypatch.context() as m:
        m.setattr(lib, "sb2_top_n_select_dev", None)            # any selection call would fail
        only = algo._top_n_fold(fold, [], [], None, None, 100, rank=True)
    assert lib.sb2_launch_count() == base                       # the rank kernel in place of the selection
    assert same_result(both[2], only[2]) and same_result(only[2], algo.rank_measures(tes))
    assert only[0] == [] and only[1] == []


def test_grid_search_ranks_as_the_definition(u1_splits):
    data = u1_splits[0]
    cv = LeaveOneOut(2, random_state=0)
    grid = {"n_factors": [5, 50], "n_epochs": [1, 10], "random_state": [0]}
    gs = GridSearchCV(sb.SVD, grid, measures=["auc", "mpr"], cv=cv)
    gs.fit(data)
    want = {"auc": [], "mpr": []}
    for params in gs.param_combinations:
        per_fold = [definition(sb.SVD(**params).fit(trs), tes, None) for trs, tes in cv.split(data)]
        for m in want:
            want[m].append(np.mean([r[m] for r in per_fold]))
    for m, pick in (("auc", np.argmax), ("mpr", np.argmin)):
        mean = gs.cv_results["mean_test_" + m]
        assert mean.tobytes() == np.array(want[m]).tobytes(), m
        assert gs.best_params[m] == gs.param_combinations[int(pick(mean))]
        assert gs.cv_results["rank_test_" + m][int(pick(mean))] == 1
