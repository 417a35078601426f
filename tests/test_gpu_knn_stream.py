"""k-NN without the dense similarity matrix: sb2_sim_build_rows_dev must give the full build's rows bit for bit, and a
model forced onto the streamed route (similarity rows built band by band at predict time) must give the dense route's
estimates, details, top-N lists, measures, search scores, neighbours, matrix and pickles, bit for bit."""
import os
import pickle

import numpy as np
import pytest

import knn_stream_oracle
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import similarities as sims  # noqa: E402
from surprise_b200 import synth  # noqa: E402
from surprise_b200.model_selection import GridSearchCV  # noqa: E402
from surprise_b200.prediction_algorithms import knns  # noqa: E402

KINDS = ("cosine", "msd", "pearson", "pearson_baseline")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


@pytest.fixture(params=("auto", "digit", "general"))
def sim_path(request, monkeypatch):
    if request.param != "auto":
        monkeypatch.setenv("SB2_SIM_PATH", request.param)
    return request.param


def _baselines(ts):
    algo = sb.BaselineOnly()
    sb.AlgoBase.fit(algo, ts)
    return algo.compute_baselines()


def _kw(kind, ts, ub):
    if kind != "pearson_baseline":
        return {}
    bu, bi = _baselines(ts)
    bx, by = (bu, bi) if ub else (bi, bu)
    return dict(global_mean=float(ts.global_mean), x_biases=bx, y_biases=by)


def _row_lists(n_x, seed=0):
    rng = np.random.RandomState(seed)
    perm = rng.permutation(n_x)
    return [np.array([n_x - 1], dtype=np.int32),
            perm[:300].astype(np.int32),                                       # unsorted, not 256-aligned
            np.concatenate((perm[:37], perm[:5], [0, n_x - 1, 257 % n_x, 257 % n_x])).astype(np.int32),   # repeats
            np.arange(n_x, dtype=np.int32)[::-1].copy()]


def _assert_rows_equal_full(kind, n_x, yr, min_support=1, **kw):
    import torch
    inp = sims.upload_inputs(kind, n_x, yr, kw.get("x_biases"), kw.get("y_biases"))
    full = sims.build_device(kind, n_x, yr, min_support, inputs=inp, **kw).cpu().numpy()
    ms = dict(global_mean=kw.get("global_mean", 0.0), shrinkage=kw.get("shrinkage", 100))
    for rows in _row_lists(n_x):
        out = torch.full((len(rows) + 3, n_x), 7.0, dtype=torch.float64, device="cuda")
        sims.build_rows_device(kind, inp, torch.as_tensor(rows, device="cuda"), out, min_support, **ms)
        got = out.cpu().numpy()
        assert np.array_equal(bits(got[:len(rows)]), bits(full[rows])), (kind, len(rows))
        assert np.all(got[len(rows):] == 7.0)                    # rows past the list untouched


@pytest.mark.parametrize("orient", ("item", "user"))
@pytest.mark.parametrize("kind", KINDS)
def test_rows_equal_full_build_u1(u1, kind, orient, sim_path):
    ts, _ = u1
    ub = orient == "user"
    n_x, yr = (ts.n_users, ts.item_csr()) if ub else (ts.n_items, ts.user_csr())
    _assert_rows_equal_full(kind, n_x, yr, **_kw(kind, ts, ub))
    if kind == "msd":
        _assert_rows_equal_full(kind, n_x, yr, min_support=5)


@pytest.mark.parametrize("kind", KINDS)
def test_rows_equal_full_build_floats_and_duplicates(floats, kind, monkeypatch):
    """Two-decimal ratings (denominator 100; the row build follows the full build's path) and, with a few (x, y)
    pairs repeated, the general path's duplicate handling."""
    ds = sb.Dataset.load_from_arrays(floats["uid"], floats["iid"], floats["rating"], sb.Reader(rating_scale=(-10, 10)))
    ts = ds.build_full_trainset()
    for ub in (False, True):
        n_x, yr = (ts.n_users, ts.item_csr()) if ub else (ts.n_items, ts.user_csr())
        kw = _kw(kind, ts, ub)
        _assert_rows_equal_full(kind, n_x, yr, 2, **kw)
        ptr, idx, val = yr
        dup = np.arange(0, len(idx), 9)                      # repeat every 9th entry right after itself
        keep = np.sort(np.concatenate((np.arange(len(idx)), dup)), kind="stable")
        seg = np.searchsorted(ptr, keep, side="right") - 1
        ptr2 = np.concatenate(([0], np.cumsum(np.bincount(seg, minlength=len(ptr) - 1)))).astype(np.int64)
        _assert_rows_equal_full(kind, n_x, (ptr2, idx[keep], val[keep]), 2, **kw)
        monkeypatch.setenv("SB2_SIM_PATH", "general")
        _assert_rows_equal_full(kind, n_x, yr, 2, **kw)
        monkeypatch.delenv("SB2_SIM_PATH")


@pytest.mark.parametrize("kind", ("cosine", "pearson_baseline"))
def test_rows_equal_full_build_skewed_synth(kind, sim_path):
    d = synth.ratings(3000, 1200, 120_000, step=0.5, seed=3, skew=True)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"], (0.5, 5.0), 0)
    for ub in (True, False):
        n_x, yr = (ts.n_users, ts.item_csr()) if ub else (ts.n_items, ts.user_csr())
        _assert_rows_equal_full(kind, n_x, yr, **_kw(kind, ts, ub))


def test_rows_errors(u1):
    import torch
    ts, _ = u1
    inp = sims.upload_inputs("msd", ts.n_items, ts.user_csr())
    out = torch.empty((2, ts.n_items), dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        sims.build_rows_device("msd", inp, torch.tensor([0, ts.n_items], dtype=torch.int32, device="cuda"), out, 1)
    with pytest.raises(ZeroDivisionError):   # some item pair without a common user
        sims.build_rows_device("msd", inp, torch.arange(2, dtype=torch.int32, device="cuda"), out, 0)


# ---- forced streaming against the dense route ------------------------------------------------------------
ALGOS = {
    "basic_cosine": (sb.KNNBasic, dict(k=40, sim_options={"name": "cosine"})),
    "means_msd": (sb.KNNWithMeans, dict(k=30, sim_options={"name": "msd"})),
    "zscore_pearson": (sb.KNNWithZScore, dict(k=20, min_k=3, sim_options={"name": "pearson"})),
    "baseline_pb": (sb.KNNBaseline, dict(k=40, sim_options={"name": "pearson_baseline"})),
}


def make(case, orient):
    cls, kw = ALGOS[case]
    kw = dict(kw, sim_options=dict(kw["sim_options"], user_based=orient == "user"))
    return cls(**kw)


def stream(monkeypatch, n_x, band):
    monkeypatch.setattr(knns, "_DENSE_SIM_FRACTION", 0.0)
    monkeypatch.setattr(knns, "_STREAM_BAND_BYTES", 8 * n_x * band)


@pytest.fixture(scope="module")
def testset(u1):
    """u1's testset, then a shuffled copy of 3000 of its rows (duplicated pairs) and unknown users / items."""
    _, tes = u1
    rng = np.random.RandomState(5)
    extra = [tes[k] for k in rng.permutation(len(tes))[:3000]]
    return list(tes) + extra + [("nobody", "1", 4.0), ("1", "no-item", 2.0), ("nobody", "x", 1.0)]


def outputs(algo, ts, tes):
    preds = algo.test(tes)
    est = np.array([p.est for p in preds])
    details = [sorted(p.details.items()) for p in preds]
    top = algo.get_top_n(10)
    top_bits = {u: [(i, int(np.float64(e).view(np.int64))) for i, e in l] for u, l in top.items()}
    meas = algo.top_n_measures(tes, 10, 3.5)
    meas = [meas[key] for key in sorted(meas)]
    x_ids = [0, 1, 17, algo.n_x - 1]
    nbrs = [algo.get_neighbors(x, k) for x in x_ids for k in (1, 10, algo.n_x)]
    return est, details, top_bits, np.array(meas), nbrs


_dense = {}


def dense_outputs(case, orient, ts, tes):
    if (case, orient) not in _dense:
        algo = make(case, orient).fit(ts)
        assert not algo._streamed
        _dense[(case, orient)] = outputs(algo, ts, tes) + (algo.sim.copy(),)
    return _dense[(case, orient)]


@pytest.mark.parametrize("band", (1, 7, 256, None))
@pytest.mark.parametrize("orient", ("user", "item"))
@pytest.mark.parametrize("case", sorted(ALGOS))
def test_streamed_equals_dense(u1, testset, case, orient, band, monkeypatch):
    import torch
    ts, _ = u1
    want = dense_outputs(case, orient, ts, testset)
    n_x = ts.n_users if orient == "user" else ts.n_items
    stream(monkeypatch, n_x, band or n_x)
    algo = make(case, orient).fit(ts)
    assert algo._streamed and algo._sim_dev is None
    got = outputs(algo, ts, testset)
    assert np.array_equal(bits(got[0]), bits(want[0]))
    assert got[1] == want[1]
    assert got[2] == want[2]
    assert np.array_equal(bits(got[3]), bits(want[3]))
    assert got[4] == want[4]
    if band in (7, None):
        back = pickle.loads(pickle.dumps(algo))
        assert back._streamed and back._sim_inputs is None and back._sim_host is None   # no matrix in the pickle
        assert np.array_equal(bits(outputs(back, ts, testset)[0]), bits(want[0]))
        assert np.array_equal(bits(algo.sim), bits(want[5]))
        torch.cuda.synchronize()


def test_streamed_golden_rmse(u1, u1_golden, monkeypatch):
    """Config 1 and its siblings through the streamed route: RMSE / MAE to the last bit."""
    ts, tes = u1
    for orient in ("item", "user"):
        n_x = ts.n_users if orient == "user" else ts.n_items
        stream(monkeypatch, n_x, 7)
        for kind in ("cosine", "msd", "pearson"):
            algo = sb.KNNBasic(sim_options={"name": kind, "user_based": orient == "user", "min_support": 1})
            preds = algo.fit(ts).test(tes)
            assert algo._streamed
            g = u1_golden["algos"]["KNNBasic_%s_%s_ms1" % (kind, orient)]
            assert repr(float(sb.accuracy.rmse(preds, verbose=False))) == g["rmse"]
            assert repr(float(sb.accuracy.mae(preds, verbose=False))) == g["mae"]


def test_streamed_grid_search_scores(u1, monkeypatch):
    reader = sb.Reader("ml-100k")
    data = sb.Dataset.load_from_folds([(os.path.join(GOLDEN, "u1_ml100k_train"),
                                        os.path.join(GOLDEN, "u1_ml100k_test"))], reader)
    grid = {"k": [10, 40], "sim_options": {"name": ["msd", "pearson_baseline"], "user_based": [True, False]}}
    measures = ["rmse", "mae", "fcp", "hr@10"]
    want = GridSearchCV(sb.KNNBaseline, grid, measures=measures, cv=sb.model_selection.PredefinedKFold())
    want.fit(data)
    stream(monkeypatch, 1682, 7)
    got = GridSearchCV(sb.KNNBaseline, grid, measures=measures, cv=sb.model_selection.PredefinedKFold())
    got.fit(data)
    keys = [key for key in want.cv_results
            if key.startswith(("split", "mean_test", "std_test")) and key.split("_")[-1] in measures]
    assert len(keys) == 3 * len(measures)
    for key in keys:
        assert np.array_equal(bits(got.cv_results[key]), bits(want.cv_results[key])), key


def test_streamed_fit_raises_and_assigned_sim(u1, monkeypatch):
    ts, tes = u1
    with pytest.raises(ZeroDivisionError):
        sb.KNNBasic(sim_options={"name": "msd", "min_support": 0, "user_based": False}).fit(ts)
    stream(monkeypatch, ts.n_items, 256)
    with pytest.raises(ZeroDivisionError):
        sb.KNNBasic(sim_options={"name": "msd", "min_support": 0, "user_based": False}).fit(ts)
    algo = sb.KNNBasic(sim_options={"name": "cosine", "user_based": False}).fit(ts)
    assert algo._streamed
    want = np.array([p.est for p in algo.test(tes)])
    algo.sim = algo.sim.copy()                 # a user-assigned matrix: back on the dense route
    assert not algo._streamed
    assert np.array_equal(bits([p.est for p in algo.test(tes)]), bits(want))


# ---- full shape: the Netflix shape, where the dense matrix would be 1.84 TB --------------------------------
def test_netflix_shape_user_based_streamed(monkeypatch):
    import torch
    d = synth.shaped("netflix", seed=0)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"], (1.0, 5.0), 0)
    tu, ti, _ = d["test"]
    rng = np.random.RandomState(0)
    sel = rng.choice(len(tu), 10_000, replace=False)
    pu, pi = tu[sel].astype(np.int32), ti[sel].astype(np.int32)
    pu[:20] = -1                                                  # unknown users
    known = (pu >= 0) & (pi >= 0)
    budget = 4 << 30
    monkeypatch.setattr(knns, "_STREAM_BAND_BYTES", budget)
    assert knns.streams_similarities(ts.n_users, knns._device_bytes())   # 1.84 TB: streamed without any patch
    for cls, kind, mode in ((sb.KNNBasic, "cosine", 0), (sb.KNNBaseline, "pearson_baseline", 1)):
        algo = cls(k=40, sim_options={"name": kind, "user_based": True})
        algo.fit(ts)
        assert algo._streamed
        want_est, want_ak = knn_stream_oracle.user_based(kind, mode, ts, u, i, r, pu, pi, 40, algo.bu, algo.bi)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        est, ak, imp = algo._knn_batch(pu, pi, *algo._knn_args())
        peak = torch.cuda.max_memory_allocated() - base
        assert peak <= budget + 64 * len(pu) + (16 << 20), peak
        ok = known & (imp == 0)
        assert np.array_equal(bits(est[ok]), bits(want_est[ok]))
        assert np.array_equal(ak[known], want_ak[known])
        if mode:
            assert np.array_equal(bits(est), bits(want_est))
        else:
            assert np.array_equal(imp[~known], np.ones((~known).sum(), dtype=np.uint8))
        del algo
        torch.cuda.empty_cache()
