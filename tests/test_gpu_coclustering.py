"""CoClustering on the device against the C oracle (itself pinned to a transcription of the reference and to the u1
golden by tests/test_coclustering_cpu.py): every fitted attribute np.array_equal, every estimate equal bit for bit."""
import os
import pickle

import numpy as np
import pytest

from conftest import GOLDEN, inner_pairs
from test_coclustering_cpu import U1_CONFIGS, custom_trainset, float_sets, oracle_estimates, oracle_fit

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import synth  # noqa: E402

ATTRS = ("cltr_u", "cltr_i", "user_mean", "item_mean", "avg_cltr_u", "avg_cltr_i", "avg_cocltr")


def check_fit(ts, pairs, n_cltr_u=3, n_cltr_i=3, n_epochs=20, random_state=0):
    """Fit on the device and with the oracle from the same seed; compare every attribute and the batched estimates."""
    algo = sb.CoClustering(n_cltr_u, n_cltr_i, n_epochs, random_state=random_state).fit(ts)
    want = oracle_fit(ts, n_cltr_u, n_cltr_i, n_epochs, random_state=random_state)
    for k in ATTRS:
        got = getattr(algo, k)
        assert isinstance(got, np.ndarray) and got.dtype == want[k].dtype, k
        assert np.array_equal(got, want[k]), k
    iu, ii = pairs
    est, details = algo._estimate_batch(iu, ii)
    assert np.array_equal(est, oracle_estimates(ts, want, iu, ii))
    assert not any(d["was_impossible"] for d in details)
    return algo, want


def test_u1_configurations(u1, cc_golden):
    ts, testset = u1
    iu, ii = inner_pairs(ts, testset)
    for cfg in U1_CONFIGS:
        algo, want = check_fit(ts, (iu, ii), *cfg, random_state=1)
        preds = algo.test(testset)
        assert np.array_equal(np.array([p.est for p in preds]),
                              np.clip(oracle_estimates(ts, want, iu, ii), *ts.rating_scale))
        if cfg == (3, 3, 20):
            assert repr(float(sb.accuracy.rmse(preds, verbose=False))) == cc_golden["u1_default_rs1"]["rmse"]
            assert repr(float(sb.accuracy.mae(preds, verbose=False))) == cc_golden["u1_default_rs1"]["mae"]


@pytest.fixture(scope="module")
def cc_golden():
    import json
    with open(os.path.join(GOLDEN, "coclustering_golden.json")) as fh:
        return json.load(fh)


def all_pairs(ts, step=1):
    iu = np.arange(-1, ts.n_users, step, dtype=np.int32).repeat(4)
    ii = np.resize(np.arange(-1, ts.n_items, dtype=np.int32), len(iu))
    return iu, ii


def test_float_and_half_star_sets(floats):
    """Negative and fractional ratings: the C-int truncation path (and the np.mean fallback of the means)."""
    for ts in float_sets(floats):
        for cfg, seed in (((3, 3, 20), 0), ((2, 5, 7), 3), ((4, 1, 4), 11), ((40, 40, 6), 5)):
            check_fit(ts, all_pairs(ts), *cfg, random_state=seed)


def test_empty_clusters_take_global_mean():
    """More clusters than users / items: empty clusters, whose averages fall back to global_mean."""
    ts = custom_trainset()
    algo, want = check_fit(ts, all_pairs(ts), 20, 9, 5, random_state=2)
    assert ts.n_users < 20 and (algo.avg_cltr_u == ts.global_mean).any()


@pytest.fixture(scope="module")
def skewed():
    d = synth.ratings(3000, 1500, 150_000, seed=21, skew=True)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    assert np.bincount(i).max() > 1500   # a 2000-rater item: the longest ordered chain
    return d, ts


def test_skewed_long_segments(skewed):
    d, ts = skewed
    tu, ti, _ = d["test"]
    for cfg in ((3, 3, 20), (5, 40, 4)):
        check_fit(ts, (tu, ti), *cfg, random_state=4)


def test_table_larger_than_shared_memory(skewed):
    """300 x 300 cells (1.4 MB of counts and sums): the global-atomic histogram and several 32-candidate groups."""
    d, ts = skewed
    tu, ti, _ = d["test"]
    check_fit(ts, (tu, ti), 300, 300, 2, random_state=6)
    check_fit(ts, (tu, ti), 33, 70, 3, random_state=7)


def test_ml1m_shape_defaults():
    d = synth.shaped("ml-1m")
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    tu, ti, _ = d["test"]
    check_fit(ts, (tu, ti), random_state=0)


def test_draw_order_and_launches(u1):
    """cltr_u is drawn before cltr_i (n_epochs=0 returns the draw); a fit is 4 launches per epoch + 3 and never
    synchronises inside the epoch loop (one status read at the end)."""
    ts, _ = u1
    algo = sb.CoClustering(4, 6, 0, random_state=9).fit(ts)
    rng = np.random.RandomState(9)
    assert np.array_equal(algo.cltr_u, rng.randint(4, size=ts.n_users))
    assert np.array_equal(algo.cltr_i, rng.randint(6, size=ts.n_items))
    for n_ep in (0, 7):
        nat.lib().sb2_reset_launch_count()
        sb.CoClustering(n_epochs=n_ep, random_state=0).fit(ts)
        assert nat.lib().sb2_launch_count() == 4 * n_ep + 3


def test_host_c_abi_equals_device_form(u1):
    ts, _ = u1
    algo = sb.CoClustering(5, 4, 6, random_state=3).fit(ts)
    up, ui, ur = ts.user_csr()
    ip, iu, ir = ts.item_csr()
    rng = np.random.RandomState(3)
    cu = rng.randint(5, size=ts.n_users).astype(np.int32)
    ci = rng.randint(4, size=ts.n_items).astype(np.int32)
    au, ai, ac = np.empty(5), np.empty(4), np.empty((5, 4))
    nat.check(nat.lib().sb2_coclustering_fit(ts.n_users, ts.n_items, nat.hptr(up), nat.hptr(ui), nat.hptr(ur),
                                             nat.hptr(ip), nat.hptr(iu), nat.hptr(ir), nat.hptr(algo.user_mean),
                                             nat.hptr(algo.item_mean), float(ts.global_mean), 5, 4, 6, nat.hptr(cu),
                                             nat.hptr(ci), nat.hptr(au), nat.hptr(ai), nat.hptr(ac)))
    assert np.array_equal(cu, algo.cltr_u) and np.array_equal(ci, algo.cltr_i)
    assert np.array_equal(au, algo.avg_cltr_u) and np.array_equal(ai, algo.avg_cltr_i)
    assert np.array_equal(ac, algo.avg_cocltr)


def test_invalid_input():
    ts = sb.Trainset.from_coo([0, 0, 1], [0, 1, 0], [1.0, 3e9, 2.0])
    with pytest.raises(OverflowError):
        sb.CoClustering(random_state=0).fit(ts)
    ts = custom_trainset()
    up, ui, ur = ts.user_csr()
    ip, iu, ir = ts.item_csr()
    cu, ci = np.zeros(ts.n_users, np.int32), np.zeros(ts.n_items, np.int32)
    means = np.zeros(max(ts.n_users, ts.n_items))
    out = np.empty(64)
    for ncu, nci, bad in ((0, 3, None), (3, -1, None), (3, 3, "u")):
        if bad:
            cu[0] = 3
        rc = nat.lib().sb2_coclustering_fit(ts.n_users, ts.n_items, nat.hptr(up), nat.hptr(ui), nat.hptr(ur),
                                            nat.hptr(ip), nat.hptr(iu), nat.hptr(ir), nat.hptr(means), nat.hptr(means),
                                            3.0, ncu, nci, 2, nat.hptr(cu), nat.hptr(ci), nat.hptr(out),
                                            nat.hptr(out), nat.hptr(out))
        assert rc == nat.ERR_INVALID


def test_unknown_ids_predict_test_pickle_dump(tmp_path):
    """reference tests/test_algorithms.py::test_unknown_user_or_item + tests/test_dump.py, and predict == test."""
    reader = sb.Reader(line_format="user item rating", sep=" ", skip_lines=3, rating_scale=(1, 5))
    data = sb.Dataset.load_from_file(os.path.join(GOLDEN, "custom_dataset"), reader)
    ts = data.build_full_trainset()
    algo = sb.CoClustering(random_state=0).fit(ts)
    for uid, iid in (("user0", "unknown_item"), ("unkown_user", "item0"), ("unkown_user", "unknown_item")):
        p = algo.predict(uid, iid, None)
        assert p.est == ts.global_mean and p.details == {"was_impossible": False}
    testset = ts.build_testset() + [("unkown_user", "item0", 3.0), ("user0", "unknown_item", 2.0)]
    preds = algo.test(testset)
    assert [p.est for p in preds] == [algo.predict(u, i, r).est for (u, i, r) in testset]
    assert [p.details for p in preds] == [algo.predict(u, i, r).details for (u, i, r) in testset]
    clone = pickle.loads(pickle.dumps(algo))
    assert clone._dev is None
    assert [p.est for p in clone.test(testset)] == [p.est for p in preds]
    for k in ATTRS:
        assert np.array_equal(getattr(clone, k), getattr(algo, k))
    path = str(tmp_path / "cc.dump")
    sb.dump.dump(path, predictions=preds, algo=algo)
    preds2, algo2 = sb.dump.load(path)
    assert preds2 == preds and [p.est for p in algo2.test(testset)] == [p.est for p in preds]


def test_cross_validate_predefined_folds(u1):
    """reference tests/test_co_clustering.py: runs through cross_validate on the u1 folds, and every parameter
    changes the RMSE."""
    from surprise_b200.model_selection import PredefinedKFold, cross_validate
    data = sb.Dataset.load_from_folds([(os.path.join(GOLDEN, "u1_ml100k_train"),
                                        os.path.join(GOLDEN, "u1_ml100k_test"))], sb.Reader("ml-100k"))

    def rmse(**kw):
        kw.setdefault("n_epochs", 1)
        return float(cross_validate(sb.CoClustering(random_state=1, **kw), data, ["rmse"], PredefinedKFold())
                     ["test_rmse"][0])

    base = rmse()
    assert base != rmse(n_cltr_u=1)
    assert base != rmse(n_cltr_i=1)
    assert base != rmse(n_epochs=2)
