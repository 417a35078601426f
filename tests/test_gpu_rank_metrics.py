"""accuracy.fcp and accuracy.precision_recall_at_k on the device: identical (values, types, key order, warnings) to
the reference's fcp loop and the FAQ recipe, the counts of the two C-ABI entry points against a numpy restatement, and
one launch per call."""
import numpy as np
import pytest

from test_rank_metrics_cpu import (CASES, NUMPY_THRESHOLDS, THRESHOLDS, assert_same_dict, assert_same_fcp,
                                   assert_same_precision_recall, call, count_oracle, group, k_eff, k_values, preds_of,
                                   random_grid, same_value)

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import accuracy  # noqa: E402
from surprise_b200.prediction_algorithms.predictions import Prediction  # noqa: E402


def launches(f, *args, **kw):
    nat.lib().sb2_reset_launch_count()
    out = f(*args, **kw)
    return out, nat.lib().sb2_launch_count()


def check_all(preds, ks=(10, 1, None), thresholds=(3.5, 4)):
    (_, n) = launches(call, accuracy.fcp, preds, verbose=False)
    assert n == 1
    assert_same_fcp(preds)
    for k in ks:
        for t in thresholds:
            (_, n) = launches(accuracy.precision_recall_at_k, preds, k, t)
            assert n == 1
            assert_same_precision_recall(preds, k, t)


@pytest.mark.parametrize("make", [lambda: sb.SVD(n_factors=20, n_epochs=5, random_state=0),
                                  lambda: sb.KNNBasic(sim_options={"name": "msd", "user_based": True}),
                                  lambda: sb.CoClustering(random_state=0)], ids=["svd", "knn", "coclustering"])
def test_u1_predictions(u1, make):
    ts, te = u1
    preds = make().fit(ts).test(te)
    check_all(preds, ks=(10, 1, 0, -3, None, 1000), thresholds=(3.5, 4, 3, np.float64(3.5), np.int64(4)))


@pytest.mark.parametrize("seed", [0, 1])
def test_random_grid(seed):
    preds = preds_of(random_grid(seed, n_users=200))
    check_all(preds, ks=(None, 0, 1, 5, -1), thresholds=(3.5, 3, 2.5))


@pytest.mark.parametrize("case", sorted(CASES))
def test_adversarial_cases(case):
    preds = preds_of(CASES[case])
    (_, n) = launches(call, accuracy.fcp, preds, verbose=False)
    assert n == 1
    assert_same_fcp(preds)
    for k in k_values(CASES[case]):
        for t in THRESHOLDS:
            (_, n) = launches(accuracy.precision_recall_at_k, preds, k, t)
            assert n == 1
            assert_same_precision_recall(preds, k, t)
    assert_same_precision_recall(preds, 1.5, 3.5)


def test_python_route_inputs_launch_nothing():
    for rows in ([("a", None, 3.0), ("a", 4.0, 2.0)], [("a", 4.0, "3.5"), ("a", 3.0, "2.0")],
                 [("a", 4.0, np.float32(0.5)), ("a", 3.0, 0.5)], [("a", 4.0, 2 ** 60), ("a", 3.0, 1.0)]):
        preds = preds_of(rows)
        (_, n) = launches(call, accuracy.fcp, preds, verbose=False)
        assert n == 0
        assert_same_fcp(preds)
        assert_same_precision_recall(preds, 2, 3.5)
    (_, n) = launches(accuracy.precision_recall_at_k, preds_of(CASES["ties"]), 2, np.float32(3.5))
    assert n == 0


@pytest.mark.parametrize("case", sorted(CASES))
def test_numpy_and_nan_thresholds(case):
    # a numpy threshold makes every compare a numpy bool: the results' types follow from the counts alone
    preds = preds_of(CASES[case])
    for k in k_values(CASES[case]):
        for t in NUMPY_THRESHOLDS + [float("nan")]:
            (_, n) = launches(accuracy.precision_recall_at_k, preds, k, t)
            assert n == 1
            assert_same_precision_recall(preds, k, t)


def test_one_entry_users_give_nan_with_warning():
    rng = np.random.RandomState(0)
    preds = preds_of([(u, float(r), float(e)) for u, (r, e) in enumerate(rng.randint(1, 6, (100_000, 2)))])
    (out, n) = launches(call, accuracy.fcp, preds, verbose=False)
    assert n == 1 and np.isnan(out[0]) and out[1] == ["RuntimeWarning"]
    assert_same_fcp(preds)
    check_all(preds[:5000], ks=(1, 0), thresholds=(3.5,))


def test_cross_validate_fcp(monkeypatch):
    import os
    from surprise_b200.model_selection import PredefinedKFold, cross_validate
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    data = sb.Dataset.load_from_folds([(os.path.join(golden, "u1_ml100k_train"),
                                        os.path.join(golden, "u1_ml100k_test"))], sb.Reader("ml-100k"))
    measures = ["rmse", "mae", "fcp"]
    calls, device_counts = [], accuracy._fcp_counts_dev
    monkeypatch.setattr(accuracy, "_fcp_counts_dev", lambda *a: calls.append(1) or device_counts(*a))
    algo = sb.KNNBasic(sim_options={"name": "msd", "user_based": False})     # a deterministic fit
    got = cross_validate(algo, data, measures, PredefinedKFold(), return_train_measures=True)
    assert len(calls) == 2                                                  # test and train predictions
    monkeypatch.setattr(accuracy, "_device_usable", lambda: False)
    want = cross_validate(algo, data, measures, PredefinedKFold(), return_train_measures=True)
    assert len(calls) == 2
    for m in measures:
        for part in ("test_", "train_"):
            assert got[part + m].tobytes() == want[part + m].tobytes(), (part, m)


def run_counts(seg_ptr, r, est, k_effs=None, threshold=0.0):
    d = [nat.to_dev(np.asarray(a), dt) for a, dt in ((seg_ptr, np.int64), (r, np.float64), (est, np.float64))]
    n_seg = len(seg_ptr) - 1
    if k_effs is None:
        out = nat.empty_dev((n_seg, 2), np.int64)
        rc = nat.lib().sb2_fcp_counts_dev(n_seg, len(r), *(nat.ptr(x) for x in d), nat.ptr(out), nat.stream())
    else:
        out = nat.empty_dev((n_seg, 3), np.int64)
        d_k = nat.to_dev(np.asarray(k_effs), np.int64)
        rc = nat.lib().sb2_precision_at_k_counts_dev(n_seg, len(r), *(nat.ptr(x) for x in d), nat.ptr(d_k),
                                                     threshold, nat.ptr(out), nat.stream())
    nat.check(rc)
    return out.cpu().numpy()


def test_entry_points_on_signed_zeros_nan_inf():
    rng = np.random.RandomState(3)
    vals = np.array([-0.0, 0.0, np.nan, np.inf, -np.inf, 1.0, -1.0])
    lens = [1, 2, 7, 300, 1, 2500, 0, 40, 700]
    seg_ptr = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    n = int(seg_ptr[-1])
    r, est = vals[rng.randint(0, len(vals), n)], vals[rng.randint(0, len(vals), n)]
    assert np.array_equal(run_counts(seg_ptr, r, est), count_oracle(seg_ptr, r, est))
    for k in (0, 1, 3, 299, -2, None):
        ks = np.array([k_eff(k, m) for m in lens])
        for t in (0.0, -0.0, 1.0, np.inf):
            want = count_oracle(seg_ptr, r, est, ks, t)
            assert np.array_equal(run_counts(seg_ptr, r, est, ks, t), want), (k, t)


def test_entry_points_reject_malformed_offsets():
    r = np.ones(10)
    for seg_ptr in ([0, 5, 4, 10], [1, 5, 10], [0, 5, 9], [0, 5, 11]):
        with pytest.raises(ValueError, match="malformed"):
            run_counts(np.array(seg_ptr), r, r)
        with pytest.raises(ValueError, match="malformed"):
            run_counts(np.array(seg_ptr), r, r, np.ones(len(seg_ptr) - 1), 0.5)
    assert np.array_equal(run_counts(np.array([0, 0, 10, 10]), r, r), [[0, 0], [0, 0], [0, 0]])


def skewed_fold(n_users, n, seed):
    """A MovieLens-like fold: log-normal user activity, ratings on a 0.5 grid, estimates = rating + noise."""
    rng = np.random.default_rng(seed)
    p = rng.lognormal(0.0, 1.0, n_users)
    u = rng.choice(n_users, n, p=p / p.sum())
    r = rng.integers(1, 11, n) * 0.5
    est = np.clip(r + rng.normal(0, 0.9, n), 0.5, 5.0)
    return u, r, est


def check_scale(u, r, est, ks=(10,), thresholds=(3.5,)):
    preds = [Prediction(a, None, b, c, None) for a, b, c in zip(u.tolist(), r.tolist(), est.tolist())]
    keys, seg_ptr, gr, ge = group(preds)
    want = count_oracle(seg_ptr, gr, ge)
    nc, nd = accuracy._fcp_counts(preds)
    assert list(nc) == keys
    assert np.array_equal(np.array([list(nc.values()), list(nd.values())]).T, want)
    c, d = np.mean(want[:, 0].tolist()), np.mean(want[:, 1].tolist())
    assert same_value(accuracy.fcp(preds, verbose=False), c / (c + d))
    m = np.diff(seg_ptr)
    for k in ks:
        for t in thresholds:
            ks_ = np.array([k_eff(k, int(x)) for x in m])
            cnt = count_oracle(seg_ptr, gr, ge, ks_, t)
            prec, rec = accuracy.precision_recall_at_k(preds, k, t)
            assert list(prec) == keys
            want_p = {u_: (c_ / b if b != 0 else 0) for u_, (_, b, c_) in zip(keys, cnt.tolist())}
            want_r = {u_: (c_ / a if a != 0 else 0) for u_, (a, _, c_) in zip(keys, cnt.tolist())}
            assert_same_dict(prec, want_p)
            assert_same_dict(rec, want_r)


def test_scale_ml20m_fold():
    u, r, est = skewed_fold(138_000, 4_000_000, seed=0)
    check_scale(u, r, est)


def test_scale_single_long_user():
    rng = np.random.default_rng(1)
    n = 50_000
    r = rng.integers(1, 11, n) * 0.5
    est = np.round(np.clip(r + rng.normal(0, 0.9, n), 0.5, 5.0), 1)
    check_scale(np.zeros(n, dtype=np.int64), r, est, ks=(10, 30_000), thresholds=(3.5,))
