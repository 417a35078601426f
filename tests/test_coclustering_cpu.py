"""CoClustering without a GPU: the C oracle (tests/coclustering_oracle.c) against a literal Python transcription of the
reference's CoClustering.fit / compute_averages / estimate (co_clustering.pyx:68-237), bit for bit; the u1 golden;
the compiled reference wherever oracle/_ref is built; constructor and argument behaviour."""
import hashlib
import json
import os

import numpy as np
import pytest

import coclustering_oracle
import oracle
from conftest import GOLDEN, inner_pairs

import surprise_b200 as sb
from surprise_b200.prediction_algorithms.algo_base import list_means
from surprise_b200.utils import get_rng

U1_CONFIGS = [(3, 3, 20), (1, 1, 5), (3, 3, 0), (2, 7, 20), (10, 10, 3)]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# ---- the transcription: Python floats are IEEE doubles; int() where the reference declares `cdef int` ------------
def compute_averages(ts, cltr_u, cltr_i, n_cltr_u, n_cltr_i):
    count_cltr_u, count_cltr_i = [0] * n_cltr_u, [0] * n_cltr_i
    count_cocltr = [[0] * n_cltr_i for _ in range(n_cltr_u)]
    sum_cltr_u, sum_cltr_i = [0.0] * n_cltr_u, [0.0] * n_cltr_i
    sum_cocltr = [[0.0] * n_cltr_i for _ in range(n_cltr_u)]
    for u, i, r in ts.all_ratings():
        r = int(r)
        uc, ic = cltr_u[u], cltr_i[i]
        count_cltr_u[uc] += 1
        count_cltr_i[ic] += 1
        count_cocltr[uc][ic] += 1
        sum_cltr_u[uc] += r
        sum_cltr_i[ic] += r
        sum_cocltr[uc][ic] += r
    gm = ts.global_mean
    avg_cltr_u = [s / c if c else gm for s, c in zip(sum_cltr_u, count_cltr_u)]
    avg_cltr_i = [s / c if c else gm for s, c in zip(sum_cltr_i, count_cltr_i)]
    avg_cocltr = [[s / c if c else gm for s, c in zip(sr, cr)] for sr, cr in zip(sum_cocltr, count_cocltr)]
    return avg_cltr_u, avg_cltr_i, avg_cocltr


def transcribed_fit(ts, n_cltr_u=3, n_cltr_i=3, n_epochs=20, random_state=None):
    rng = get_rng(random_state)
    cltr_u = rng.randint(n_cltr_u, size=ts.n_users).tolist()
    cltr_i = rng.randint(n_cltr_i, size=ts.n_items).tolist()
    ur, ir = ts.ur, ts.ir
    user_mean = [float(np.mean([r for (_, r) in ur[u]])) for u in ts.all_users()]
    item_mean = [float(np.mean([r for (_, r) in ir[i]])) for i in ts.all_items()]
    for _ in range(n_epochs):
        avg_cltr_u, avg_cltr_i, avg_cocltr = compute_averages(ts, cltr_u, cltr_i, n_cltr_u, n_cltr_i)
        for u in ts.all_users():
            errors = [0.0] * n_cltr_u
            for uc in range(n_cltr_u):
                for i, r in ur[u]:
                    r = int(r)
                    ic = cltr_i[i]
                    est = avg_cocltr[uc][ic] + user_mean[u] - avg_cltr_u[uc] + item_mean[i] - avg_cltr_i[ic]
                    errors[uc] += (r - est) ** 2
            cltr_u[u] = int(np.argmin(errors))
        for i in ts.all_items():
            errors = [0.0] * n_cltr_i
            for ic in range(n_cltr_i):
                for u, r in ir[i]:
                    r = int(r)
                    uc = cltr_u[u]
                    est = avg_cocltr[uc][ic] + user_mean[u] - avg_cltr_u[uc] + item_mean[i] - avg_cltr_i[ic]
                    errors[ic] += (r - est) ** 2
            cltr_i[i] = int(np.argmin(errors))
    avg_cltr_u, avg_cltr_i, avg_cocltr = compute_averages(ts, cltr_u, cltr_i, n_cltr_u, n_cltr_i)
    return dict(cltr_u=np.array(cltr_u, dtype=np.int64), cltr_i=np.array(cltr_i, dtype=np.int64),
                user_mean=np.array(user_mean), item_mean=np.array(item_mean), avg_cltr_u=np.array(avg_cltr_u),
                avg_cltr_i=np.array(avg_cltr_i), avg_cocltr=np.array(avg_cocltr).reshape(n_cltr_u, n_cltr_i))


def transcribed_estimate(ts, m, u, i):
    if not (0 <= u < ts.n_users and 0 <= i < ts.n_items):
        return ts.global_mean
    uc, ic = m["cltr_u"][u], m["cltr_i"][i]
    return float(m["avg_cocltr"][uc, ic] + m["user_mean"][u] - m["avg_cltr_u"][uc] + m["item_mean"][i]
                 - m["avg_cltr_i"][ic])


def oracle_fit(ts, n_cltr_u=3, n_cltr_i=3, n_epochs=20, random_state=None):
    """What CoClustering.fit computes, with the C oracle for the epoch loop."""
    rng = get_rng(random_state)
    cu0 = rng.randint(n_cltr_u, size=ts.n_users)
    ci0 = rng.randint(n_cltr_i, size=ts.n_items)
    um, im = list_means(*ts.user_csr()[::2]), list_means(*ts.item_csr()[::2])
    cu, ci, au, ai, ac = coclustering_oracle.fit(ts.n_users, ts.n_items, ts.user_csr(), ts.item_csr(), um, im,
                                          ts.global_mean, n_cltr_u, n_cltr_i, n_epochs, cu0, ci0)
    return dict(cltr_u=cu, cltr_i=ci, user_mean=um, item_mean=im, avg_cltr_u=au, avg_cltr_i=ai, avg_cocltr=ac)


def oracle_estimates(ts, m, iu, ii):
    return coclustering_oracle.estimate(iu, ii, m["cltr_u"], m["cltr_i"], m["user_mean"], m["item_mean"],
                                        m["avg_cltr_u"], m["avg_cltr_i"], m["avg_cocltr"], ts.global_mean)


def accuracy_of(ts, testset, est):
    """AlgoBase.test + accuracy.rmse / mae on the given raw estimates (offset, clipping, Prediction tuples)."""
    lo, hi = ts.rating_scale
    preds = [sb.Prediction(u, i, r - ts.offset, max(lo, min(hi, e - ts.offset)), {})
             for (u, i, r), e in zip(testset, np.asarray(est).tolist())]
    return repr(float(sb.accuracy.rmse(preds, verbose=False))), repr(float(sb.accuracy.mae(preds, verbose=False)))


def assert_same_model(got, want):
    for k in ("cltr_u", "cltr_i", "user_mean", "item_mean", "avg_cltr_u", "avg_cltr_i", "avg_cocltr"):
        assert got[k].dtype == want[k].dtype, k
        assert np.array_equal(got[k], want[k]), k


def float_sets(floats):
    out = []
    for pre, scale in (("", (-10, 10)), ("half_", (0.5, 5))):
        ds = sb.Dataset.load_from_arrays(floats[pre + "uid"], floats[pre + "iid"], floats[pre + "rating"],
                                         sb.Reader(rating_scale=scale))
        out.append(ds.build_full_trainset())
    return out


def custom_trainset():
    reader = sb.Reader(line_format="user item rating", sep=" ", skip_lines=3, rating_scale=(1, 5))
    return sb.Dataset.load_from_file(os.path.join(GOLDEN, "custom_dataset"), reader).build_full_trainset()


# ---- oracle == transcription ------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", U1_CONFIGS)
def test_oracle_matches_transcription_u1(u1, cfg):
    ts, testset = u1
    n_cu, n_ci, n_ep = cfg
    want = transcribed_fit(ts, n_cu, n_ci, n_ep, random_state=1)
    got = oracle_fit(ts, n_cu, n_ci, n_ep, random_state=1)
    assert_same_model(got, want)
    iu, ii = inner_pairs(ts, testset)
    est = oracle_estimates(ts, got, iu, ii)
    assert np.array_equal(est, [transcribed_estimate(ts, want, int(a), int(b)) for a, b in zip(iu, ii)])


def test_oracle_matches_transcription_small_sets(floats):
    """custom_dataset, the float (negative, fractional: truncation toward zero) and the half-star sets."""
    for ts in [custom_trainset()] + float_sets(floats):
        for cfg, seed in (((3, 3, 20), 0), ((2, 5, 7), 3), ((4, 1, 4), 11)):
            want = transcribed_fit(ts, *cfg, random_state=seed)
            got = oracle_fit(ts, *cfg, random_state=seed)
            assert_same_model(got, want)
            iu = np.arange(-1, ts.n_users, dtype=np.int32).repeat(3)
            ii = np.resize(np.arange(-1, ts.n_items, dtype=np.int32), len(iu))
            est = oracle_estimates(ts, got, iu, ii)
            assert np.array_equal(est, [transcribed_estimate(ts, want, int(a), int(b)) for a, b in zip(iu, ii)])


def test_list_means_is_np_mean(floats):
    """The shared per-list mean (SlopeOne and CoClustering): both the exact fast path and the np.mean loop."""
    for ts in [custom_trainset()] + float_sets(floats):
        for ptr, _, val in (ts.user_csr(), ts.item_csr()):
            want = [np.mean(val[ptr[k]:ptr[k + 1]].tolist()) for k in range(len(ptr) - 1)]
            assert np.array_equal(list_means(ptr, val), want)


# ---- golden ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cc_golden():
    with open(os.path.join(GOLDEN, "coclustering_golden.json")) as fh:
        return json.load(fh)


def test_u1_golden(u1, cc_golden):
    ts, testset = u1
    m = oracle_fit(ts, random_state=1)
    g = cc_golden["u1_default_rs1"]
    for k in ("cltr_u", "cltr_i", "avg_cltr_u", "avg_cltr_i", "avg_cocltr"):
        assert sha(m[k]) == g["sha256"][k], k
    rmse, mae = accuracy_of(ts, testset, oracle_estimates(ts, m, *inner_pairs(ts, testset)))
    assert (rmse, mae) == (g["rmse"], g["mae"])


@pytest.mark.skipif(oracle.reference_path() is None, reason="the compiled reference (oracle/_ref) is not built here")
def test_compiled_reference(u1, cc_golden, floats):
    """The compiled reference's CoClustering against the oracle: u1 (and its golden) and the fractional ratings, which
    also settle the reading of `[r for (_, r) in ur[u]]` under `cdef int r` (untruncated means)."""
    ref = oracle.import_reference()
    from surprise.model_selection import PredefinedKFold
    data = ref.Dataset.load_from_folds([(os.path.join(GOLDEN, "u1_ml100k_train"),
                                         os.path.join(GOLDEN, "u1_ml100k_test"))], ref.Reader("ml-100k"))
    rtrain, rtest = next(PredefinedKFold().split(data))
    ts, testset = u1
    for cfg in U1_CONFIGS:
        algo = ref.CoClustering(*cfg, random_state=1)
        algo.fit(rtrain)
        want = oracle_fit(ts, *cfg, random_state=1)
        for k in ("cltr_u", "cltr_i", "avg_cltr_u", "avg_cltr_i", "avg_cocltr"):
            assert np.array_equal(np.asarray(getattr(algo, k)), want[k]), (cfg, k)
        if cfg == (3, 3, 20):
            preds = algo.test(rtest)
            g = cc_golden["u1_default_rs1"]
            assert repr(float(ref.accuracy.rmse(preds, verbose=False))) == g["rmse"]
    import pandas as pd
    rdata = ref.Dataset.load_from_df(pd.DataFrame({"u": floats["uid"], "i": floats["iid"], "r": floats["rating"]}),
                                     ref.Reader(rating_scale=(-10, 10)))
    algo = ref.CoClustering(random_state=0).fit(rdata.build_full_trainset())
    want = oracle_fit(float_sets(floats)[0], random_state=0)
    for k in ("cltr_u", "cltr_i", "user_mean", "item_mean", "avg_cltr_u", "avg_cltr_i", "avg_cocltr"):
        assert np.array_equal(np.asarray(getattr(algo, k)), want[k]), k


# ---- API ---------------------------------------------------------------------------------------------------------
def test_constructor_defaults():
    algo = sb.CoClustering()
    assert (algo.n_cltr_u, algo.n_cltr_i, algo.n_epochs, algo.random_state, algo.verbose) == (3, 3, 20, None, False)
    assert isinstance(algo, sb.AlgoBase) and algo.sim_options == {"user_based": True} and algo.bsl_options == {}
    algo = sb.CoClustering(4, 5, 6, 7, True)
    assert (algo.n_cltr_u, algo.n_cltr_i, algo.n_epochs, algo.random_state, algo.verbose) == (4, 5, 6, 7, True)


@pytest.mark.parametrize("kw", [dict(n_cltr_u=0), dict(n_cltr_i=0)])
def test_zero_clusters_raise_value_error(kw):
    """rng.randint(0, ...) raises ValueError in the reference; it happens before any device work here too."""
    with pytest.raises(ValueError):
        sb.CoClustering(random_state=0, **kw).fit(custom_trainset())


def test_oracle_rejects_ratings_outside_c_int():
    ts = sb.Trainset.from_coo([0, 0, 1], [0, 1, 0], [1.0, 3e9, 2.0])
    with pytest.raises(OverflowError):
        oracle_fit(ts, random_state=0)
