"""AlgoBase.get_top_n on the device: equal, as dicts in key order and est bit for bit, to the reference FAQ's get_top_n
over algo.test(trainset.build_anti_testset()); the factor scorer bit-identical to sb2_mf_predict_dev."""
import pickle

import numpy as np
import pytest

from test_top_n_cpu import assert_same_top_n, faq_get_top_n

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import synth  # noqa: E402
from surprise_b200.prediction_algorithms.algo_base import rank_top_n  # noqa: E402


def u1_algos():
    knn = [(cls, ub) for cls in (sb.KNNBasic, sb.KNNWithMeans, sb.KNNWithZScore, sb.KNNBaseline) for ub in (True, False)]
    return ([lambda: sb.SVD(n_factors=20, n_epochs=5, random_state=0),
             lambda: sb.SVD(n_factors=20, n_epochs=5, biased=False, random_state=0),
             lambda: sb.SVDpp(n_factors=10, n_epochs=2, random_state=0),
             lambda: sb.NMF(n_factors=15, n_epochs=5, random_state=0),
             lambda: sb.NMF(n_factors=15, n_epochs=5, biased=True, random_state=0),
             lambda: sb.BaselineOnly(bsl_options={"method": "als"}),
             lambda: sb.BaselineOnly(bsl_options={"method": "sgd"}),
             lambda: sb.CoClustering(random_state=0),
             lambda: sb.SlopeOne()]
            + [(lambda c=cls, u=ub: c(sim_options={"name": "msd", "user_based": u})) for cls, ub in knn])


def check_contract(algo, ts, ns=None, preds=None):
    preds = algo.test(ts.build_anti_testset()) if preds is None else preds
    for n in ns or (1, 10, ts.n_items + 5):
        assert_same_top_n(algo.get_top_n(n), faq_get_top_n(preds, n))
    return preds


@pytest.mark.parametrize("k", range(len(u1_algos())))
def test_u1_full_contract(u1, k):
    ts, _ = u1
    algo = u1_algos()[k]().fit(ts)
    check_contract(algo, ts)


F_LIST = (0, 1, 15, 20, 31, 32, 33, 64, 100, 128, 200)


@pytest.mark.parametrize("f", F_LIST)
def test_scorer_bits_match_mf_predict(f):
    import torch
    rng = np.random.RandomState(f)
    n_u, n_i = 37, 301
    lens = rng.randint(1, 40, n_u)
    up = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    ui = np.concatenate([rng.choice(n_i, m, replace=False) for m in lens]).astype(np.int32)
    pu, qi, yj = (rng.normal(0, 1, (n, f)) for n in (n_u, n_i, n_i))
    bu, bi = rng.normal(0, 1, n_u), rng.normal(0, 1, n_i)
    d = {k: nat.to_dev(v, np.float64) for k, v in dict(pu=pu, qi=qi, yj=yj, bu=bu, bi=bi).items()}
    d_up, d_ui = nat.to_dev(up, np.int64), nat.to_dev(ui, np.int32)
    rows = np.array([5, 0, 36, 7, 7, 12] + list(range(n_u)), dtype=np.int32)
    d_rows = nat.to_dev(rows, np.int32)
    pu_ptr = nat.ptr(d["pu"]) if f else None
    qi_ptr = nat.ptr(d["qi"]) if f else None
    for biased in (0, 1):
        for with_yj in ((False, True) if f else (False,)):
            yj_ptr, up_ptr, ui_ptr = (nat.ptr(d["yj"]), nat.ptr(d_up), nat.ptr(d_ui)) if with_yj else (None,) * 3
            ld = n_i + 3
            scores = torch.full((len(rows), ld), 7.0, dtype=torch.float64, device="cuda")
            nat.check(nat.lib().sb2_mf_score_block_dev(len(rows), nat.ptr(d_rows), n_i, f, biased, 3.5, pu_ptr,
                                                       qi_ptr, nat.ptr(d["bu"]), nat.ptr(d["bi"]), yj_ptr, up_ptr,
                                                       ui_ptr, nat.ptr(scores), ld, nat.stream()))
            d_u = d_rows.repeat_interleave(n_i)
            d_i = torch.arange(n_i, dtype=torch.int32, device="cuda").repeat(len(rows))
            est = torch.empty(len(d_u), dtype=torch.float64, device="cuda")
            imp = torch.empty(len(d_u), dtype=torch.uint8, device="cuda")
            nat.check(nat.lib().sb2_mf_predict_dev(len(d_u), nat.ptr(d_u), nat.ptr(d_i), f, biased, 3.5, pu_ptr,
                                                   qi_ptr, nat.ptr(d["bu"]), nat.ptr(d["bi"]), yj_ptr, up_ptr,
                                                   ui_ptr, nat.ptr(est), nat.ptr(imp), nat.stream()))
            got = scores[:, :n_i].contiguous().view(torch.int64).cpu().numpy().reshape(-1)
            want = est.view(torch.int64).cpu().numpy()
            assert np.array_equal(got, want), (f, biased, with_yj, int((got != want).sum()))
            assert (scores[:, n_i:] == 7.0).all()          # nothing written past n_items


def test_ties_at_high_and_assigned_factors(u1):
    ts, _ = u1
    algo = sb.SVD(n_factors=10, n_epochs=3, random_state=0).fit(ts)
    algo.get_top_n(5)                                 # fills the device cache
    bi = algo.bi.copy()
    bi[::3] += 10.0                                   # a third of the items clip at high for every user
    algo.bi = bi
    items, est, count = algo.top_n_inner(50)
    assert (est[:, :10] == ts.rating_scale[1]).all()
    assert (np.diff(items[:, :10], axis=1) > 0).all()  # ties in ascending inner id
    check_contract(algo, ts, ns=(10, 50))


def offset_trainset(seed=0, n_u=60, n_i=80, n=1500):
    d = synth.ratings(n_u, n_i, n, seed=seed)
    u, i, r = d["train"]
    r = np.round(r * 4 - 11)                          # ratings on (-10, 10)
    return sb.Trainset.from_coo(u, i, r + 11, d["n_users"], d["n_items"], (-10, 10), 11)


def test_offset_scale_and_zero_scores():
    ts = offset_trainset()
    for algo in (sb.SVD(n_factors=8, n_epochs=5, random_state=1), sb.KNNBasic(), sb.SlopeOne()):
        algo.fit(ts)
        check_contract(algo, ts)
    algo = sb.SVD(n_factors=8, n_epochs=1, random_state=1, biased=False).fit(ts)
    pu = algo.pu.copy()
    pu[::2] = -0.0                                    # -0.0 factor products; the chains still sum to +0.0
    algo.pu = pu
    algo.qi = np.abs(algo.qi)
    check_contract(algo, ts)
    base = sb.SVD(n_factors=4, n_epochs=1, random_state=1).fit(ts)
    base.bu = np.full(ts.n_users, 11.0 - ts.global_mean)
    base.bi = np.zeros_like(base.bi)
    base.pu = np.zeros_like(base.pu)
    check_contract(base, ts)                          # est near 0.0 after the offset, many ties


def full_rater_trainset():
    d = synth.ratings(40, 30, 400, seed=3)
    u, i, r = d["train"]
    keep = u != 0
    u, i, r = u[keep], i[keep], r[keep]
    u = np.concatenate((np.zeros(30, np.int32), u))
    i = np.concatenate((np.arange(30, dtype=np.int32), i))
    r = np.concatenate((np.full(30, 3.0), r))
    return sb.Trainset.from_coo(u, i, r, int(u.max()) + 1, 30)


@pytest.mark.parametrize("make", [lambda: sb.SVD(n_factors=5, n_epochs=2, random_state=0), lambda: sb.KNNBasic()])
def test_user_who_rated_everything(make):
    ts = full_rater_trainset()
    algo = make().fit(ts)
    items, est, count = algo.top_n_inner(5)
    assert count[0] == 0 and (items[0] == -1).all() and np.isnan(est[0]).all()
    check_contract(algo, ts)
    assert ts.to_raw_uid(0) not in algo.get_top_n(5)


def test_uids_subsets_and_unknown(u1):
    ts, _ = u1
    algo = sb.SVD(n_factors=10, n_epochs=3, random_state=0).fit(ts)
    preds = algo.test(ts.build_anti_testset())
    by_user = {}
    for p in preds:
        by_user.setdefault(p.uid, []).append(p)
    raw = [ts.to_raw_uid(u) for u in range(ts.n_users)]
    for uids in (raw[10:400:7], raw[::-1][:50], [raw[3], raw[900], raw[0]]):
        sub = [p for u in uids for p in by_user[u]]
        assert_same_top_n(algo.get_top_n(10, uids=uids), faq_get_top_n(sub, 10))
    with pytest.raises(ValueError):
        algo.get_top_n(10, uids=[raw[0], "not a user"])


def test_non_batched_subclass_goes_through_test(u1):
    ts, _ = u1

    class MySVD(sb.SVD):
        def estimate(self, u, i):
            return sb.SVD.estimate(self, u, i)

    algo = MySVD(n_factors=5, n_epochs=2, random_state=0).fit(ts)
    assert not algo._batched()
    uids = [ts.to_raw_uid(u) for u in (4, 1)]
    ref = sb.SVD(n_factors=5, n_epochs=2, random_state=0).fit(ts)
    assert_same_top_n(algo.get_top_n(7, uids=uids), ref.get_top_n(7, uids=uids))


@pytest.mark.parametrize("make", [lambda: sb.SVDpp(n_factors=5, n_epochs=2, random_state=0),
                                  lambda: sb.KNNBaseline(), lambda: sb.CoClustering(random_state=0), sb.SlopeOne,
                                  lambda: sb.BaselineOnly()])
def test_pickle_round_trip(u1, make):
    ts, _ = u1
    algo = make().fit(ts)
    want = algo.get_top_n(10)
    assert_same_top_n(pickle.loads(pickle.dumps(algo)).get_top_n(10), want)


@pytest.mark.parametrize("make", [lambda: sb.SVDpp(n_factors=5, n_epochs=2, random_state=0),
                                  lambda: sb.KNNBasic(sim_options={"user_based": False})])
def test_block_boundaries_are_invisible(u1, make):
    ts, _ = u1
    algo = make().fit(ts)
    users = np.r_[np.arange(0, ts.n_users, 3), [5, 5, 0]].astype(np.int32)
    want = algo.top_n_inner(12, users)
    for rows in (1, 7, 100, 10 ** 6):
        got = algo.top_n_inner(12, users, _block_rows=rows)
        for g, w in zip(got, want):
            assert np.array_equal(g.view(np.uint8), w.view(np.uint8)), rows


def test_launches_per_block(u1):
    ts, _ = u1
    for algo, per_block in ((sb.SVD(n_factors=5, n_epochs=1, random_state=0).fit(ts), 4),
                            (sb.CoClustering(random_state=0).fit(ts), 2)):
        algo.top_n_inner(3)
        for rows, blocks in ((100, 10), (300, 4), (10 ** 6, 1)):
            nat.lib().sb2_reset_launch_count()
            algo.top_n_inner(3, _block_rows=rows)
            assert nat.lib().sb2_launch_count() == per_block * blocks, (type(algo).__name__, rows)


def test_zero_division_is_raised():
    ts = offset_trainset(seed=2)
    algo = sb.KNNBasic(k=5, min_k=0).fit(ts)
    algo.sim = np.zeros((ts.n_users, ts.n_users))     # no positive neighbour anywhere: 0 / 0 with min_k = 0
    with pytest.raises(ZeroDivisionError):
        algo.test(ts.build_anti_testset())
    with pytest.raises(ZeroDivisionError):
        algo.get_top_n(5)


def test_select_signed_zeros_nan_and_default():
    """sb2_top_n_select_dev on hand-built rows: -0.0 ties +0.0 (ascending item), NaN after every number, code 1
    replaced by default_est, every est with the bits AlgoBase.test's numpy clipping gives."""
    import torch
    nz, nan = -0.0, np.nan
    scores = np.array([[nz, 0.0, nan, 0.5, nz, 0.0, -0.5, nan, 0.25, nz, 2.0, -3.0],
                       [0.0, nz, 1.0, nan, 7.0, nz, 0.0, 0.5, nz, -2.0, nan, 1.0]])
    codes = np.zeros(scores.shape, np.uint8)
    codes[0, 8] = codes[1, 4] = 1                     # impossible: default_est = -0.0
    up, ui = np.array([0, 1, 1], np.int64), np.array([3], np.int32)   # user 0 rated item 3, user 1 nothing
    low, high, default = -1.0, 1.0, -0.0
    val = np.maximum(low, np.minimum(high, np.where(codes == 1, default, scores) - 0.0))
    d_sc, d_imp = nat.to_dev(scores, np.float64), nat.to_dev(codes, np.uint8)
    d_rows, d_up, d_ui = nat.to_dev(np.array([0, 1], np.int32), np.int32), nat.to_dev(up, np.int64), nat.to_dev(ui, np.int32)
    n_i = scores.shape[1]
    for n in (1, 3, 6, n_i, n_i + 8):
        items = torch.empty((2, n), dtype=torch.int32, device="cuda")
        est = torch.empty((2, n), dtype=torch.float64, device="cuda")
        count = torch.empty(2, dtype=torch.int32, device="cuda")
        nat.check(nat.lib().sb2_top_n_select_dev(2, nat.ptr(d_rows), n_i, nat.ptr(d_sc), n_i, nat.ptr(d_imp), default,
                                                 0.0, low, high, nat.ptr(d_up), nat.ptr(d_ui), n, nat.ptr(items),
                                                 nat.ptr(est), nat.ptr(count), nat.stream()))
        items, est, count = items.cpu().numpy(), est.cpu().numpy(), count.cpu().numpy()
        for r in range(2):
            cand = np.setdiff1d(np.arange(n_i), ui[up[r]:up[r + 1]])
            order = cand[rank_top_n(val[r, cand], cand)][:n]
            c = len(order)
            assert count[r] == c
            assert items[r, :c].tolist() == order.tolist()
            got, want = est[r, :c], val[r, order]
            assert np.array_equal(np.isnan(got), np.isnan(want))      # NaN payloads are the device's own
            num = ~np.isnan(want)
            assert np.array_equal(got[num].view(np.int64), want[num].view(np.int64))
            assert (items[r, c:] == -1).all() and np.isnan(est[r, c:]).all()


def reference_top_n(algo, ts, users, n):
    """_estimate_dev over every (user, item) pair of `users` plus the numpy ordering rule, without get_top_n's code."""
    import torch
    d_u = torch.as_tensor(np.repeat(users, ts.n_items), device="cuda")
    d_i = torch.as_tensor(np.tile(np.arange(ts.n_items, dtype=np.int32), len(users)), device="cuda")
    est, _ = algo._estimate_dev(d_u, d_i)
    est = np.maximum(ts.rating_scale[0], np.minimum(ts.rating_scale[1], est.cpu().numpy() - ts.offset))
    est = est.reshape(len(users), ts.n_items)
    ptr, idx, _ = ts.user_csr()
    out_i = np.full((len(users), n), -1, np.int32)
    out_e = np.full((len(users), n), np.nan)
    for k, u in enumerate(users.tolist()):
        cand = np.setdiff1d(np.arange(ts.n_items), idx[ptr[u]:ptr[u + 1]])
        order = rank_top_n(est[k, cand], cand)[:n]
        out_i[k, :len(order)], out_e[k, :len(order)] = cand[order], est[k, cand[order]]
    return out_i, out_e


@pytest.mark.parametrize("shape", ["ml-1m", "ml-20m"])
def test_scale(shape):
    d = synth.shaped(shape, seed=0)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"], (0.5, 5.0) if shape == "ml-20m" else (1, 5))
    algo = sb.SVD(n_factors=100, n_epochs=2, random_state=0).fit(ts)
    cnt = np.diff(ts.user_csr()[0])
    if shape == "ml-1m":
        users = np.arange(ts.n_users, dtype=np.int32)
    else:
        rng = np.random.RandomState(0)
        users = np.unique(np.r_[np.argsort(cnt)[:20], np.argsort(cnt)[-20:], rng.choice(ts.n_users, 260, False)])
        users = users.astype(np.int32)
    for n in (10, 100):
        items, est, count = algo.top_n_inner(n, users)
        want_i, want_e = reference_top_n(algo, ts, users, n)
        assert np.array_equal(items, want_i)
        assert np.array_equal(est.view(np.int64), want_e.view(np.int64))
        assert np.array_equal(count, np.minimum(n, ts.n_items - cnt[users]))


@pytest.mark.parametrize("make", [lambda: sb.SVD(n_factors=20, n_epochs=2, random_state=0),
                                  lambda: sb.CoClustering(random_state=0)])
def test_selection_passes_beyond_2048(make):
    """n past the 2048 entries one selection pass keeps: a second and a third pass, on the factor route and on the
    estimate-kernel route, bitwise against the per-pair reference (count included) and against the FAQ."""
    d = synth.ratings(300, 5000, 60_000, seed=7)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    assert ts.n_items > 4096
    algo = make().fit(ts)
    users = np.arange(ts.n_users, dtype=np.int32)
    cnt = np.diff(ts.user_csr()[0])
    for n, block_rows in ((2048, None), (2049, None), (4097, 64), (ts.n_items + 5, 7)):
        items, est, count = algo.top_n_inner(n, users, _block_rows=block_rows)
        width = min(n, ts.n_items)
        want_i, want_e = reference_top_n(algo, ts, users, width)
        assert np.array_equal(count, np.minimum(width, ts.n_items - cnt))
        assert np.array_equal(items, want_i), n
        assert np.array_equal(est.view(np.int64), want_e.view(np.int64)), n
    check_contract(algo, ts, ns=(2049, ts.n_items + 5))
