"""Parity tests proper: the CUDA path (through the C-ABI / the reference-shaped Python API) against the
C oracle and the golden vectors.  Bit-exact for similarities on integer / half-integer ratings, NMF
factors, ALS / SGD baselines and k-NN estimates; 1e-9 absolute for pearson_baseline and float ratings;
held-out RMSE / MAE within 0.005 for SVD (stratified update order)."""
import ctypes as C
import hashlib
import os
import pickle

import numpy as np
import pytest

import oracle
from conftest import GOLDEN, inner_pairs, rmse_mae

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import similarities as sims  # noqa: E402
from surprise_b200 import synth  # noqa: E402

KINDS = ("cosine", "msd", "pearson", "pearson_baseline")
PB_ATOL = 1e-9  # north_star: stated tolerance for the floating-point similarity path


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(params=("digit", "general"))
def sim_path(request, monkeypatch):
    """Both implementations of the similarity functions (csrc/sim.cu: int8 tensor-core contractions; csrc/sim_general.cu:
    the reference's loop nest in fp64) must pass the same parity tests; without this the cost model would pick one."""
    monkeypatch.setenv("SB2_SIM_PATH", request.param)
    return request.param


def test_device_is_blackwell():
    sm, maj, mnr, mem = C.c_int(), C.c_int(), C.c_int(), C.c_int64()
    nat.check(nat.lib().sb2_device_info(C.byref(sm), C.byref(maj), C.byref(mnr), C.byref(mem)))
    assert maj.value == 10, "kernels are built for sm_100a only"


@pytest.mark.parametrize("shape", [(256, 256, 128), (256, 512, 1024), (768, 256, 4096 + 128)])
def test_tcgen05_gemm_against_dp4a_and_numpy(shape):
    import torch
    m, n, k = shape
    rng = np.random.RandomState(m + n + k)
    a = rng.randint(0, 256, (m, k)).astype(np.uint8)
    b = rng.randint(0, 256, (n, k)).astype(np.uint8)
    da, db = nat.to_dev(a, np.uint8), nat.to_dev(b, np.uint8)
    c_tc = nat.empty_dev((m, n), np.int32)
    c_ref = nat.empty_dev((m, n), np.int32)
    nat.check(nat.lib().sb2_gemm_u8_selftest_dev(1, m, n, k, nat.ptr(da), nat.ptr(db), nat.ptr(c_tc), nat.stream()))
    nat.check(nat.lib().sb2_gemm_u8_selftest_dev(0, m, n, k, nat.ptr(da), nat.ptr(db), nat.ptr(c_ref), nat.stream()))
    torch.cuda.synchronize()
    want = a.astype(np.int64) @ b.astype(np.int64).T
    assert np.array_equal(c_ref.cpu().numpy(), want)
    assert np.array_equal(c_tc.cpu().numpy(), want)


# ---- similarities -----------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("ms", (1, 4))
def test_toy_similarities(toy, kind, ms, sim_path):
    yr = (toy["y_ptr"], toy["x_idx"], toy["r"])
    if kind == "pearson_baseline":
        got = sims.pearson_baseline(8, yr, ms, float(toy["global_mean"]), toy["bx"], toy["by"])
        assert np.allclose(got, toy["%s_%d" % (kind, ms)], rtol=0, atol=PB_ATOL)
        assert np.array_equal(got == 0, toy["%s_%d" % (kind, ms)] == 0)  # freq / min_support mask is exact
    else:
        got = getattr(sims, kind)(8, yr, ms)
        assert np.array_equal(got, toy["%s_%d" % (kind, ms)])
    assert np.array_equal(got, got.T) and np.all(np.diag(got) == 1)


def test_toy_dict_input_and_shuffle(toy, sim_path):
    """The reference API takes a dict of lists; order inside a list must not matter."""
    import random
    yr = {0: [(0, 3), (1, 3), (2, 3), (5, 1), (6, 1.5), (7, 3)], 1: [(0, 4), (1, 4), (2, 4)],
          2: [(2, 5), (3, 2), (4, 3)], 3: [(1, 1), (2, 4), (3, 2), (4, 3), (5, 3), (6, 3.5), (7, 2)],
          4: [(1, 5), (2, 1), (5, 2), (6, 2.5), (7, 2.5)]}
    random.seed(0)
    for v in yr.values():
        random.shuffle(v)
    assert np.array_equal(sims.cosine(8, yr, 1), toy["cosine_1"])
    assert np.array_equal(sims.msd(8, yr, 1), toy["msd_1"])
    assert np.array_equal(sims.pearson(8, yr, 4), toy["pearson_4"])
    s0 = sims.pearson_baseline(8, yr, 1, 3, toy["bx"], toy["by"], 0)
    assert np.allclose(s0, toy["pearson_baseline_shr0"], rtol=0, atol=PB_ATOL)
    s7 = sims.pearson_baseline(8, yr, 2, 3, toy["bx"], toy["by"], shrinkage=7.5)
    assert np.allclose(s7, toy["pearson_baseline_shr7p5"], rtol=0, atol=PB_ATOL)


@pytest.mark.parametrize("orient", ("item", "user"))
def test_u1_similarities_bit_exact(u1, u1_golden, u1_arrays, orient, sim_path):
    ts, _ = u1
    ub = orient == "user"
    n_x = ts.n_users if ub else ts.n_items
    yr = ts.item_csr() if ub else ts.user_csr()
    for kind in ("cosine", "msd", "pearson"):
        got = getattr(sims, kind)(n_x, yr, 1)
        g = u1_golden["sims"]["%s_%s_ms1" % (kind, orient)]
        assert sha(got) == g["sha256"], kind
        assert int(np.count_nonzero(got)) == g["nnz"]
    assert sha(sims.cosine(n_x, yr, 3)) == u1_golden["sims"]["cosine_%s_ms3" % orient]["sha256"]
    bu, bi = u1_arrays["als_bu"], u1_arrays["als_bi"]
    bx, by = (bu, bi) if ub else (bi, bu)
    got = sims.pearson_baseline(n_x, yr, 1, float(ts.global_mean), bx, by)
    want = oracle.similarity("pearson_baseline", n_x, *yr, 1, float(ts.global_mean), bx, by, 100.0)
    assert sha(want) == u1_golden["sims"]["pearson_baseline_%s_ms1" % orient]["sha256"]
    assert np.allclose(got, want, rtol=0, atol=PB_ATOL)
    assert np.array_equal(got == 0, want == 0)
    assert np.array_equal(got, got.T)


def test_u1_row_shard_equals_full(u1, sim_path):
    ts, _ = u1
    yr = ts.user_csr()
    full = sims.cosine(ts.n_items, yr, 1)
    for kind in ("cosine", "pearson"):
        full = getattr(sims, kind)(ts.n_items, yr, 1)
        for (b, e) in ((0, 256), (256, 768), (1024, ts.n_items)):
            blk = sims.build_device(kind, ts.n_items, yr, 1, row_begin=b, row_end=e).cpu().numpy()
            assert np.array_equal(blk, full[b:e]), (kind, b, e)


def test_float_ratings_similarities(floats, sim_path):
    """Jester-style two-decimal ratings run on the digit-split exact-integer path (denominator 100)."""
    ds = sb.Dataset.load_from_arrays(floats["uid"], floats["iid"], floats["rating"], sb.Reader(rating_scale=(-10, 10)))
    ts = ds.build_full_trainset()
    assert sims.rating_denominator(ts.user_csr()[2]) == 100
    for ub, o in ((False, "item"), (True, "user")):
        n_x = ts.n_users if ub else ts.n_items
        yr = ts.item_csr() if ub else ts.user_csr()
        bx, by = (floats["als_bu"], floats["als_bi"]) if ub else (floats["als_bi"], floats["als_bu"])
        for kind in KINDS:
            if kind == "pearson_baseline":
                got = sims.pearson_baseline(n_x, yr, 2, float(ts.global_mean), bx, by)
            else:
                got = getattr(sims, kind)(n_x, yr, 2)
            want = floats["sim_%s_%s" % (kind, o)]
            assert np.allclose(got, want, rtol=0, atol=PB_ATOL, equal_nan=True), (kind, o, np.abs(got - want).max())


@pytest.mark.parametrize("kind", KINDS)
def test_sim_upper_shards_assemble_to_full(u1, kind, sim_path):
    """Symmetric multi-rank build emulated on one GPU: the upper-only shards of 3 ranks (sb2_sim_build_upper_dev),
    completed by the transposes the NCCL exchange would deliver, equal the single-GPU matrix bit for bit."""
    from surprise_b200 import distributed as D
    ts, _ = u1
    n_x, yr = ts.n_items, ts.user_csr()
    kw = {}
    if kind == "pearson_baseline":
        algo = sb.BaselineOnly()
        sb.AlgoBase.fit(algo, ts)
        bu, bi = algo.compute_baselines()
        kw = dict(global_mean=float(ts.global_mean), x_biases=bi, y_biases=bu)
    want = sims.build_device(kind, n_x, yr, 1, **kw).cpu().numpy()
    ranges = D.sim_tri_ranges(n_x, 3)
    blocks = [sims.build_device(kind, n_x, yr, 1, row_begin=b, row_end=e, upper=True, **kw).cpu().numpy() for b, e in ranges]
    for k, (b, e) in enumerate(ranges):
        assert np.all(blocks[k][:, :b] == 0)            # untouched
        for j in range(k):
            bj, ej = ranges[j]
            blocks[k][:, bj:ej] = blocks[j][:, b:e].T     # what sim_exchange delivers
    assert np.array_equal(np.concatenate(blocks, axis=0), want, equal_nan=True)


def test_rating_denominator_on_device():
    """sb2_rating_denominator_dev == similarities.rating_denominator (host) on every supported grid."""
    rng = np.random.RandomState(0)
    for d in (1, 2, 4, 5, 10, 20, 100, 1000):
        r = rng.randint(0, 5 * d + 1, 5000) / d
        r[0] = 1.0 / d                                  # make sure the finest step is present
        got = C.c_int(-1)
        nat.check(nat.lib().sb2_rating_denominator_dev(nat.ptr(nat.to_dev(r, np.float64)), len(r), C.byref(got), nat.stream()))
        assert got.value == sims.rating_denominator(r) == d
    got = C.c_int(-1)
    nat.check(nat.lib().sb2_rating_denominator_dev(nat.ptr(nat.to_dev(np.array([np.pi, 2.0]), np.float64)), 2, C.byref(got), nat.stream()))
    assert got.value == 0


@pytest.mark.parametrize("band_rows", (256, 512))
def test_sim_banded_planes_bit_identical(u1, monkeypatch, band_rows):
    monkeypatch.setenv("SB2_SIM_PATH", "digit")
    """The fp64 accumulator planes cover one band of row blocks at a time (bounded footprint); forcing 3 / 5 bands on
    the 1187-item fixture must not change one bit of any matrix: single-GPU symmetric build, plain row shard,
    upper-only shard, SlopeOne."""
    from surprise_b200 import distributed as D
    ts, _ = u1
    n_x, yr = ts.n_items, ts.user_csr()
    algo = sb.BaselineOnly()
    sb.AlgoBase.fit(algo, ts)
    bu, bi = algo.compute_baselines()

    def build_all():
        out = []
        for kind in KINDS:
            kw = dict(global_mean=float(ts.global_mean), x_biases=bi, y_biases=bu) if kind == "pearson_baseline" else {}
            out.append(sims.build_device(kind, n_x, yr, 1, **kw).cpu().numpy())
            out.append(sims.build_device(kind, n_x, yr, 1, row_begin=256, row_end=1100, **kw).cpu().numpy())
            out.append(sims.build_device(kind, n_x, yr, 1, row_begin=256, row_end=n_x, upper=True, **kw).cpu().numpy())
        so = sb.SlopeOne().fit(ts)
        out += [so.freq.astype(np.float64), np.nan_to_num(so.dev, nan=123.0)]
        return out
    monkeypatch.delenv("SB2_SIM_BAND_ROWS", raising=False)
    want = build_all()
    monkeypatch.setenv("SB2_SIM_BAND_ROWS", str(band_rows))
    got = build_all()
    for k, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b, equal_nan=True), k


def test_similarity_errors():
    with pytest.raises(ZeroDivisionError):
        sims.msd(2, {0: [(0, 3.0)], 1: [(1, 4.0)]}, 0)
    empty = sims.cosine(3, {}, 1)
    assert np.array_equal(empty, np.eye(3))


def _random_yr(rng, n_x, n_y, nnz, ratings, dup=0):
    """yr CSR with unique (x, y) pairs (+ `dup` repeated pairs appended to random segments), list order shuffled."""
    lin = rng.choice(n_x * n_y, nnz, replace=False)
    y, x = lin // n_x, lin % n_x
    if dup:
        k = rng.choice(nnz, dup, replace=True)
        y, x = np.concatenate((y, y[k])), np.concatenate((x, x[k]))
    r = ratings(len(x))
    o = rng.permutation(len(x))
    y, x, r = y[o], x[o], r[o]
    o = np.argsort(y, kind="stable")
    y, x, r = y[o], x[o], r[o]
    ptr = np.concatenate(([0], np.cumsum(np.bincount(y, minlength=n_y)))).astype(np.int64)
    return ptr, x.astype(np.int32), r.astype(np.float64)


@pytest.mark.parametrize("case", ("irrational", "negative", "duplicates", "duplicates_grid", "wide_range"))
def test_general_similarity_path_bit_exact(case):
    """Ratings the integer-digit panels cannot hold -- arbitrary doubles, negative values, 12 orders of magnitude of
    dynamic range, duplicated (x, y) pairs (which the reference counts as separate co-ratings,
    similarities.pyx:78-84) -- go through the general fp64 path in the reference's own summation order: every kind,
    both min_support settings, EQUAL BIT FOR BIT to the oracle's restatement of the reference loops."""
    rng = np.random.RandomState({"irrational": 1, "negative": 2, "duplicates": 3, "duplicates_grid": 4, "wide_range": 5}[case])
    n_x, n_y = 150, 90
    gen = {"irrational": lambda k: rng.uniform(0.5, 5.0, k) * np.pi / 3,
           "negative": lambda k: rng.normal(0, 2.0, k),
           "duplicates": lambda k: rng.uniform(1, 5, k),
           "duplicates_grid": lambda k: rng.randint(1, 6, k).astype(np.float64),
           "wide_range": lambda k: 10.0 ** rng.uniform(-6, 6, k)}[case]
    ptr, idx, val = _random_yr(rng, n_x, n_y, 2500, gen, dup=120 if case.startswith("dup") else 0)
    mu = float(np.mean(val))
    bx, by = rng.normal(0, .3, n_x), rng.normal(0, .3, n_y)
    yr = (ptr, idx, val)
    for kind in KINDS:
        for ms in (1, 3):
            kw = (mu, bx, by, 50.0) if kind == "pearson_baseline" else ()
            want = oracle.similarity(kind, n_x, ptr, idx, val, ms, *kw)
            got = getattr(sims, kind)(n_x, yr, ms, *kw)
            assert np.array_equal(got, want, equal_nan=True), (case, kind, ms, float(np.nanmax(np.abs(got - want))))
    # a row shard equals the rows of the full build (the multi-rank similarity build on such ratings)
    full = sims.build_device("pearson", n_x, yr, 1).cpu().numpy()
    part = sims.build_device("pearson", n_x, yr, 1, row_begin=0, row_end=77).cpu().numpy()
    assert np.array_equal(part, full[:77], equal_nan=True)
    # dict input with a duplicated pair, as a user would pass it
    d = {0: [(0, 3.0), (0, 4.0), (1, 2.0)], 1: [(1, np.pi), (0, 2.0)]}
    p2, i2, v2 = oracle.flatten_yr(d, 2)
    assert np.array_equal(sims.cosine(2, d, 1), oracle.similarity("cosine", 2, p2, i2, v2, 1))


def test_general_path_forced_on_grid_ratings_matches_digit_path(u1, monkeypatch):
    """SB2_SIM_PATH=general sends grid ratings through the general path too: on the reference's fixture both paths must
    produce the same bits (cosine / msd / pearson: both exact; pearson_baseline: the general path IS the reference's
    arithmetic, the digit path is within 1e-9 of it)."""
    ts, _ = u1
    yr = ts.user_csr()
    mu = float(ts.global_mean)
    bu, bi = oracle.baseline_als(ts.n_users, ts.n_items, *ts.user_csr(), *ts.item_csr(), mu)
    monkeypatch.setenv("SB2_SIM_PATH", "digit")
    digit = {k: getattr(sims, k)(ts.n_items, yr, 1, *((mu, bi, bu) if k == "pearson_baseline" else ())) for k in KINDS}
    monkeypatch.setenv("SB2_SIM_PATH", "general")
    for k in KINDS:
        got = getattr(sims, k)(ts.n_items, yr, 1, *((mu, bi, bu) if k == "pearson_baseline" else ()))
        if k == "pearson_baseline":
            want = oracle.similarity(k, ts.n_items, *yr, 1, mu, bi, bu, 100.0)
            assert np.array_equal(got, want)
            assert np.allclose(got, digit[k], rtol=0, atol=PB_ATOL)
        else:
            assert np.array_equal(got, digit[k]), k


def test_synthetic_half_star_similarity_sampled(sim_path):
    """ml-20M-style half-star ratings at a reduced shape: sampled entries against the oracle (bit-exact
    for the integer kinds), plus symmetry / diagonal / bounds on the whole matrix."""
    d = synth.ratings(3000, 1500, 200_000, step=0.5, seed=3)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"], (0.5, 5.0), 0)
    yr = ts.user_csr()
    n_x = ts.n_items
    o = np.lexsort((u, i))
    xptr = np.concatenate(([0], np.cumsum(np.bincount(i, minlength=n_x)))).astype(np.int64)
    rng = np.random.RandomState(0)
    pi, pj = rng.randint(0, n_x, 20000), rng.randint(0, n_x, 20000)
    mu = float(ts.global_mean)
    bu, bi = oracle.baseline_als(ts.n_users, ts.n_items, *ts.user_csr(), *ts.item_csr(), mu)
    for kind in KINDS:
        if kind == "pearson_baseline":
            got = sims.pearson_baseline(n_x, yr, 1, mu, bi, bu)
        else:
            got = getattr(sims, kind)(n_x, yr, 2)
        want = oracle.similarity_pairs(kind, pi, pj, xptr, u[o], r[o], 1 if kind == "pearson_baseline" else 2, mu,
                                       bi, bu, 100.0)
        if kind == "pearson_baseline":
            assert np.allclose(got[pi, pj], want, rtol=0, atol=PB_ATOL), np.abs(got[pi, pj] - want).max()
        else:
            assert np.array_equal(got[pi, pj], want), kind
        assert np.array_equal(got, got.T) and np.all(np.diag(got) == 1)
        assert np.nanmax(np.abs(got)) <= 1 + 1e-12


# ---- baselines ----------------------------------------------------------------------------------------
def test_u1_baselines_bit_exact(u1, u1_golden):
    ts, _ = u1
    algo = sb.BaselineOnly()
    algo.fit(ts)
    assert sha(algo.bu) == u1_golden["baseline_als"]["bu_sha256"]
    assert sha(algo.bi) == u1_golden["baseline_als"]["bi_sha256"]
    algo = sb.BaselineOnly(bsl_options={"method": "sgd"})
    algo.fit(ts)
    assert sha(algo.bu) == u1_golden["baseline_sgd"]["bu_sha256"]
    assert sha(algo.bi) == u1_golden["baseline_sgd"]["bi_sha256"]
    with pytest.raises(ValueError):
        sb.BaselineOnly(bsl_options={"method": "nope"}).fit(ts)


def test_u1_baseline_only_predictions(u1, u1_golden):
    """BaselineOnly.test is batched through the estimate kernel with zero factors: (mu + b_u) + b_i with unknown ids
    skipped, the reference's additions in the reference's order -- RMSE / MAE equal the golden to the last digit."""
    ts, testset = u1
    for method, tag in (("als", "BaselineOnly_als"), ("sgd", "BaselineOnly_sgd")):
        algo = sb.BaselineOnly(bsl_options={"method": method}).fit(ts)
        preds = algo.test(testset)
        g = u1_golden["algos"][tag]
        assert repr(float(sb.accuracy.rmse(preds, verbose=False))) == g["rmse"]
        assert repr(float(sb.accuracy.mae(preds, verbose=False))) == g["mae"]
        assert sum(p.details["was_impossible"] for p in preds) == g["n_impossible"] == 0
        uid, iid, _ = testset[3]
        assert algo.predict(uid, iid).est == preds[3].est
        assert pickle.loads(pickle.dumps(algo)).predict(uid, iid).est == preds[3].est


# ---- k-NN -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("orient", ("item", "user"))
@pytest.mark.parametrize("kind", KINDS)
def test_u1_knnbasic_end_to_end(u1, u1_golden, u1_arrays, kind, orient):
    ts, testset = u1
    algo = sb.KNNBasic(sim_options={"name": kind, "user_based": orient == "user", "min_support": 1})
    preds = algo.fit(ts).test(testset)
    tag = "KNNBasic_%s_%s_ms1" % (kind, orient)
    g = u1_golden["algos"][tag]
    est = np.array([p.est for p in preds])
    ak = np.array([p.details.get("actual_k", -1) for p in preds])
    assert sum(p.details["was_impossible"] for p in preds) == g["n_impossible"]
    if kind == "pearson_baseline":
        assert np.allclose(est, u1_arrays[tag + "_est"], rtol=0, atol=1e-6)
        assert abs(float(sb.accuracy.rmse(preds, verbose=False)) - float(g["rmse"])) < 1e-7
    else:
        assert np.array_equal(est, u1_arrays[tag + "_est"])
        assert np.array_equal(ak, u1_arrays[tag + "_actual_k"])
        assert repr(float(sb.accuracy.rmse(preds, verbose=False))) == g["rmse"]   # config 1: to the last bit
        assert repr(float(sb.accuracy.mae(preds, verbose=False))) == g["mae"]
    for p in preds:
        if not p.details["was_impossible"]:
            assert algo.min_k <= p.details["actual_k"] <= algo.k


@pytest.mark.parametrize("orient", ("item", "user"))
def test_u1_knn_kernel_against_oracle_on_same_sim(u1, u1_arrays, orient):
    """Select + ordered-sum kernel in isolation: same sim matrix in, bit-identical estimates out."""
    ts, testset = u1
    ub = orient == "user"
    iu, ii = inner_pairs(ts, testset)
    x, y = (iu, ii) if ub else (ii, iu)
    n_x = ts.n_users if ub else ts.n_items
    ptr, idx, val = ts.item_csr() if ub else ts.user_csr()
    mu = float(ts.global_mean)
    bu, bi = u1_arrays["als_bu"], u1_arrays["als_bi"]
    bx, by = (bu, bi) if ub else (bi, bu)
    sim = oracle.similarity("pearson_baseline", n_x, ptr, idx, val, 1, mu, bx, by, 100.0)
    for (k, min_k, mode) in ((40, 1, 0), (5, 2, 0), (40, 1, 1 if ub else 2), (10, 3, 1 if ub else 2), (1, 1, 0)):
        want = oracle.knn_estimate(x, y, sim, ptr, idx, val, k, min_k, mode, mu, bx, by)
        est = np.empty(len(x)); ak = np.empty(len(x), dtype=np.int32); imp = np.empty(len(x), dtype=np.uint8)
        n_y = len(ptr) - 1
        rc = nat.lib().sb2_knn_predict(len(x), nat.hptr(np.ascontiguousarray(x)), nat.hptr(np.ascontiguousarray(y)),
                                       n_x, n_y, nat.hptr(sim), nat.hptr(ptr), nat.hptr(idx), nat.hptr(val), k, min_k,
                                       mode, mu, nat.hptr(np.ascontiguousarray(bx)), nat.hptr(np.ascontiguousarray(by)),
                                       nat.hptr(est), nat.hptr(ak), nat.hptr(imp))
        nat.check(rc)
        assert np.array_equal(imp, want[2]), (k, min_k, mode)
        assert np.array_equal(ak, want[1]), (k, min_k, mode)
        assert np.array_equal(est, want[0]), (k, min_k, mode)


@pytest.mark.parametrize("orient", ("item", "user"))
def test_u1_knnbaseline_end_to_end(u1, u1_golden, u1_arrays, orient):
    ts, testset = u1
    ub = orient == "user"
    algo = sb.KNNBaseline(k=10, min_k=3, sim_options={"name": "msd", "user_based": ub})
    preds = algo.fit(ts).test(testset)
    tag = "KNNBaseline_msd_k10_mk3_" + orient
    assert np.array_equal(np.array([p.est for p in preds]), u1_arrays[tag + "_est"])
    assert np.array_equal(np.array([p.details.get("actual_k", -1) for p in preds]), u1_arrays[tag + "_actual_k"])
    assert repr(float(sb.accuracy.rmse(preds, verbose=False))) == u1_golden["algos"][tag]["rmse"]
    algo = sb.KNNBaseline(sim_options={"name": "pearson_baseline", "user_based": ub})
    preds = algo.fit(ts).test(testset)
    tag = "KNNBaseline_pb_" + orient
    assert np.allclose(np.array([p.est for p in preds]), u1_arrays[tag + "_est"], rtol=0, atol=1e-6)
    assert abs(float(sb.accuracy.rmse(preds, verbose=False)) - float(u1_golden["algos"][tag]["rmse"])) < 1e-7


@pytest.mark.parametrize("orient", ("item", "user"))
def test_u1_knn_means_zscore_end_to_end(u1, u1_golden, u1_arrays, orient):
    ts, testset = u1
    ub = orient == "user"
    for algo, tag in ((sb.KNNWithMeans(sim_options={"name": "msd", "user_based": ub}), "KNNWithMeans_msd_" + orient),
                      (sb.KNNWithZScore(k=20, min_k=2, sim_options={"name": "pearson", "user_based": ub}),
                       "KNNWithZScore_pearson_k20_mk2_" + orient)):
        preds = algo.fit(ts).test(testset)
        assert np.array_equal(np.array([p.est for p in preds]), u1_arrays[tag + "_est"]), tag
        assert np.array_equal(np.array([p.details.get("actual_k", -1) for p in preds]), u1_arrays[tag + "_actual_k"])
        assert repr(float(sb.accuracy.rmse(preds, verbose=False))) == u1_golden["algos"][tag]["rmse"]
        assert sum(p.details["was_impossible"] for p in preds) == u1_golden["algos"][tag]["n_impossible"]


def test_get_neighbors_matches_stable_sort(u1):
    """AlgoBase.get_neighbors (algo_base.py:303-334): stable descending sort of the sim row, self excluded --
    item-based cosine on the fixture has many exact ties (1.0 and 0.0), which pins the tie order."""
    ts, _ = u1
    algo = sb.KNNBasic(sim_options={"name": "cosine", "user_based": False}).fit(ts)
    sim = algo.sim
    n = ts.n_items
    for iid in (0, 1, 17, 500, n - 1):
        others = [(x, sim[iid, x]) for x in range(n) if x != iid]
        others.sort(key=lambda t: t[1], reverse=True)
        for k in (1, 10, 40, 300):
            assert algo.get_neighbors(iid, k) == [j for (j, _) in others[:k]], (iid, k)
    assert len(algo.get_neighbors(3, 10 * n)) == n - 1


# ---- SlopeOne ("next" row 4) -----------------------------------------------------------------------------
def _nan0(a):
    return np.where(np.isnan(a), 0.0, a)


def test_u1_slope_one_end_to_end(u1, u1_golden, u1_arrays):
    """freq / dev from the tensor-core contractions and the warp-per-pair estimate: bit-identical to the
    reference on the fixture (NaN where freq == 0, sign of NaN aside)."""
    ts, testset = u1
    algo = sb.SlopeOne().fit(ts)
    g = u1_golden["slope_one"]
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
    assert algo.freq.dtype == np.int64 and sha(algo.freq) == g["freq_sha256"]
    assert sha(_nan0(algo.dev)) == g["dev_nan0_sha256"] and int(np.isnan(algo.dev).sum()) == g["n_nan"]
    assert np.array_equal(np.array(algo.user_mean), u1_arrays["SlopeOne_user_mean"])
    preds = algo.test(testset)
    assert np.array_equal(np.array([p.est for p in preds]), u1_arrays["SlopeOne_est"])
    assert repr(float(sb.accuracy.rmse(preds, verbose=False))) == u1_golden["algos"]["SlopeOne"]["rmse"]
    assert sum(p.details["was_impossible"] for p in preds) == u1_golden["algos"]["SlopeOne"]["n_impossible"]
    # single-pair API and pickling
    uid, iid, _ = testset[0]
    assert algo.predict(uid, iid).est == preds[0].est
    clone = pickle.loads(pickle.dumps(algo))
    assert clone.predict(uid, iid).est == preds[0].est


def test_slope_one_truncation_and_c_abi(floats):
    """Ratings are truncated to C ints (slope_one.pyx:52): float and half-star goldens; host-buffer C-ABI form."""
    n_u, n_i = 40, 60
    tp = [(int(a), int(b), 0.0) for a in range(0, n_u, 3) for b in range(0, n_i, 7)]
    hp = [(int(a), int(b), 0.0) for a in range(30) for b in range(0, 25, 3)]
    for uid, iid, rat, scale, pre, pairs in ((floats["uid"], floats["iid"], floats["rating"], (-10, 10), "", tp),
                                             (floats["half_uid"], floats["half_iid"], floats["half_rating"], (0.5, 5), "half_", hp)):
        ts = sb.Dataset.load_from_arrays(uid, iid, rat, sb.Reader(rating_scale=scale)).build_full_trainset()
        algo = sb.SlopeOne().fit(ts)
        assert np.array_equal(algo.freq, floats[pre + "slope_freq"])
        assert np.array_equal(_nan0(algo.dev), _nan0(floats[pre + "slope_dev"]))
        assert np.array_equal(np.isnan(algo.dev), np.isnan(floats[pre + "slope_dev"]))
        preds = algo.test(pairs)
        assert np.array_equal(np.array([p.est for p in preds]), floats[pre + "slope_est"])
        ptr, idx, val = ts.user_csr()
        freq = np.empty((ts.n_items, ts.n_items), dtype=np.int64); dev = np.empty((ts.n_items, ts.n_items))
        nat.check(nat.lib().sb2_slope_one_fit(ts.n_items, ts.n_users, nat.hptr(ptr), nat.hptr(idx), nat.hptr(val),
                                              nat.hptr(freq), nat.hptr(dev)))
        assert np.array_equal(freq, algo.freq) and np.array_equal(dev, algo.dev, equal_nan=True)


def test_slope_one_synthetic_vs_oracle():
    """Half-star synthetic at a size spanning several 256-row tiles and 128-byte k-blocks, against the oracle."""
    d = synth.ratings(1500, 700, 60_000, step=0.5, seed=8)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"], (0.5, 5.0), 0)
    algo = sb.SlopeOne().fit(ts)
    ptr, idx, val = ts.user_csr()
    freq, dev = oracle.slope_one_fit(ts.n_items, ptr, idx, val)
    assert np.array_equal(algo.freq, freq)
    assert np.array_equal(_nan0(algo.dev), _nan0(dev)) and np.array_equal(np.isnan(algo.dev), np.isnan(dev))
    tu, ti, _ = d["test"]
    want, wimp = oracle.slope_one_estimate(tu, ti, freq, dev, ptr, idx, np.array(algo.user_mean))
    got, details = algo._estimate_batch(np.asarray(tu, dtype=np.int32), np.asarray(ti, dtype=np.int32))
    assert np.array_equal(np.array([x["was_impossible"] for x in details]), wimp > 0)
    assert np.array_equal(got[wimp == 0], want[wimp == 0])


def test_knn_long_lists_and_ties():
    """Lists longer than the per-warp cache and many tied similarities (stable selection order)."""
    rng = np.random.RandomState(1)
    n_x, n_y = 1500, 3
    ptr = np.array([0, 1400, 1400 + 900, 1400 + 900 + 5], dtype=np.int64)
    idx = np.concatenate([rng.permutation(n_x)[:1400], rng.permutation(n_x)[:900], rng.permutation(n_x)[:5]]).astype(np.int32)
    val = rng.randint(1, 6, len(idx)).astype(np.float64)
    sim = np.round(rng.rand(n_x, n_x) * 8) / 8 - 0.25   # heavy ties, some <= 0
    sim = (sim + sim.T) / 2
    np.fill_diagonal(sim, 1)
    x = rng.randint(0, n_x, 300).astype(np.int32); y = rng.randint(0, n_y, 300).astype(np.int32)
    x[:5] = -1
    bx = rng.normal(0, 1, n_x); by = rng.normal(0, 1, n_y)
    for (k, min_k, mode) in ((40, 1, 0), (1000, 1, 0), (40, 1, 1), (3, 5, 2)):
        want = oracle.knn_estimate(x, y, sim, ptr, idx, val, k, min_k, mode, 3.1, bx, by)
        est = np.empty(len(x)); ak = np.empty(len(x), dtype=np.int32); imp = np.empty(len(x), dtype=np.uint8)
        nat.check(nat.lib().sb2_knn_predict(len(x), nat.hptr(x), nat.hptr(y), n_x, n_y, nat.hptr(sim), nat.hptr(ptr),
                                            nat.hptr(idx), nat.hptr(val), k, min_k, mode, 3.1, nat.hptr(bx),
                                            nat.hptr(by), nat.hptr(est), nat.hptr(ak), nat.hptr(imp)))
        assert np.array_equal(imp, want[2]) and np.array_equal(ak, want[1]) and np.array_equal(est, want[0])


def test_knn_threshold_select_on_nearly_equal_similarities():
    """The short-list select bisects on the high 32 bits of the similarity keys first: similarities that differ only in
    their low mantissa bits (same high word), exact ties among them, and groups straddling the k-th place must still
    come out in heapq.nlargest order -- every list length from 1 to a few hundred, several k."""
    rng = np.random.RandomState(5)
    n_x = 400
    lens = np.concatenate([np.arange(1, 70), rng.randint(70, 400, 40)])
    n_y = len(lens)
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    idx = np.concatenate([rng.permutation(n_x)[:ln] for ln in lens]).astype(np.int32)
    val = rng.randint(1, 6, len(idx)).astype(np.float64)
    base = np.array([0.5, 0.5, 0.5, 0.25, 0.75, 1.0, 0.1])          # few high words ...
    sim = base[rng.randint(0, len(base), (n_x, n_x))] + rng.randint(0, 6, (n_x, n_x)) * 2.0 ** -45   # ... many low words, ties
    sim[rng.rand(n_x, n_x) < 0.05] = -0.3
    sim[rng.rand(n_x, n_x) < 0.02] = 0.0
    sim = np.triu(sim) + np.triu(sim, 1).T
    np.fill_diagonal(sim, 1)
    x = rng.randint(0, n_x, 4000).astype(np.int32); y = rng.randint(0, n_y, 4000).astype(np.int32)
    bx = rng.normal(0, 1, n_x); by = rng.normal(0, 1, n_y)
    for (k, min_k, mode) in ((40, 1, 0), (1, 1, 0), (7, 1, 1), (128, 2, 2), (33, 1, 3)):
        want = oracle.knn_estimate(x, y, sim, ptr, idx, val, k, min_k, mode, 3.1, bx, by)
        est = np.empty(len(x)); ak = np.empty(len(x), dtype=np.int32); imp = np.empty(len(x), dtype=np.uint8)
        nat.check(nat.lib().sb2_knn_predict(len(x), nat.hptr(x), nat.hptr(y), n_x, n_y, nat.hptr(sim), nat.hptr(ptr),
                                            nat.hptr(idx), nat.hptr(val), k, min_k, mode, 3.1, nat.hptr(bx),
                                            nat.hptr(by), nat.hptr(est), nat.hptr(ak), nat.hptr(imp)))
        assert np.array_equal(imp, want[2]) and np.array_equal(ak, want[1]) and np.array_equal(est, want[0])


# ---- NMF ------------------------------------------------------------------------------------------------
def test_u1_nmf_bit_exact(u1, u1_golden, u1_arrays):
    ts, testset = u1
    algo = sb.NMF(random_state=0).fit(ts)
    g = u1_golden["algos"]["NMF_rs0"]
    assert sha(algo.pu) == g["pu_sha256"] and sha(algo.qi) == g["qi_sha256"]
    preds = algo.test(testset)
    assert abs(float(sb.accuracy.rmse(preds, verbose=False)) - float(g["rmse"])) < 1e-12
    assert sum(p.details["was_impossible"] for p in preds) == g["n_impossible"]
    algo = sb.NMF(random_state=3, n_factors=7, n_epochs=3, reg_pu=.1, reg_qi=.02).fit(ts)
    g = u1_golden["algos"]["NMF_rs3_f7_e3"]
    assert sha(algo.pu) == g["pu_sha256"] and sha(algo.qi) == g["qi_sha256"]
    algo = sb.NMF(random_state=0, biased=True).fit(ts)
    assert np.array_equal(algo.bu, u1_arrays["NMF_rs0_biased_bu"])
    preds = algo.test(testset)
    assert abs(float(sb.accuracy.rmse(preds, verbose=False)) - float(u1_golden["algos"]["NMF_rs0_biased"]["rmse"])) < 1e-12
    with pytest.raises(ValueError):
        sb.NMF(init_low=-1)


@pytest.mark.parametrize("f", (3, 8, 15, 16, 24, 32, 40))
def test_synthetic_nmf_bit_exact_host_abi(f):
    """Through the host-buffer C-ABI, ragged segments, every group width of the fused pass (4 / 8 / 16 / 32 lanes) and
    the three-kernel path (f > 32, and the biased model)."""
    d = synth.ratings(700, 300, 30_000, seed=f)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    uu, ii, rr = ts.coo()
    rng = np.random.RandomState(f)
    pu0 = rng.uniform(0, 1, (ts.n_users, f)); qi0 = rng.uniform(0, 1, (ts.n_items, f))
    for biased in (False, True):
        want = oracle.nmf_sgd(ts.n_users, ts.n_items, uu, ii, rr, np.diff(ts.user_csr()[0]), np.diff(ts.item_csr()[0]),
                              pu0, qi0, 4, biased, float(ts.global_mean), .06, .05, .02, .03, .005, .004)
        pu, qi = pu0.copy(), qi0.copy()
        bu, bi = np.empty(ts.n_users), np.empty(ts.n_items)
        prm = nat.NmfParams(n_factors=f, n_epochs=4, biased=int(biased), reserved=0, global_mean=float(ts.global_mean),
                            reg_pu=.06, reg_qi=.05, reg_bu=.02, reg_bi=.03, lr_bu=.005, lr_bi=.004)
        nat.check(nat.lib().sb2_nmf_fit(ts.n_users, ts.n_items, len(rr), nat.hptr(uu), nat.hptr(ii), nat.hptr(rr),
                                        C.byref(prm), nat.hptr(pu), nat.hptr(qi), nat.hptr(bu), nat.hptr(bi)))
        for got, w, name in ((pu, want[0], "pu"), (qi, want[1], "qi"), (bu, want[2], "bu"), (bi, want[3], "bi")):
            assert np.array_equal(got, w), (f, biased, name)


# ---- SVD ------------------------------------------------------------------------------------------------
RMSE_TOL = 0.005  # north_star: SVD / SVD++ held-out RMSE / MAE within 0.005 of the reference


@pytest.mark.parametrize("tag,kw", [("SVD_rs0", {}), ("SVD_rs0_f20_e5", {"n_factors": 20, "n_epochs": 5})])
def test_u1_svd_rmse(u1, u1_golden, tag, kw):
    ts, testset = u1
    algo = sb.SVD(random_state=0, **kw).fit(ts)
    assert algo.pu.shape == (ts.n_users, algo.n_factors) and algo.pu.dtype == np.float64
    preds = algo.test(testset)
    g = u1_golden["algos"][tag]
    assert abs(float(sb.accuracy.rmse(preds, verbose=False)) - float(g["rmse"])) <= RMSE_TOL
    assert abs(float(sb.accuracy.mae(preds, verbose=False)) - float(g["mae"])) <= RMSE_TOL
    assert sum(p.details["was_impossible"] for p in preds) == g["n_impossible"]


def test_u1_svd_unbiased_rmse(u1, u1_golden):
    """SVD(biased=False) on the 8000-rating fixture is far from converged after 20 epochs (RMSE 2.28), and in
    that regime the reference's OWN result depends on the order of its input by more than 0.005: sequential
    SGD (the oracle) on permutations of the same ratings gives 2.2826..2.2842 against 2.2754 in file order
    (DESIGN.md "SVD parity").  The stratified kernel is therefore held to 0.005 of the sequential algorithm on a
    permuted order, and to 0.012 of the file-order golden."""
    ts, testset = u1
    algo = sb.SVD(random_state=0, biased=False).fit(ts)
    preds = algo.test(testset)
    got = float(sb.accuracy.rmse(preds, verbose=False))
    g = u1_golden["algos"]["SVD_rs0_unbiased"]
    assert sum(p.details["was_impossible"] for p in preds) == g["n_impossible"]
    assert abs(got - float(g["rmse"])) <= 0.012
    u, i, r = ts.coo()
    iu, ii = inner_pairs(ts, testset)
    mu = float(ts.global_mean)
    band = []
    for seed in (0, 1):
        o = np.random.RandomState(seed).permutation(len(r))
        rng = np.random.RandomState(0)
        pu0 = rng.normal(0, .1, (ts.n_users, 100)); qi0 = rng.normal(0, .1, (ts.n_items, 100))
        pu, qi, bu, bi = oracle.svd_sgd(u[o], i[o], r[o], pu0, qi0, 20, False, mu, *([.005] * 4), *([.02] * 4))
        est, imp = oracle.mf_estimate(iu, ii, False, mu, pu, qi, bu, bi)
        band.append(rmse_mae(np.where(imp > 0, mu, est), testset, ts, mu)[0])
    assert abs(got - np.mean(band)) <= RMSE_TOL, (got, band)


def test_svd_zero_epochs_returns_init(u1):
    ts, _ = u1
    algo = sb.SVD(random_state=5, n_epochs=0, n_factors=10).fit(ts)
    rng = np.random.RandomState(5)
    pu0 = rng.normal(0, .1, (ts.n_users, 10))
    assert np.allclose(algo.pu, pu0.astype(np.float32), rtol=0, atol=0) and np.all(algo.bu == 0)


@pytest.mark.parametrize("f", (8, 20, 100))
def test_synthetic_svd_rmse_vs_oracle(f):
    """ml-1M-style synthetic at reduced size: same seed, same hyper-parameters, held-out RMSE vs the oracle's
    sequential SGD.  Also: one epoch on a conflict-free input must equal the oracle to fp32 accuracy."""
    d = synth.ratings(2000, 1200, 150_000, seed=10 + f)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    uu, ii, rr = ts.coo()
    tu, ti, tr_ = d["test"]
    mu = float(ts.global_mean)
    algo = sb.SVD(n_factors=f, n_epochs=10, random_state=1).fit(ts)
    rng = np.random.RandomState(1)
    pu0 = rng.normal(0, .1, (ts.n_users, f)); qi0 = rng.normal(0, .1, (ts.n_items, f))
    pu, qi, bu, bi = oracle.svd_sgd(uu, ii, rr, pu0, qi0, 10, True, mu, *([.005] * 4), *([.02] * 4))
    want, _ = oracle.mf_estimate(tu, ti, True, mu, pu, qi, bu, bi)
    got, _ = oracle.mf_estimate(tu, ti, True, mu, algo.pu, algo.qi, algo.bu, algo.bi)
    rm_w = np.sqrt(np.mean((np.clip(want, 1, 5) - tr_) ** 2)); rm_g = np.sqrt(np.mean((np.clip(got, 1, 5) - tr_) ** 2))
    ma_w = np.mean(np.abs(np.clip(want, 1, 5) - tr_)); ma_g = np.mean(np.abs(np.clip(got, 1, 5) - tr_))
    assert abs(rm_w - rm_g) <= RMSE_TOL and abs(ma_w - ma_g) <= RMSE_TOL, (rm_w, rm_g)


@pytest.mark.parametrize("f", (3, 50, 150, 300))
def test_svd_lane_shapes_rmse_vs_oracle(f):
    """Every (lanes, chunks-per-lane) shape of the update: f=3 -> 1 lane x 1 chunk, 50 -> 4 x 4, 150 -> 16 x 3 (512-thread
    CTAs), 300 -> 32 lanes striding the row.  Held-out RMSE within 0.005 of the sequential oracle, and one epoch on a
    conflict-free input equal to the oracle to fp32 rounding."""
    d = synth.ratings(1500, 900, 60_000, seed=30 + f)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    uu, ii, rr = ts.coo()
    tu, ti, tr_ = d["test"]
    mu = float(ts.global_mean)
    algo = sb.SVD(n_factors=f, n_epochs=6, random_state=3).fit(ts)
    rng = np.random.RandomState(3)
    pu0 = rng.normal(0, .1, (ts.n_users, f)); qi0 = rng.normal(0, .1, (ts.n_items, f))
    pu, qi, bu, bi = oracle.svd_sgd(uu, ii, rr, pu0, qi0, 6, True, mu, *([.005] * 4), *([.02] * 4))
    want, _ = oracle.mf_estimate(tu, ti, True, mu, pu, qi, bu, bi)
    got, _ = oracle.mf_estimate(tu, ti, True, mu, algo.pu, algo.qi, algo.bu, algo.bi)
    rm = lambda e: float(np.sqrt(np.mean((np.clip(e, 1, 5) - tr_) ** 2)))
    assert abs(rm(want) - rm(got)) <= RMSE_TOL, (f, rm(want), rm(got))
    n = 400
    rs = np.random.RandomState(2)
    pu_, pi_ = np.arange(n, dtype=np.int32), rs.permutation(n).astype(np.int32)
    pr_ = rs.randint(1, 6, n).astype(np.float64)
    tsp = sb.Trainset.from_coo(pu_, pi_, pr_, n, n)
    a2 = sb.SVD(n_factors=f, n_epochs=2, random_state=4).fit(tsp)
    rs = np.random.RandomState(4)
    p0 = rs.normal(0, .1, (n, f)); q0 = rs.normal(0, .1, (n, f))
    p1, q1, b1, c1 = oracle.svd_sgd(pu_, pi_, pr_, p0, q0, 2, True, float(tsp.global_mean), *([.005] * 4), *([.02] * 4))
    assert np.allclose(a2.pu, p1, rtol=0, atol=3e-6) and np.allclose(a2.qi, q1, rtol=0, atol=3e-6)
    assert np.allclose(a2.bu, b1, rtol=0, atol=3e-6) and np.allclose(a2.bi, c1, rtol=0, atol=3e-6)


@pytest.mark.parametrize("f", (40, 150))
def test_svdpp_wide_factors_rmse_vs_oracle(f):
    """SVD++ user rows are [p | z | g] = 3 x the factor row: f=40 -> 4 lanes x 3 chunks, f=150 -> 16 x 3 with user rows
    too long to stage every block in shared memory."""
    d = synth.ratings(800, 500, 25_000, seed=40 + f)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    uu, ii, rr = ts.coo()
    ptr, idx, _ = ts.user_csr()
    tu, ti, tr_ = d["test"]
    mu = float(ts.global_mean)
    algo = sb.SVDpp(n_factors=f, n_epochs=5, random_state=0).fit(ts)
    rng = np.random.RandomState(0)
    pu0 = rng.normal(0, .1, (ts.n_users, f)); qi0 = rng.normal(0, .1, (ts.n_items, f)); yj0 = rng.normal(0, .1, (ts.n_items, f))
    pu, qi, yj, bu, bi = oracle.svdpp_sgd(uu, ii, rr, ptr, idx, pu0, qi0, yj0, 5, mu, *([.007] * 5), *([.02] * 5))
    want, _ = oracle.mf_estimate(tu, ti, True, mu, pu, qi, bu, bi, yj, ptr, idx)
    got, _ = oracle.mf_estimate(tu, ti, True, mu, algo.pu, algo.qi, algo.bu, algo.bi, algo.yj, ptr, idx)
    rm = lambda e: float(np.sqrt(np.mean((np.clip(e, 1, 5) - tr_) ** 2)))
    assert abs(rm(want) - rm(got)) <= RMSE_TOL, (f, rm(want), rm(got))


def test_svd_conflict_free_input_matches_oracle():
    """A permutation matrix of ratings (no two share a user or an item) makes SGD order-independent:
    the stratified kernel must then reproduce the sequential oracle up to fp32 rounding."""
    n = 500
    rng = np.random.RandomState(2)
    u = np.arange(n, dtype=np.int32); i = rng.permutation(n).astype(np.int32)
    r = rng.randint(1, 6, n).astype(np.float64)
    ts = sb.Trainset.from_coo(u, i, r, n, n)
    for biased in (True, False):
        algo = sb.SVD(n_factors=12, n_epochs=3, random_state=4, biased=biased).fit(ts)
        rs = np.random.RandomState(4)
        pu0 = rs.normal(0, .1, (n, 12)); qi0 = rs.normal(0, .1, (n, 12))
        pu, qi, bu, bi = oracle.svd_sgd(u, i, r, pu0, qi0, 3, biased, float(ts.global_mean), *([.005] * 4), *([.02] * 4))
        assert np.allclose(algo.pu, pu, rtol=0, atol=2e-6) and np.allclose(algo.qi, qi, rtol=0, atol=2e-6)
        assert np.allclose(algo.bu, bu, rtol=0, atol=2e-6) and np.allclose(algo.bi, bi, rtol=0, atol=2e-6)
    # SVD++: each y_j has one rater, who rates nothing else, so its relaxation is exact here as well
    algo = sb.SVDpp(n_factors=12, n_epochs=3, random_state=4).fit(ts)
    rs = np.random.RandomState(4)
    pu0, qi0, yj0 = (rs.normal(0, .1, (n, 12)) for _ in range(3))
    ptr, idx, _ = ts.user_csr()
    want = oracle.svdpp_sgd(u, i, r, ptr, idx, pu0, qi0, yj0, 3, float(ts.global_mean), *([.007] * 5), *([.02] * 5))
    for name, w in zip(("pu", "qi", "yj", "bu", "bi"), want):
        assert np.allclose(getattr(algo, name), w, rtol=0, atol=2e-6), name
    assert np.abs(algo.yj - yj0).max() > 1e-4


def test_svd_split_launches_bit_identical(monkeypatch):
    """A launch may cover any range of strata (the SVD++ path applies y_j between ranges): running every epoch
    as n launches performs the same updates in the same order, so the factors must not change by one bit --
    this pins the hand-over of item blocks across launch boundaries (cluster ring + L2 mailboxes)."""
    d = synth.ratings(3000, 1500, 200_000, seed=3)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    monkeypatch.delenv("SB2_DSGD_SPLIT", raising=False)
    base = sb.SVD(n_factors=24, n_epochs=3, random_state=2).fit(ts)
    for split in (2, 3, 7, 16, 10_000):
        monkeypatch.setenv("SB2_DSGD_SPLIT", str(split))
        algo = sb.SVD(n_factors=24, n_epochs=3, random_state=2).fit(ts)
        for name in ("pu", "qi", "bu", "bi"):
            assert np.array_equal(getattr(algo, name), getattr(base, name)), (split, name)


def test_u1_svdpp_rmse(u1, u1_golden):
    ts, testset = u1
    algo = sb.SVDpp(random_state=0).fit(ts)
    assert algo.yj.shape == (ts.n_items, 20) and algo.yj.dtype == np.float64
    preds = algo.test(testset)
    g = u1_golden["algos"]["SVDpp_rs0"]
    assert abs(float(sb.accuracy.rmse(preds, verbose=False)) - float(g["rmse"])) <= RMSE_TOL
    assert abs(float(sb.accuracy.mae(preds, verbose=False)) - float(g["mae"])) <= RMSE_TOL
    # estimate() path of SVD++ (implicit term recomputed from yj) against the oracle on the fitted factors
    iu, ii = inner_pairs(ts, testset)
    ptr, idx, _ = ts.user_csr()
    want, _ = oracle.mf_estimate(iu, ii, True, float(ts.global_mean), algo.pu, algo.qi, algo.bu, algo.bi, algo.yj, ptr, idx)
    got, _ = algo._estimate_batch(iu, ii)
    assert np.allclose(got, want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("shape", [(600, 400, 30_000, 10), (3000, 300, 200_000, 10)])
def test_synthetic_svdpp_rmse_vs_oracle(shape):
    """Second shape: every item has ~670 raters -- the regime where adding a whole epoch of y_j gradients without
    integrating the (1 - lr reg) decay overshoots by 0.017 (tools/proto/svdpp_variants.py); with the decay
    integrated exactly the once-per-epoch application stays within 0.005 of the per-rating reference."""
    nu, ni, n, epochs = shape
    d = synth.ratings(nu, ni, n, seed=5)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    uu, ii, rr = ts.coo()
    ptr, idx, _ = ts.user_csr()
    tu, ti, tr_ = d["test"]
    mu = float(ts.global_mean)
    algo = sb.SVDpp(n_epochs=epochs, random_state=0).fit(ts)
    rng = np.random.RandomState(0)
    f = 20
    pu0 = rng.normal(0, .1, (ts.n_users, f)); qi0 = rng.normal(0, .1, (ts.n_items, f)); yj0 = rng.normal(0, .1, (ts.n_items, f))
    pu, qi, yj, bu, bi = oracle.svdpp_sgd(uu, ii, rr, ptr, idx, pu0, qi0, yj0, epochs, mu, *([.007] * 5), *([.02] * 5))
    want, _ = oracle.mf_estimate(tu, ti, True, mu, pu, qi, bu, bi, yj, ptr, idx)
    got, _ = oracle.mf_estimate(tu, ti, True, mu, algo.pu, algo.qi, algo.bu, algo.bi, algo.yj, ptr, idx)
    rm = lambda e: float(np.sqrt(np.mean((np.clip(e, 1, 5) - tr_) ** 2)))
    ma = lambda e: float(np.mean(np.abs(np.clip(e, 1, 5) - tr_)))
    assert abs(rm(want) - rm(got)) <= RMSE_TOL and abs(ma(want) - ma(got)) <= RMSE_TOL, (rm(want), rm(got))


@pytest.mark.parametrize("scale", (0.5, 1.0))
def test_svdpp_ml10m_shape_vs_stored_oracle(scale):
    """BASELINE configs[3] (SVD++ f=20, 20 epochs, ml-10M shape) and its half-scale version: held-out RMSE within
    0.005 of the sequential oracle's, which took 4 / 32 CPU-minutes to produce (tests/golden/svdpp_oracle_rmse.json,
    generated by tools/oracle_svdpp_rmse.py on the same seeded workload)."""
    import json
    with open(os.path.join(GOLDEN, "svdpp_oracle_rmse.json")) as fh:
        want = {r["scale"]: r for r in json.load(fh)["runs"]}[scale]
    d = synth.shaped("ml-10m", seed=0, scale=scale)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"], (0.5, 5.0), 0)
    assert ts.n_ratings == want["n_ratings"]
    algo = sb.SVDpp(random_state=0).fit(ts)
    tu, ti, tr_ = d["test"]
    est, _ = algo._estimate_batch(tu, ti)
    got = float(np.sqrt(np.mean((np.clip(est, 0.5, 5) - tr_) ** 2)))
    assert abs(got - want["oracle_svdpp_heldout_rmse"]) <= RMSE_TOL, (got, want["oracle_svdpp_heldout_rmse"])


def test_mf_predict_against_oracle(u1):
    ts, testset = u1
    iu, ii = inner_pairs(ts, testset)
    rng = np.random.RandomState(0)
    for f in (1, 15, 100, 130):
        pu = rng.normal(0, 1, (ts.n_users, f)); qi = rng.normal(0, 1, (ts.n_items, f))
        bu = rng.normal(0, 1, ts.n_users); bi = rng.normal(0, 1, ts.n_items)
        for biased in (True, False):
            want, wimp = oracle.mf_estimate(iu, ii, biased, 3.5, pu, qi, bu, bi)
            est = np.empty(len(iu)); imp = np.empty(len(iu), dtype=np.uint8)
            nat.check(nat.lib().sb2_mf_predict(len(iu), nat.hptr(iu), nat.hptr(ii), ts.n_users, ts.n_items, f,
                                               int(biased), 3.5, nat.hptr(pu), nat.hptr(qi), nat.hptr(bu), nat.hptr(bi),
                                               None, None, None, nat.hptr(est), nat.hptr(imp)))
            assert np.array_equal(imp, wimp)
            assert np.allclose(est, want, rtol=1e-12, atol=1e-12)


# ---- API behaviour ----------------------------------------------------------------------------------------
def test_unknown_user_or_item_and_pickle(tmp_path):
    """reference tests/test_algorithms.py::test_unknown_user_or_item + tests/test_dump.py."""
    reader = sb.Reader(line_format="user item rating", sep=" ", skip_lines=3, rating_scale=(1, 5))
    data = sb.Dataset.load_from_file(os.path.join(GOLDEN, "custom_dataset"), reader)
    ts = data.build_full_trainset()
    for klass in (sb.SVD, sb.SVDpp, sb.NMF, sb.KNNBasic, sb.KNNBaseline, sb.KNNWithMeans, sb.KNNWithZScore, sb.BaselineOnly):
        algo = klass()
        algo.fit(ts)
        algo.predict("user0", "unknown_item", None)
        algo.predict("unkown_user", "item0", None)
        p = algo.predict("unkown_user", "unknown_item", None)
        assert 1 <= p.est <= 5
        q = algo.predict("user0", "item0", 4)
        sb.dump.dump(str(tmp_path / "a.pkl"), algo=algo)
        _, algo2 = sb.dump.load(str(tmp_path / "a.pkl"))
        assert algo2.predict("user0", "item0", 4).est == q.est
    with pytest.raises(NameError):
        sb.KNNBasic(sim_options={"name": "wrong"}).fit(ts)


# ---- stress variant of SURVEY 8d: Zipf item popularity x log-normal user activity ------------------------------------
@pytest.fixture(scope="module")
def skewed():
    d = synth.ratings(3000, 1500, 150_000, seed=21, skew=True)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    assert np.bincount(i).max() > 1500 and np.bincount(u).max() > 300   # a 2000-rater item, 500-rating users
    return d, ts


def test_skewed_similarities_and_knn_bit_exact(skewed, sim_path):
    """Popular items / heavy users: long neighbour lists (beyond the per-lane buffers: refills) and large co-rating
    counts, item-based; every similarity kind against the oracle's full matrix, k-NN estimates bit for bit."""
    d, ts = skewed
    yr = ts.user_csr()
    n_x = ts.n_items
    algo = sb.BaselineOnly()
    sb.AlgoBase.fit(algo, ts)
    bu, bi = algo.compute_baselines()
    mu = float(ts.global_mean)
    for kind in KINDS:
        kw = dict(global_mean=mu, x_biases=bi, y_biases=bu) if kind == "pearson_baseline" else {}
        got = sims.build_device(kind, n_x, yr, 1, **kw).cpu().numpy()
        want = oracle.similarity(kind, n_x, *yr, 1, mu, bi, bu, 100.0)
        if kind == "pearson_baseline":
            assert np.allclose(got, want, rtol=0, atol=PB_ATOL, equal_nan=True), np.nanmax(np.abs(got - want))
        else:
            assert np.array_equal(got, want, equal_nan=True), kind
    sim = oracle.similarity("msd", n_x, *yr, 1)
    tu, ti, _ = d["test"]
    x, y = np.asarray(ti, dtype=np.int32), np.asarray(tu, dtype=np.int32)
    for (k, min_k, mode) in ((40, 1, 0), (300, 1, 0), (40, 1, 2)):
        want = oracle.knn_estimate(x, y, sim, *yr, k, min_k, mode, mu, bi, bu)
        est = np.empty(len(x)); ak = np.empty(len(x), dtype=np.int32); imp = np.empty(len(x), dtype=np.uint8)
        nat.check(nat.lib().sb2_knn_predict(len(x), nat.hptr(x), nat.hptr(y), n_x, ts.n_users, nat.hptr(sim), nat.hptr(yr[0]),
                                            nat.hptr(yr[1]), nat.hptr(yr[2]), k, min_k, mode, mu, nat.hptr(bi), nat.hptr(bu),
                                            nat.hptr(est), nat.hptr(ak), nat.hptr(imp)))
        ok = want[2] == 0
        assert np.array_equal(imp, want[2]) and np.array_equal(ak[ok], want[1][ok]) and np.array_equal(est[ok], want[0][ok]), (k, mode)


def test_skewed_nmf_bit_exact(skewed):
    """Item segments of 2000+ entries next to segments of one entry."""
    _, ts = skewed
    uu, ii, rr = ts.coo()
    f = 15
    rng = np.random.RandomState(0)
    pu0 = rng.uniform(0, 1, (ts.n_users, f)); qi0 = rng.uniform(0, 1, (ts.n_items, f))
    want = oracle.nmf_sgd(ts.n_users, ts.n_items, uu, ii, rr, np.diff(ts.user_csr()[0]), np.diff(ts.item_csr()[0]), pu0, qi0, 4,
                          False, 0.0, .06, .06, .02, .02, .005, .005)
    pu, qi = pu0.copy(), qi0.copy()
    bu, bi = np.empty(ts.n_users), np.empty(ts.n_items)
    prm = nat.NmfParams(n_factors=f, n_epochs=4, biased=0, reserved=0, global_mean=0.0, reg_pu=.06, reg_qi=.06, reg_bu=.02,
                        reg_bi=.02, lr_bu=.005, lr_bi=.005)
    nat.check(nat.lib().sb2_nmf_fit(ts.n_users, ts.n_items, len(rr), nat.hptr(uu), nat.hptr(ii), nat.hptr(rr), C.byref(prm),
                                    nat.hptr(pu), nat.hptr(qi), nat.hptr(bu), nat.hptr(bi)))
    assert np.array_equal(pu, want[0]) and np.array_equal(qi, want[1])


def test_skewed_svd_and_svdpp_rmse_vs_oracle(skewed):
    """Cells with a 2000-rater item overflow the 63 colours (sequential tail); SVD++: y_j of a popular item decays
    thousands of times per epoch.  Held-out RMSE / MAE within 0.005 of the sequential oracle."""
    d, ts = skewed
    uu, ii, rr = ts.coo()
    ptr, idx, _ = ts.user_csr()
    tu, ti, tr_ = d["test"]
    mu = float(ts.global_mean)
    rm = lambda e: float(np.sqrt(np.mean((np.clip(e, 1, 5) - tr_) ** 2)))
    ma = lambda e: float(np.mean(np.abs(np.clip(e, 1, 5) - tr_)))
    f = 20
    rng = np.random.RandomState(0)
    pu0 = rng.normal(0, .1, (ts.n_users, f)); qi0 = rng.normal(0, .1, (ts.n_items, f))
    pu, qi, bu, bi = oracle.svd_sgd(uu, ii, rr, pu0, qi0, 10, True, mu, *([.005] * 4), *([.02] * 4))
    want, _ = oracle.mf_estimate(tu, ti, True, mu, pu, qi, bu, bi)
    algo = sb.SVD(n_factors=f, n_epochs=10, random_state=0).fit(ts)
    got, _ = oracle.mf_estimate(tu, ti, True, mu, algo.pu, algo.qi, algo.bu, algo.bi)
    assert abs(rm(want) - rm(got)) <= RMSE_TOL and abs(ma(want) - ma(got)) <= RMSE_TOL, ("svd", rm(want), rm(got))
    rng = np.random.RandomState(0)
    pu0 = rng.normal(0, .1, (ts.n_users, f)); qi0 = rng.normal(0, .1, (ts.n_items, f)); yj0 = rng.normal(0, .1, (ts.n_items, f))
    pu, qi, yj, bu, bi = oracle.svdpp_sgd(uu, ii, rr, ptr, idx, pu0, qi0, yj0, 10, mu, *([.007] * 5), *([.02] * 5))
    want, _ = oracle.mf_estimate(tu, ti, True, mu, pu, qi, bu, bi, yj, ptr, idx)
    algo = sb.SVDpp(n_epochs=10, random_state=0).fit(ts)
    got, _ = oracle.mf_estimate(tu, ti, True, mu, algo.pu, algo.qi, algo.bu, algo.bi, algo.yj, ptr, idx)
    assert abs(rm(want) - rm(got)) <= RMSE_TOL and abs(ma(want) - ma(got)) <= RMSE_TOL, ("svdpp", rm(want), rm(got))

