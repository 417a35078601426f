"""The streamed k-NN route's host logic, without a GPU: the band planner, the route decision, pickling of a streamed
model, and the C-ABI declarations of the row build and the row-indexed k-NN estimate."""
import os
import pickle
import re

import numpy as np
import pytest
import torch

from conftest import ROOT

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200.prediction_algorithms import knns  # noqa: E402


def check_plan(x, per):
    x_t = torch.as_tensor(np.asarray(x, dtype=np.int32))
    order, inv, rows, slot, bands = knns.plan_bands(x_t, per)
    x = np.asarray(x, dtype=np.int32)
    n = len(x)
    order, inv, rows, slot = order.numpy(), inv.numpy(), rows.numpy(), slot.numpy()
    assert sorted(order.tolist()) == list(range(n))
    xs = x[order]
    assert np.array_equal(xs[inv], x)                              # inverse permutation
    assert np.array_equal(order, np.argsort(x, kind="stable"))     # grouped by x, input order inside a group
    assert rows.dtype == np.int32 and slot.dtype == np.int32
    assert np.array_equal(rows, np.unique(x[x >= 0]))
    if n == 0:
        assert bands == []
        return bands
    # bands tile the grouped pairs and the rows, in order, at most `per` rows each
    assert bands[0][0] == 0 and bands[-1][1] == n
    assert bands[0][2] == 0 and bands[-1][3] == len(rows)
    for (p0, p1, r0, r1), nxt in zip(bands, bands[1:] + [None]):
        assert 0 < r1 - r0 <= per or (len(rows) == 0 and r0 == r1 == 0)
        if nxt is not None:
            assert nxt[0] == p1 and nxt[2] == r1
        band_rows = rows[r0:r1]
        for p in range(p0, p1):
            if xs[p] < 0:
                assert p0 == 0 and slot[p] == 0                # unknown x: first band, reads nothing
            else:
                assert band_rows[slot[p]] == xs[p]              # the pair's row inside its band's block
    return bands


@pytest.mark.parametrize("per", (1, 2, 3, 7, 1000))
def test_plan_bands(per):
    rng = np.random.RandomState(per)
    for x in ([5, -1, 3, 5, 9, 3, -1, 7, 9, 9], rng.randint(-1, 50, 400), rng.randint(0, 3, 17), [4], [-1, -1, -1],
              rng.permutation(300) - 1, []):
        check_plan(x, per)


def test_plan_bands_shapes():
    assert check_plan([-1, -1], 4) == [(0, 2, 0, 0)]
    assert check_plan([2, 0, 2, -1, 1], 2) == [(0, 3, 0, 2), (3, 5, 2, 3)]


def test_route_decision(monkeypatch):
    gib = 1 << 30
    b200 = 180 * gib
    assert not knns.streams_similarities(27_000, b200)      # ml-20M item-based: 5.8 GB dense
    assert not knns.streams_similarities(100_000, b200)     # 80 GB: half the device or less
    assert knns.streams_similarities(138_000, b200)         # ml-20M user-based: 152 GB
    assert knns.streams_similarities(480_000, b200)         # Netflix shape user-based: 1.84 TB
    monkeypatch.setattr(knns, "_DENSE_SIM_FRACTION", 0.0)
    assert knns.streams_similarities(1, b200)
    assert knns.band_rows(480_000, b200) == (b200 // 8) // (8 * 480_000)
    monkeypatch.setattr(knns, "_STREAM_BAND_BYTES", 8 * 943 * 7)
    assert knns.band_rows(943, b200) == 7
    monkeypatch.setattr(knns, "_STREAM_BAND_BYTES", 1)
    assert knns.band_rows(943, b200) == 1


def test_streamed_state_pickles_without_device():
    u = np.array([0, 0, 1, 2], dtype=np.int32)
    i = np.array([0, 1, 1, 0], dtype=np.int32)
    ts = sb.Trainset.from_coo(u, i, np.array([1.0, 2.0, 3.0, 4.0]), 3, 2, (1.0, 5.0), 0)
    algo = sb.KNNBaseline(sim_options={"name": "pearson_baseline"})
    sb.AlgoBase.fit(algo, ts)
    algo.n_x, algo.n_y = 3, 2
    algo.bu, algo.bi = np.zeros(3), np.zeros(2)
    algo._sim_dev = algo._sim_host = algo._yr_dev = None
    algo._streamed = True
    algo._sim_kind = ("pearson_baseline", 1, float(ts.global_mean), 100)
    algo._sim_inputs = {"ptr": object()}                    # stands for device arrays: must not be pickled
    back = pickle.loads(pickle.dumps(algo))
    assert back._streamed and back._sim_inputs is None and back._sim_host is None and back._sim_dev is None
    assert back._sim_kind == algo._sim_kind
    back.sim = np.eye(3)                                    # an assigned matrix puts the model on the dense route
    assert not back._streamed and np.array_equal(back.sim, np.eye(3))


def test_header_declares_row_build_and_row_predict():
    hdr = open(os.path.join(ROOT, "include", "surprise_b200.h")).read()
    for name in ("sb2_sim_build_rows_dev", "sb2_knn_predict_rows_dev"):
        assert re.search(r"\bint %s\(" % name, hdr), name
        assert name in nat.SIGNATURES
    decl = re.search(r"int sb2_sim_build_rows_dev\((.*?)\);", hdr, re.S).group(1)
    assert len(decl.split(",")) == len(nat.SIGNATURES["sb2_sim_build_rows_dev"][1]) == 18
    decl = re.search(r"int sb2_knn_predict_rows_dev\((.*?)\);", hdr, re.S).group(1)
    assert "const int32_t* sim_row" in decl
    assert len(decl.split(",")) == len(nat.SIGNATURES["sb2_knn_predict_rows_dev"][1]) == 20
