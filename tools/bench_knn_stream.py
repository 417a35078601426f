"""k-NN without the dense similarity matrix (DESIGN.md section 3.10): what the streamed route costs where the dense matrix
fits, and what it does where it cannot.

  * item-based KNNBasic(cosine) and KNNBaseline(pearson_baseline) at the ml-1M and ml-20M shapes: dense against forced
    streaming (default band budget), fit and test() on the 10 % fold, alternated in this process, median of --reps;
  * user-based KNNBasic(cosine) at the ml-20M shape and at the Netflix shape (streamed by default): fit, test() on the
    10 % fold, peak device memory (torch's allocator) and bands.

Before any time is reported: forced-streaming estimates must equal the dense ones bit for bit (every pair of the fold),
and the user-based estimates of --check pairs must equal the oracle's (orc_similarity_pairs for the entries they read,
then orc_knn_estimate's k-NN step restated, tests/knn_stream_oracle.py).  The card's name, power limit and max SM clock
are read in the same run.

    python tools/bench_knn_stream.py [--out RESULT.json] [--shapes ml-1m,ml-20m,netflix] [--reps 3] [--check 2000]

One JSON line per measurement goes to stdout; --out also writes the whole report to a file.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import synth  # noqa: E402
from surprise_b200.prediction_algorithms import knns  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def sync_time(fn):
    import torch
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t


def load(shape):
    d = synth.shaped(shape, seed=0)
    u, i, r = d["train"]
    step = synth.SHAPES[shape][3]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"], (step, 5.0), 0)
    tu, ti, _ = d["test"]
    return ts, (u, i, r), tu.astype(np.int32), ti.astype(np.int32)


def run(cls, kind, ub, ts, tu, ti, streamed):
    """(est, fit s, test s, streamed?) of one fit and one estimate pass over the fold's pairs."""
    saved = knns._DENSE_SIM_FRACTION
    if streamed:
        knns._DENSE_SIM_FRACTION = 0.0
    try:
        algo = cls(k=40, sim_options={"name": kind, "user_based": ub})
        _, t_fit = sync_time(lambda: algo.fit(ts))
        (est, _, _), t_test = sync_time(lambda: algo._knn_batch(tu, ti, *algo._knn_args()))
        return est, t_fit, t_test, algo._streamed
    finally:
        knns._DENSE_SIM_FRACTION = saved


def item_based(shape, reps, report):
    ts, _, tu, ti = load(shape)
    for cls, kind in ((sb.KNNBasic, "cosine"), (sb.KNNBaseline, "pearson_baseline")):
        want = run(cls, kind, False, ts, tu, ti, False)[0]
        got = run(cls, kind, False, ts, tu, ti, True)[0]
        same = bool(np.array_equal(want.view(np.int64), got.view(np.int64)))
        times = {False: [], True: []}
        for _ in range(reps):
            for streamed in (False, True):        # alternated
                est, t_fit, t_test, s = run(cls, kind, False, ts, tu, ti, streamed)
                assert s == streamed
                same = same and bool(np.array_equal(est.view(np.int64), want.view(np.int64)))
                times[streamed].append((t_fit, t_test))
        if not same:
            raise SystemExit("streamed estimates differ from the dense ones: %s %s" % (shape, kind))
        med = {s: np.median(np.array(v), axis=0) for s, v in times.items()}
        line = dict(workload="item-based %s %s" % (cls.__name__, kind), shape=shape, pairs=len(tu),
                    n_x=ts.n_items, bit_identical=same,
                    dense_fit_s=float(med[False][0]), dense_test_s=float(med[False][1]),
                    streamed_fit_s=float(med[True][0]), streamed_test_s=float(med[True][1]),
                    band_rows=knns.band_rows(ts.n_items, knns._device_bytes()))
        print(json.dumps(line), flush=True)
        report.append(line)


def user_based(shape, n_check, report):
    import knn_stream_oracle
    import torch
    ts, (u, i, r), tu, ti = load(shape)
    algo = sb.KNNBasic(k=40, sim_options={"name": "cosine", "user_based": True})
    _, t_fit = sync_time(lambda: algo.fit(ts))
    assert algo._streamed, "the dense matrix fits: not a streaming workload"
    rng = np.random.RandomState(0)
    sel = rng.choice(len(tu), min(n_check, len(tu)), replace=False)
    (est_s, ak_s, imp_s), _ = sync_time(lambda: algo._knn_batch(tu[sel], ti[sel], 0))
    want_est, want_ak = knn_stream_oracle.user_based("cosine", 0, ts, u, i, r, tu[sel], ti[sel], 40)
    known = (tu[sel] >= 0) & (ti[sel] >= 0)
    ok = known & (imp_s == 0)
    same = bool(np.array_equal(est_s[ok].view(np.int64), want_est[ok].view(np.int64))
                and np.array_equal(ak_s[known], want_ak[known]))
    if not same:
        raise SystemExit("streamed estimates differ from the oracle's: %s" % shape)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    _, t_test = sync_time(lambda: algo._knn_batch(tu, ti, 0))
    peak = torch.cuda.max_memory_allocated()
    per = knns.band_rows(ts.n_users, knns._device_bytes())
    rows = len(np.unique(tu[(tu >= 0) & (ti >= 0)]))
    line = dict(workload="user-based KNNBasic cosine, streamed", shape=shape, n_x=ts.n_users,
                dense_matrix_gb=8 * ts.n_users ** 2 / 1e9, pairs=len(tu), oracle_checked_pairs=int(known.sum()),
                bit_identical_to_oracle=same, fit_s=t_fit, test_s=t_test, rows_built=rows, band_rows=per,
                bands=-(-rows // per), peak_torch_gb=peak / 1e9, resident_before_test_gb=base / 1e9)
    print(json.dumps(line), flush=True)
    report.append(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--shapes", default="ml-1m,ml-20m,netflix")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check", type=int, default=2000)
    a = ap.parse_args()
    report = [dict(gpu=gpu_info())]
    print(json.dumps(report[0]), flush=True)
    shapes = a.shapes.split(",")
    for shape in ("ml-1m", "ml-20m"):
        if shape in shapes:
            item_based(shape, a.reps, report)
    for shape in ("ml-20m", "netflix"):
        if shape in shapes:
            user_based(shape, a.check, report)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(report, fh, indent=1)


if __name__ == "__main__":
    main()
