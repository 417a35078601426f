"""GridSearchCV against the loop a user would otherwise write: per candidate and fold, fit, algo.test(testset) and
accuracy.rmse / mae on the Prediction tuples (the tuple route).

Workloads (synthetic, synth.ratings(..., seed=0); KFold(3, random_state=0); measures rmse and mae):
  svd_ml1m        SVD, 18 candidates (n_factors 50/100/150 x lr_all 0.002/0.005/0.01 x reg_all 0.02/0.1), ml-1M shape
  knnbaseline_ml1m  KNNBaseline, item-based pearson_baseline, k = 10/20/40/80, ml-1M shape
  svd_ml20m       SVD, 4 candidates (n_factors 50/100 x lr_all 0.005/0.01), ml-20M shape; the tuple route runs on
                  fold 0 only (seconds per task there) and its loop time is extrapolated from those tasks
The tuple route refits every candidate (the fits are deterministic) and each of its scores must equal, bit for bit,
the score GridSearchCV reported for that candidate and fold; any difference fails the run before anything is
reported.  Reported per workload: search wall time (synchronised), its fit and non-fit parts, per-task fit and score
times of both routes, the tuple loop's time and the speedup, with the GPU's name and power limit read in the same run.
One JSON line per workload on stdout; --out FILE writes the whole report.  Nothing is written into the tree.

    python tools/bench_search.py [--out FILE] [--only svd_ml1m,knnbaseline_ml1m,svd_ml20m]
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

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import accuracy, synth  # noqa: E402
from surprise_b200.model_selection import GridSearchCV, KFold  # noqa: E402

MEASURES = ["rmse", "mae"]
WORKLOADS = {
    "svd_ml1m": ("ml-1m", sb.SVD, {"n_factors": [50, 100, 150], "lr_all": [0.002, 0.005, 0.01],
                                   "reg_all": [0.02, 0.1], "random_state": [0]}, None),
    "knnbaseline_ml1m": ("ml-1m", sb.KNNBaseline, {"k": [10, 20, 40, 80],
                                                   "sim_options": {"name": ["pearson_baseline"],
                                                                   "user_based": [False]}}, None),
    "svd_ml20m": ("ml-20m", sb.SVD, {"n_factors": [50, 100], "lr_all": [0.005, 0.01], "random_state": [0]}, [0]),
}
N_FOLDS = 3


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi: %s)" % q.stderr.strip()


def sync():
    nat.torch_cuda().cuda.synchronize()


def dataset(shape):
    nu, ni, nr, step = synth.SHAPES[shape]
    u, i, r = synth.ratings(nu, ni, nr, step=step, seed=0)["train"]
    lo = 0.5 if step == 0.5 else 1.0
    return sb.Dataset.load_from_arrays(u, i, r, sb.Reader(rating_scale=(lo, 5.0)))


def bench(name):
    shape, cls, grid, check_folds = WORKLOADS[name]
    # warm-up: module loads and first launches of every kernel this algorithm uses, on other data
    warm = dataset("ml-100k")
    GridSearchCV(cls, {k: v[:1] if isinstance(v, list) else v for k, v in grid.items()}, measures=MEASURES,
                 cv=2).fit(warm)
    data = dataset(shape)
    gs = GridSearchCV(cls, grid, measures=MEASURES, cv=KFold(N_FOLDS, random_state=0))
    sync()
    t0 = time.perf_counter()
    gs.fit(data)
    sync()
    search_s = time.perf_counter() - t0
    res = gs.cv_results
    n_c = len(gs.param_combinations)
    search_fit_s = float(res["mean_fit_time"].sum() * N_FOLDS)

    # the tuple route on the same folds: each score checked against the search's before anything is reported
    check_folds = list(range(N_FOLDS)) if check_folds is None else check_folds
    t0 = time.perf_counter()
    folds = []
    for f, fold in enumerate(KFold(N_FOLDS, random_state=0).split(data)):
        if f in check_folds:
            folds.append((f, fold))
    split_s = time.perf_counter() - t0
    fit_t, score_t = [], []
    for c, params in enumerate(gs.param_combinations):
        for f, (trs, tes) in folds:
            algo = cls(**params)
            sync()
            t0 = time.perf_counter()
            algo.fit(trs)
            sync()
            t1 = time.perf_counter()
            preds = algo.test(tes)
            scores = {m: getattr(accuracy, m)(preds, verbose=False) for m in MEASURES}
            t2 = time.perf_counter()
            fit_t.append(t1 - t0)
            score_t.append(t2 - t1)
            for m in MEASURES:
                got = res["split%d_test_%s" % (f, m)][c]
                if np.float64(got).tobytes() != np.float64(scores[m]).tobytes():
                    raise SystemExit("%s: candidate %d fold %d %s: search %r != tuple route %r"
                                     % (name, c, f, m, got, scores[m]))
            del algo, preds
    n_tasks = n_c * N_FOLDS
    tuple_fit, tuple_score = float(np.mean(fit_t)), float(np.mean(score_t))
    tuple_loop_s = split_s + (tuple_fit + tuple_score) * n_tasks      # split_s covers all the folds
    return dict(workload=name, gpu=gpu_info(), shape=shape, candidates=n_c, folds=N_FOLDS,
                test_pairs_per_fold=int(synth.SHAPES[shape][2] // N_FOLDS), checked_tasks=len(fit_t),
                checked="bit-identical rmse and mae on %d of %d tasks" % (len(fit_t), n_tasks),
                search_wall_s=search_s, search_fit_s=search_fit_s, search_non_fit_s=search_s - search_fit_s,
                search_fit_per_task_s=search_fit_s / n_tasks,
                search_non_fit_per_task_s=(search_s - search_fit_s) / n_tasks,
                tuple_fit_per_task_s=tuple_fit, tuple_score_per_task_s=tuple_score,
                tuple_split_s=split_s, tuple_loop_s=tuple_loop_s,
                tuple_loop_extrapolated=len(folds) < N_FOLDS,
                speedup=tuple_loop_s / search_s,
                best_rmse=float(gs.best_score["rmse"]), best_params_rmse=repr(gs.best_params["rmse"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=",".join(WORKLOADS))
    args = ap.parse_args()
    nat.torch_cuda()
    report = []
    for name in args.only.split(","):
        rep = bench(name)
        print(json.dumps(rep), flush=True)
        report.append(rep)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(report, fh, indent=1)


if __name__ == "__main__":
    main()
