"""AUC, MRR and MPR over the full ranking on a LeaveOneOut split: AlgoBase.rank_measures (device route) against the
definition, accuracy.rank_measures over get_top_n(n_items), for SVD f=100 at the ml-1M shape (fitted) and the ml-20M
shape (factors drawn, as tools/bench_top_n.py does: the ranking only reads them), and item-based
KNNBaseline(pearson_baseline) at the ml-1M shape.

Before any time is reported, the device route's result must equal the definition's (same keys, same float bits): over
every held-out user at the ml-1M shape, and over a fixed sample of 1 000 held-out users at the ml-20M shape, where the
definition over every user does not fit in host memory (138 000 x 26 700 tuples).  Every timed call's result must equal
the checked one.  The device route is synchronised wall time, median of --reps warm calls; the scorer and the rank call
(sb2_top_n_ranks_dev, one per block) are CUDA events around each block, summed over the pass, median of 5 passes; the
definition (get_top_n + accuracy.rank_measures) is timed once where it runs.

    python tools/bench_rank_eval.py [--out RESULT.json] [--workloads svd-ml-1m,svd-ml-20m,knn-ml-1m] [--reps 3]

One JSON line per workload goes to stdout; --out also writes the whole report to a file.
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
from surprise_b200.model_selection import LeaveOneOut  # noqa: E402
from surprise_b200.model_selection.validation import Fold  # noqa: E402

SAMPLE_USERS = 1000


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def same_result(a, b):
    return list(a) == list(b) and all(np.float64(a[k]).tobytes() == np.float64(b[k]).tobytes() for k in a)


def timed(fn, reps, check=lambda o: True):
    """Median wall time (ms, synchronised) of `reps` calls after one warm-up call, and whether `check` accepted the
    output of every timed call."""
    import torch
    fn()
    ms, ok = [], True
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        o = fn()
        torch.cuda.synchronize()
        ms.append((time.perf_counter() - t) * 1e3)
        ok = ok and check(o)
    return float(np.median(ms)), ok


def pass_event_ms(algo, tes):
    """(scorer ms, rank-call ms, blocks): CUDA events around each block's scoring and its sb2_top_n_ranks_dev call,
    summed over one pass over every evaluated user, median of 5 warm passes."""
    ts = algo.trainset
    iu, _, rel_ptr, rel_idx = Fold(ts, tes).test_pairs().relevant(None, ts.n_items)
    users = iu[iu >= 0]
    d_csr = algo._user_csr_dev()
    hook, _ = algo._rank_counter(len(users), rel_ptr, rel_idx, d_csr)
    algo._top_n_dev(1, users, on_scores=hook, select=False, d_csr=d_csr)
    score, rank = [], []
    for _ in range(5):
        ev = []
        algo._top_n_dev(1, users, _events=ev, on_scores=hook, select=False, d_csr=d_csr)
        ev[-1][2].synchronize()
        score.append(sum(e[0].elapsed_time(e[1]) for e in ev))
        rank.append(sum(e[1].elapsed_time(e[2]) for e in ev))
    return float(np.median(score)), float(np.median(rank)), len(ev)


def split(shape):
    if shape == "ml-1m":
        d = synth.ratings(*synth.SHAPES["ml-1m"][:3], seed=0)
        scale = (1, 5)
    else:
        d = synth.shaped(shape, seed=0)
        scale = (0.5, 5.0)
    u, i, r = d["train"]
    data = sb.Dataset.load_from_arrays(u, i, r, sb.Reader(rating_scale=scale))
    return next(LeaveOneOut(1, random_state=0).split(data))


def model(name, trs):
    if name == "knn":
        return sb.KNNBaseline(sim_options={"name": "pearson_baseline", "user_based": False}).fit(trs)
    if trs.n_users < 10 ** 5:
        return sb.SVD(n_factors=100, random_state=0).fit(trs)
    algo = sb.SVD(n_factors=100)        # drawn factors: the ranking reads pu / qi / bu / bi only
    sb.AlgoBase.fit(algo, trs)
    rng = np.random.RandomState(0)
    algo.pu, algo.qi = rng.normal(0, .3, (trs.n_users, 100)), rng.normal(0, .3, (trs.n_items, 100))
    algo.bu, algo.bi = rng.normal(0, .3, trs.n_users), rng.normal(0, .3, trs.n_items)
    return algo


def workload(label, reps):
    name, shape = label.split("-", 1)
    trs, tes = split(shape)
    algo = model(name, trs)
    tes = list(tes)
    res = dict(workload=label, n_users=trs.n_users, n_items=trs.n_items, n_ratings=trs.n_ratings, held_out=len(tes),
               gpu=gpu_info())
    if shape == "ml-1m":
        check_tes, check_users = tes, None
    else:
        rng = np.random.RandomState(0)
        users = sorted(set(u for u, _, _ in tes))
        keep = set(rng.choice(len(users), SAMPLE_USERS, replace=False).tolist())
        keep = set(users[k] for k in keep)
        check_tes = [row for row in tes if row[0] in keep]
        check_users = [u for u in dict.fromkeys(u for u, _, _ in check_tes) if trs.to_inner_uids([u])[0] >= 0]
    res["checked_users"] = len(set(u for u, _, _ in check_tes))
    t = time.perf_counter()
    want = accuracy.rank_measures(algo.get_top_n(trs.n_items, check_users), check_tes, trs, verbose=False)
    res["definition_ms" if check_users is None else "definition_sample_ms"] = (time.perf_counter() - t) * 1e3
    got = algo.rank_measures(check_tes)
    res["equal_to_definition"] = same_result(got, want)
    if not res["equal_to_definition"]:
        res.update(device=got, definition=want)
        print(json.dumps(res), flush=True)
        return res
    full = algo.rank_measures(tes)
    res["measures"] = full
    res["device_route_ms"], res["timed_outputs_match"] = timed(lambda: algo.rank_measures(tes), reps,
                                                               lambda o: same_result(o, full))
    res["scorer_ms"], res["rank_call_ms"], res["blocks"] = pass_event_ms(algo, tes)
    res["score_bytes"] = 8 * len(set(u for u, _, _ in tes)) * trs.n_items
    if "definition_ms" in res:
        res["speedup_vs_definition"] = res["definition_ms"] / res["device_route_ms"]
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--workloads", default="svd-ml-1m,svd-ml-20m,knn-ml-1m")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    nat.torch_cuda()
    report = dict(gpu=gpu_info(), results=[workload(w, a.reps) for w in a.workloads.split(",")])
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(report, fh, indent=1)


if __name__ == "__main__":
    main()
