"""Coverage, novelty and diversity of top-N lists: AlgoBase.top_n_list_measures (device route) against the dict route,
accuracy.top_n_list_measures over get_top_n, for SVD f=100 over every user of the training part of `synth` data (seed 0)
at the ml-1M shape (fitted) and the ml-20M shape (factors drawn, as tools/bench_top_n.py does: top-N only reads them),
n = 10 and 100.  Diversity reads the item-item cosine of an item-based KNNBasic fitted on the same trainset, passed as
the model (its device matrix is read in place); the definition reads its .sim array.

Before any time is reported, the device route's result must equal the definition's (same keys, same float bits), and
every timed device call's result must equal that checked result.  Where the Python definition over every user would
take minutes (diversity is quadratic in n), both routes are compared on a fixed sample of users (``uids``, drawn with
seed 0) and the definition's time over every user is an extrapolation from the sample, reported as such.  Device route
times are synchronised wall time, median of --reps warm calls; the dict route is timed once.  The list kernel
(sb2_top_n_lists_dev over every user, one launch, with diversity) is timed with CUDA events, median of 5 warm calls.

    python tools/bench_top_n_lists.py [--out RESULT.json] [--shapes ml-1m,ml-20m] [--n 10,100] [--reps 3]
        [--max-pairs 3e7] [--sample 2000]

One JSON line per (shape, n) goes to stdout; --out also writes the whole report to a file.
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def same_result(a, b):
    return list(a) == list(b) and all(np.float64(a[k]).tobytes() == np.float64(b[k]).tobytes() for k in a)


def sync_ms(fn):
    import torch
    torch.cuda.synchronize()
    t = time.perf_counter()
    o = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, o


def timed(fn, reps, check=lambda o: True):
    """Median wall time (ms, synchronised) of `reps` calls after one warm-up call, and whether `check` accepted the
    output of every timed call."""
    fn()
    ms, ok = [], True
    for _ in range(reps):
        t, o = sync_ms(fn)
        ms.append(t)
        ok = ok and check(o)
    return float(np.median(ms)), ok


def list_kernel_ms(algo, knn, n):
    """sb2_top_n_lists_dev over every user in one launch, with diversity (CUDA events, median of 5 warm calls), and
    the pairs it sums: sum over users of c(c - 1) / 2, each one scattered 8-byte read of the similarity matrix."""
    import torch
    ts = algo.trainset
    users = np.arange(ts.n_users, dtype=np.int32)
    width = min(n, ts.n_items)
    items, est, count = algo._top_n_dev(width, users)
    d_info = nat.to_dev(accuracy._novelty_table(ts), np.float64)
    sim = knn._sim_device()
    cov, nov, ils = (nat.empty_dev((len(users),), t) for t in (np.int32, np.float64, np.float64))
    seen = torch.zeros(ts.n_items, dtype=torch.uint8, device=nat.device())

    def call():
        nat.check(nat.lib().sb2_top_n_lists_dev(len(users), nat.ptr(items), width, nat.ptr(est), nat.ptr(count),
                                                width, 0, 0.0, ts.n_items, nat.ptr(d_info), nat.ptr(sim),
                                                nat.ptr(cov), nat.ptr(nov), nat.ptr(ils), nat.ptr(seen),
                                                nat.stream()))

    call()
    ms = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    c = count.cpu().numpy().astype(np.int64)
    return float(np.median(ms)), int((c * (c - 1) // 2).sum())


def workload(shape, ns, reps, max_pairs, sample):
    if shape == "ml-1m":
        d = synth.ratings(*synth.SHAPES["ml-1m"][:3], seed=0)
        scale = (1, 5)
    else:
        d = synth.shaped(shape, seed=0)
        scale = (0.5, 5.0)
    u, i, r = d["train"]
    ts = sb.Dataset.load_from_arrays(u, i, r, sb.Reader(rating_scale=scale)).build_full_trainset()
    if shape == "ml-1m":
        algo = sb.SVD(n_factors=100, random_state=0).fit(ts)
    else:     # drawn factors: top-N reads pu / qi / bu / bi only
        algo = sb.SVD(n_factors=100)
        sb.AlgoBase.fit(algo, ts)
        rng = np.random.RandomState(0)
        algo.pu, algo.qi = rng.normal(0, .3, (ts.n_users, 100)), rng.normal(0, .3, (ts.n_items, 100))
        algo.bu, algo.bi = rng.normal(0, .3, ts.n_users), rng.normal(0, .3, ts.n_items)
    knn = sb.KNNBasic(sim_options={"name": "cosine", "user_based": False}).fit(ts)
    sim_host = knn.sim
    raw_all = [ts.to_raw_uid(k) for k in range(ts.n_users)]
    rng = np.random.RandomState(0)
    sampled = [raw_all[k] for k in np.sort(rng.choice(ts.n_users, min(sample, ts.n_users), replace=False)).tolist()]
    out = []
    for n in ns:
        res = dict(shape=shape, n=n, n_users=ts.n_users, n_items=ts.n_items, n_ratings=ts.n_ratings, gpu=gpu_info())
        width = min(n, ts.n_items)
        full = ts.n_users * width * (width - 1) // 2 <= max_pairs
        uids = None if full else sampled
        res["definition_users"] = ts.n_users if full else len(sampled)
        dict_ms, want = sync_ms(lambda: accuracy.top_n_list_measures(algo.get_top_n(n, uids), ts, n, uids, None,
                                                                     sim_host, verbose=False))
        got = algo.top_n_list_measures(n, uids, sim=knn)
        res["equal_to_definition"] = same_result(got, want)
        res["measures_checked"] = got
        if not res["equal_to_definition"]:
            res["definition"] = want
            out.append(res)
            print(json.dumps(res), flush=True)
            continue
        if full:
            res["dict_route_ms"] = dict_ms
            check = lambda o: same_result(o, want)  # noqa: E731
        else:
            res["dict_route_ms_sample"] = dict_ms
            res["dict_route_ms_extrapolated_to_all_users"] = dict_ms * ts.n_users / len(sampled)
            res["measures_all_users"] = algo.top_n_list_measures(n, sim=knn)
            check = lambda o: same_result(o, res["measures_all_users"])  # noqa: E731
        res["device_route_ms"], res["timed_outputs_match"] = timed(lambda: algo.top_n_list_measures(n, sim=knn),
                                                                   reps, check)
        res["top_n_inner_ms"], _ = timed(lambda: algo.top_n_inner(n), reps)
        res["list_kernel_ms"], res["list_kernel_pairs"] = list_kernel_ms(algo, knn, n)
        res["list_kernel_sim_sector_bytes"] = 32 * res["list_kernel_pairs"]
        out.append(res)
        print(json.dumps(res), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--shapes", default="ml-1m,ml-20m")
    ap.add_argument("--n", default="10,100")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-pairs", type=float, default=3e7,
                    help="run the definition over every user when it sums at most this many similarity pairs")
    ap.add_argument("--sample", type=int, default=2000, help="users of the fixed sample otherwise")
    a = ap.parse_args()
    nat.torch_cuda()
    report = dict(gpu=gpu_info(), results=[])
    for shape in a.shapes.split(","):
        report["results"] += workload(shape, [int(x) for x in a.n.split(",")], a.reps, a.max_pairs, a.sample)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(report, fh, indent=1)


if __name__ == "__main__":
    main()
