"""Top-N recommendations on the GPU: scorer, selection and end-to-end time of top_n_inner, end-to-end time of
get_top_n, achieved DFMA/s of the factor scorer against the FP64 data-sheet rate, and the per-pair baseline route
(sb2_mf_predict_dev / the algorithm's _estimate_dev on materialised anti-pairs, then a stable torch sort) on the same
users.  Before any time is reported, top_n_inner's output for all users is compared with the baseline route (items,
est bits, counts), and every timed call's output (top_n_inner arrays, get_top_n dicts) with that checked output.

    python tools/bench_top_n.py [--out RESULT.json] [--workloads svd_f100_ml-1m,...] [--n 10,100,3000]
                                [--baseline-users 1000] [--reps 3]

n = 3000 is past the 2048 entries one selection pass keeps, so it runs two passes per row.

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
from surprise_b200 import synth  # noqa: E402

DFMA_PER_S = 37e12 / 2  # HGX B200 data sheet, one GPU: 37 TFLOP/s FP64


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def trainset(shape):
    d = synth.shaped(shape, seed=0)
    u, i, r = d["train"]
    scale = (1, 5) if shape == "ml-1m" else (0.5, 5.0)
    return sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"], scale, 0)


def baseline(algo, users, width):
    """Per-pair route: every (user, item) pair of `users` through _estimate_dev (sb2_mf_predict_dev for the factor
    models), offset and clipping, rated items to -inf, a stable descending torch sort.  Returns (items, est) of the
    first `width` entries per user, on the device."""
    import torch
    ts = algo.trainset
    n_i = ts.n_items
    ptr, idx, _ = ts.user_csr()
    d_users = nat.to_dev(users, np.int32)
    d_u = d_users.repeat_interleave(n_i)
    d_i = torch.arange(n_i, dtype=torch.int32, device="cuda").repeat(len(users))
    est, _ = algo._estimate_dev(d_u, d_i)
    low, high = ts.rating_scale
    est = torch.clamp(est[:len(d_u)] - ts.offset, low, high).view(len(users), n_i)
    rated_u = np.repeat(np.arange(len(users)), np.diff(ptr)[users])
    rated_i = np.concatenate([idx[ptr[u]:ptr[u + 1]] for u in users])
    est[torch.as_tensor(rated_u, device="cuda"), torch.as_tensor(rated_i.astype(np.int64), device="cuda")] = -np.inf
    order = torch.sort(est, dim=1, descending=True, stable=True).indices[:, :width]
    return order.to(torch.int32), torch.gather(est, 1, order)


def matches_baseline(algo, out, width, chunk_pairs=1 << 26):
    """top_n_inner's output for all users against the per-pair route, user chunk by user chunk: items, est bits and
    count."""
    ts = algo.trainset
    items, est, count = out
    cnt = np.diff(ts.user_csr()[0])
    if not np.array_equal(count, np.minimum(width, ts.n_items - cnt)):
        return False
    chunk = max(1, chunk_pairs // ts.n_items)
    for u0 in range(0, ts.n_users, chunk):
        users = np.arange(u0, min(u0 + chunk, ts.n_users), dtype=np.int32)
        b_i, b_e = baseline(algo, users, width)
        b_i, b_e = b_i.cpu().numpy(), b_e.cpu().numpy()
        valid = np.arange(width)[None, :] < count[users, None]
        if not (np.array_equal(np.where(valid, items[users], -1), np.where(valid, b_i, -1)) and
                np.array_equal(np.where(valid, est[users], 0.0).view(np.int64), np.where(valid, b_e, 0.0).view(np.int64))):
            return False
    return True


def same_arrays(a, b):
    return all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


def dict_matches(top, out):
    """get_top_n's dict against top_n_inner's arrays (raw ids are the inner ids of these trainsets)."""
    items, est, count = out
    keys = np.flatnonzero(count).tolist()
    if list(top.keys()) != keys:
        return False
    return all(top[u] == list(zip(items[u, :count[u]].tolist(), est[u, :count[u]].tolist())) for u in keys)


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
        del o
    return float(np.median(ms)), ok


def workload(name, shape, make, ns, baseline_users, reps):
    ts = trainset(shape)
    if make == "assigned":     # drawn factors: top-N reads pu / qi / bu / bi only
        algo = sb.SVD(n_factors=100)
        sb.AlgoBase.fit(algo, ts)
        rng = np.random.RandomState(0)
        algo.pu, algo.qi = rng.normal(0, .3, (ts.n_users, 100)), rng.normal(0, .3, (ts.n_items, 100))
        algo.bu, algo.bi = rng.normal(0, .3, ts.n_users), rng.normal(0, .3, ts.n_items)
    else:
        algo = make().fit(ts)
    rng = np.random.RandomState(0)
    bl_users = np.sort(rng.choice(ts.n_users, min(baseline_users, ts.n_users), replace=False)).astype(np.int32)
    f = int(getattr(algo, "n_factors", 0)) if algo._top_n_scorer() is not None else 0
    out = []
    for n in ns:
        width = min(n, ts.n_items)
        res = dict(workload=name, shape=shape, n_users=ts.n_users, n_items=ts.n_items, n=n, gpu=gpu_info())
        # correctness first: all users against the per-pair route; every timed output must equal this one
        ref = algo.top_n_inner(n)
        res["matches_baseline"] = matches_baseline(algo, ref, width)
        if not res["matches_baseline"]:
            out.append(res)
            print(json.dumps(res), flush=True)
            continue
        events = []

        def inner():
            events.clear()
            return algo.top_n_inner(n, _events=events)

        sc, se = [], []

        def check_inner(o):
            sc.append(sum(e[0].elapsed_time(e[1]) for e in events))
            se.append(sum(e[1].elapsed_time(e[2]) for e in events))
            return same_arrays(o, ref)

        res["top_n_inner_ms"], res["timed_outputs_match"] = timed(inner, reps, check_inner)
        res.update(blocks=len(events), scorer_ms=float(np.median(sc)), select_ms=float(np.median(se)))
        if f:
            dfma = float(ts.n_users) * ts.n_items * f
            res["dfma_per_s"] = dfma / (res["scorer_ms"] * 1e-3)
            res["dfma_share_of_fp64_datasheet"] = res["dfma_per_s"] / DFMA_PER_S
        if n <= 100:      # get_top_n builds n Python tuples per user
            res["get_top_n_ms"], ok = timed(lambda: algo.get_top_n(n), reps, lambda t: dict_matches(t, ref))
            res["timed_outputs_match"] = res["timed_outputs_match"] and ok
        # the per-pair route on a user sample, warm, extrapolated linearly to all users
        res["baseline_ms"], _ = timed(lambda: baseline(algo, bl_users, width), reps)
        res["baseline_users"] = len(bl_users)
        res["baseline_ms_all_users_extrapolated"] = res["baseline_ms"] * ts.n_users / len(bl_users)
        res["speedup_vs_baseline_all_users"] = res["baseline_ms_all_users_extrapolated"] / res["top_n_inner_ms"]
        out.append(res)
        print(json.dumps(res), flush=True)
    return out


WORKLOADS = {
    "svd_f100_ml-1m": ("ml-1m", lambda: sb.SVD(n_factors=100, n_epochs=2, random_state=0)),
    "svd_f100_ml-20m": ("ml-20m", "assigned"),
    "svdpp_f20_ml-10m": ("ml-10m", lambda: sb.SVDpp(n_factors=20, n_epochs=1, random_state=0)),
    "coclustering_ml-1m": ("ml-1m", lambda: sb.CoClustering(random_state=0)),
    "knnbaseline_item_ml-1m": ("ml-1m", lambda: sb.KNNBaseline(sim_options={"name": "pearson_baseline",
                                                                               "user_based": False})),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--n", default="10,100,3000")
    ap.add_argument("--baseline-users", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    nat.torch_cuda()
    report = dict(gpu=gpu_info(), results=[])
    ns = [int(x) for x in a.n.split(",")]
    for name in a.workloads.split(","):
        shape, make = WORKLOADS[name]
        report["results"] += workload(name, shape, make, ns, a.baseline_users, a.reps)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(report, fh, indent=1)


if __name__ == "__main__":
    main()
