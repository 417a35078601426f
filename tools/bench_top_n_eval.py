"""Top-N measures against a LeaveOneOut split: AlgoBase.top_n_measures (device route) against the dict route,
accuracy.top_n_measures over get_top_n, for SVD f=100 at the ml-1M shape (fitted) and the ml-20M shape (factors drawn,
as tools/bench_top_n.py does: top-N only reads them), n = 10 and 100.

Before any time is reported, the device route's result must equal the dict route's (same keys, same float bits), and
every timed call's result must equal that checked result.  Route times are synchronised wall time, median of --reps
warm calls.  The hit kernel (sb2_top_n_hits_dev over every evaluated user, one launch) is timed with CUDA events around
the call, median of 5 warm calls.  The LeaveOneOut split of the array-backed dataset is timed once per shape.

    python tools/bench_top_n_eval.py [--out RESULT.json] [--shapes ml-1m,ml-20m] [--n 10,100] [--reps 3]

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
from surprise_b200.model_selection import LeaveOneOut  # noqa: E402
from surprise_b200.model_selection.validation import Fold  # noqa: E402


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


def hit_kernel_ms(algo, tes, n):
    """sb2_top_n_hits_dev over every evaluated user of the split in one launch (CUDA events, median of 5 warm calls),
    and the bytes it must read: the rows' items up to the cutoff plus the relevant lists and offsets."""
    import torch
    ts = algo.trainset
    iu, n_rel, rel_ptr, rel_idx = Fold(ts, tes).test_pairs().relevant(None, ts.n_items)
    users = iu[iu >= 0]
    width = min(n, ts.n_items)
    items, _, count = algo._top_n_dev(width, users)
    inv, disc, _ = accuracy._rank_tables(width)
    d_inv, d_disc = nat.to_dev(inv, np.float64), nat.to_dev(disc, np.float64)
    d_ptr, d_idx = nat.to_dev(rel_ptr, np.int64), nat.to_dev(rel_idx, np.int32)
    out = [nat.empty_dev((len(users),), t) for t in (np.int32, np.float64, np.float64)]

    def call():
        nat.check(nat.lib().sb2_top_n_hits_dev(len(users), nat.ptr(items), width, nat.ptr(count), width,
                                               nat.ptr(d_ptr), nat.ptr(d_idx), len(rel_idx), nat.ptr(d_inv),
                                               nat.ptr(d_disc), *(nat.ptr(o) for o in out), nat.stream()))

    call()
    ms = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    read = len(users) * (width * 4 + 4 + 8) + rel_idx.nbytes
    return float(np.median(ms)), read


def workload(shape, ns, reps):
    if shape == "ml-1m":
        d = synth.ratings(*synth.SHAPES["ml-1m"][:3], seed=0)
        scale = (1, 5)
    else:
        d = synth.shaped(shape, seed=0)
        scale = (0.5, 5.0)
    u, i, r = d["train"]
    data = sb.Dataset.load_from_arrays(u, i, r, sb.Reader(rating_scale=scale))
    t = time.perf_counter()
    trs, tes = next(LeaveOneOut(1, random_state=0).split(data))
    split_s = time.perf_counter() - t
    if shape == "ml-1m":
        algo = sb.SVD(n_factors=100, random_state=0).fit(trs)
    else:     # drawn factors: top-N reads pu / qi / bu / bi only
        algo = sb.SVD(n_factors=100)
        sb.AlgoBase.fit(algo, trs)
        rng = np.random.RandomState(0)
        algo.pu, algo.qi = rng.normal(0, .3, (trs.n_users, 100)), rng.normal(0, .3, (trs.n_items, 100))
        algo.bu, algo.bi = rng.normal(0, .3, trs.n_users), rng.normal(0, .3, trs.n_items)
    out = []
    for n in ns:
        res = dict(shape=shape, n=n, n_users=trs.n_users, n_items=trs.n_items, n_ratings=trs.n_ratings,
                   held_out=len(tes), leave_one_out_split_s=split_s, gpu=gpu_info())
        want = accuracy.top_n_measures(algo.get_top_n(n), tes, n, offset=trs.offset, verbose=False)
        got = algo.top_n_measures(tes, n)
        res["equal_to_definition"] = same_result(got, want)
        res["measures"] = got
        if not res["equal_to_definition"]:
            res["definition"] = want
            out.append(res)
            print(json.dumps(res), flush=True)
            continue
        res["device_route_ms"], ok1 = timed(lambda: algo.top_n_measures(tes, n), reps, lambda o: same_result(o, want))
        res["dict_route_ms"], ok2 = timed(lambda: accuracy.top_n_measures(algo.get_top_n(n), tes, n, offset=trs.offset,
                                                                           verbose=False),
                                          reps, lambda o: same_result(o, want))
        res["timed_outputs_match"] = ok1 and ok2
        res["top_n_inner_ms"], _ = timed(lambda: algo.top_n_inner(n), reps)
        res["hit_kernel_ms"], res["hit_kernel_bytes_read"] = hit_kernel_ms(algo, tes, n)
        res["speedup_vs_dict_route"] = res["dict_route_ms"] / res["device_route_ms"]
        out.append(res)
        print(json.dumps(res), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--shapes", default="ml-1m,ml-20m")
    ap.add_argument("--n", default="10,100")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    nat.torch_cuda()
    report = dict(gpu=gpu_info(), results=[])
    for shape in a.shapes.split(","):
        report["results"] += workload(shape, [int(x) for x in a.n.split(",")], a.reps)
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(report, fh, indent=1)


if __name__ == "__main__":
    main()
