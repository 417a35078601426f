"""accuracy.fcp and accuracy.precision_recall_at_k (k=10, threshold=3.5) on the device against the Python code.

Workloads (synthetic, synth.ratings(..., skew=True); est = r_ui + N(0, 0.9) clipped to the scale, string uids as a
file-loaded dataset has them):
  ml1m_fold   one 20 % test fold at the ml-1M shape (200 k predictions)
  ml1m_train  the whole ml-1M-shaped trainset, as cross_validate(return_train_measures=True) scores it (1 M)
  ml20m_fold  one 20 % test fold at the ml-20M shape (4 M)
  long_user   a single user with 50 000 predictions (spans 196 CTAs: the cross-CTA reduction)
Before any time is reported, the device output is checked against the Python code (the three fold workloads) or a
chunked numpy restatement of the counts (long_user, where the Python loop would take minutes).  Reported per
workload: host extraction + grouping time, count-call time from CUDA events, the kernel's own time from
torch.profiler (mean of 5 calls), end-to-end times, the Python times, sum of m^2, pair visits per second of the
kernel and launches per call, with the GPU's name and power limit read in the same run.
One JSON line per workload on stdout; --out FILE writes the whole report.  Nothing is written into the tree.

    python tools/bench_rank_metrics.py [--out FILE] [--only ml1m_fold,long_user]
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

from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import accuracy, synth  # noqa: E402
from surprise_b200.prediction_algorithms.predictions import Prediction  # noqa: E402
from test_rank_metrics_cpu import count_oracle, group  # noqa: E402

K, THRESHOLD = 10, 3.5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi: %s)" % q.stderr.strip()


def predictions(name):
    rng = np.random.default_rng(7)
    if name == "long_user":
        n = 50_000
        u, r = np.zeros(n, dtype=np.int64), rng.integers(1, 11, n) * 0.5
    else:
        nu, ni, nr, step = synth.SHAPES["ml-20m" if name == "ml20m_fold" else "ml-1m"]
        if name == "ml1m_train":
            d = synth.ratings(nu, ni, nr, step=step, seed=0, skew=True)
            u, _, r = d["train"]
        else:   # a 20 % fold: 80 % train, the rest held out
            d = synth.ratings(nu, ni, int(nr * 0.8), step=step, seed=0, holdout=0.25, skew=True)
            u, _, r = d["test"]
    est = np.clip(r + rng.normal(0, 0.9, len(r)), 0.5, 5.0)
    uids = ["u%d" % x for x in u.tolist()]
    return [Prediction(a, None, b, c, None) for a, b, c in zip(uids, r.tolist(), est.tolist())]


def wall(f, reps):
    ts, out = [], None
    for _ in range(reps):
        nat.torch_cuda().cuda.synchronize()
        t0 = time.perf_counter()
        out = f()
        nat.torch_cuda().cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def python_route(f, *args):
    usable, accuracy._device_usable = accuracy._device_usable, lambda: False
    try:
        t0 = time.perf_counter()
        out = f(*args)
        return time.perf_counter() - t0, out
    finally:
        accuracy._device_usable = usable


def same(a, b):
    return type(a) is type(b) and (a == b or (a != a and b != b))


def same_dicts(a, b):
    return list(a) == list(b) and all(same(a[u], b[u]) for u in b)


def bench(name):
    torch = nat.torch_cuda()
    preds = predictions(name)
    n = len(preds)
    # host extraction + grouping (the O(n) pass over the tuples, then the device segment CSR)
    t_host, (keys, code, r_ui, est, _) = wall(lambda: accuracy._exact_columns(preds), 3)
    t_group, (seg_ptr, d_r, d_e) = wall(lambda: accuracy._segments(code, len(keys), r_ui, est), 3)
    m = np.bincount(code, minlength=len(keys))
    sum_m2 = int(np.sum(m.astype(np.int64) ** 2))
    n_seg = len(keys)
    k_eff = nat.to_dev(np.minimum(m, K), np.int64)

    def count_call(mode):
        out = nat.empty_dev((n_seg, 2 if mode == "fcp" else 3), np.int64)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        if mode == "fcp":
            rc = nat.lib().sb2_fcp_counts_dev(n_seg, n, nat.ptr(seg_ptr), nat.ptr(d_r), nat.ptr(d_e), nat.ptr(out),
                                              nat.stream())
        else:
            rc = nat.lib().sb2_precision_at_k_counts_dev(n_seg, n, nat.ptr(seg_ptr), nat.ptr(d_r), nat.ptr(d_e),
                                                         nat.ptr(k_eff), THRESHOLD, nat.ptr(out), nat.stream())
        ev[1].record()
        nat.check(rc)
        ev[1].synchronize()
        return ev[0].elapsed_time(ev[1]) * 1e-3, out

    rep = dict(workload=name, gpu=gpu_info(), predictions=n, users=n_seg, max_user=int(m.max()), sum_m2=sum_m2)
    # correctness first
    nat.lib().sb2_reset_launch_count()
    fcp_dev = accuracy.fcp(preds, verbose=False)
    rep["launches_per_fcp"] = int(nat.lib().sb2_launch_count())
    nat.lib().sb2_reset_launch_count()
    pr_dev = accuracy.precision_recall_at_k(preds, K, THRESHOLD)
    rep["launches_per_precision_recall"] = int(nat.lib().sb2_launch_count())
    if name == "long_user":
        _, gseg, gr, ge = group(preds)
        counts = count_call("fcp")[1].cpu().numpy()
        assert np.array_equal(counts, count_oracle(gseg, gr, ge)), "fcp counts differ from the numpy oracle"
        counts = count_call("precision")[1].cpu().numpy()
        assert np.array_equal(counts, count_oracle(gseg, gr, ge, [min(K, n)], THRESHOLD)), "precision counts differ"
        rep["checked_against"] = "numpy oracle (counts)"
    else:
        rep["python_fcp_s"], fcp_py = python_route(accuracy.fcp, preds, False)
        assert same(fcp_dev, fcp_py), (fcp_dev, fcp_py)
        rep["python_precision_recall_s"], pr_py = python_route(accuracy.precision_recall_at_k, preds, K, THRESHOLD)
        assert same_dicts(pr_dev[0], pr_py[0]) and same_dicts(pr_dev[1], pr_py[1]), "precision_recall differs"
        rep["checked_against"] = "Python code (bit-identical fcp, identical dicts)"
    rep["fcp"] = float(fcp_dev)
    # times
    for mode in ("fcp", "precision"):
        count_call(mode)                                                     # warm
        ts = sorted(count_call(mode)[0] for _ in range(5))
        rep["%s_count_call_ms" % mode] = ts[2] * 1e3
    rep["host_extract_s"], rep["host_group_to_device_s"] = t_host, t_group
    rep["fcp_end_to_end_s"], out = wall(lambda: accuracy.fcp(preds, verbose=False), 3)
    assert same(out, fcp_dev)
    rep["precision_recall_end_to_end_s"], out = wall(lambda: accuracy.precision_recall_at_k(preds, K, THRESHOLD), 3)
    assert same_dicts(out[0], pr_dev[0]) and same_dicts(out[1], pr_dev[1])
    # the kernel alone: device time of rank_metrics_kernel under torch.profiler, in a pass of its own (the count call
    # above also holds the stream-ordered allocation, two memsets and the synchronising read of the offsets check)
    from torch.profiler import ProfilerActivity, profile
    for mode in ("fcp", "precision"):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                count_call(mode)
        kern = [e for e in prof.key_averages() if "rank_metrics_kernel" in e.key]
        assert len(kern) == 1 and kern[0].count == 5, [(e.key, e.count) for e in kern]
        rep["%s_kernel_ms" % mode] = kern[0].device_time_total / kern[0].count * 1e-3
    rep["fcp_pair_visits_per_s"] = sum_m2 / (rep["fcp_kernel_ms"] * 1e-3)
    if "python_fcp_s" in rep:
        rep["fcp_speedup_end_to_end"] = rep["python_fcp_s"] / rep["fcp_end_to_end_s"]
        rep["precision_recall_speedup_end_to_end"] = (rep["python_precision_recall_s"] /
                                                      rep["precision_recall_end_to_end_s"])
    return rep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default="ml1m_fold,ml1m_train,ml20m_fold,long_user")
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
