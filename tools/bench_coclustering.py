"""CoClustering fit on the GPU: wall time (Python API and resident device arrays), per-kernel time, launches per fit,
algorithmic bytes per pass against HBM bandwidth and the longest ordered chain, and the C oracle's single-core time.
Every device result is compared with the oracle bit for bit at the timed sizes.

    python tools/bench_coclustering.py [--out RESULT.json] [--reps 5] [--no-oracle-20m]

One JSON line per shape goes to stdout; --out also writes the whole report to a file.
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

import coclustering_oracle  # noqa: E402
import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import synth  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def pass_bytes(nnz, n_seg, n_other):
    """Bytes one assignment pass has to move at least: the CSR entries (int32 index + int32 truncated rating), the
    segment offsets / means / new clusters, and the other side's clusters and means read once."""
    return nnz * 8 + (n_seg + 1) * 8 + n_seg * 12 + n_other * 12


def run_shape(name, n_cu, n_ci, n_epochs, reps, with_oracle):
    import torch
    d = synth.shaped(name)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"])
    up, ui, ur = ts.user_csr()
    ip, iu, ir = ts.item_csr()
    nnz = len(ur)
    res = dict(shape=name, n_users=ts.n_users, n_items=ts.n_items, n_ratings=nnz, n_cltr_u=n_cu, n_cltr_i=n_ci,
               n_epochs=n_epochs, longest_user=int(np.diff(up).max()), longest_item=int(np.diff(ip).max()))

    # Python API, synchronised (includes means, uploads, downloads)
    sb.CoClustering(n_cu, n_ci, n_epochs, random_state=0).fit(ts)  # warm-up
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        algo = sb.CoClustering(n_cu, n_ci, n_epochs, random_state=0).fit(ts)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t)
    res["fit_python_api_s"] = sorted(times)[len(times) // 2]
    res["fit_python_api_all_s"] = times

    # resident device arrays: the C-ABI fit alone (it ends with its own stream synchronisation)
    rng = np.random.RandomState(0)
    cu0 = nat.to_dev(rng.randint(n_cu, size=ts.n_users), np.int32)
    ci0 = nat.to_dev(rng.randint(n_ci, size=ts.n_items), np.int32)
    dev = dict(up=nat.to_dev(up, np.int64), ui=nat.to_dev(ui, np.int32), ur=nat.to_dev(ur, np.float64),
               ip=nat.to_dev(ip, np.int64), iu=nat.to_dev(iu, np.int32), ir=nat.to_dev(ir, np.float64),
               um=nat.to_dev(algo.user_mean, np.float64), im=nat.to_dev(algo.item_mean, np.float64))
    cu, ci = cu0.clone(), ci0.clone()
    au, ai = nat.empty_dev((n_cu,), np.float64), nat.empty_dev((n_ci,), np.float64)
    ac = nat.empty_dev((n_cu, n_ci), np.float64)

    def fit_resident():
        cu.copy_(cu0)
        ci.copy_(ci0)
        nat.check(nat.lib().sb2_coclustering_fit_dev(
            ts.n_users, ts.n_items, nnz, nat.ptr(dev["up"]), nat.ptr(dev["ui"]), nat.ptr(dev["ur"]), nat.ptr(dev["ip"]),
            nat.ptr(dev["iu"]), nat.ptr(dev["ir"]), nat.ptr(dev["um"]), nat.ptr(dev["im"]), float(ts.global_mean),
            n_cu, n_ci, n_epochs, nat.ptr(cu), nat.ptr(ci), nat.ptr(au), nat.ptr(ai), nat.ptr(ac), nat.stream()))

    fit_resident()
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fit_resident()
        times.append(time.perf_counter() - t)
    res["fit_resident_s"] = sorted(times)[len(times) // 2]
    res["fit_resident_all_s"] = times
    nat.lib().sb2_reset_launch_count()
    fit_resident()
    res["launches_per_fit"] = int(nat.lib().sb2_launch_count())

    # per-kernel device time over one resident fit, in a run of the profiler of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fit_resident()
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        if "cc_" in ev.key:
            tag = ("user_pass" if "cc_assign_kernel<false>" in ev.key else "item_pass" if "cc_assign_kernel<true>"
                   in ev.key else ev.key.split("(")[0].replace("void sb2::", ""))
            dt = getattr(ev, "device_time_total", None)
            if dt is None:
                dt = ev.cuda_time_total
            kernels[tag] = dict(count=ev.count, total_us=dt, mean_us=dt / max(ev.count, 1))
    res["kernels"] = kernels
    for side, n_seg, n_other, longest in (("user_pass", ts.n_users, ts.n_items, res["longest_user"]),
                                          ("item_pass", ts.n_items, ts.n_users, res["longest_item"])):
        if side in kernels:
            b = pass_bytes(nnz, n_seg, n_other)
            t = kernels[side]["mean_us"] * 1e-6
            kernels[side].update(algorithmic_bytes=b, hbm_bound_us=b / HBM_BYTES_PER_S * 1e6,
                                 hbm_share=b / HBM_BYTES_PER_S / t, longest_segment=longest,
                                 ns_per_entry_of_longest_chain=t * 1e9 / longest)

    # bit-exactness at the timed size, and the oracle's time on one host core
    if with_oracle:
        rng = np.random.RandomState(0)
        cu_h, ci_h = rng.randint(n_cu, size=ts.n_users), rng.randint(n_ci, size=ts.n_items)
        t = time.perf_counter()
        want = coclustering_oracle.fit(ts.n_users, ts.n_items, (up, ui, ur), (ip, iu, ir), algo.user_mean,
                                       algo.item_mean, ts.global_mean, n_cu, n_ci, n_epochs, cu_h, ci_h)
        res["oracle_fit_one_core_s"] = time.perf_counter() - t
        got = (algo.cltr_u, algo.cltr_i, algo.avg_cltr_u, algo.avg_cltr_i, algo.avg_cocltr)
        res["bit_identical_to_oracle"] = all(np.array_equal(g, w) for g, w in zip(got, want))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the whole report (JSON) to this file")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-oracle-20m", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_coclustering needs a CUDA device")
    out = dict(gpu=gpu_info(), host_cpu_count=os.cpu_count(), oracle_threads=1, results=[])
    for name, n_cu, n_ci, with_oracle in (("ml-1m", 3, 3, True), ("ml-1m", 50, 50, True),
                                          ("ml-20m", 3, 3, not a.no_oracle_20m)):
        r = run_shape(name, n_cu, n_ci, 20, a.reps, with_oracle)
        print(json.dumps(r), flush=True)
        out["results"].append(r)
    out["gpu_after"] = gpu_info()
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)
        print("wrote", a.out)


if __name__ == "__main__":
    main()
