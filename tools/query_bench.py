#!/usr/bin/env python
"""scema_query_compare / scema_query_knn against the bench's 10^6 c4 rows, next to today's workaround (scema_compare on
the concatenation [Q; R]) and scema_compare on R alone.

  python tools/query_bench.py --out FILE [--reps 3] [--histories 1000000] [--queries 1000,10000,100000,1000000]

R is generated and resampled on the device as bench.py does. The queries are half rows of R perturbed far below the
threshold (the same population) and half c4 histories of another seed, resampled on a second context; they stay on the
device and are passed by pointer. For every query count m, in the same process: query_compare(1e-6), query_knn at k = 1
and k = 8 (and k = 8 on the exact top-k kernel alone, up to 10^10 pairs), scema_compare on [Q; R] and on R alone, each
once to warm up and --reps times timed (host clock around the call, which ends in a device synchronise; median, min,
max). Each query call is split into its phases with the stats of
the call (CUDA events: scratch copy [Q; R], operand prep, filter, exact recompute, sort, compaction / selection, exact
top-k kernel). Prints the card name, power limit and max SM clock read in the same call and writes everything to --out
as JSON."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:
        out = f"nvidia-smi unavailable ({e})"
    return out


def timed(fn, reps):
    fn()
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ms.append(1000.0 * (time.perf_counter() - t0))
    return {"ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms), "reps": reps}


def spline_of(seed, n, w):
    import torch
    import bench
    import scema_b200
    from scema_b200 import synth
    hc = scema_b200.HistCluster(0)
    off = synth.device_offsets(seed, n, bench.CLUSTER, w["lmin"], w["lmax"])
    steps = synth.device_histories(seed, n, bench.CLUSTER, bench.wl_amp(w), synth.default_pert(bench.THR, w["P"]), off,
                                   device=torch.device("cuda", 0), **bench.wl_model(w))
    hc.set_histories(None, off, device_ptr=steps.data_ptr())
    hc.resample(w["P"])
    torch.cuda.synchronize()
    del steps
    return hc


def main():
    import numpy as np
    import torch
    import bench
    import scema_b200
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--histories", type=int, default=1000000)
    ap.add_argument("--queries", default="1000,10000,100000,1000000")
    ap.add_argument("--out", required=True, help="JSON file to write")
    args = ap.parse_args()
    sizes = [int(x) for x in args.queries.split(",")]
    res = {"card": card(), "n": args.histories, "threshold": bench.THR, "queries": {}}
    print("card:", res["card"], flush=True)
    w = bench.WORKLOADS["c4"]
    hc = spline_of(bench.SEED, args.histories, w)
    n, K, r_ptr = hc.spline_info()
    R = torch.empty((n, K), dtype=torch.float64, device="cuda")
    R.copy_(torch.from_numpy(hc.get_spline()))
    mmax = max(sizes)
    other = spline_of(bench.SEED + 1, mmax - mmax // 2, w)
    g = torch.Generator(device="cuda").manual_seed(7)
    pick = torch.randint(0, n, (mmax // 2,), device="cuda", generator=g)
    near = R[pick] + 2e-9 * torch.randn((mmax // 2, K), dtype=torch.float64, device="cuda", generator=g)
    Qall = torch.empty((mmax, K), dtype=torch.float64, device="cuda")
    Qall[0::2] = near
    Qall[1::2] = torch.from_numpy(other.get_spline()).cuda()
    other.close()
    torch.cuda.synchronize()
    res["compare_R"] = timed(lambda: hc.compare(bench.THR), args.reps)
    res["compare_R"]["edges"] = hc.n_edges
    res["compare_R"]["counters"] = hc.counters()
    print("compare R", json.dumps(res["compare_R"]), flush=True)
    cat_ctx = scema_b200.HistCluster(0)
    for m in sizes:
        Q = Qall[:m].contiguous()
        torch.cuda.synchronize()
        e = {"m": m}
        out = {}

        def qc():
            out["qc"] = hc.query_compare(None, bench.THR, device_ptr=Q.data_ptr(), m=m)

        e["query_compare"] = timed(qc, args.reps)
        e["query_compare"]["stats"] = hc.query_last_stats()
        e["query_compare"]["edges"] = len(out["qc"][0])
        for k in (1, 8):
            t = timed(lambda: hc.query_knn(None, k, device_ptr=Q.data_ptr(), m=m), args.reps)
            t["stats"] = hc.query_last_stats()
            e[f"query_knn_k{k}"] = t
        if m * n <= 10 ** 10:   # the exact top-k kernel on every query: the other side of KNN_QUERY_EXACT_PAIRS
            t = timed(lambda: hc.query_knn(None, 8, scema_b200.PAIRS_EXACT, device_ptr=Q.data_ptr(), m=m), args.reps)
            t["stats"] = hc.query_last_stats()
            t["pairs_per_s"] = m * n / (t["ms_median"] * 1e-3)
            e["query_knn_k8_exact_kernel"] = t
        cat = torch.cat([Q, R])
        torch.cuda.synchronize()
        cat_ctx.set_spline(device_ptr=cat.data_ptr(), n=m + n, k=K)
        e["compare_concat"] = timed(lambda: cat_ctx.compare(bench.THR), args.reps)
        a, b, d = cat_ctx.get_edges()
        keep = (a < m) & (b >= m)
        j, i, dq = out["qc"]
        e["compare_concat"]["edges"] = int(len(a))
        e["compare_concat"]["counters"] = cat_ctx.counters()
        e["cross_list_equal"] = bool(np.array_equal(a[keep], j) and np.array_equal(b[keep] - m, i)
                                     and np.array_equal(d[keep].view(np.uint64), dq.view(np.uint64)))
        e["speedup_vs_concat"] = e["compare_concat"]["ms_median"] / e["query_compare"]["ms_median"]
        del cat
        res["queries"][str(m)] = e
        print(m, json.dumps(e), flush=True)
    cat_ctx.close()
    hc.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
