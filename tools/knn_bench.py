#!/usr/bin/env python
"""scema_knn on the bench's c4 and c4s rows, next to scema_compare at the bench threshold and scema_nearest.

  python tools/knn_bench.py --out FILE [--reps 3] [--histories 1000000] [--nearest-rows 200000]

For each workload the rows are generated and resampled on the device as bench.py does, then in the same process:
scema_compare(1e-6) and scema_knn for k = 1 and k = 8, each once to warm up and --reps times timed (host clock around the
call, which ends in a device synchronise), with the stats of the query (rounds, radius per round, rows open after
round 1, survivors, edges, exact pairs). Then scema_nearest and scema_knn(k = 1) on the first --nearest-rows c4 rows, timed the same
way, with their outputs compared (IDs and distance bits). Prints the card name and power limit read in the same call
and writes everything to --out as JSON."""
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


def rows_of(wl_name, n):
    import torch
    import bench
    import scema_b200
    from scema_b200 import synth
    w = bench.WORKLOADS[wl_name]
    hc = scema_b200.HistCluster(0)
    off = synth.device_offsets(bench.SEED, n, bench.CLUSTER, w["lmin"], w["lmax"])
    steps = synth.device_histories(bench.SEED, n, bench.CLUSTER, bench.wl_amp(w), synth.default_pert(bench.THR, w["P"]), off,
                                   device=torch.device("cuda", 0), **bench.wl_model(w))
    hc.set_histories(None, off, device_ptr=steps.data_ptr())
    hc.resample(w["P"])
    torch.cuda.synchronize()
    return hc, steps


def main():
    import numpy as np
    import bench
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--histories", type=int, default=1000000)
    ap.add_argument("--nearest-rows", type=int, default=200000)
    ap.add_argument("--out", required=True, help="JSON file to write")
    args = ap.parse_args()
    res = {"card": card(), "workloads": {}}
    print("card:", res["card"], flush=True)
    for wl in ("c4", "c4s"):
        hc, steps = rows_of(wl, args.histories)
        entry = {"n": args.histories, "compare": timed(lambda: hc.compare(bench.THR), args.reps)}
        entry["compare"]["edges"] = hc.n_edges
        for k in (1, 8):
            t = timed(lambda: hc.knn(k), args.reps)
            t["stats"] = hc.knn_last_stats()
            t["open_after_round1"] = args.histories - t["stats"]["rows_round1"] if t["stats"]["rounds"] else args.histories
            entry[f"knn_k{k}"] = t
        res["workloads"][wl] = entry
        print(wl, json.dumps(entry), flush=True)
        hc.close()
        del steps
    hc, steps = rows_of("c4", args.histories)
    hc.select_rows(np.arange(args.nearest_rows, dtype=np.uint32))
    got = {}

    def nearest():
        got["nearest"] = hc.nearest()

    def knn1():
        got["knn"] = hc.knn(1)

    cmp = {"n": args.nearest_rows, "nearest": timed(nearest, 1), "knn_k1": timed(knn1, args.reps)}
    cmp["knn_k1"]["stats"] = hc.knn_last_stats()
    nid, nd = got["nearest"]
    idx, d = got["knn"]
    ids = np.arange(args.nearest_rows, dtype=np.uint32)
    kid = np.where(idx[:, 0] == 0xffffffff, np.uint32(0xffffffff), ids[np.minimum(idx[:, 0], args.nearest_rows - 1)])
    cmp["ids_equal"] = bool(np.array_equal(kid, nid))
    cmp["diff_bits_equal"] = bool(np.array_equal(d[:, 0].view(np.uint64), nd.view(np.uint64)))
    cmp["speedup"] = cmp["nearest"]["ms_median"] / cmp["knn_k1"]["ms_median"]
    res["nearest_vs_knn1"] = cmp
    print("nearest vs knn(1)", json.dumps(cmp), flush=True)
    hc.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
