#!/usr/bin/env python
"""The tcgen05 filter kernel alone, 64-column one-slice copies vs projected 16-column copies, on the bench's c4 and c4s
rows and on isotropic rows generated from a seed.

  python tools/filter_ab.py [--rounds 3] [--min-seconds 1.0] [--histories 1000000] [--out FILE]

Every (workload, filter) runs in a process of its own (SCEMA_TC_SLICES=1 / 3 pins the filter; "auto" lets the survivor
sample choose), alternated round by round. One warm-up compare builds the operand copies; then compare is repeated on
the same rows (the copies are reused) until the CUDA-event time of the filter launch alone adds up to --min-seconds.
Prints the card name and power limit read in the same call, the filter time per (workload, filter), the executed tensor
FLOP/s and the per-tile cycle budget of the MMA (dense fp16 rate) against the epilogue's TMEM reads (861 B/clk/SM,
profiles/r02_tmem_probe.json) next to the measured cycles per tile."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ISO_SEED = 77
ISO_SIGMA = 1e-3
MODES = {"1": "64 columns, one slice", "3": "projected, 16 columns", "auto": "survivor sample decides"}


def one(wl, n, min_s):
    import torch
    import bench
    import scema_b200
    from scema_b200 import synth
    dev = torch.device("cuda", 0)
    hc = scema_b200.HistCluster(0)
    if wl == "iso":
        g = torch.Generator(device=dev)
        g.manual_seed(ISO_SEED)
        rows = torch.randn((n, 60), generator=g, device=dev, dtype=torch.float64) * ISO_SIGMA
        hc.set_spline(device_ptr=rows.data_ptr(), n=n, k=60)
        thr = 0.5 * math.sqrt(120.0) * ISO_SIGMA   # half the typical distance: |z_a - z_b| keeps ~11/60 of it
        k = 60
    else:
        w = bench.WORKLOADS[wl]
        off = synth.device_offsets(bench.SEED, n, bench.CLUSTER, w["lmin"], w["lmax"])
        steps = synth.device_histories(bench.SEED, n, bench.CLUSTER, bench.wl_amp(w), synth.default_pert(bench.THR, w["P"]), off,
                                       device=dev, **bench.wl_model(w))
        hc.set_histories(None, off, device_ptr=steps.data_ptr())
        hc.resample(w["P"])
        thr = bench.THR
        k = 6 * w["P"]
    torch.cuda.synchronize()
    hc.compare(thr)
    prep_ms = hc.timings()["prep"]
    sampler = bench.ClockSampler(0)
    sampler.start()
    times = []
    while sum(times) < 1000.0 * min_s:
        hc.compare(thr)
        times.append(hc.timings()["filter"])
    clocks = sampler.stop()
    c, plan = hc.counters(), hc.tc_last_plan()
    hc.close()
    return {"workload": wl, "n": n, "k": k, "reps": len(times), "filter_ms_median": statistics.median(times),
            "filter_ms_min": min(times), "filter_ms_max": max(times), "prep_ms": prep_ms, "survivors": c["survivors"],
            "tc_slices": c["tc_slices"], "projected": plan["projected_chosen"], "plan": plan, "clocks": clocks}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:
        out = f"nvidia-smi unavailable ({e})"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--one", nargs=2, metavar=("WORKLOAD", "MODE"))
    ap.add_argument("--workloads", default="c4,c4s,iso")
    ap.add_argument("--modes", default="1,3,auto")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--histories", type=int, default=1000000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if args.one:
        print(json.dumps(one(args.one[0], args.histories, args.min_seconds)))
        return
    print("card:", card(), flush=True)
    runs = []
    modes = args.modes.split(",")
    for r in range(args.rounds):
        order = modes if r % 2 == 0 else modes[::-1]
        for wl in args.workloads.split(","):
            for mode in order:
                env = dict(os.environ)
                env.pop("SCEMA_TC_SLICES", None)
                if mode != "auto":
                    env["SCEMA_TC_SLICES"] = mode
                t0 = time.time()
                p = subprocess.run([sys.executable, __file__, "--one", wl, mode, "--histories", str(args.histories),
                                    "--min-seconds", str(args.min_seconds)], env=env, capture_output=True, text=True)
                if p.returncode != 0:
                    print(p.stdout[-2000:], p.stderr[-4000:], file=sys.stderr)
                    raise SystemExit(f"filter_ab: {wl} / {mode} failed")
                res = json.loads(p.stdout.strip().splitlines()[-1])
                res.update(mode=mode, round=r)
                runs.append(res)
                print(f"round {r} {wl:4s} {MODES[mode]:26s} filter {res['filter_ms_median']:8.3f} ms (min {res['filter_ms_min']:.3f}, "
                      f"max {res['filter_ms_max']:.3f}, {res['reps']} reps) prep {res['prep_ms']:.3f} ms survivors {res['survivors']} "
                      f"projected={res['projected']} sm {res['clocks'].get('sm_mhz')} MHz {res['clocks'].get('reasons')} "
                      f"[{time.time() - t0:.0f} s]", flush=True)
    # summary: executed flops and per-tile cycles (a 256 x 256 tile is one MMA group of a CTA pair: 128 rows per SM)
    summary = {}
    for wl in args.workloads.split(","):
        for mode in modes:
            rs = [x for x in runs if x["workload"] == wl and x["mode"] == mode]
            if not rs:
                continue
            ms = statistics.median(x["filter_ms_median"] for x in rs)
            kexec = 16 if rs[0]["projected"] else 64
            nt = (rs[0]["n"] + 255) // 256
            tiles = nt * (nt + 1) // 2
            mhz = statistics.median(x["clocks"]["sm_mhz"] for x in rs if x["clocks"].get("sm_mhz")) if any(
                x["clocks"].get("sm_mhz") for x in rs) else None
            flops = tiles * 256.0 * 256.0 * kexec * 2.0
            row = {"filter_ms": ms, "spread_ms": [min(x["filter_ms_median"] for x in rs), max(x["filter_ms_median"] for x in rs)],
                   "k_executed": kexec, "tiles": tiles, "executed_tflops": flops / (ms * 1e-3) / 1e12, "sm_mhz": mhz,
                   "mma_cycles_per_tile": 128.0 * 256.0 * kexec / 4096.0,       # 128 x 256 x K MACs per SM, 4096 fp16 MAC/clk/SM
                   "epilogue_cycles_per_tile": 128.0 * 256.0 * 4.0 / 861.0,    # 128 x 256 fp32 per SM from TMEM at 861 B/clk
                   "projected": rs[0]["projected"], "survivors": rs[0]["survivors"]}
            if mhz:
                row["measured_cycles_per_tile"] = ms * 1e-3 * mhz * 1e6 * 74 / tiles
            summary[f"{wl}/{mode}"] = row
            print(f"{wl}/{mode}: " + json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"card": card(), "runs": runs, "summary": summary}, f, indent=1)


if __name__ == "__main__":
    main()
