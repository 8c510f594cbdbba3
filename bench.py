#!/usr/bin/env python
"""bench.py — history pair comparisons / second of the MD-redundancy clustering hot path.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (+ DIR/<name>.npy: results of the last timed step)

A "step" is one pass of the hot path over the synthetic batch: K1 ragged spline resample of every
history -> (N>1: one NCCL all-gather of the resampled rows) -> K2 all-pairs GEMM-form filter (tcgen05
split-fp16 tensor-core filter; --variant dmma selects the FP64 DMMA filter)
+ exact recompute of the survivors -> K3 edge compaction -> canonical sort (-> N>1: all-gather of
the edge counts). Workload (BASELINE.json configs[3], the one the 1/2/4/8 scaling is quoted on; it
fits one GPU): 1M histories x 6 components x 10 spline points, all-pairs = 5.0e11 unordered pairs,
tile-sharded over the ranks (strong scaling: total work fixed). `value` = pairs / second over the
whole job with the raw histories resident in HBM; `e2e` = the same through the C ABI with HOST
buffers (pinned host -> device copy of the histories and device -> host read of the edge list
inside the timed region).

The reference arm (--impl reference) times the reference's own CPU code (oracle/_ref, the
unmodified header compiled with -O2 and OpenMP over rows) on a bounded sample of the same
workload, on all host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

THR = 1e-6
AMP = 5e-3
CLUSTER = 16
SEED = 4
WORKLOADS = {
    # name: n, spline points, raw history length range (model 0 = cluster population of include/scema_synth.h)
    "c2": dict(n=16384, P=10, lmin=8, lmax=64, desc="BASELINE configs[1]: 16k histories x 6 x 10"),
    "c3": dict(n=200000, P=10, lmin=6, lmax=200, desc="BASELINE configs[2]: 200k ragged histories (6..200 steps)"),
    "c4": dict(n=1000000, P=10, lmin=8, lmax=64, desc="BASELINE configs[3]: 1M histories x 6 x 10 spline points"),
    "c5": dict(n=4000000, P=50, lmin=8, lmax=64, desc="BASELINE configs[4]: 4M histories x 6 x 50 spline points"),
    # production shape (SURVEY 8d C1; reference input_configurations/inputs_dogbone_cuboid.json, FE_problem.h:1091-1103):
    # every quadrature point on nearly the same stretch path (model 1: 2 % stretch, groups of 16 symmetric points
    # 0.5 % of the norm apart), all histories equally long
    "c4s": dict(n=1000000, P=10, lmin=36, lmax=36, model=1, amp=2e-2, spread=5e-3,
                desc="production-shaped: 1M histories on one common stretch path (dogbone emulation), 36 steps each, x 6 x 10 spline points"),
}


def wl_model(wl):
    return dict(model=wl.get("model", 0), spread=wl.get("spread", 0.0))


def wl_amp(wl):
    return wl.get("amp", AMP)


def wl_config(wl, wl_name):
    """The workload as both arms print it (identical keys and values: the driver compares the two config objects)."""
    return {"workload": f"{wl_name}: {wl['desc']}", "histories": wl["n"], "spline_points": wl["P"], "threshold": THR,
            "raw_steps_per_history": [wl["lmin"], wl["lmax"]], "cluster_size": CLUSTER, "population_model": wl.get("model", 0),
            "l2": "inputs (raw histories + spline matrix) larger than L2"}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v == "Active":
                    reasons.add(nm)
        busy = [x for x in sm if x > 300] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ------------------------------------------------------------------------------------------------
def cpu_reference_rows(wl, m, timed):
    """First m histories of the workload, generated with the numpy twin and resampled by the
    reference's own splinify. -> (rows, lib, kind, splinify_seconds)."""
    from scema_b200 import synth
    from oracle.pyoracle import Oracle, Reference, have_reference
    if have_reference():
        lib, kind = Reference(), "reference"
    else:
        lib, kind = Oracle(), "port"
    off = synth.offsets(SEED, m, CLUSTER, wl["lmin"], wl["lmax"])
    steps = synth.histories(SEED, m, CLUSTER, wl_amp(wl), synth.default_pert(THR, wl["P"]), off, **wl_model(wl))
    t0 = time.perf_counter()
    rows = lib.splinify_batch(steps, off, wl["P"], host_threads())
    return rows, lib, kind, time.perf_counter() - t0


def host_threads():
    """All host cores this process may use. Asked for explicitly: torch.distributed.run exports OMP_NUM_THREADS=1
    to every rank, which would silently turn the CPU arm into a single-core run."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_pairs_step(lib, rows, r0, r1):
    t0 = time.perf_counter()
    edges, pairs = lib.all_pairs(rows, THR, r0, r1, host_threads(), count_only=True)
    return pairs, time.perf_counter() - t0, edges


def cpu_pairs_step_threads(lib, rows, r0, r1, nthreads):
    t0 = time.perf_counter()
    edges, pairs = lib.all_pairs(rows, THR, r0, r1, nthreads, count_only=True)
    return pairs, time.perf_counter() - t0, edges


def run_reference(args, wl, wl_name):
    rank = env_int("RANK", 0)
    if rank != 0:
        return  # the CPU reference runs once, on rank 0
    m = min(wl["n"], 65536)
    rows, lib, kind, t_spl = cpu_reference_rows(wl, m, True)
    cores = host_threads()
    # calibrate the per-step sample: whole run ~ 100 s at most
    pairs, dt, _ = cpu_pairs_step(lib, rows, 0, 64)
    rate = pairs / dt
    budget = max(1.0, min(8.0, 100.0 / (args.steps + args.warmup)))
    rows_per_step = int(max(16, min(m // 2, rate * budget / m)))
    cursor = 0

    def one():
        nonlocal cursor
        if cursor + rows_per_step >= m // 2:
            cursor = 0
        r = cpu_pairs_step(lib, rows, cursor, cursor + rows_per_step)
        cursor += rows_per_step
        return r

    for _ in range(args.warmup):
        one()
    tot_p, tot_t = 0, 0.0
    for _ in range(args.steps):
        p, t, _ = one()
        tot_p += p
        tot_t += t
    value = tot_p / tot_t
    sample = (f"first {m} of {wl['n']} histories (numpy twin of the generator, resampled by the reference's "
              f"splinify: {m / t_spl:.0f} histories/s); each step = rows [r, r+{rows_per_step}) against all later "
              f"rows = {tot_p // args.steps} pairs; compare_L2_norm + strict threshold, OpenMP over rows")
    line = {
        "impl": "reference", "metric": "history pair comparisons/sec", "value": value, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": wl_config(wl, wl_name),
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
# verification of the measured path (after the timed regions; the oracle is only ever the checker)
# ------------------------------------------------------------------------------------------------
def edge_checksums(a, b, d, n):
    """Order-independent fingerprints of an edge list: the same for any number of shards iff the union is the same."""
    keys = a.astype(np.uint64) * np.uint64(n) + b.astype(np.uint64)
    with np.errstate(over="ignore"):
        ck = int(np.sum(keys, dtype=np.uint64))
    cd = int(np.bitwise_xor.reduce(np.ascontiguousarray(d, dtype=np.float64).view(np.uint64))) if len(d) else 0
    return {"edges": int(len(a)), "sum_keys_mod_2_64": ck, "xor_distance_bits": cd}


DUMP_EDGES = 3 << 19   # 1.5 Mi edges x 4 arrays x 8 bytes = 48 MiB
DUMP_ROWS = 4096


class DeviceRows:
    """A [n, k] float64 matrix in device memory owned by the library, visible to torch without a copy."""

    def __init__(self, ptr, n, k):
        self.__cuda_array_interface__ = {"shape": (n, k), "typestr": "<f8", "data": (ptr, False), "strides": None,
                                         "version": 3}


def dump_outputs(out_dir, a, b, d, rows):
    """--dump-outputs: the edge list (a, b, d) and the resampled rows (a [n, K] float64 CUDA tensor) as float64 .npy
    files in out_dir. Longer lists and larger matrices are represented by fixed samples (seed 0) whose positions are
    stored beside them, so that two builds given the same arguments can be compared file for file. At most 58 MiB
    (K = 300)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    m, n = len(a), rows.shape[0]
    rng = np.random.default_rng(0)
    pos = np.sort(rng.choice(m, DUMP_EDGES, replace=False)) if m > DUMP_EDGES else np.arange(m)
    ridx = np.sort(rng.choice(n, DUMP_ROWS, replace=False)) if n > DUMP_ROWS else np.arange(n)
    sample = rows[torch.from_numpy(ridx).to(rows.device)].cpu().numpy()
    out = {"edge_count": np.array([m]), "edge_sample_position": pos, "edge_a": a[pos], "edge_b": b[pos],
           "edge_distance": d[pos], "spline_row_index": ridx, "spline_rows": sample}
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(arr, dtype=np.float64))


def verify_run(args, hc, sc, world, rank, dev, n, P, variant, stream_mode, level, gloo=None):
    """One more, untimed, pass of exactly the path that was timed (same context, same variant, same sharding), then:
      (i)   every rank's list sorted and unique; the union of the ranks' lists unique;
      (ii)  EVERY emitted edge re-derived on the CPU by direct differences in the reference's order (oracle.check_edges:
            distance bits and strict threshold);
      (iii) completeness: `rows` random complete rows of the pair matrix recomputed on the CPU, no edge missing or extra;
      (iv)  N > 1: the union of the shards == the list ONE GPU produces for the whole matrix (ids, order, distance bits);
            N = 1: the FP64 DMMA filter on the first 200k histories == the same sub-matrix of the tcgen05 list;
      (v)   level "full" (config 5): 64 random 1024 x 1024 tiles of the pair matrix recomputed on the CPU.
    -> dict for the JSON line (rank 0), None elsewhere."""
    import torch
    import scema_b200
    from scema_b200.distributed import gather_edges
    from oracle.pyoracle import Oracle
    t0 = time.perf_counter()
    got = []

    def vsink(a, b, d):
        got.append((a, b, d))

    if world > 1:
        if getattr(sc, "side_group", None) is not None and not stream_mode:
            ne, counts, offs, full = sc.run_overlapped(n, P, THR)   # the path that was timed
        else:
            ne, counts, offs, full = sc.run(n, P, THR, variant, sink=vsink if stream_mode else None)
    else:
        hc.resample(P)
        ne = hc.compare_stream(THR, vsink, variant) if stream_mode else hc.compare(THR, variant)
        counts, full = [ne], None
    if stream_mode:
        a, b, d = (np.concatenate([g[k] for g in got]) if got else np.zeros(0, dtype=(np.uint32, np.uint32, np.float64)[k]) for k in range(3))
    else:
        a, b, d = hc.get_edges()
    key = a.astype(np.int64) * n + b
    local_ok = bool(len(a) == ne and np.all(a < b) and np.all(np.diff(key) > 0))
    if world > 1:
        flags = torch.tensor([int(local_ok)], dtype=torch.int64, device=dev)
        torch.distributed.all_reduce(flags, op=torch.distributed.ReduceOp.MIN)
        local_ok = bool(flags.item())
        A, B, D = gather_edges(a, b, d, n, counts, dev)
    else:
        A, B, D = a, b, d
    if rank != 0:
        if world > 1:
            torch.distributed.barrier(group=gloo)   # host-side wait: rank 0's CPU checks may take minutes
        return None
    out = {"level": level, "per_rank_lists_sorted_unique": local_ok, "per_rank_edges": [int(c) for c in counts]}
    out.update(edge_checksums(A, B, D, n))
    ukey = A.astype(np.int64) * n + B
    out["union_unique"] = bool(np.all(np.diff(ukey) > 0))
    n_rows, K, ptr = hc.spline_info()
    rows = full.cpu().numpy() if full is not None else hc.get_spline()
    o = Oracle()
    out["cpu_recheck_bad_edges"] = int(o.check_edges(rows, THR, A, B, D, host_threads()))
    rng = np.random.default_rng(12345)
    # complete rows in random blocks of 16 consecutive rows (the oracle threads over the rows of a call), within a time budget
    n_check = 208 if level != "full" else 1008
    bad_rows, done_rows, t_rows = 0, 0, time.perf_counter()
    budget = 60.0 if level != "full" else 240.0
    for r0 in rng.choice(max(n - 16, 1), size=min(n_check // 16, max(n - 16, 1)), replace=False).tolist():
        r1 = min(n, r0 + 16)
        ei, ej, ed, _ = o.all_pairs(rows, THR, r0, r1, host_threads())
        lo, hi = np.searchsorted(A, r0), np.searchsorted(A, r1)
        if not (np.array_equal(A[lo:hi], ei) and np.array_equal(B[lo:hi], ej) and np.array_equal(D[lo:hi].view(np.uint64), ed.view(np.uint64))):
            bad_rows += r1 - r0
        done_rows += r1 - r0
        if time.perf_counter() - t_rows > budget:
            break
    out["complete_rows_checked"] = int(done_rows)
    out["complete_rows_bad"] = int(bad_rows)
    if level == "full":
        # the filter-free exact kernel against the tcgen05 list on the first rows (1/16 of the pairs at 4M histories)
        m16 = min(n, 1000000)
        hc.set_spline(device_ptr=(full.data_ptr() if full is not None else ptr), n=m16, k=K)
        hc.compare(THR, scema_b200.PAIRS_EXACT)
        ax, bx, dx = hc.get_edges()
        hx = np.searchsorted(A, m16)
        selx = B[:hx] < m16
        out["exact_kernel_equals_on_first_rows"] = bool(np.array_equal(ax, A[:hx][selx]) and np.array_equal(bx, B[:hx][selx]) and
                                                        np.array_equal(dx.view(np.uint64), D[:hx][selx].view(np.uint64)))
        out["exact_kernel_rows"] = int(m16)
        bad_tiles, T = 0, 1024
        nt = (n + T - 1) // T
        for _ in range(64):
            I = int(rng.integers(0, nt)); J = int(rng.integers(I, nt))
            ri = np.arange(I * T, min(n, (I + 1) * T)); rj = np.arange(J * T, min(n, (J + 1) * T))
            idx = ri if I == J else np.concatenate([ri, rj])
            ei, ej, ed, _ = o.all_pairs(rows[idx], THR, 0, len(ri), host_threads())
            if I != J:
                keep = ej >= len(ri)
                ei, ej, ed = ei[keep], ej[keep], ed[keep]
            want = set(zip(idx[ei].tolist(), idx[ej].tolist(), ed.view(np.uint64).tolist()))
            lo, hi = np.searchsorted(A, I * T), np.searchsorted(A, min(n, (I + 1) * T))
            sel = (B[lo:hi] >= J * T) & (B[lo:hi] < min(n, (J + 1) * T))
            have = set(zip(A[lo:hi][sel].tolist(), B[lo:hi][sel].tolist(), D[lo:hi][sel].view(np.uint64).tolist()))
            bad_tiles += int(want != have)
        out["tiles_1024_checked"] = 64
        out["tiles_1024_bad"] = bad_tiles
    # (iv) an independent GPU list
    if world > 1:
        hc.set_spline(device_ptr=full.data_ptr(), n=n, k=K)
        got1 = []
        if stream_mode:
            hc.compare_stream(THR, lambda x, y, z: got1.append((x, y, z)), variant)
            a1, b1, d1 = (np.concatenate([g[k] for g in got1]) for k in range(3))
        else:
            hc.compare(THR, variant)
            a1, b1, d1 = hc.get_edges()
        out["union_equals_single_gpu_list"] = bool(len(a1) == len(A) and np.array_equal(a1, A) and np.array_equal(b1, B) and
                                                   np.array_equal(d1.view(np.uint64), D.view(np.uint64)))
        out["single_gpu"] = edge_checksums(a1, b1, d1, n)
    else:
        m = min(n, 200000)
        hc.set_spline(device_ptr=ptr, n=m, k=K)
        hc.compare(THR, scema_b200.PAIRS_DMMA)
        a1, b1, d1 = hc.get_edges()
        t = hc.timings()
        sel = B < m
        hi = np.searchsorted(A, m)
        sel[hi:] = False
        out["fp64_dmma_list_equals_on_first_rows"] = bool(np.array_equal(a1, A[sel]) and np.array_equal(b1, B[sel]) and
                                                          np.array_equal(d1.view(np.uint64), D[sel].view(np.uint64)))
        out["_fp64"] = {"rows": m, "filter_ms": t["filter"], "K": K}
    out["ok"] = bool(local_ok and out["union_unique"] and out["cpu_recheck_bad_edges"] == 0 and bad_rows == 0 and
                     out.get("tiles_1024_bad", 0) == 0 and out.get("union_equals_single_gpu_list", True) and
                     out.get("exact_kernel_equals_on_first_rows", True) and
                     out.get("fp64_dmma_list_equals_on_first_rows", True))
    out["seconds"] = time.perf_counter() - t0
    if world > 1:
        torch.distributed.barrier(group=gloo)
    return out


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, wl, wl_name):
    import torch
    import torch.distributed as dist
    import scema_b200
    from scema_b200 import synth
    from scema_b200.distributed import ShardedCluster, aligned_shard_bounds, shard_bounds

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    gloo = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        gloo = dist.new_group(backend="gloo")   # host-side barrier while rank 0 drives all GPUs through the library
    n, P = wl["n"], wl["P"]
    K = 6 * P
    variant = {"dmma": 0, "fma": 1, "exact": 2, "tc": 3}[args.variant]
    # the tcgen05 filter takes rows of up to 10 chunks of 64 columns; wider rows take the DMMA filter
    eff_variant = "dmma" if (args.variant == "tc" and K > 636) else args.variant
    pert = synth.default_pert(THR, P)
    # N > 1: the plain sequence (all-gather of the FP64 rows, then every rank prepares and filters) is the default.
    # SCEMA_SHARD_OVERLAP=1 selects the overlapped exchange (ShardedCluster.run_overlapped: own-row operand images
    # all-gathered, FP64 rows pulled by copy engines on a side stream) — measured on 2 GPUs it gains nothing: the filter is
    # power-capped and clocks lower by what the overlap saves (filter 16.8 -> 18.1 ms), DESIGN.md section 4
    overlapped = (world > 1 and args.variant == "tc" and K <= 636 and not args.stream and n >= 4096 * world and
                  os.environ.get("SCEMA_SHARD_OVERLAP", "0") == "1" and not args.norm_band)
    all_bounds = aligned_shard_bounds(n, world)[1] if overlapped else shard_bounds(n, world)
    b, e = all_bounds[rank]
    n_local = e - b

    # one explicit (non-default) stream carries everything: the library's kernels, the NCCL
    # collectives and the timing events
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    hc = scema_b200.HistCluster(local_rank, stream.cuda_stream)
    assert hc.stream_ptr() == stream.cuda_stream
    off = synth.device_offsets(SEED, n_local, CLUSTER, wl["lmin"], wl["lmax"], first=b)
    d_steps = synth.device_histories(SEED, n_local, CLUSTER, wl_amp(wl), pert, off, first=b, device=dev, **wl_model(wl))
    steps_bytes = d_steps.numel() * 8
    h_steps = torch.empty(d_steps.shape, dtype=torch.float64, pin_memory=True)
    h_steps.copy_(d_steps)
    torch.cuda.synchronize()
    h_steps_np = h_steps.numpy()
    sc = ShardedCluster(hc, side_group=dist.new_group(backend="nccl") if overlapped else None, bounds=all_bounds) if world > 1 else None
    total_pairs = n * (n - 1) // 2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    acc = {"filter": 0.0, "resample": 0.0, "exact": 0.0, "sort": 0.0, "prep": 0.0, "allgather": 0.0, "steps": 0,
           "edges": 0, "survivors": 0}

    streamed = {"edges": 0, "chunks": 0}
    # what the latest resident step handed its caller (--dump-outputs): the shard counts and full rows (N > 1) and,
    # streamed, the edge chunks (collected only while "chunks" is present)
    last = {}

    def sink(a, b, d):
        streamed["edges"] += len(a)
        streamed["chunks"] += 1
        if "chunks" in last:
            last["chunks"].append((a, b, d))

    def step_resident(record):
        if args.dump_outputs and args.stream:
            last["chunks"] = []
        if world > 1:
            if overlapped:
                ne, counts, offs, full = sc.run_overlapped(n, P, THR)
            else:
                ne, counts, offs, full = sc.run(n, P, THR, variant, sink=sink if args.stream else None)
            last["counts"], last["full"] = counts, full
            tot = sum(counts)
        else:
            hc.resample(P)
            t_res = hc.timings()["resample"] if record else 0.0
            ne = hc.compare_stream(THR, sink, variant) if args.stream else hc.compare(THR, variant)
            tot = ne
        if record:
            t = hc.timings()
            for k in ("filter", "exact", "sort", "prep"):
                acc[k] += t[k]
            acc["resample"] += t["resample"] if world > 1 else t_res
            if world > 1:
                acc["allgather"] += sc.gather_events[0].elapsed_time(sc.gather_events[1])  # hc.timings() synchronised
            acc["steps"] += 1
            acc["edges"] = tot
            cn = hc.counters()
            acc["survivors"] = cn["survivors"]
            acc["passes"] = cn["passes"]
            acc["band_tiles"] = cn.get("band_tiles", 0)
            acc["plan"] = dict(hc.tc_last_plan(), slices=cn["tc_slices"])
        return tot

    # result buffers of the end-to-end path: pinned, allocated once and reused like a real caller would
    e2e_out = {"cap": 0, "bufs": None}

    def e2e_buffers(m):
        if m > e2e_out["cap"]:
            cap = int(m * 1.25) + 1024
            ta = torch.empty(cap, dtype=torch.int32, pin_memory=True)
            tb = torch.empty(cap, dtype=torch.int32, pin_memory=True)
            td = torch.empty(cap, dtype=torch.float64, pin_memory=True)
            e2e_out["keep"] = (ta, tb, td)
            e2e_out["bufs"] = (ta.numpy().view(np.uint32), tb.numpy().view(np.uint32), td.numpy())
            e2e_out["cap"] = cap
        return e2e_out["bufs"]

    def step_e2e():
        if world == 1 and not args.stream:
            # the one-call host API (scema_cluster): pinned host -> device copy, K1, K2, K3 — pipelined range by
            # range inside the library when the tcgen05 filter applies
            ne = hc.cluster(h_steps_np, off, None, P, THR, variant)
            hc.get_edges(out=e2e_buffers(ne))        # device -> host read of the result
            return ne
        hc.set_histories(h_steps_np, off)            # pinned host -> device inside the timed region
        if world > 1 and overlapped:
            ne, counts, offs, _ = sc.run_overlapped(n, P, THR)
        elif world > 1:
            ne, counts, offs, _ = sc.run(n, P, THR, variant, sink=sink if args.stream else None)
        else:
            hc.resample(P)
            # streamed: every chunk of edges lands in host memory through the sink
            ne = hc.compare_stream(THR, sink, variant) if args.stream else hc.compare(THR, variant)
        if not args.stream:
            hc.get_edges(out=e2e_buffers(ne))        # device -> host read of the result
        return ne

    # ---- device-resident timing: the raw histories are handed over once (borrowed device pointer)
    hc.set_histories(None, off, device_ptr=d_steps.data_ptr())
    for _ in range(args.warmup):
        step_resident(False)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = hc.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step_resident(True)
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = hc.kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = total_pairs * args.steps / (ms * 1e-3)

    if args.dump_outputs:
        # what the last timed step computed, read back after the timed region
        if args.stream:
            ch = last.pop("chunks")
            a, b, d = (np.concatenate([c[k] for c in ch]) if ch else np.zeros(0, dtype=(np.uint32, np.uint32, np.float64)[k])
                       for k in range(3))
        else:
            a, b, d = hc.get_edges()
        if world > 1:
            from scema_b200.distributed import gather_edges
            a, b, d = gather_edges(a, b, d, n, last["counts"], dev)
        if rank == 0:
            if world > 1:
                rows = last["full"]
            else:
                n_rows, K_rows, ptr = hc.spline_info()
                rows = torch.as_tensor(DeviceRows(ptr, n_rows, K_rows), device=dev)
            dump_outputs(args.dump_outputs, a, b, d, rows)
        if world > 1:
            dist.barrier()

    # ---- end-to-end timing (host buffers)
    e2e_steps = args.steps
    step_e2e()
    barrier()
    ev0.record(stream)
    ne_local = 0
    for _ in range(e2e_steps):
        ne_local = step_e2e()
    ev1.record(stream)
    barrier()
    ms_e2e = ev0.elapsed_time(ev1)
    e2e_pipeline_ranges = hc.counters().get("pipeline_ranges", 0) if world == 1 else 0   # of the last e2e step, before later calls reset the counters
    if world > 1:
        t = torch.tensor([ms_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    e2e_value = total_pairs * e2e_steps / (ms_e2e * 1e-3)
    h2d = steps_bytes + off.nbytes
    d2h = ne_local * 16

    # ---- N > 1, end to end through the LIBRARY's own multi-GPU entry point (scema_multi_cluster: one process, one host
    # thread + context per GPU, NCCL inside the library, host buffers in, merged sorted edge list out to pinned host
    # memory). Rank 0 drives all N GPUs; the other ranks keep their GPUs idle behind a host-side (gloo) barrier.
    e2e_lib = None
    if world > 1 and not args.stream and not args.no_library_e2e:
        torch.cuda.synchronize()
        dist.barrier(group=gloo)
        if rank == 0:
            off_all = synth.device_offsets(SEED, n, CLUSTER, wl["lmin"], wl["lmax"])
            h_all = torch.empty((int(off_all[-1]), 6), dtype=torch.float64, pin_memory=True)
            for (sb, se) in all_bounds:
                so = (off_all[sb:se + 1] - off_all[sb]).astype(np.uint64)
                part = synth.device_histories(SEED, se - sb, CLUSTER, wl_amp(wl), pert, so, first=sb, device=dev, **wl_model(wl))
                h_all[int(off_all[sb]):int(off_all[se])].copy_(part)
                del part
            torch.cuda.synchronize()
            mc = scema_b200.MultiCluster(list(range(world)))
            s0 = torch.cuda.ExternalStream(mc.first.stream_ptr(), device=dev)
            h_all_np = h_all.numpy()
            for _ in range(2):
                ne_m = mc.cluster(h_all_np, off_all, None, P, THR, variant)
                mc.first.get_edges(out=e2e_buffers(ne_m))
            lev0, lev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_wall = time.perf_counter()
            lev0.record(s0)
            for _ in range(e2e_steps):
                ne_m = mc.cluster(h_all_np, off_all, None, P, THR, variant)
                ma, mb, md = mc.first.get_edges(out=e2e_buffers(ne_m))
            lev1.record(s0)
            lev1.synchronize()
            wall_ms = (time.perf_counter() - t_wall) * 1e3
            lib_ms = lev0.elapsed_time(lev1)
            e2e_lib = {"value": total_pairs * e2e_steps / (lib_ms * 1e-3), "unit": "pairs/s", "ms_per_step": lib_ms / e2e_steps,
                       "wall_ms_per_step": wall_ms / e2e_steps, "h2d_bytes_per_step": int(h_all.numel() * 8 + off_all.nbytes),
                       "d2h_bytes_per_step": int(ne_m * 16), "steps": e2e_steps, "phases_ms": mc.last_ms(),
                       "checksums": edge_checksums(ma, mb, md, n),
                       "api": "scema_multi_cluster + scema_get_edges (C ABI, one process, %d host threads, NCCL inside the library); "
                              "timed with CUDA events on the first GPU's stream, which also receives the other shards' edges last" % world}
            mc.close()
            del h_all
        dist.barrier(group=gloo)

    # ---- verification of what was just timed (untimed; CPU oracle as the checker)
    verified = None
    if args.verify != "off":
        hc.set_histories(None, off, device_ptr=d_steps.data_ptr())
        verified = verify_run(args, hc, sc, world, rank, dev, n, P, variant, bool(args.stream), args.verify, gloo)

    if rank == 0:
        # ---- roofline of the dominant kernel (K2 filter): algorithmic 2*K flops per unordered pair
        pairs_this_rank = total_pairs / world
        filt_ms = acc["filter"] / max(acc["steps"], 1)
        achieved = pairs_this_rank * 2 * K / (filt_ms * 1e-3) / 1e12 if filt_ms > 0 else None
        if args.norm_band and acc.get("band_tiles", 0):
            # the roofline describes the kernel on the tiles it walked (128 x 256 pairs each), not the pairs the
            # norm bound dismissed beforehand
            tile_rows = 128 if os.environ.get("SCEMA_TC_CG") == "1" else 256
            achieved = acc["band_tiles"] * tile_rows * 256 * 2 * K / (filt_ms * 1e-3) / 1e12 if filt_ms > 0 else None
        NT = (n + 255) // 256
        if eff_variant == "tc":
            # tensor roofline: the denominators are the driver-measured cuBLAS bf16 figures (fp16 runs at the
            # same rate). `achieved` stays ALGORITHMIC (2K flops per unordered pair); the filter executes 3
            # sliced products of 64 columns over whole 256 x 256 tiles of the upper triangle = `executed`.
            mp, src = {}, "fallback"
            try:
                mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
                src = "measured"
            except Exception:
                mp = {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
            peak = float(mp.get("bf16_tflops", 1590.0))
            tc_slices = (acc.get("plan") or {}).get("slices") or 1   # of the timed steps (the verification ran other filters since)
            n_products = 1 if tc_slices == 1 else 3
            n_chunks = (K + 4 + 63) // 64
            executed = ((NT * (NT + 1) / 2) / world * 256 * 256 * n_products * 64 * n_chunks * 2 / (filt_ms * 1e-3) / 1e12
                        if filt_ms > 0 else None)
            extra = {"tc_slices": tc_slices, "executed_tflops": executed, "frac_executed": (executed / peak) if executed else None,
                     "peak_sustained": mp.get("bf16_tflops_sustained"),
                     "kernel": "k_filter_tc (K2 GEMM-form filter on tcgen05, split fp16, fp32 accumulate in TMEM)",
                     "peak_source": "of %s: MEASURED_PEAKS.json bf16_tflops (cuBLAS bf16 8192^3 burst); the kernel is timed "
                                    "alone per launch (CUDA events around it); sustained figure beside it" % src}
            if tc_slices == 1:
                extra["limiter"] = {"what": "tensor pipe under the board's power cap: executed flops exceed the cuBLAS bf16 burst figure "
                                            "(ncu: tensor pipe ~80 % active at the capped SM clock; round 1's 'TMEM read-out ceiling' was the "
                                            "issue loop of the MMA warp, tools/tmem_probe.cu measures >= 860 B/clk/SM of read-out)"}
            else:
                extra["limiter"] = {"what": "tensor pipe (ncu: 90 % busy, SM clock pulled to 1.70 GHz by the power cap)"}
            fp64 = max(hc.fp64_peak()["dmma_tflops"] for _ in range(2))
            extra["fp64_dmma_peak_tflops"] = fp64
            extra["achieved_over_fp64_peak"] = (achieved / fp64) if achieved else None
            tkey = f"tc:{wl_name}:{n}"
        else:
            # issue-rate probe, taken twice (the first call also warms the clocks back up after the host-side
            # bookkeeping above); the better of the two is the denominator
            peaks = [hc.fp64_peak() for _ in range(2)]
            key = "dmma_tflops" if eff_variant == "dmma" else "dfma_tflops"
            peak = max(p[key] for p in peaks)
            extra = {"kernel": "k_filter (K2 GEMM-form filter, %s)" % eff_variant,
                     "peak_source": "measured live on this GPU: FP64 %s issue-rate probe (scema_fp64_peak); "
                                    "MEASURED_PEAKS.json has no FP64 figure" % ("DMMA m8n8k4" if eff_variant == "dmma" else "DFMA")}
            tkey = f"{wl_name}:{n}"
        traffic = None
        tfile = os.path.join(ROOT, "profiles", "filter_traffic.json")
        if world == 1 and os.path.exists(tfile):
            try:
                traffic = json.load(open(tfile)).get(tkey)
            except Exception:
                traffic = None
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                    "launch_ms": filt_ms,
                    "other_kernels_ms": {k: acc[k] / max(acc["steps"], 1)
                                         for k in ("resample", "prep", "exact", "sort") + (("allgather",) if world > 1 else ())}}
        roofline.update(extra)
        # K1 (ragged spline resample) is the HBM-bound kernel of the step: 48 bytes per raw step read + 8 K bytes per history written
        res_ms = acc["resample"] / max(acc["steps"], 1)
        try:
            hbm_peak, hbm_src = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured"
        except Exception:
            hbm_peak, hbm_src = 6650.0, "fallback"
        k1_bytes = steps_bytes + n_local * K * 8
        roofline_resample = {"bound": "hbm", "achieved": k1_bytes / (res_ms * 1e-3) / 1e9 if res_ms > 0 else None, "peak": hbm_peak,
                             "unit": "GB/s", "frac": (k1_bytes / (res_ms * 1e-3) / 1e9 / hbm_peak) if res_ms > 0 else None,
                             "launch_ms": res_ms, "kernel": "k_resample_pair (K1; SCEMA_K1_KERNEL=stream selects the first-generation kernel), launches per length class summed",
                             "peak_source": "of %s: MEASURED_PEAKS.json hbm_gbs" % hbm_src,
                             "traffic": 3.50e9 * (k1_bytes / 2.207e9) if wl_name in ("c4", "c4s") else None,
                             "note": "bound by the forward-sweep result z (as large as the input) that the backward sweep reads back: DRAM moves "
                                     "~1.6x the algorithmic bytes at the number of chains whose z rows L2 can hold (ncu: profiles/r02_ncu_resample_pair_c4.txt, "
                                     "3.50 GB for 2.21 GB at 1M histories; traffic here is that capture scaled to this launch), issue slots 49 %, FP64 pipe 32 %"}
        # BASELINE's metric is quoted as a fraction of the FP64 peak: the true FP64 contraction (DMMA filter) on a bounded
        # sample of the same rows, timed by its own CUDA events, against the DMMA issue-rate probe
        roofline_fp64 = None
        if verified and verified.get("_fp64"):
            f = verified.pop("_fp64")
            dm = max(hc.fp64_peak()["dmma_tflops"] for _ in range(2))
            pr = f["rows"] * (f["rows"] - 1) / 2
            ach = pr * 2 * f["K"] / (f["filter_ms"] * 1e-3) / 1e12 if f["filter_ms"] > 0 else None
            roofline_fp64 = {"bound": "tensor", "achieved": ach, "peak": dm, "unit": "TFLOP/s", "frac": (ach / dm) if ach else None,
                             "traffic": None, "launch_ms": f["filter_ms"],
                             "kernel": "k_filter_ws (K2 GEMM-form filter on FP64 DMMA, --variant dmma), first %d histories of the workload "
                                       "(%.3g pairs), after the timed region" % (f["rows"], pr),
                             "peak_source": "measured live: FP64 DMMA m8n8k4 issue-rate probe (scema_fp64_peak)"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            m = min(n, 65536)
            rows, lib, kind, t_spl = cpu_reference_rows(wl, m, True)
            pairs, dt, _ = cpu_pairs_step(lib, rows, 0, 64)
            rps = int(max(64, min(m // 2, (pairs / dt) * 12.0 / m)))
            pairs, dt, _ = cpu_pairs_step(lib, rows, 0, rps)
            cpu = {"value": pairs / dt, "unit": "pairs/s", "cores": host_threads(), "kind": kind,
                   "sample": f"first {m} of {n} histories; rows [0,{rps}) x all later rows = {pairs} pairs in {dt:.1f} s; "
                             f"reference splinify {m / t_spl:.0f} histories/s"}
            # one core, for scale: the -O2 build and the as-shipped build (clustering/Makefile has no -O)
            try:
                p1, d1, _ = cpu_pairs_step_threads(lib, rows, 0, 24, 1)
                cpu["single_core_O2"] = p1 / d1
                if kind == "reference":
                    from oracle.pyoracle import Reference
                    lib0 = Reference(o0=True)
                    p0, d0, _ = cpu_pairs_step_threads(lib0, rows, 0, 8, 1)
                    cpu["single_core_O0_as_shipped"] = p0 / d0
            except Exception as e:  # noqa: BLE001 - the extra figures are optional
                cpu["single_core_note"] = repr(e)
        line = {
            "metric": "history pair comparisons/sec", "value": value, "unit": "pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": wl_config(wl, wl_name),
            "run": {"variant": eff_variant, "parallelism": f"tile-shard x{world}",
                    "exchange": (sc.path if (world > 1 and overlapped) else ("plain" if world > 1 else None)),
                    "filter_arithmetic": ("fp16 split operands (centred copies) on tcgen05, fp32 accumulate; every survivor and every "
                                          "emitted distance recomputed in f64 in the reference's operation order")
                    if eff_variant == "tc" else "f64",
                    "edges": acc["edges"], "survivors_last_rank0": acc["survivors"], "passes_last_rank0": acc.get("passes", 0),
                    "filter_plan_rank0": acc.get("plan"), "norm_band": bool(args.norm_band),
                    "band_tiles_last_rank0": acc.get("band_tiles", 0)},
            "clocks": clocks,
            "e2e": ({"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                     "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps,
                     "pipeline_ranges": e2e_pipeline_ranges,
                     "api": "scema_cluster + scema_get_edges (C ABI)" if world == 1 and not args.stream else
                            "scema_set_histories + resample + NCCL all-gather (torch.distributed) + sharded compare, one process per GPU"}
                    if e2e_lib is None else e2e_lib),
            "e2e_process_per_gpu": None if e2e_lib is None else
            {"value": e2e_value, "unit": "pairs/s", "ms_per_step": ms_e2e / e2e_steps, "h2d_bytes_per_step": int(h2d) * world,
             "d2h_bytes_per_step": int(d2h) * world,
             "api": "scema_set_histories + resample + NCCL all-gather (torch.distributed) + sharded compare, one process per GPU"},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "roofline_fp64": roofline_fp64,
            "roofline_resample": roofline_resample,
            "verified": verified,
            "cpu_baseline": cpu,
        }
        emit(line)
    hc.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def claim_stdout():
    """Libraries (NCCL's version banner, for one) write to file descriptor 1. The contract is ONE JSON
    line on stdout, so everything else is sent to stderr and only emit() reaches the real stdout."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--variant", default="tc", choices=["tc", "dmma", "fma", "exact"])
    ap.add_argument("--histories", type=int, default=0, help="override the workload's history count")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--norm-band", action="store_true",
                    help="opt-in exact shortcut (SCEMA_NORM_BAND=1): rows sorted by norm, tiles out of the threshold's reach skipped; "
                         "NOT part of the default line")
    ap.add_argument("--no-library-e2e", action="store_true", help="N > 1: skip the end-to-end figure through scema_multi_cluster")
    ap.add_argument("--verify", default="on", choices=["off", "on", "full"],
                    help="after the timed regions: CPU re-check of every edge, complete rows, union of the shards == one GPU's list "
                         "(full: 1000 rows and 64 tiles of 1024 x 1024, the config-5 checks of SURVEY 8d)")
    ap.add_argument("--stream", type=int, default=-1,
                    help="1: edges leave the device chunk by chunk through scema_compare_stream (default for c5), 0: one-shot compare")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the edge list and resampled rows of the last timed step to DIR/<name>.npy (float64, "
                         "fixed seeded samples when larger than ~50 MB) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = dict(WORKLOADS[args.workload])
    if args.stream < 0:
        args.stream = 1 if args.workload == "c5" else 0
    if args.histories:
        wl["n"] = args.histories
    if args.norm_band:
        os.environ["SCEMA_NORM_BAND"] = "1"
    if args.impl == "reference":
        run_reference(args, wl, args.workload)
    else:
        run_ours(args, wl, args.workload)


if __name__ == "__main__":
    main()
