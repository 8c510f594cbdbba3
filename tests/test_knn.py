"""scema_knn: exact k nearest neighbours of every history, filtered on the tensor cores.

CPU: the CPU top-k (tests/knn_oracle.c, on the oracle's compare_l2) against a numpy brute force with the reference's
operation order.
GPU: k = 1 against scema_nearest, every k and variant against the oracle, each path of the query (round 1, later filter
rounds, the exact kernel) on data built to take it, ties, dense data, wide rows, the caller's compare results left
untouched, the store path, the tcgen05 kernel selections, and 1M c4 rows."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


NONE = np.uint32(0xffffffff)
THR = 1e-6
VARIANTS = {"TC": 3, "DMMA": 0, "FMA": 1, "EXACT": 2}


class KnnOracle:
    """tests/knn_oracle.c compiled into a temporary directory (the tree may be read-only), linked against
    oracle/liboracle.so for the oracle's compare_l2."""

    def __init__(self, tmpdir):
        import ctypes as C
        from oracle.pyoracle import Oracle
        Oracle()   # builds oracle/liboracle.so when it is missing
        odir = os.path.join(ROOT, "oracle")
        so = os.path.join(tmpdir, "libknn_oracle.so")
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-Wall", "-o", so,
                               os.path.join(ROOT, "tests", "knn_oracle.c"), "-L" + odir, "-l:liboracle.so",
                               "-Wl,-rpath," + odir, "-lm"])
        self.lib = C.CDLL(so)
        u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
        f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
        self.lib.knn_oracle.restype = None
        self.lib.knn_oracle.argtypes = [f64p, C.c_uint64, C.c_uint32, C.c_uint32, u32p, C.c_uint64, C.c_uint64, u32p, f64p]

    def knn(self, rows, k, ids=None, row_begin=0, row_end=None):
        """k nearest neighbours of rows [row_begin, row_end) among all rows -> (index [m, k], diff [m, k])"""
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        n, K = rows.shape
        ids = np.arange(n, dtype=np.uint32) if ids is None else np.ascontiguousarray(ids, dtype=np.uint32)
        row_end = n if row_end is None else min(row_end, n)
        m = max(row_end - row_begin, 0)
        index = np.empty((m, k), dtype=np.uint32)
        diff = np.empty((m, k), dtype=np.float64)
        if m and k:
            self.lib.knn_oracle(rows, n, K, k, ids, row_begin, row_end, index, diff)
        return index, diff


@pytest.fixture(scope="module")
def oracle(tmp_path_factory):
    return KnnOracle(str(tmp_path_factory.mktemp("knn_oracle")))


def numpy_knn(rows, k, ids):
    """Brute force, column by column (s = s + (a - b)^2, then sqrt): the reference's order, no FMA."""
    n = len(rows)
    index = np.full((n, k), NONE, dtype=np.uint32)
    diff = np.full((n, k), np.inf)
    with np.errstate(all="ignore"):
        for i in range(n):
            s = np.zeros(n)
            for c in range(rows.shape[1]):
                s = s + (rows[i, c] - rows[:, c]) ** 2
            d = np.sqrt(s)
            cand = sorted((float(d[j]), int(ids[j]), j) for j in range(n) if j != i and not math.isnan(d[j]))
            for slot, (dd, _, j) in enumerate(cand[:k]):
                index[i, slot] = j
                diff[i, slot] = dd
    return index, diff


def same(a, b):
    """(index, diff) pairs identical, diffs bit for bit"""
    return np.array_equal(a[0], b[0]) and np.array_equal(np.asarray(a[1]).view(np.uint64), np.asarray(b[1]).view(np.uint64))


# ------------------------------------------------------------------------------------------------ CPU
def _cpu_cases():
    rng = np.random.default_rng(11)
    cases = []
    for n in (0, 1, 2):
        cases.append(("n%d" % n, rng.standard_normal((n, 6)), None, 3))
    r = rng.standard_normal((40, 6))
    cases.append(("random", r, None, 5))
    lat = rng.integers(0, 3, (50, 6)) * 0.25                     # exact ties and duplicate rows
    cases.append(("lattice", lat, rng.permutation(50)[::-1] // 3, 7))   # repeated, non-ascending IDs
    sp = rng.standard_normal((30, 12))
    sp[3] = np.nan
    sp[5, 2] = np.inf
    sp[6, 4] = -np.inf
    sp[7] = 1e200
    sp[8] = 1e200
    sp[9] = 1e-170 * rng.standard_normal(12)
    sp[10] = sp[11]
    cases.append(("special", sp, rng.integers(0, 10, 30), 4))
    cases.append(("k_ge_n", rng.standard_normal((5, 6)), None, 8))
    return cases


@pytest.mark.parametrize("name,rows,ids,k", _cpu_cases(), ids=[c[0] for c in _cpu_cases()])
def test_oracle_knn_matches_numpy(oracle, name, rows, ids, k):
    n = len(rows)
    ids = np.arange(n, dtype=np.uint32) if ids is None else np.asarray(ids, dtype=np.uint32)
    got = oracle.knn(rows, k, ids)
    assert got[0].shape == (n, k)
    assert same(got, numpy_knn(rows, k, ids))
    if n >= 2:   # the row range gives the same rows
        part = oracle.knn(rows, k, ids, row_begin=1, row_end=n)
        assert same(part, (got[0][1:], got[1][1:]))


def test_oracle_knn_special_rules(oracle):
    rows = np.zeros((4, 6))
    rows[1] = np.nan
    rows[2, 0] = np.inf
    idx, d = oracle.knn(rows, 3, np.array([5, 4, 3, 2], dtype=np.uint32))
    assert np.all(idx[1] == NONE) and np.all(np.isinf(d[1]))          # NaN row: nothing
    assert list(idx[0]) == [3, 2, NONE] and d[0, 0] == 0.0 and np.isinf(d[0, 1])   # +inf partners listed, tie by ID


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def hc():
    import scema_b200
    h = scema_b200.HistCluster(0)
    yield h
    h.close()


def nearest_equal(hc, ids):
    nid, nd = hc.nearest()
    idx, d = hc.knn(1)
    got_ids = np.where(idx[:, 0] == NONE, NONE, np.asarray(ids, dtype=np.uint32)[np.minimum(idx[:, 0], len(ids) - 1)])
    return np.array_equal(got_ids, nid) and np.array_equal(d[:, 0].view(np.uint64), nd.view(np.uint64))


def special_rows(n=4000):
    from scema_b200 import synth
    rng = np.random.default_rng(5)
    rows = synth.rows(7, n, 8, 10, 5e-3, synth.default_pert(THR, 10))
    rows[10] = np.nan
    rows[20, 3] = np.inf
    rows[30] = rows[31]
    rows[40] = 1e200
    rows[41] = 1e200
    rows[50:60] = rows[50:60] * 0 + 3.0
    rows[60:70] = 1e-170 * rng.standard_normal((10, 60))
    return rows


@pytest.mark.gpu
def test_knn1_equals_nearest(hc):
    from scema_b200 import synth
    rows = synth.rows(3, 16384, 16, 10, 5e-3, synth.default_pert(THR, 10))          # c2-shaped
    hc.set_spline(rows)
    assert nearest_equal(hc, np.arange(len(rows)))
    off = synth.offsets(9, 20000, 16, 6, 200)                                         # ragged histories, resampled
    steps = synth.histories(9, 20000, 16, 5e-3, synth.default_pert(THR, 10), off)
    ids = np.random.default_rng(2).permutation(20000).astype(np.uint32)
    hc.set_histories(steps, off, ids)
    hc.resample(10)
    assert nearest_equal(hc, ids)
    for n in (600, 4000):                                                             # special values, exact-only and rounds
        rows = special_rows(n)
        ids = np.random.default_rng(n).integers(0, 50, n).astype(np.uint32)
        hc.set_spline(rows, ids)
        assert nearest_equal(hc, ids)
    hc.set_spline(synth.rows(4, 6000, 16, 10, 5e-3, synth.default_pert(THR, 10)))     # repeated IDs after select_rows
    sel = np.concatenate([np.arange(0, 6000, 2), np.arange(0, 3000, 3)]).astype(np.uint32)
    hc.select_rows(sel)
    assert nearest_equal(hc, sel)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1000, 20000])
def test_knn_matches_oracle_all_variants(hc, oracle, n):
    from scema_b200 import synth
    rows = synth.rows(12, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
    ids = np.random.default_rng(n).permutation(n).astype(np.uint32)
    want = oracle.knn(rows, 32, ids)
    hc.set_spline(rows, ids)
    for k in (1, 2, 8, 32):
        first = None
        for vname, v in VARIANTS.items():
            got = hc.knn(k, v)
            assert same(got, (want[0][:, :k], want[1][:, :k])), (n, k, vname, hc.knn_last_stats())
            first = first or got
            assert same(got, first)


def path_rows(seed=21):
    """200k rows of 60 columns: 160k in tight clusters of 32 (closed in round 1), 39.9k in looser clusters of 16 (too
    loose for round 1's radius, closed in a later round: |U| n is above the exact-kernel cutoff), 90 far outliers, 5 NaN
    rows and 5 rows with an inf entry (left to the exact kernel)."""
    rng = np.random.default_rng(seed)
    K, s1, s2 = 60, 1e-3, 2e-3
    a = np.repeat(rng.random((5000, K)), 32, axis=0) + s1 * rng.standard_normal((160000, K))
    b = np.repeat(rng.random((2494, K)), 16, axis=0) + s2 * rng.standard_normal((39904, K))
    c = 1e3 * (1.0 + rng.random((96, K)))
    rows = np.concatenate([a, b, c])
    rows[-96:-91] = np.nan
    rows[-91:-86, 7] = np.inf
    perm = rng.permutation(len(rows))
    return rows[perm], perm


@pytest.mark.gpu
def test_knn_every_path(hc, oracle):
    rows, perm = path_rows()
    n = len(rows)
    k = 8
    hc.set_spline(rows)
    got = hc.knn(k)
    st = hc.knn_last_stats()
    assert st["rows_round1"] > 0 and st["rows_later_rounds"] > 0 and st["rows_exact"] > 0, st
    assert st["rows_round1"] + st["rows_later_rounds"] + st["rows_exact"] == n, st
    inv = np.argsort(perm)
    # rows of every population: the first of each kind in the original order, plus a seeded range
    check = np.unique(np.concatenate([inv[0:64], inv[160000:160064], inv[-96:], np.arange(1000, 1128)]))
    for r in check:
        want = oracle.knn(rows, k, None, int(r), int(r) + 1)
        assert same((got[0][r:r + 1], got[1][r:r + 1]), want), (int(r), st)
    nan_rows = inv[-96:-91]
    assert np.all(got[0][nan_rows] == NONE)


@pytest.mark.gpu
def test_knn_ties_lattice(hc, oracle):
    rng = np.random.default_rng(8)
    n = 3000
    rows = rng.integers(0, 4, (n, 6)) * 0.125
    ids = (rng.permutation(n) // 3).astype(np.uint32)
    hc.set_spline(rows, ids)
    want = oracle.knn(rows, 16, ids)
    for vname, v in VARIANTS.items():
        got = hc.knn(16, v)
        assert same(got, want), (vname, hc.knn_last_stats())
    idx, d = got
    for i in range(0, n, 97):   # slot order (diff, ID, index)
        keys = [(d[i, s], ids[idx[i, s]], idx[i, s]) for s in range(16)]
        assert keys == sorted(keys)


@pytest.mark.gpu
def test_knn_dense_isotropic(hc, oracle):
    n, k = 20000, 8
    rows = np.random.default_rng(31).standard_normal((n, 60))
    hc.set_spline(rows)
    got = hc.knn(k)
    st = hc.knn_last_stats()
    assert st["rows_exact"] > 0 and st["exact_pairs"] >= st["rows_exact"] * (n - 1), st
    assert st["edges"] <= 8 * n * k + (1 << 20), st      # no O(n^2) edge list
    want = oracle.knn(rows, k)
    assert same(got, want), st


@pytest.mark.gpu
@pytest.mark.parametrize("P", [50, 110])
def test_knn_wide_rows(hc, oracle, P):
    from scema_b200 import synth
    rows = synth.rows(13, 5000, 16, P, 5e-3, synth.default_pert(THR, P))
    hc.set_spline(rows)
    want = oracle.knn(rows, 8)
    got = hc.knn(8)
    assert same(got, want), hc.knn_last_stats()
    assert same(hc.knn(8, VARIANTS["EXACT"]), want)


@pytest.mark.gpu
def test_knn_leaves_compare_results(hc, tmp_path):
    import scema_b200
    from scema_b200 import synth
    n = 20000
    rows = synth.rows(14, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
    hc.set_spline(rows)
    hc.compare(THR)

    def snapshot(tag):
        d = tmp_path / tag
        d.mkdir()
        hc.write_similar_hist(str(d / "last.%u.similar_hist"))
        files = {f: (d / f).read_bytes() for f in sorted(os.listdir(d))}
        e = hc.get_edges()
        return (e[0].copy(), e[1].copy(), e[2].copy().view(np.uint64)), hc.get_degrees(n), files, hc.counters()

    before = snapshot("before")
    hc.knn(8)
    with pytest.raises(scema_b200.ScemaError):
        hc.knn(0)
    after = snapshot("after")
    for x, y in zip(before, after):
        if isinstance(x, tuple):
            assert all(np.array_equal(p, q) for p, q in zip(x, y))
        elif isinstance(x, np.ndarray):
            assert np.array_equal(x, y)
        else:
            assert x == y
    ne = hc.compare(THR)
    a, b, d = hc.get_edges()
    assert ne == len(before[0][0]) and np.array_equal(a, before[0][0]) and np.array_equal(b, before[0][1])


@pytest.mark.gpu
def test_knn_store_path(hc):
    from scema_b200 import synth
    n, P = 8000, 10
    off = synth.offsets(15, n, 16, 12, 12)
    steps = synth.histories(15, n, 16, 5e-3, synth.default_pert(THR, P), off).reshape(n, 12, 6)
    ids = (np.arange(n, dtype=np.uint32) * 7) % 5003
    hc.store_reset(n, ids)
    for t in range(12):
        hc.store_append(np.ascontiguousarray(steps[:, t, :]))
    hc.store_resample(P)
    sel = np.arange(0, n, 3, dtype=np.uint32)
    hc.select_rows(sel)
    got = hc.knn(8)
    rows = hc.get_spline()
    hc.set_spline(rows, ids[sel])
    assert same(got, hc.knn(8))


_SELECTION_SCRIPT = r"""
import hashlib, sys
sys.path.insert(0, sys.argv[1])
import numpy as np, scema_b200
from scema_b200 import synth
hc = scema_b200.HistCluster(0)
hc.set_spline(synth.rows(16, 20000, 16, 10, 5e-3, synth.default_pert(1e-6, 10)))
i, d = hc.knn(8)
print(hashlib.sha256(i.tobytes() + d.tobytes()).hexdigest(), hc.knn_last_stats()["rounds"])
"""


@pytest.mark.gpu
def test_knn_kernel_selections():
    """SCEMA_TC_SLICES / SCEMA_TC_CG are read once per process: each setting in a process of its own."""
    out = {}
    for name, env in (("default", {}), ("s1", {"SCEMA_TC_SLICES": "1"}), ("s2", {"SCEMA_TC_SLICES": "2"}),
                      ("s3", {"SCEMA_TC_SLICES": "3"}), ("cg1", {"SCEMA_TC_CG": "1"})):
        e = {k: v for k, v in os.environ.items() if not k.startswith("SCEMA_TC")}
        e.update(env)
        r = subprocess.run([sys.executable, "-c", _SELECTION_SCRIPT, ROOT], env=e, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        out[name] = r.stdout.split()
    assert all(v[0] == out["default"][0] for v in out.values()), out
    assert int(out["default"][1]) >= 1


@pytest.mark.gpu
def test_knn_c4_million(hc, oracle):
    import torch
    import bench
    from scema_b200 import synth
    w = bench.WORKLOADS["c4"]
    n = w["n"]
    off = synth.device_offsets(bench.SEED, n, bench.CLUSTER, w["lmin"], w["lmax"])
    steps = synth.device_histories(bench.SEED, n, bench.CLUSTER, bench.wl_amp(w), synth.default_pert(bench.THR, w["P"]), off,
                                   device=torch.device("cuda", 0), **bench.wl_model(w))
    hc.set_histories(None, off, device_ptr=steps.data_ptr())
    hc.resample(w["P"])
    torch.cuda.synchronize()
    idx, d = hc.knn(8)
    st = hc.knn_last_stats()
    i1, d1 = hc.knn(1)
    assert same((idx[:, :1], d[:, :1]), (i1, d1)), st
    rows = hc.get_spline()
    del steps
    r0 = int(np.random.default_rng(17).integers(0, n - 256))
    want = oracle.knn(rows, 8, None, r0, r0 + 256)
    assert same((idx[r0:r0 + 256], d[r0:r0 + 256]), want), json.dumps(st)
    print("knn c4 stats", json.dumps(st))
