"""scema_query_compare / scema_query_knn: a second set of histories (the queries) against the spline matrix.

CPU: the cross oracle (tests/query_oracle.c, on the oracle's compare_l2) against a numpy brute force with the reference's
operation order, and the compaction rule of the [Q; R] prefix on index grids.
GPU: every variant against the oracle at panel-boundary sizes and row widths, near-threshold and special-value rows in
both sets, host and device query rows, select_rows and the store path, properties against scema_compare / scema_knn,
every path of query_knn, pinned kernel selections, a queue overflow, the planner's pair count, the caller's state left
untouched, the error codes, and 10^6 c4 rows."""
import ctypes as C
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
PANEL = 2048


class QueryOracle:
    """tests/query_oracle.c compiled into a temporary directory (the tree may be read-only), linked against
    oracle/liboracle.so for the oracle's compare_l2."""

    def __init__(self, tmpdir):
        from oracle.pyoracle import Oracle
        Oracle()   # builds oracle/liboracle.so when it is missing
        odir = os.path.join(ROOT, "oracle")
        so = os.path.join(tmpdir, "libquery_oracle.so")
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-Wall", "-o", so,
                               os.path.join(ROOT, "tests", "query_oracle.c"), "-L" + odir, "-l:liboracle.so",
                               "-Wl,-rpath," + odir, "-lm"])
        self.lib = C.CDLL(so)
        u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
        u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
        f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
        L = self.lib
        L.query_radius_count.restype = C.c_uint64
        L.query_radius_count.argtypes = [f64p, C.c_uint64, f64p, C.c_uint64, C.c_uint32, C.c_double, u64p]
        L.query_radius_fill.restype = None
        L.query_radius_fill.argtypes = [f64p, C.c_uint64, f64p, C.c_uint64, C.c_uint32, C.c_double, u64p, u32p, u32p, f64p]
        L.query_knn_oracle.restype = None
        L.query_knn_oracle.argtypes = [f64p, C.c_uint64, u32p, f64p, C.c_uint64, C.c_uint32, C.c_uint32, u32p, f64p]

    @staticmethod
    def _prep(R, Q):
        R = np.ascontiguousarray(R, dtype=np.float64)
        Q = np.ascontiguousarray(Q, dtype=np.float64)
        K = R.shape[1] if R.ndim == 2 and R.shape[1] else Q.shape[1]
        return R.reshape(-1, K) if R.size else np.zeros((0, K)), Q.reshape(-1, K) if Q.size else np.zeros((0, K)), K

    def radius(self, R, Q, thr):
        """-> (query_index, row_index, diff) sorted by (j, i)"""
        R, Q, K = self._prep(R, Q)
        n, m = len(R), len(Q)
        per = np.zeros(max(m, 1), dtype=np.uint64)
        if n == 0 or m == 0:
            return np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(0)
        tot = int(self.lib.query_radius_count(R, n, Q, m, K, float(thr), per))
        off = np.concatenate([[0], np.cumsum(per[:m])]).astype(np.uint64)
        j = np.empty(max(tot, 1), np.uint32)
        i = np.empty(max(tot, 1), np.uint32)
        d = np.empty(max(tot, 1))
        self.lib.query_radius_fill(R, n, Q, m, K, float(thr), off, j, i, d)
        return j[:tot], i[:tot], d[:tot]

    def knn(self, R, Q, k, ids=None):
        R, Q, K = self._prep(R, Q)
        n, m = len(R), len(Q)
        ids = np.arange(n, dtype=np.uint32) if ids is None else np.ascontiguousarray(ids, dtype=np.uint32)
        index = np.full((m, k), NONE, dtype=np.uint32)
        diff = np.full((m, k), np.inf)
        if m and n:
            self.lib.query_knn_oracle(R, n, ids if n else np.zeros(1, np.uint32), Q, m, K, k, index, diff)
        return index, diff


@pytest.fixture(scope="module")
def oracle(tmp_path_factory):
    return QueryOracle(str(tmp_path_factory.mktemp("query_oracle")))


def numpy_dist(R, Q):
    """[m, n] distances, column by column (s = s + (r - q)^2, then sqrt): the reference's order, no FMA."""
    s = np.zeros((len(Q), len(R)))
    with np.errstate(all="ignore"):
        for c in range(R.shape[1]):
            s = s + (R[None, :, c] - Q[:, None, c]) ** 2
        return np.sqrt(s)


def numpy_radius(R, Q, thr):
    if len(R) == 0 or len(Q) == 0:
        return np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(0)
    d = numpy_dist(R, Q)
    with np.errstate(invalid="ignore"):
        j, i = np.nonzero(d < thr)      # row-major: (j, i) order
    return j.astype(np.uint32), i.astype(np.uint32), d[j, i]


def numpy_knn(R, Q, k, ids):
    m = len(Q)
    index = np.full((m, k), NONE, dtype=np.uint32)
    diff = np.full((m, k), np.inf)
    if len(R) == 0:
        return index, diff
    d = numpy_dist(R, Q)
    for j in range(m):
        cand = sorted((float(d[j, i]), int(ids[i]), i) for i in range(len(R)) if not np.isnan(d[j, i]))
        for s, (dd, _, i) in enumerate(cand[:k]):
            index[j, s] = i
            diff[j, s] = dd
    return index, diff


def same_list(a, b):
    return (len(a[0]) == len(b[0]) and np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
            and np.array_equal(np.asarray(a[2]).view(np.uint64), np.asarray(b[2]).view(np.uint64)))


def same_knn(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(np.asarray(a[1]).view(np.uint64), np.asarray(b[1]).view(np.uint64))


def specials(rows, rng, at):
    rows = rows.copy()
    K = rows.shape[1]
    rows[at[0]] = np.nan
    rows[at[1], min(3, K - 1)] = np.inf
    rows[at[2], 0] = -np.inf
    rows[at[3]] = 1e200
    rows[at[4]] = 1e-170 * rng.standard_normal(K)
    return rows


# ------------------------------------------------------------------------------------------------ CPU
def _cpu_cases():
    rng = np.random.default_rng(41)
    cases = []
    cases.append(("empty_q", rng.standard_normal((30, 6)), np.zeros((0, 6)), None, 1.0))
    cases.append(("empty_r", np.zeros((0, 6)), rng.standard_normal((7, 6)), None, 1.0))
    cases.append(("m_much_larger", rng.standard_normal((3, 6)), rng.standard_normal((200, 6)), None, 2.5))
    cases.append(("m_much_smaller", rng.standard_normal((300, 12)), rng.standard_normal((2, 12)), None, 4.0))
    lat_r = rng.integers(0, 3, (60, 6)) * 0.25
    lat_q = rng.integers(0, 3, (25, 6)) * 0.25
    cases.append(("lattice", lat_r, lat_q, (rng.permutation(60)[::-1] // 3).astype(np.uint32), 0.6))
    r = specials(rng.standard_normal((40, 12)), rng, (1, 2, 3, 4, 5))
    q = specials(rng.standard_normal((20, 12)), rng, (6, 7, 8, 9, 10))
    q[11] = r[12]           # a query equal to a retained row: listed at 0
    q[13] = r[4]            # a tiny retained row
    cases.append(("special", r, q, rng.integers(0, 9, 40).astype(np.uint32), 5.0))
    return cases


@pytest.mark.parametrize("name,R,Q,ids,thr", _cpu_cases(), ids=[c[0] for c in _cpu_cases()])
def test_oracle_matches_numpy(oracle, name, R, Q, ids, thr):
    ids = np.arange(len(R), dtype=np.uint32) if ids is None else ids
    for t in (thr, thr * 0.5, 0.0, -1.0, np.nan, np.inf):     # threshold sweep
        assert same_list(oracle.radius(R, Q, t), numpy_radius(R, Q, t)), (name, t)
    for k in (1, 3, 8):
        got = oracle.knn(R, Q, k, ids)
        assert got[0].shape == (len(Q), k)
        assert same_knn(got, numpy_knn(R, Q, k, ids)), (name, k)


def test_oracle_special_rules(oracle):
    R = np.zeros((4, 6))
    R[1] = np.nan
    R[2, 0] = np.inf
    Q = np.zeros((2, 6))
    Q[1] = np.nan
    idx, d = oracle.knn(R, Q, 4, np.array([5, 4, 3, 2], dtype=np.uint32))
    assert list(idx[0]) == [3, 0, 2, NONE] and d[0, 0] == 0.0 and d[0, 1] == 0.0 and np.isinf(d[0, 2])
    assert np.all(idx[1] == NONE)
    j, i, dd = oracle.radius(R, Q, 1.0)
    assert list(j) == [0, 0] and list(i) == [0, 3] and np.all(dd == 0.0)


def compact(m, N):
    """The host statement of the compaction: the (a, b) pairs a < b of an N-row matrix in the prefix compare's (sorted)
    order, the rule a < m <= b, the remap (j, i) = (a, b - m)."""
    a, b = np.triu_indices(N, 1)
    keep = (a < m) & (b >= m)
    return a[keep], b[keep] - m


@pytest.mark.parametrize("m,n", [(0, 5), (5, 0), (1, 1), (3, 7), (7, 3), (16, 16), (33, 2)])
def test_compaction_rule(m, n):
    j, i = compact(m, m + n)
    want_j, want_i = np.divmod(np.arange(m * n), max(n, 1))
    assert np.array_equal(j, want_j[:len(j)]) and np.array_equal(i, want_i[:len(i)]) and len(j) == m * n
    # order preserved: ascending (j, i) is ascending packed key
    key = j.astype(np.uint64) * (n + 1) + i
    assert np.all(np.diff(key.astype(np.int64)) > 0)


def test_filter_pair_bound():
    """The panels [0, ceil(m / 2048)) of [Q; R] hold at most m n + m (m - 1) / 2 + 2048 n pairs, and every Q x R pair."""
    for m in (1, 2, 2047, 2048, 2049, 8193, 10 ** 4):
        for n in (1, 2, 2047, 2049, 8193, 10 ** 6):
            N = m + n
            r1 = min(N, -(-m // PANEL) * PANEL)
            pairs = r1 * N - r1 * (r1 + 1) // 2
            assert m * n <= pairs <= m * n + m * (m - 1) // 2 + 2048 * n


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def hc():
    import scema_b200
    h = scema_b200.HistCluster(0)
    yield h
    h.close()


def clustered(seed, n, K, n_centres=None, spread=None):
    """Rows around shared centres, spread so that about half of the pairs of a centre lie below THR."""
    rng = np.random.default_rng(seed)
    n_centres = n_centres or max(1, n // 8)
    spread = spread if spread is not None else THR / np.sqrt(2.0 * K)
    centres = np.random.default_rng(1000 + K).random((max(n_centres, 1), K))
    return centres[rng.integers(0, len(centres), n)] + spread * rng.standard_normal((n, K))


def plant(R, Q, rng, count=12):
    """Queries at THR (1 + e) from retained rows, e a few ulp either side: the computed distance straddles THR."""
    Q = Q.copy()
    if len(R) == 0 or len(Q) == 0:
        return Q
    K = R.shape[1]
    for t in range(min(count, len(Q))):
        u = rng.standard_normal(K)
        u /= np.linalg.norm(u)
        e = (t - count // 2) * 2.0 ** -52
        Q[(t * 7919) % len(Q)] = R[(t * 104729) % len(R)] + THR * (1.0 + e) * u
    return Q


def filter_pairs_ok(st, m, n):
    return st["filter_pairs"] <= st["rounds"] * (m * n + m * (m - 1) // 2 + 2048 * n)


def check_all_variants(hc, oracle, R, Q, k=8, ids=None, thr=THR):
    m, n = len(Q), len(R)
    want_e = oracle.radius(R, Q, thr)
    want_k = oracle.knn(R, Q, k, ids)
    for vname, v in VARIANTS.items():
        got = hc.query_compare(Q, thr, v)
        st = hc.query_last_stats()
        assert same_list(got, want_e), (m, n, R.shape[1], vname, st)
        assert st["cross_edges"] == len(want_e[0]) and filter_pairs_ok(st, m, n), st
        got = hc.query_knn(Q, k, v)
        st = hc.query_last_stats()
        assert same_knn(got, want_k), (m, n, R.shape[1], vname, st)
        assert filter_pairs_ok(st, m, n), st
    return want_e, want_k


SIZES = [(1, 8193), (2, 2049), (2047, 2048), (2048, 2047), (2049, 2), (8193, 1), (2049, 8193), (8193, 2048)]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [6, 16, 30, 60, 66])
def test_query_matches_oracle(hc, oracle, K):
    rng = np.random.default_rng(K)
    for m, n in SIZES:
        R = clustered(K * 31 + n, n, K, n_centres=max(1, (m + n) // 16))
        Q = plant(R, clustered(K * 37 + m, m, K, n_centres=max(1, (m + n) // 16)), rng)
        hc.set_spline(R)
        check_all_variants(hc, oracle, R, Q)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [300, 642])
def test_query_wide_rows(hc, oracle, K):
    rng = np.random.default_rng(K)
    for m, n in [(1, 2049), (2049, 2), (2049, 2048)]:
        R = clustered(K + n, n, K, n_centres=max(1, (m + n) // 16))
        Q = plant(R, clustered(K + m + 1, m, K, n_centres=max(1, (m + n) // 16)), rng)
        hc.set_spline(R)
        check_all_variants(hc, oracle, R, Q)


@pytest.mark.gpu
def test_query_special_values(hc, oracle):
    rng = np.random.default_rng(3)
    for m, n in [(300, 5000), (5000, 300)]:
        R = clustered(5 + n, n, 60, n_centres=max(1, n // 8))
        Q = clustered(6 + m, m, 60, n_centres=max(1, n // 8))
        R[100:120] = 3.0
        Q[50:60] = 3.0                          # exact duplicates across the sets: listed at distance 0
        R = specials(R, rng, (10, 11, 12, 13, 14))
        R[15] = 1e200
        Q = specials(Q, rng, (20, 21, 22, 23, 24))
        Q[25] = R[15]
        Q[26] = R[14]
        ids = rng.integers(0, 40, n).astype(np.uint32)
        hc.set_spline(R, ids)
        check_all_variants(hc, oracle, R, Q, k=16, ids=ids)
        check_all_variants(hc, oracle, R, Q, k=4, ids=ids, thr=1e-3)


@pytest.mark.gpu
def test_query_device_rows(hc, oracle):
    import torch
    R = clustered(71, 9000, 30)
    Q = plant(R, clustered(72, 3000, 30), np.random.default_rng(1))
    hc.set_spline(R)
    want = hc.query_compare(Q, THR)
    want_k = hc.query_knn(Q, 8)
    assert same_list(want, oracle.radius(R, Q, THR))
    qd = torch.from_numpy(Q).cuda()
    torch.cuda.synchronize()
    for v in VARIANTS.values():
        assert same_list(hc.query_compare(None, THR, v, device_ptr=qd.data_ptr(), m=len(Q)), want)
        assert same_knn(hc.query_knn(None, 8, v, device_ptr=qd.data_ptr(), m=len(Q)), want_k)
    # raw query histories resampled on a second context, passed by its device pointer
    import scema_b200
    from scema_b200 import synth
    off = synth.offsets(9, 4000, 16, 6, 60)
    steps = synth.histories(9, 4000, 16, 5e-3, synth.default_pert(THR, 10), off)
    hc.set_histories(steps[:int(off[2500])], off[:2501])
    hc.resample(10)
    R2 = hc.get_spline()
    q = scema_b200.HistCluster(0)
    q.set_histories(steps, off)
    q.resample(10)
    n2, k2, ptr = q.spline_info()
    got = hc.query_compare(None, THR, device_ptr=ptr, m=n2)
    Q2 = q.get_spline()
    assert same_list(got, oracle.radius(R2, Q2, THR))
    assert np.count_nonzero(got[1] == got[0]) == 2500        # the first 2500 queries are the retained rows themselves
    q.close()


@pytest.mark.gpu
def test_query_select_rows_and_store(hc, oracle):
    from scema_b200 import synth
    rows = clustered(81, 6000, 60)
    hc.set_spline(rows)
    sel = np.concatenate([np.arange(0, 6000, 2), np.arange(0, 3000, 3)]).astype(np.uint32)
    hc.select_rows(sel)
    Q = plant(rows[sel], clustered(82, 2500, 60), np.random.default_rng(2))
    R = rows[sel]
    check_all_variants(hc, oracle, R, Q, ids=sel)        # repeated rows and IDs
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
    R = hc.get_spline()
    Q = plant(R, R[::5] + 1e-8, np.random.default_rng(3))
    check_all_variants(hc, oracle, R, Q, ids=ids[sel])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [8192, 80000])
def test_query_properties(hc, n):
    from scema_b200 import synth
    rows = synth.rows(23, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
    rows = rows[np.sort(np.unique(rows, axis=0, return_index=True)[1])]     # no duplicate rows
    n = len(rows)
    hc.set_spline(rows)
    ne = hc.compare(THR)
    a, b, d = hc.get_edges()
    # Q = R: both directions of scema_compare's list plus the finite diagonal
    j, i, dq = hc.query_compare(rows, THR)
    jj = np.concatenate([a, b, np.arange(n, dtype=np.uint32)])
    ii = np.concatenate([b, a, np.arange(n, dtype=np.uint32)])
    dd = np.concatenate([d, d, np.zeros(n)])
    o = np.lexsort((ii, jj))
    assert same_list((j, i, dq), (jj[o], ii[o], dd[o])), (ne, len(j))
    # Q = R, no duplicate rows: query_knn(k + 1) without the self slot is scema_knn(k)
    for k in (1, 8):
        qi, qd = hc.query_knn(rows, k + 1)
        assert np.array_equal(qi[:, 0], np.arange(n)) and np.all(qd[:, 0] == 0.0)
        assert same_knn((qi[:, 1:], qd[:, 1:]), hc.knn(k)), hc.query_last_stats()
    # Q = the first rows of a c4-shaped matrix: the cross part of scema_compare on the concatenation
    m = min(n // 4, 5000)
    Q = rows[:m] + 3e-7 * np.random.default_rng(4).standard_normal((m, rows.shape[1]))
    cat = np.concatenate([Q, rows])
    hc.set_spline(cat)
    hc.compare(THR)
    a, b, d = hc.get_edges()
    keep = (a < m) & (b >= m)
    hc.set_spline(rows)
    got = hc.query_compare(Q, THR)
    assert same_list(got, (a[keep], b[keep] - m, d[keep]))


def path_rows(seed=21):
    """R: 200k rows of 60 columns in tight clusters of 32 and looser clusters of 16, plus outliers. Queries drawn the same
    way: those of tight clusters close in round 1, those of loose ones in a later round (open queries * n stays above the
    exact cutoff), the outliers, NaN and inf queries go to the exact kernel."""
    rng = np.random.default_rng(seed)
    K, s1, s2 = 60, 1e-3, 2e-3
    ca, cb = rng.random((5000, K)), rng.random((2494, K))
    R = np.concatenate([np.repeat(ca, 32, axis=0) + s1 * rng.standard_normal((160000, K)),
                        np.repeat(cb, 16, axis=0) + s2 * rng.standard_normal((39904, K)),
                        1e3 * (1.0 + rng.random((96, K)))])
    R = R[rng.permutation(len(R))]
    Q = np.concatenate([ca[rng.integers(0, 5000, 8000)] + s1 * rng.standard_normal((8000, K)),
                        cb[rng.integers(0, 2494, 3000)] + s2 * rng.standard_normal((3000, K)),
                        1e3 * (1.0 + rng.random((100, K)))])
    Q[-100:-95] = np.nan
    Q[-95:-90, 7] = np.inf
    return R, Q


@pytest.mark.gpu
def test_query_knn_every_path(hc, oracle):
    R, Q = path_rows()
    m, n, k = len(Q), len(R), 8
    hc.set_spline(R)
    got = hc.query_knn(Q, k)
    st = hc.query_last_stats()
    assert st["rows_round1"] > 0 and st["rows_later_rounds"] > 0 and st["rows_exact"] > 0, st
    assert st["rows_round1"] + st["rows_later_rounds"] + st["rows_exact"] == m, st
    assert filter_pairs_ok(st, m, n), st
    assert same_knn(got, hc.query_knn(Q, k, VARIANTS["EXACT"]))
    check = np.unique(np.concatenate([np.arange(0, 96), np.arange(8000, 8096), np.arange(m - 100, m)]))
    assert same_knn((got[0][check], got[1][check]), oracle.knn(R, Q[check], k)), st
    assert np.all(got[0][m - 100:m - 95] == NONE)


@pytest.mark.gpu
def test_query_queue_overflow(hc, oracle):
    """R isotropic and far apart, except 4000 rows in a tiny ball; the queries sit in the same ball. The survivor
    sample of [Q; R] sees mostly the far pairs, so the queue sized from it overflows and the compare has to re-decide."""
    rng = np.random.default_rng(91)
    n, m, K = 131072, 2048, 30
    R = rng.random((n, K))
    ball = rng.choice(n, 4000, replace=False)
    R[ball] = 0.5 + 2e-8 * rng.standard_normal((4000, K))
    Q = 0.5 + 2e-8 * rng.standard_normal((m, K))
    hc.set_spline(R)
    got = hc.query_compare(Q, THR)
    st = hc.query_last_stats()
    assert st["passes"] >= 2, st
    assert len(got[0]) == m * 4000
    assert same_list(got, hc.query_compare(Q, THR, VARIANTS["EXACT"]))
    sub = np.arange(0, m, 97)
    want = oracle.radius(R, Q[sub], THR)
    keep = np.isin(got[0], sub)
    assert same_list((np.searchsorted(sub, got[0][keep]).astype(np.uint32), got[1][keep], got[2][keep]), want)


@pytest.mark.gpu
def test_query_planner_pairs(hc):
    """10^6 rows of 6 columns in 25 tight clusters: 4 % of all pairs are edges. Planned for the whole triangle, no
    tensor-core (or DMMA) queue could hold the survivors and the filter-free kernel would run; planned for the query's own
    panels, the tensor-core filter runs."""
    import scema_b200
    import torch
    rng = np.random.default_rng(17)
    n, m, K = 1000000, 256, 6
    centres = rng.random((25, K))
    R = centres[rng.integers(0, 25, n)] + 1e-7 * rng.random((n, K))
    Q = centres[rng.integers(0, 25, m)] + 1e-7 * rng.random((m, K))
    hc.set_spline(R)
    got = hc.query_compare(Q, THR)
    st = hc.query_last_stats()
    assert st["variant"] == VARIANTS["TC"], st
    assert same_list(got, hc.query_compare(Q, THR, VARIANTS["EXACT"]))
    # what the whole-triangle plan of the same rows decides, from the same survivor sample
    cat = np.concatenate([Q, R])
    h2 = scema_b200.HistCluster(0)
    h2.set_spline(cat)

    def stop(a, b, d):
        raise StopIteration

    with pytest.raises(StopIteration):
        h2.compare_stream(THR, stop, panels_per_chunk=1)
    p = h2.tc_last_plan()
    h2.close()
    counts = [p["one_slice"], p["two_slices"], p["one_slice_raw"], p["two_slices_raw"], p["dmma"], p["projected"]]
    N = n + m
    total = torch.cuda.get_device_properties(0).total_memory
    whole = scema_b200.binding.tc_choose(N * (N - 1) // 2, K, counts, p["sample"], total // 2)
    assert whole[0] == -1, (whole, p)
    prefix = scema_b200.binding.tc_choose(st["filter_pairs"], K, counts, p["sample"], total // 2)
    assert prefix[0] in (1, 2, 3), (prefix, p)


_SELECTION_SCRIPT = r"""
import hashlib, sys
sys.path.insert(0, sys.argv[1])
import numpy as np, scema_b200
rng = np.random.default_rng(5)
c = rng.random((400, 60))
R = c[rng.integers(0, 400, 20000)] + 1e-7 * rng.standard_normal((20000, 60))
Q = c[rng.integers(0, 400, 3000)] + 1e-7 * rng.standard_normal((3000, 60))
hc = scema_b200.HistCluster(0)
hc.set_spline(R)
j, i, d = hc.query_compare(Q, 1e-6)
st = hc.query_last_stats()
ix, dk = hc.query_knn(Q, 8)
print(hashlib.sha256(j.tobytes() + i.tobytes() + d.tobytes() + ix.tobytes() + dk.tobytes()).hexdigest(), len(j), st["variant"])
"""


@pytest.mark.gpu
def test_query_kernel_selections():
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
    assert int(out["default"][1]) > 0 and all(int(v[2]) == VARIANTS["TC"] for v in out.values()), out


@pytest.mark.gpu
def test_query_leaves_context_state(hc, tmp_path):
    import scema_b200
    from scema_b200 import synth
    n = 20000
    rows = synth.rows(14, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
    Q = rows[:3000] + 1e-7
    hc.set_spline(rows)
    hc.knn(4)
    knn_stats = hc.knn_last_stats()
    hc.compare(THR)

    def snapshot(tag):
        d = tmp_path / tag
        d.mkdir()
        hc.write_similar_hist(str(d / "last.%u.similar_hist"))
        files = {f: (d / f).read_bytes() for f in sorted(os.listdir(d))}
        e = hc.get_edges()
        return ((e[0].copy(), e[1].copy(), e[2].copy().view(np.uint64)), hc.get_degrees(n), files, hc.counters(), hc.timings(),
                hc.last_audit(), hc.knn_last_stats())

    before = snapshot("before")
    assert before[-1] == knn_stats
    cross = hc.query_compare(Q, THR)
    hc.query_knn(Q, 8)
    with pytest.raises(scema_b200.ScemaError):
        hc.query_knn(Q, 0)
    with pytest.raises(scema_b200.ScemaError):
        hc.query_compare(Q[:, :10], THR)
    after = snapshot("after")
    for x, y in zip(before, after):
        if isinstance(x, tuple):
            assert all(np.array_equal(p, q) for p, q in zip(x, y))
        elif isinstance(x, np.ndarray):
            assert np.array_equal(x, y)
        else:
            assert x == y
    # the cross edges: kept across scema_compare, scema_knn and scema_query_knn, replaced by the next query_compare,
    # gone after a failing one
    cross = hc.query_compare(Q, THR)
    hc.compare(THR)
    hc.knn(2)
    hc.query_knn(Q, 3)
    hc.set_spline(rows[:5000])
    assert same_list(hc.query_edges(len(cross[0])), cross)
    with pytest.raises(scema_b200.ScemaError):
        hc.query_compare(Q, THR, 7)
    with pytest.raises(scema_b200.ScemaError) as e:
        hc.query_edges(1)
    assert e.value.code == 5


@pytest.mark.gpu
def test_query_errors(hc):
    import scema_b200
    INVALID, STATE = 1, 5
    fresh = scema_b200.HistCluster(0)
    for call in (lambda: fresh.query_compare(np.zeros((2, 6)), THR), lambda: fresh.query_knn(np.zeros((2, 6)), 2)):
        with pytest.raises(scema_b200.ScemaError) as e:
            call()
        assert e.value.code == STATE
    fresh.close()
    hc.set_spline(np.random.default_rng(0).random((100, 6)))
    q = np.zeros((3, 6))
    L = hc._L
    for call in (lambda: hc.query_compare(np.zeros((3, 7)), THR), lambda: hc.query_compare(q, THR, 4),
                 lambda: hc.query_compare(q, THR, -1), lambda: hc.query_knn(q, 0), lambda: hc.query_knn(q, 33),
                 lambda: hc.query_knn(np.zeros((3, 5)), 2), lambda: hc.query_knn(q, 2, 9),
                 lambda: hc._ck(L.scema_query_compare(hc._h, None, 0, 3, 6, THR, 3, None)),
                 lambda: hc._ck(L.scema_query_knn(hc._h, None, 0, 3, 6, 2, 3, None, None)),
                 lambda: hc._ck(L.scema_query_compare(hc._h, q.ctypes.data, 1, (1 << 32) - 100, 6, THR, 3, None))):
        with pytest.raises(scema_b200.ScemaError) as e:
            call()
        assert e.value.code == INVALID
    # empty results
    for t in (0.0, -1.0, float("nan")):
        assert len(hc.query_compare(q, t)[0]) == 0
    assert len(hc.query_compare(np.zeros((0, 6)), THR)[0]) == 0
    assert hc.query_knn(np.zeros((0, 6)), 3)[0].shape == (0, 3)
    hc.set_spline(np.zeros((0, 6)))
    assert len(hc.query_compare(q, THR)[0]) == 0
    idx, d = hc.query_knn(q, 3)
    assert np.all(idx == NONE) and np.all(np.isinf(d))


@pytest.mark.gpu
def test_query_c4_million(hc, oracle):
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
    R = hc.get_spline()
    del steps
    rng = np.random.default_rng(29)
    m = 10000
    near = R[rng.integers(0, n, m // 2)] + 2e-8 * rng.standard_normal((m // 2, R.shape[1]))   # below the threshold
    other = synth.rows(77, m - m // 2, bench.CLUSTER, w["P"], bench.wl_amp(w), synth.default_pert(bench.THR, w["P"]))
    Q = np.concatenate([near, other])
    got = hc.query_compare(Q, bench.THR)
    st = hc.query_last_stats()
    assert filter_pairs_ok(st, m, n) and len(got[0]) >= m // 2, st
    hc.set_spline(np.concatenate([Q, R]))
    hc.compare(bench.THR)
    a, b, d = hc.get_edges()
    keep = (a < m) & (b >= m)
    assert same_list(got, (a[keep], b[keep] - m, d[keep])), st
    e = rng.choice(len(got[0]), min(2000, len(got[0])), replace=False)
    for t in e[:200]:
        j, i = int(got[0][t]), int(got[1][t])
        ww = oracle.radius(R[i:i + 1], Q[j:j + 1], bench.THR)
        assert len(ww[0]) == 1 and ww[2][0].view(np.uint64) == got[2][t].view(np.uint64)
