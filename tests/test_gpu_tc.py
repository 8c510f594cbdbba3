"""The tcgen05 filter (SCEMA_PAIRS_TC): operand layout, fold columns, the accumulation-error model its
guard band relies on, and edge-list parity on inputs chosen to stress it (wide dynamic range, heavy
cancellation, pairs planted a few ulp either side of the threshold at several norm scales).

The filter's soundness argument (DESIGN.md "K2-TC") ASSUMES that one tcgen05.mma kind::f16 step returns
c + sum of 16 exact products with an error of at most 2^-18 (|c| + sum |products|). The first test pins
that assumption on the hardware with a 4x margin; everything else is bit-exact parity with the oracle.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import scema_b200
from scema_b200 import synth, PAIRS_TC, PAIRS_EXACT

pytestmark = pytest.mark.gpu
THR = 1e-6
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def edges_equal(got, want):
    return (len(got[0]) == len(want[0]) and np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
            and np.array_equal(bits(got[2]), bits(want[2])))


def unswizzle(buf, n_pad):
    """operand bytes as they sit in memory -> (hi, lo) float64 [n_pad, 64]"""
    b = buf.reshape(n_pad // 128, 2, 128, 8, 16)  # block, slice, row, stored 16-byte chunk, bytes
    out = np.empty_like(b)
    r = np.arange(128)
    for c in range(8):
        out[:, :, r, c, :] = b[:, :, r, c ^ (r & 7), :]
    h = out.reshape(n_pad // 128, 2, 128, 128).view(np.float16).astype(np.float64)
    return h[:, 0].reshape(n_pad, 64), h[:, 1].reshape(n_pad, 64)


def datasets():
    rng = np.random.default_rng(3)
    n = 1100
    yield "clusters", synth.rows(11, n, 16, 10, 5e-3, synth.default_pert(THR, 10)), THR
    yield "gauss", rng.standard_normal((n, 60)) * 1e-3, 1e-3
    alt = np.tile(np.array([1.0, -1.0]), 30)[None, :] * (1e-2 + 1e-6 * rng.standard_normal((n, 60)))
    yield "cancel", alt * np.where(rng.random((n, 1)) < 0.5, 1.0, -1.0), 1e-5   # a.b = +-|a||b|: worst cancellation
    yield "ranges", rng.standard_normal((n, 60)) * 10.0 ** rng.integers(-12, -2, size=(n, 1)), 1e-7
    yield "k18", rng.standard_normal((n, 18)) * 1e-2, 1e-2
    # ten decades INSIDE every row and a larger matrix (16.8M accumulators): most products are far below the running sum
    yield "inrow", rng.standard_normal((4096, 60)) * 10.0 ** rng.uniform(-10, 0, size=(4096, 60)), 1e-4


@pytest.mark.parametrize("slices", [2, 1])
@pytest.mark.parametrize("name,rows,thr", list(datasets()), ids=[d[0] for d in datasets()])
def test_tc_accumulators_match_sliced_fp64(hc, name, rows, thr, slices):
    """Every accumulator the tensor core produced == the same sliced products summed in FP64 from the
    operand copies, within a quarter of the error the guard band budgets for; the operand copies
    reproduce s*a to 2^-22 and fold -h_i-h_j as documented; and no true edge has a negative accumulator."""
    n, K = rows.shape
    rows0 = rows
    hc.set_spline(rows)
    acc, ha, hb = hc.tc_debug(thr, n, slices)
    n_pad = acc.shape[0]
    ahi, alo = unswizzle(ha, n_pad)
    bhi, blo = unswizzle(hb, n_pad)
    want = ahi @ bhi.T
    absum = np.abs(ahi) @ np.abs(bhi).T
    if slices == 2:
        want = want + alo @ bhi.T + ahi @ blo.T
        absum = absum + np.abs(alo) @ np.abs(bhi).T + np.abs(ahi) @ np.abs(blo).T
    steps = 12 if slices == 2 else 4
    ti = np.arange(n_pad)[:, None] // 256
    tj = np.arange(n_pad)[None, :] // 256
    must = tj >= ti
    assert not np.any(np.isnan(acc[must])), "a tile of the upper triangle was not written"
    assert np.all(np.isnan(acc[~must])), "a tile below the diagonal was computed"
    err = np.abs(acc.astype(np.float64) - want)
    budget = (steps + 1) * 2.0 ** -18 * absum
    assert np.all(err[must] <= 0.25 * budget[must] + 1e-30), float(np.max(err[must] / np.maximum(budget[must], 1e-300)))
    # data columns: hi + lo == s * (a - m) to 2^-22 relative (+ the fp16 subnormal floor), same in both copies;
    # m = the column means of the (sampled) rows
    m = hc.tc_centre()
    assert m.shape == (K,) and np.array_equal(m, np.sort(rows, axis=0)[(n - 1) // 2])   # all n <= 4096 rows are sampled
    rows = rows - m[None, :]
    finite = np.isfinite((rows ** 2).sum(1))
    M = np.abs(rows[finite]).max()
    s = 2.0 ** (11 - int(np.floor(np.log2(M))))
    a_s = np.zeros((n_pad, 64))
    a_s[:n, :K] = rows * s
    if slices == 2:
        rec = (ahi + alo)[:, :60]
        assert np.all(np.abs(rec[:n] - a_s[:n, :60]) <= 2.0 ** -22 * np.abs(a_s[:n, :60]) + 2.0 ** -13)
        assert np.array_equal(alo[:, :60], blo[:, :60])
    else:  # the lo halves are neither written nor read with one slice
        assert np.all(np.abs(ahi[:n, :60] - a_s[:n, :60]) <= 2.0 ** -11 * np.abs(a_s[:n, :60]) + 2.0 ** -13)
    assert np.array_equal(ahi[:, :60], bhi[:, :60])
    assert np.abs(ahi[:n, :60]).max() < 4096
    # no fp16 subnormal anywhere in the operands (the prep flushes them; the bound budgets for that)
    for arr in ((ahi, alo, bhi, blo) if slices == 2 else (ahi, bhi)):
        nz = np.abs(arr[arr != 0])
        assert nz.size == 0 or nz.min() >= 2.0 ** -14
    # fold columns: P x0 + Q x1 (+ Q x2) == -h_i, h_i as documented (guard 2^-13 / 2^-9)
    P, Q = 32768.0, 8.0
    cg = 2.0 ** -13 if slices == 2 else 2.0 ** -9
    nrm = (a_s[:n] ** 2).sum(1)
    T0 = thr * thr * (1 + (2 * K + 16) * 2.0 ** -53) * (1 + 4 * 2.0 ** -53) * s * s
    h = 0.5 * (nrm * (1 - cg) - T0 * (0.5 + 2 * cg) - K * 2.0 ** -7)
    fold_a = P * ahi[:n, 60] + Q * ahi[:n, 61]
    fold_b = P * bhi[:n, 62] + Q * bhi[:n, 63]
    if slices == 2:
        fold_a = fold_a + Q * alo[:n, 61]
        fold_b = fold_b + Q * blo[:n, 63]
    normal = -h <= 32768.0 * P
    rel = 2.0 ** -30 if slices == 2 else 2.0 ** -21
    assert np.all(np.abs(fold_a[normal] + h[normal]) <= rel * np.abs(h[normal]) + 2.0 ** -10)
    assert np.array_equal(fold_a, fold_b)
    assert np.all(ahi[:n, 62] == P) and np.all(ahi[:n, 63] == Q) and np.all(bhi[:n, 60] == P) and np.all(bhi[:n, 61] == Q)
    if slices == 2:
        assert np.all(alo[:, 60] == 0) and np.all(alo[:, 62:] == 0) and np.all(blo[:, 60:63] == 0)
    assert np.all(ahi[n:, 60] == -65504.0)  # padding rows can never survive
    # soundness on this data: every true edge (FP64 direct differences) has a non-negative accumulator
    for r0 in range(0, n, 64):
        d2 = ((rows0[r0:r0 + 64, None, :] - rows0[None, :, :]) ** 2).sum(-1)
        edge = (np.sqrt(d2) < thr) & (np.arange(r0, min(r0 + 64, n))[:, None] < np.arange(n)[None, :])
        a_blk = acc[r0:r0 + 64, :n][: edge.shape[0]]
        assert not np.any(edge & (np.signbit(a_blk))), "a true edge was rejected by the filter"


def two_blobs(n, spread, seed=2):
    """Two tight blobs at +-base (so the mean is ~0 and centring changes nothing): pairs inside a blob lie `spread`
    of the norm apart, i.e. inside a guard band wider than that and outside a narrower one."""
    rng = np.random.default_rng(seed)
    base = 5e-3 * rng.standard_normal(60)
    rows = base[None, :] * (1 + spread / np.sqrt(2) * rng.standard_normal((n, 60)))
    rows[1::2] *= -1.0
    rows[::50] = rows[2::50][: len(rows[::50])] + 1e-8 * rng.standard_normal((len(rows[::50]), 60))  # a few true edges
    return rows


def test_tc_filter_is_chosen_up_front_from_a_sample():
    """The survivor-density sample decides BEFORE the first launch (one pass, no overflow-and-retry): blobs 3 % of
    their norm wide sit inside the one-slice band (6 %) and outside the two-slice band (1.6 %) -> two slices;
    blobs 0.1 % wide defeat both -> the FP64 DMMA filter; clustered rows -> one slice. Same edge list every time."""
    from oracle.pyoracle import Oracle
    o = Oracle()
    n = 2600
    for name, rows, slices_want in (("3pct", two_blobs(n, 0.03), 2), ("0.1pct", two_blobs(n, 0.001), 0),
                                    ("clusters", synth.rows(3, n, 16, 10, 5e-3, synth.default_pert(THR, 10)), 1)):
        want = o.all_pairs(rows, THR)
        h = scema_b200.HistCluster(0)  # fresh context: default queue capacity
        h.set_spline(rows)
        assert h.compare(THR, PAIRS_TC) == len(want[0]), name
        assert edges_equal(h.get_edges(), want), name
        c, plan = h.counters(), h.tc_last_plan()
        assert c["tc_slices"] == slices_want and c["passes"] == 1 and len(want[0]) >= 40, (name, c, plan)
        assert plan["sample"] == 8192
        if name == "3pct":
            assert plan["one_slice"] > 3000 and plan["two_slices"] < 300 and c["survivors"] < n * 40, plan
            # the same rows and threshold again keep the decision without sampling again
            assert h.compare(THR, PAIRS_TC) == len(want[0]) and h.counters()["passes"] == 1 and h.counters()["tc_slices"] == 2
        if name == "0.1pct":
            assert plan["two_slices"] > 3000 and plan["two_slices_raw"] > 3000 and plan["dmma"] < 50, plan
        h.close()


def test_tc_production_shaped_rows_keep_the_one_slice_filter(oracle):
    """SURVEY 8d C1 / FE_problem.h:1091-1103: every quadrature point follows nearly the same stretch path (model 1 of
    the generator: groups 0.5 % of the norm apart). The guard band of the raw rows would keep every pair; the centred
    filter copies keep only group mates. Edge list identical to the oracle, one pass, one slice; with the centring
    switched off (SCEMA_TC_CENTRE=0 in a child process) the sample sends the same rows to the DMMA filter."""
    n, P = 20000, 10
    rows = synth.rows(7, n, 16, P, 2e-2, synth.default_pert(THR, P), model=1, spread=5e-3)
    nrm = np.linalg.norm(rows, axis=1)
    assert nrm.min() > 0.9 * nrm.max()                       # all on the same path
    want = oracle.all_pairs(rows, THR)
    h = scema_b200.HistCluster(0)
    h.set_spline(rows)
    assert h.compare(THR, PAIRS_TC) == len(want[0]) and len(want[0]) > n
    assert edges_equal(h.get_edges(), want)
    c = h.counters()
    assert c["tc_slices"] == 1 and c["passes"] == 1 and c["survivors"] < 40 * n, c
    h.close()
    code = (
        "import numpy as np, scema_b200\n"
        "from scema_b200 import synth, PAIRS_TC, PAIRS_EXACT\n"
        "rows = synth.rows(7, 6000, 16, 10, 2e-2, synth.default_pert(1e-6, 10), model=1, spread=5e-3)\n"
        "hc = scema_b200.HistCluster(0); hc.set_spline(rows)\n"
        "n1 = hc.compare(1e-6, PAIRS_TC); e1 = hc.get_edges(); c = hc.counters(); plan = hc.tc_last_plan()\n"
        "assert c['tc_slices'] == 0 and c['passes'] == 1 and plan['one_slice'] > 8000 and plan['one_slice_raw'] > 8000 and plan['dmma'] < 50, (c, plan)\n"
        "n2 = hc.compare(1e-6, PAIRS_EXACT); e2 = hc.get_edges()\n"
        "assert n1 == n2 and all(np.array_equal(x.view(np.uint64) if x.dtype == np.float64 else x, y.view(np.uint64) if y.dtype == np.float64 else y) for x, y in zip(e1, e2))\n"
        "print('ok')\n")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, SCEMA_TC_CENTRE="0", PYTHONPATH=ROOT), capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("ok"), (r.stdout, r.stderr)


def test_tc_pinned_one_slice_grows_the_queue():
    """SCEMA_TC_SLICES=1 pins the hi-slice filter: survivors that overflow the queue make it grow (second pass), the
    edge list stays the oracle's."""
    code = (
        "import numpy as np, scema_b200, sys, importlib.util\n"
        "spec = importlib.util.spec_from_file_location('t', %r); t = importlib.util.module_from_spec(spec); spec.loader.exec_module(t)\n"
        "from oracle.pyoracle import Oracle\n"
        "rows = t.two_blobs(2600, 0.03); want = Oracle().all_pairs(rows, 1e-6)\n"
        "h = scema_b200.HistCluster(0); h.set_spline(rows)\n"
        "assert h.compare(1e-6, scema_b200.PAIRS_TC) == len(want[0]) and t.edges_equal(h.get_edges(), want)\n"
        "c = h.counters(); assert c['tc_slices'] == 1 and c['passes'] == 2 and c['survivors'] >= 1300 * 1299, c\n"
        "print('ok')\n") % os.path.abspath(__file__)
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, SCEMA_TC_SLICES="1", PYTHONPATH=ROOT), capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("ok"), (r.stdout, r.stderr)


@pytest.mark.parametrize("scale", [1.0, 1e-150, 1e140, 1e-300])
def test_tc_edges_across_magnitudes(hc, oracle, scale):
    """Same clustered problem at very different magnitudes (rows and threshold scaled together by a power
    of two would be exactly equivalent; a decimal factor is not) — the edge list must equal the oracle's."""
    # at 1e-300 every squared difference underflows in the reference: ALL pairs are edges there
    n = 3000 if scale != 1e-300 else 1200
    rows = synth.rows(21, n, 16, 10, 5e-3, synth.default_pert(THR, 10)) * scale
    thr = THR * scale
    rng = np.random.default_rng(4)
    for q in range(300):  # pairs a few ulp either side of the threshold
        a = int(rng.integers(0, n)); b = (a + n // 2) % n
        u = rng.standard_normal(60); u /= np.linalg.norm(u)
        rows[b] = rows[a] + u * thr * (1 + (q - 150) * 3e-16)
    want = oracle.all_pairs(rows, thr)
    hc.set_spline(rows)
    assert hc.compare(thr, PAIRS_TC) == len(want[0])
    assert edges_equal(hc.get_edges(), want)
    assert len(want[0]) > 1000
    if scale == 1e-300:
        assert len(want[0]) == n * (n - 1) // 2


def test_tc_mixed_norm_scales_and_dense_neighbourhoods(hc, oracle):
    """Rows of very different norms in one batch (the guard band scales with each row's own norm), small
    rows whose fp16 image is zero, and a dense cloud well inside the guard band but outside the threshold."""
    rng = np.random.default_rng(8)
    n = 4000
    rows = rng.standard_normal((n, 60)) * 10.0 ** rng.integers(-5, -1, size=(n, 1))
    rows[:600] = 0.3 + 2e-6 * rng.standard_normal((600, 60))        # |a| ~ 2.3, distances ~ 2e-5: all inside the guard band
    rows[600:900] = 1e-14 * rng.standard_normal((300, 60))          # vanish in fp16 next to the 0.3 rows; all mutual edges
    rows[900] = rows[901] = 0.0
    for q in range(400):
        a = int(rng.integers(1000, n)); b = int(rng.integers(1000, n))
        if a == b:
            continue
        u = rng.standard_normal(60); u /= np.linalg.norm(u)
        rows[b] = rows[a] + u * THR * (1 + (q - 200) * 2e-16)
    want = oracle.all_pairs(rows, THR)
    hc.set_spline(rows)
    assert hc.compare(THR, PAIRS_TC) == len(want[0])
    assert edges_equal(hc.get_edges(), want)
    c = hc.counters()
    # the cloud goes through the exact path whenever a tcgen05 filter runs (the up-front sample may prefer the DMMA
    # filter on rows like these: its band separates the cloud)
    assert c["tc_slices"] == 0 or c["survivors"] >= 600 * 599 // 2
    assert len(want[0]) >= 300 * 299 // 2 + 150


def test_tc_threshold_beyond_all_distances(hc, oracle):
    """thr so large relative to the data that the folded row term saturates: every pair must survive."""
    rows = synth.rows(1, 900, 16, 10, 5e-3, 1e-7)
    for thr in (10.0, 1e30, float("inf")):
        hc.set_spline(rows)
        assert hc.compare(thr, PAIRS_TC) == 900 * 899 // 2
    want = oracle.all_pairs(rows, 10.0)
    hc.compare(10.0, PAIRS_TC)
    assert edges_equal(hc.get_edges(), want)


@pytest.mark.parametrize("P", [11, 32, 50, 64, 106, 107])
def test_tc_wide_rows(hc, oracle, P):
    """K > 60: the row is cut into 64-column chunks (hi slices only, the fold columns in the last chunk, scale one or
    two binades lower so the norms still fit); up to 10 chunks (P <= 106), beyond that the DMMA filter runs."""
    n = 1500
    rows = synth.rows(5, n, 16, P, 5e-3, synth.default_pert(THR, P))
    rng = np.random.default_rng(P)
    for q in range(150):
        a = int(rng.integers(0, n)); b = (a + n // 2) % n
        u = rng.standard_normal(6 * P); u /= np.linalg.norm(u)
        rows[b] = rows[a] + u * THR * (1 + (q - 75) * 3e-16)
    rows[7] = np.nan
    rows[9, 5] = 1e200
    want = oracle.all_pairs(rows, THR)
    hc.set_spline(rows)
    assert hc.compare(THR, PAIRS_TC) == len(want[0])
    assert edges_equal(hc.get_edges(), want)
    assert hc.counters()["tc_slices"] == (1 if P <= 106 else 0)
    assert len(want[0]) > n
    with pytest.raises(scema_b200.ScemaError):
        hc.tc_debug(THR, n)


def test_tc_wide_rows_dense_take_the_filter_free_kernel(oracle):
    """Every pair an edge (wide rows): the sample sees that no filter can help and the filter-free kernel runs at once."""
    n = 2200
    rows = 1e-3 + 1e-9 * np.random.default_rng(0).standard_normal((n, 300))
    h = scema_b200.HistCluster(0)
    h.set_spline(rows)
    assert h.compare(THR, PAIRS_TC) == n * (n - 1) // 2
    assert h.counters()["tc_slices"] == 0 and h.tc_last_plan()["dmma"] > 8000
    want = oracle.all_pairs(rows, THR)
    assert edges_equal(h.get_edges(), want)
    h.close()


def test_tc_threshold_change_rebuilds_operands(hc, oracle):
    """The threshold is baked into the operand copies; a second compare with another threshold on the same
    rows must not reuse them."""
    rows = synth.rows(6, 2500, 16, 10, 5e-3, synth.default_pert(THR, 10))
    hc.set_spline(rows)
    for thr in (THR, 0.3 * THR, 40 * THR, THR):
        want = oracle.all_pairs(rows, thr)
        assert hc.compare(thr, PAIRS_TC) == len(want[0])
        assert edges_equal(hc.get_edges(), want)


def test_tc_single_cta_kernel_and_pinned_slices_match(tmp_path):
    """SCEMA_TC_CG=1 selects the single-CTA kernel (128 x 256 tile per SM; the default is cta_group::2, an SM pair per
    256 x 256 tile), SCEMA_TC_SLICES pins the number of fp16 slices (3: the projected 16-column filter); every
    combination emits the exact kernel's edge list."""
    code = (
        "import numpy as np, scema_b200\n"
        "from scema_b200 import synth, PAIRS_TC, PAIRS_EXACT\n"
        "rows = synth.rows(31, 7000, 16, 10, 5e-3, synth.default_pert(1e-6, 10))\n"
        "hc = scema_b200.HistCluster(0); hc.set_spline(rows)\n"
        "pin = int(__import__('os').environ['SCEMA_TC_SLICES'])\n"
        "n1 = hc.compare(1e-6, PAIRS_TC); e1 = hc.get_edges(); assert hc.counters()['tc_slices'] == (1 if pin == 3 else pin)\n"
        "assert hc.tc_last_plan()['projected_chosen'] == (pin == 3)\n"
        "n2 = hc.compare(1e-6, PAIRS_EXACT); e2 = hc.get_edges()\n"
        "assert n1 == n2 and n1 > 7000\n"
        "assert all(np.array_equal(x.view(np.uint64) if x.dtype == np.float64 else x, y.view(np.uint64) if y.dtype == np.float64 else y) for x, y in zip(e1, e2))\n"
        "print('ok', n1)\n")
    for cg, sl in (("1", "1"), ("1", "2"), ("1", "3"), ("2", "1"), ("2", "2"), ("2", "3")):
        env = dict(os.environ, SCEMA_TC_CG=cg, SCEMA_TC_SLICES=sl, PYTHONPATH=ROOT)
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0 and r.stdout.startswith("ok"), (cg, sl, r.stdout, r.stderr)


def test_tc_single_cta_kernel_on_the_other_paths():
    """The non-default single-CTA kernel (SCEMA_TC_CG=1) through the wide-row, host-buffer-pipeline and norm-band
    paths: same edge list as the filter-free kernel."""
    code = (
        "import os, numpy as np, scema_b200\n"
        "from scema_b200 import synth, PAIRS_TC, PAIRS_EXACT\n"
        "def same(e1, e2):\n"
        "    return all(np.array_equal(x.view(np.uint64) if x.dtype == np.float64 else x, y.view(np.uint64) if y.dtype == np.float64 else y) for x, y in zip(e1, e2))\n"
        "hc = scema_b200.HistCluster(0)\n"
        "rows = synth.rows(32, 5000, 16, 50, 5e-3, synth.default_pert(1e-6, 50))\n"   # K = 300: five chunks
        "hc.set_spline(rows); n1 = hc.compare(1e-6, PAIRS_TC); e1 = hc.get_edges(); n2 = hc.compare(1e-6, PAIRS_EXACT)\n"
        "assert n1 == n2 and n1 > 5000 and same(e1, hc.get_edges()), 'wide'\n"
        "off = synth.offsets(13, 21000, 16, 6, 90); st = synth.histories(13, 21000, 16, 5e-3, synth.default_pert(1e-6, 10), off)\n"
        "n1 = hc.cluster(st, off, None, 10, 1e-6); e1 = hc.get_edges(); assert hc.counters()['pipeline_ranges'] == 2\n"
        "n2 = hc.compare(1e-6, PAIRS_EXACT); assert n1 == n2 and same(e1, hc.get_edges()), 'pipeline'\n"
        "os.environ['SCEMA_NORM_BAND'] = '1'\n"
        "rows = synth.rows(33, 9000, 16, 10, 5e-3, synth.default_pert(1e-6, 10)); hc.set_spline(rows)\n"
        "n1 = hc.compare(1e-6, PAIRS_TC); e1 = hc.get_edges(); assert hc.counters()['band_tiles'] > 0\n"
        "n2 = hc.compare(1e-6, PAIRS_EXACT); assert n1 == n2 and same(e1, hc.get_edges()), 'band'\n"
        "print('ok')\n")
    env = dict(os.environ, SCEMA_TC_CG="1", SCEMA_PIPELINE_MIN_N="4096", PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("ok"), (r.stdout, r.stderr)


def test_cluster_from_host_buffers_is_pipelined_and_identical(oracle, monkeypatch):
    """scema_cluster on a large host batch copies, resamples and compares range by range (cluster_pipelined):
    same spline matrix and edge list as the step-by-step calls; rows that outgrow the scale frozen after the
    first range, and a batch whose survivors overflow the queue (fall back to the ordinary path), included."""
    monkeypatch.setenv("SCEMA_PIPELINE_MIN_N", "4096")
    P = 10
    n = 21000  # ranges of 12288 + 8712 histories
    off = synth.offsets(13, n, 16, 6, 90)
    steps = synth.histories(13, n, 16, 5e-3, synth.default_pert(THR, P), off)
    cases = {"plain": steps}
    big = steps.copy()
    big[int(off[15000]):int(off[15020])] *= 3000.0      # later rows 3000x larger than anything in the first range
    big[int(off[20000]):int(off[20004])] *= 1e6
    cases["outgrows_scale"] = big
    for name, st in cases.items():
        h = scema_b200.HistCluster(0)
        ne = h.cluster(st, off, None, P, THR)
        c = h.counters()
        assert c["pipeline_ranges"] == 2, (name, c)
        got, sp = h.get_edges(), h.get_spline()
        want_sp = oracle.splinify_batch(st, off, P)
        assert np.array_equal(bits(sp), bits(want_sp)), name
        h.set_histories(st, off)
        h.resample(P)
        assert h.compare(THR, PAIRS_EXACT) == ne and edges_equal(h.get_edges(), got), name
        assert ne > n // 4
        # a second call on the same context reuses streams/events
        assert h.cluster(st, off, None, P, THR) == ne and edges_equal(h.get_edges(), got)
        h.close()
    # survivors overflow the queue -> the pipeline hands over to the ordinary path (which grows the buffers)
    n2 = 6000
    off2 = (np.arange(n2 + 1, dtype=np.uint64) * 7)
    st2 = np.tile(np.linspace(0, 1e-3, 7)[:, None], (n2, 6)) + 1e-10 * np.random.default_rng(0).standard_normal((n2 * 7, 6))
    h = scema_b200.HistCluster(0)
    assert h.cluster(st2, off2, None, P, THR) == n2 * (n2 - 1) // 2
    assert h.counters()["pipeline_ranges"] == 0
    h.close()
    monkeypatch.setenv("SCEMA_PIPELINE", "0")
    h = scema_b200.HistCluster(0)
    assert h.cluster(steps, off, None, P, THR) > 0 and h.counters()["pipeline_ranges"] == 0
    h.close()


def test_norm_band_mode(oracle, monkeypatch):
    """SCEMA_NORM_BAND=1: rows sorted by norm, tiles out of the threshold's reach skipped (triangle inequality). Same
    edge list as always — on clustered rows (norms spread: nearly everything skipped), on rows of equal norm (nothing
    can be skipped), with pairs a few ulp either side of the threshold, sharded, and with a NaN row (dense order)."""
    monkeypatch.setenv("SCEMA_NORM_BAND", "1")
    rng = np.random.default_rng(12)
    n = 20000
    clustered = synth.rows(41, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
    for q in range(400):
        a = int(rng.integers(0, n)); b = (a + n // 2) % n
        u = rng.standard_normal(60); u /= np.linalg.norm(u)
        clustered[b] = clustered[a] + u * THR * (1 + (q - 200) * 3e-16)
    sphere = rng.standard_normal((6000, 60))
    sphere *= 5e-3 / np.linalg.norm(sphere, axis=1)[:, None]        # equal norms
    sphere[1::2] = sphere[::2] + 2e-7 * rng.standard_normal((3000, 60)) / np.sqrt(60)
    for name, rows in (("clustered", clustered), ("sphere", sphere)):
        want = oracle.all_pairs(rows, THR)
        h = scema_b200.HistCluster(0)
        h.set_spline(rows)
        assert h.compare(THR, PAIRS_TC) == len(want[0]), name
        assert edges_equal(h.get_edges(), want), name
        c = h.counters()
        nt = (len(rows) + 255) // 256
        assert c["band_tiles"] > 0
        if name == "clustered":
            assert c["band_tiles"] < nt * (nt + 1) // 2 // 5      # most of the triangle is out of reach
        # (rows of equal norm: the filter copies are centred, so their norms differ a little and part of the triangle
        # may still go; what matters is the edge list above)
        # sharded: union of the shards
        parts = []
        for r in range(3):
            h.compare(THR, PAIRS_TC, shard=r, n_shards=3)
            parts.append(h.get_edges())
        a = np.concatenate([p[0] for p in parts]); b = np.concatenate([p[1] for p in parts]); d = np.concatenate([p[2] for p in parts])
        o = np.lexsort((b, a))
        assert edges_equal((a[o], b[o], d[o]), want), name
        # the streamed compare needs row order: the operand copies are rebuilt, same list
        chunks = []
        h.compare_stream(THR, lambda x, y, z: chunks.append((x, y, z)), PAIRS_TC, panels_per_chunk=2)
        assert edges_equal(tuple(np.concatenate([ch[k] for ch in chunks]) for k in range(3)), want), name
        h.close()
    # a pipelined scema_cluster on a context whose last compare ran in norm order must not inherit that order
    monkeypatch.setenv("SCEMA_PIPELINE_MIN_N", "4096")
    off = synth.offsets(13, 9000, 16, 6, 60)
    steps = synth.histories(13, 9000, 16, 5e-3, synth.default_pert(THR, 10), off)
    h = scema_b200.HistCluster(0)
    h.set_histories(steps, off)
    h.resample(10)
    ne = h.compare(THR, PAIRS_TC)
    ref = h.get_edges()
    assert h.counters()["band_tiles"] > 0
    assert h.cluster(steps, off, None, 10, THR) == ne and edges_equal(h.get_edges(), ref)
    assert h.counters()["pipeline_ranges"] >= 2 and h.counters()["band_tiles"] == 0
    assert h.compare(THR, PAIRS_TC) == ne and edges_equal(h.get_edges(), ref) and h.counters()["band_tiles"] > 0
    h.close()
    bad = clustered[:5000].copy()
    bad[17] = np.nan
    want = oracle.all_pairs(bad, THR)
    h = scema_b200.HistCluster(0)
    h.set_spline(bad)
    assert h.compare(THR, PAIRS_TC) == len(want[0]) and edges_equal(h.get_edges(), want)
    assert h.counters()["band_tiles"] == 0
    h.close()


def test_tc_scale_ignores_a_few_outlier_rows(oracle):
    """Five rows nine decades above the rest must not push everybody else into the flushed range of fp16 (where every
    pair would survive and the compare would end on the filter-free kernel): the scale is taken from the rest and the
    outliers are handled like rows with a non-finite norm. Also with the outliers only moderately larger (no gap: the
    largest magnitude rules as before)."""
    n = 3000
    for factor, few_passes in ((1e9, True), (40.0, True)):
        rows = synth.rows(33, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
        rows[[5, 700, 701, 1500, 2999]] *= factor
        rows[701] = rows[700] * (1 + 1e-12)          # two of the large rows nearly equal (the oracle decides whether that is an edge)
        want = oracle.all_pairs(rows, THR)
        h = scema_b200.HistCluster(0)
        h.set_spline(rows)
        assert h.compare(THR, PAIRS_TC) == len(want[0])
        assert edges_equal(h.get_edges(), want)
        c = h.counters()
        assert c["passes"] == 1 and c["survivors"] < 40 * n, (factor, c)
        assert len(want[0]) > n
        h.close()


def test_queue_capacity_follows_the_batch_size():
    """A context that started on a small batch must not read the overflow of its small survivor queue on a later, larger
    batch as 'the one-slice band keeps too much' (and fall back to two slices at half the speed): the capacity is 32
    survivors per history of the CURRENT batch."""
    h = scema_b200.HistCluster(0)
    small = synth.rows(3, 1000, 16, 10, 5e-3, synth.default_pert(THR, 10))
    h.set_spline(small)
    h.compare(THR, PAIRS_TC)
    n = 200000
    d_rows = synth.device_rows(4, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
    h.set_spline(device_ptr=d_rows.data_ptr(), n=n, k=60)
    ne = h.compare(THR, PAIRS_TC)
    c = h.counters()
    assert c["survivors"] > (1 << 20) and c["tc_slices"] == 1 and c["passes"] == 1, c
    assert ne > n
    h.close()


def test_run_time_audit_catches_a_missing_edge(oracle):
    """SCEMA_AUDIT=<samples>: sampled pairs are recomputed exactly after the compare and every reference edge among them
    must be in the list. Green on a sound compare; and it does catch a missing edge — checked by auditing a compare that
    ran with a SMALLER threshold (so true edges of the larger threshold are absent) through the same kernel."""
    code = (
        "import numpy as np, scema_b200\n"
        "from scema_b200 import synth, PAIRS_TC\n"
        "rows = synth.rows(3, 5000, 16, 10, 5e-3, synth.default_pert(1e-6, 10))\n"
        "hc = scema_b200.HistCluster(0); hc.set_spline(rows)\n"
        "ne = hc.compare(1e-6, PAIRS_TC); a = hc.last_audit(); assert a[0] > 100 and a[1] == 0, a\n"
        "print('ok', ne, a)\n")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, SCEMA_AUDIT="300000", PYTHONPATH=ROOT), capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("ok"), (r.stdout, r.stderr)
    # the audit's threshold can be moved by a test hook (SCEMA_AUDIT_THR_FACTOR): edges of 1.5 thr are then "missing"
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, SCEMA_AUDIT="300000", SCEMA_AUDIT_THR_FACTOR="1.5", PYTHONPATH=ROOT),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "audit:" in r.stderr and "missing from the emitted list" in r.stderr, (r.stdout, r.stderr)
