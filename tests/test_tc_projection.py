"""The projected tcgen05 filter: rows centred on the sample's column medians, written as 11 coordinates in an orthonormal
basis of the sample's leading principal directions plus the norm of the residual, one fp16 slice, 16 columns.

For an orthonormal basis |z_a - z_b| <= |a - b|, so the projected filter is exactly as conservative as the 64-column one
whatever the basis; the basis only decides how many pairs survive (DESIGN.md "K2-TC", projection). The CPU part restates
centre -> basis -> projection -> residual -> scale -> fp16 -> fold in numpy and checks that no reference edge gets a
negative accumulator even after the whole budgeted tensor-core error is taken off; the GPU part checks the hardware's
accumulators against the same contraction and the edge lists against the other filters."""
import os
import subprocess
import sys

import numpy as np
import pytest

import scema_b200
from scema_b200 import binding, synth

THR = 1e-6
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 11
CG1 = 2.0 ** -9          # one-slice guard band
CPROJ = 2.0 ** -32       # FP64 rounding of the projection, relative to |a'|^2
T0_PROJ = 1.0 + 2.0 ** -30
SAMPLE = 4096


def h16z(v):
    """fp16 rounding with subnormal results flushed to zero (k_tc_prep, k_tc_prep_proj)."""
    f = np.asarray(v, dtype=np.float64).astype(np.float16).astype(np.float64)
    return np.where(np.abs(f) < 2.0 ** -14, 0.0, f)


def sample_rows(rows):
    n = rows.shape[0]
    ns = min(n, SAMPLE)
    return rows[np.arange(ns) * (n // ns)]


def centre_of(rows):
    """column medians of the sample, non-finite entries skipped (k_tc_centre_median)"""
    smp = sample_rows(rows)
    m = np.zeros(rows.shape[1])
    for k in range(rows.shape[1]):
        v = np.sort(smp[:, k][np.isfinite(smp[:, k])])
        m[k] = v[(len(v) - 1) // 2] if len(v) else 0.0
    return m


def moments_of(rows, m):
    """second moments about m of the sample, products that are not finite skipped (k_tc_cov)"""
    x = sample_rows(rows) - m
    p = x[:, :, None] * x[:, None, :]
    p = np.where(np.isfinite(p), p, 0.0)
    return p.sum(0)


def projected_image(rows, thr, basis=None):
    """numpy restatement of the operand preparation: -> (A [n, 16], B [n, 16], |z|^2 scaled, survivor-always mask)"""
    n, K = rows.shape
    m = centre_of(rows)
    if basis is None:
        got = binding.tc_basis(moments_of(rows, m))
        assert got is not None
        basis, delta = got
        assert delta <= 2.0 ** -32
    a = rows - m
    with np.errstate(all="ignore"):
        nrm = (a * a).sum(1)
        wild = ~np.isfinite(nrm)
        a0 = np.where(wild[:, None], 0.0, a)
        y = a0 @ basis.T
        rho = np.sqrt(((a0 - y @ basis) ** 2).sum(1))
    maxabs = np.abs(a0[~wild]).max() if np.any(~wild) else 0.0
    s = 2.0 ** (11 - int(np.floor(np.log2(maxabs)))) if maxabs > 0 else 1.0
    s /= 8.0
    z = np.concatenate([y, rho[:, None]], axis=1) * s
    big = np.any(~(np.abs(z) < 4096.0), axis=1) & ~wild
    z[big | wild] = 0.0
    nz = (z * z).sum(1)
    eps = 2.0 ** -53
    T0 = thr * thr * (1 + (2 * K + 16) * eps) * (1 + 4 * eps) + (2 * K + 4) * 4.9406564584124654e-324
    T0s = T0 * T0_PROJ * s * s
    nfull = np.where(wild, 0.0, nrm) * s * s
    h = 0.5 * (nz * (1 - CG1) - CPROJ * nfull - T0s * (0.5 + 2 * CG1) - K * 2.0 ** -7)
    P, Q = 32768.0, 8.0
    always = wild | big | ~(-h <= 32768.0 * P)
    x0 = np.where(always, 65504.0, h16z(-h / P))
    x1 = np.where(always, 0.0, h16z((-h - P * x0) / Q))
    zh = h16z(z)
    A = np.concatenate([zh, x0[:, None], x1[:, None], np.full((n, 1), P), np.full((n, 1), Q)], axis=1)
    B = np.concatenate([zh, np.full((n, 1), P), np.full((n, 1), Q), x0[:, None], x1[:, None]], axis=1)
    return A, B, always


def check_sound(rows, thr, basis=None):
    """Every reference edge keeps a non-negative accumulator after the exact sliced sum is pushed down by the budgeted
    error of one K = 16 tensor-core step (2 x 2^-18 of the sum of the magnitudes of the products). -> fraction of the
    non-edge pairs the filter rejects."""
    A, B, always = projected_image(rows, thr, basis)
    n = rows.shape[0]
    rejected = total = 0
    for r0 in range(0, n, 256):
        r1 = min(n, r0 + 256)
        acc = A[r0:r1] @ B.T
        mag = np.abs(A[r0:r1]) @ np.abs(B).T
        low = acc - 2.0 * 2.0 ** -18 * mag
        with np.errstate(all="ignore"):
            d = np.sqrt(((rows[r0:r1, None, :] - rows[None, :, :]) ** 2).sum(-1))
        upper = np.arange(r0, r1)[:, None] < np.arange(n)[None, :]
        edge = (d < thr) & upper
        assert not np.any(edge & (low < 0)), "a reference edge was rejected by the projected filter"
        rejected += int(np.sum((acc < 0) & upper & ~edge))
        total += int(np.sum(upper & ~edge))
    return rejected / max(total, 1)


def c4_rows(n, seed=11):
    return synth.rows(seed, n, 16, 10, 5e-3, synth.default_pert(THR, 10))


def c4s_rows(n, seed=12):
    return synth.rows(seed, n, 16, 10, 2e-2, synth.default_pert(THR, 10), model=1, spread=5e-3)


def plant(rows, rng, count, scales=(1 - 4e-16, 1 - 2e-16, 1.0, 1 + 2e-16, 1 + 4e-16), thr=THR):
    """pairs planted a few ulp either side of the threshold: row 2q + 1 = row 2q + thr * f * u for a unit u"""
    out = rows.copy()
    for q in range(count):
        u = rng.standard_normal(rows.shape[1])
        u /= np.linalg.norm(u)
        out[2 * q + 1] = out[2 * q] + thr * scales[q % len(scales)] * u
    return out


# ------------------------------------------------------------------------------------------------ CPU


@pytest.mark.parametrize("model", ["c4", "c4s"])
def test_projection_sound_on_workload_rows(model):
    rng = np.random.default_rng(1)
    rows = c4_rows(3000) if model == "c4" else c4s_rows(3000)
    rows = plant(rows, rng, 200)
    assert check_sound(rows, THR) > 0.99   # and it still filters


def test_projection_sound_off_span_and_missed_cluster():
    rng = np.random.default_rng(2)
    n, K = 3000, 60
    # most of the energy outside any 11-dimensional basis: a low-rank sample, full-rank rows elsewhere
    rows = rng.standard_normal((n, 3)) @ rng.standard_normal((3, K)) * 1e-4
    rows[n // 2:] += rng.standard_normal((n - n // 2, K)) * 1e-5
    check_sound(plant(rows, rng, 100, thr=3e-5), 3e-5)
    # a basis taken from a sample that misses a whole cluster: the sampled rows (every 2nd) lie in one cluster, the
    # others in a second one far away in directions the basis does not contain
    n2 = 2 * SAMPLE
    rows2 = c4_rows(n2, seed=5)
    far = rng.standard_normal(K)
    rows2[1::2] += 1e-3 * far / np.linalg.norm(far) + rng.standard_normal((SAMPLE, K)) * 1e-7
    check_sound(plant(rows2[:3000], rng, 100), THR, basis=binding.tc_basis(moments_of(rows2, centre_of(rows2)))[0])


def test_projection_sound_isotropic_offsets_and_nonfinite():
    rng = np.random.default_rng(3)
    iso = rng.standard_normal((2500, 60)) * 1e-3
    check_sound(plant(iso, rng, 100, scales=(1 - 1e-15, 1.0, 1 + 1e-15), thr=0.9e-3), 0.9e-3)
    shifted = c4_rows(2500, seed=7) + 1e3            # large common offset: centring removes it
    check_sound(plant(shifted, rng, 100), THR)
    bad = plant(c4_rows(2500, seed=8), rng, 100)
    bad[300] = np.nan
    bad[301, 5] = np.inf
    bad[302, :] = -np.inf
    A, B, always = projected_image(bad, THR)
    assert always[300] and always[301] and always[302] and always.sum() == 3
    acc = A @ B.T
    assert np.all(acc[300, :] >= 0) and np.all(acc[:, 301] >= 0)   # rows with a non-finite norm survive against everybody
    check_sound(bad, THR)


def test_basis_is_deterministic_and_orthonormal():
    rows = c4_rows(20000)
    C = moments_of(rows, centre_of(rows))
    b1, d1 = binding.tc_basis(C)
    b2, d2 = binding.tc_basis(C.copy())
    assert np.array_equal(b1.view(np.uint64), b2.view(np.uint64)) and d1 == d2
    assert b1.shape == (R, 60) and d1 <= 2.0 ** -40
    assert np.abs(b1 @ b1.T - np.eye(R)).max() < 1e-14
    # the leading eigenvectors' span: the basis captures what an exact eigendecomposition captures
    w, V = np.linalg.eigh(C)
    top = V[:, ::-1][:, :R]
    assert np.trace(b1 @ C @ b1.T) >= (1 - 1e-9) * np.trace(top.T @ C @ top)
    for k in range(R):                                   # sign: largest-magnitude component positive
        assert b1[k, np.argmax(np.abs(b1[k]))] > 0
    assert binding.tc_basis(C[:12, :12]) is None         # rows narrower than 16 columns keep the 64-column filter
    C2 = C.copy()
    C2[3, 4] = np.nan
    assert binding.tc_basis(C2) is None
    assert binding.tc_basis(np.zeros((60, 60))) is not None   # degenerate moments: still an orthonormal basis


def test_choice_with_the_projected_count():
    P = 1000000 * 999999 // 2
    big = 1 << 40
    ch = binding.tc_choose
    assert ch(P, 60, (8, 0, 8192, 8192, 0, 8), 8192, big)[:2] == (3, 1)            # as selective as one slice: cheaper
    assert ch(P, 60, (8, 0, 8192, 8192, 0), 8192, big)[:2] == (1, 1)               # five counts: never projected
    assert ch(P, 60, (8, 0, 8192, 8192, 0, 8192), 8192, big)[:2] == (1, 1)         # isotropic rows: the projection keeps everybody
    assert ch(P, 60, (8, 0, 8192, 8192, 0, 4000), 8192, big)[:2] == (1, 1)
    assert ch(P, 12, (8, 0, 8192, 8192, 0, 0), 8192, big)[:2] == (1, 1)            # narrower than 16 columns: not a candidate
    assert ch(P, 300, (8, 8, 8192, 8192, 0, 0), 8192, big)[:2] == (1, 1)           # wider than one chunk: not a candidate
    assert ch(P, 60, (4000, 3, 8192, 8192, 0, 4000), 8192, big)[:2] == (2, 1)


# ------------------------------------------------------------------------------------------------ GPU


def unswizzle32(buf, n_pad):
    """projected operand bytes as they sit in memory -> float64 [n_pad, 16]"""
    b = buf.reshape(n_pad // 128, 128, 2, 16)
    out = np.empty_like(b)
    r = np.arange(128)
    for c in range(2):
        out[:, r, c, :] = b[:, r, c ^ ((r >> 2) & 1), :]
    return out.reshape(n_pad, 32).view(np.float16).astype(np.float64)


@pytest.fixture
def hc():
    h = scema_b200.HistCluster(0)
    yield h
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["c4", "c4s", "iso"])
def test_projected_accumulators_match_fp64(hc, model):
    rng = np.random.default_rng(4)
    n = 4000
    rows = {"c4": lambda: c4_rows(n), "c4s": lambda: c4s_rows(n), "iso": lambda: rng.standard_normal((n, 60)) * 1e-3}[model]()
    thr = 1e-3 if model == "iso" else THR
    rows = plant(rows, rng, 100, thr=thr)
    hc.set_spline(rows)
    acc, ha, hb = hc.tc_debug(thr, n, 3)
    n_pad = acc.shape[0]
    A, B = unswizzle32(ha, n_pad), unswizzle32(hb, n_pad)
    want = A @ B.T
    absum = np.abs(A) @ np.abs(B).T
    ti = np.arange(n_pad)[:, None] // 256
    tj = np.arange(n_pad)[None, :] // 256
    must = tj >= ti
    assert not np.any(np.isnan(acc[must])) and np.all(np.isnan(acc[~must]))
    err = np.abs(acc.astype(np.float64) - want)
    budget = 2 * 2.0 ** -18 * absum
    assert np.all(err[must] <= 0.25 * budget[must] + 1e-30), float(np.max(err[must] / np.maximum(budget[must], 1e-300)))
    # the image is the numpy restatement's (same centre, basis, scale and fold; FP64 sums in another order may move a
    # coordinate across an fp16 rounding boundary: one fp16 ulp)
    A_np, B_np, _ = projected_image(rows, thr)
    assert np.all(np.abs(A[:n, :12] - A_np[:, :12]) <= 2.0 ** -10 * np.abs(A_np[:, :12]) + 2.0 ** -24)
    assert np.array_equal(A[:, :12], B[:, :12])
    P, Q = 32768.0, 8.0
    fold, fold_np = P * A[:n, 12] + Q * A[:n, 13], P * A_np[:, 12] + Q * A_np[:, 13]
    assert np.all(np.abs(fold - fold_np) <= 2.0 ** -20 * np.abs(fold_np) + 2.0 ** -6)
    assert np.array_equal(A[:, 12:14], B[:, 14:16]) and np.all(A[:n, 14] == P) and np.all(B[:n, 12] == P)
    assert np.all(A[n:, 12] == -65504.0)
    for r0 in range(0, n, 128):
        d = np.sqrt(((rows[r0:r0 + 128, None, :] - rows[None, :, :]) ** 2).sum(-1))
        edge = (d < thr) & (np.arange(r0, min(r0 + 128, n))[:, None] < np.arange(n)[None, :])
        assert not np.any(edge & np.signbit(acc[r0:r0 + 128, :n][: edge.shape[0]])), "a true edge was rejected"


def _run(code, args, **env):
    r = subprocess.run([sys.executable, "-c", code, *args], env=dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.path.join(ROOT, "tests"), **env), capture_output=True,
                       text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), (r.stdout[-3000:], r.stderr[-3000:])
    return r.stdout


_PINNED = (
    "import numpy as np, sys\n"
    "import scema_b200\n"
    "from scema_b200 import PAIRS_TC, PAIRS_DMMA\n"
    "from test_tc_projection import c4_rows, c4s_rows, plant\n"
    "rng = np.random.default_rng(9)\n"
    "hc = scema_b200.HistCluster(0)\n"
    "for name, rows in (('c4', c4_rows(16384)), ('c4s', c4s_rows(16384))):\n"
    "    rows = plant(rows, rng, 400)\n"
    "    hc.set_spline(rows)\n"
    "    n = hc.compare(1e-6, PAIRS_TC); a, b, d = hc.get_edges(); c = hc.counters(); plan = hc.tc_last_plan()\n"
    "    np.save('%s/%s_%s.npy' % (sys.argv[1], name, sys.argv[2]), np.stack([a.astype(np.float64), b.astype(np.float64), d]))\n"
    "    assert c['tc_slices'] == 1 or sys.argv[2] == '2', c\n"
    "    assert plan['projected_chosen'] == (sys.argv[2] == '3'), plan\n"
    "    assert hc.last_audit()[1] == 0\n"
    "    print(name, n, c['survivors'], plan)\n"
    "print('ok')\n")


@pytest.mark.gpu
def test_pinned_filters_give_identical_edges(tmp_path):
    """Config-2-sized rows of both models with planted guard-band pairs: the projected filter, one slice and the DMMA
    filter emit the same edge list (ids, order, distance bits); the run-time audit stays green."""
    for pin in ("3", "1"):
        _run(_PINNED, [str(tmp_path), pin], SCEMA_TC_SLICES=pin, SCEMA_AUDIT="200000")
    h = scema_b200.HistCluster(0)
    rng = np.random.default_rng(9)
    for name, rows in (("c4", c4_rows(16384)), ("c4s", c4s_rows(16384))):
        rows = plant(rows, rng, 400)
        h.set_spline(rows)
        h.compare(THR, scema_b200.PAIRS_DMMA)
        a, b, d = h.get_edges()
        want = np.stack([a.astype(np.float64), b.astype(np.float64), d])
        for pin in ("3", "1"):
            got = np.load(tmp_path / f"{name}_{pin}.npy")
            assert got.shape == want.shape and np.array_equal(got.view(np.uint64), want.view(np.uint64)), (name, pin)
        assert len(a) > 400
    h.close()


@pytest.mark.gpu
def test_automatic_choice_takes_the_projection_on_workload_rows(hc):
    """c4- and c4s-shaped rows: the sample's sixth count is as small as the one-slice count, the cost model takes the
    projected filter, and the edges equal the filter-free kernel's. Isotropic rows keep the 64-column filter."""
    rng = np.random.default_rng(5)
    for rows in (c4_rows(20000), c4s_rows(20000)):
        hc.set_spline(plant(rows, rng, 200))
        n = hc.compare(THR, scema_b200.PAIRS_TC)
        got = hc.get_edges()
        plan = hc.tc_last_plan()
        assert plan["projected_chosen"] and hc.counters()["tc_slices"] == 1, plan
        assert hc.compare(THR, scema_b200.PAIRS_EXACT) == n
        want = hc.get_edges()
        assert all(np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)) for x, y in zip(got, want))
    # isotropic rows, threshold at half the typical distance: |z_a - z_b| keeps ~ 11/60 of it, most pairs survive
    hc.set_spline(rng.standard_normal((20000, 60)) * 1e-3)
    hc.compare(0.5 * np.sqrt(120.0) * 1e-3, scema_b200.PAIRS_TC)
    plan = hc.tc_last_plan()
    assert not plan["projected_chosen"] and plan["projected"] > 8 * plan["one_slice"] // 10, plan


@pytest.mark.gpu
def test_pipelined_cluster_with_late_rows_outside_the_span(oracle, monkeypatch):
    """scema_cluster range by range: the basis is frozen after the first range; later histories of another shape (outside
    its span) land in the residual coordinate. Same edges as the oracle."""
    monkeypatch.setenv("SCEMA_PIPELINE_MIN_N", "4096")
    P = 10
    n = 21000
    off = synth.offsets(13, n, 16, 36, 36)
    st = synth.histories(13, n, 16, 2e-2, synth.default_pert(THR, P), off, model=1, spread=5e-3)
    late = synth.histories(14, n, 16, 5e-3, synth.default_pert(THR, P), off)
    cut = int(off[15000])
    st[cut:] = late[cut:] * 3.0
    h = scema_b200.HistCluster(0)
    ne = h.cluster(st, off, None, P, THR)
    c, plan = h.counters(), h.tc_last_plan()
    assert c["pipeline_ranges"] == 2 and plan["projected_chosen"], (c, plan)
    a, b, d = h.get_edges()
    wi, wj, wd, _ = oracle.all_pairs(oracle.splinify_batch(st, off, P), THR)
    assert ne == len(wi) and np.array_equal(a, wi) and np.array_equal(b, wj)
    assert np.array_equal(d.view(np.uint64), wd.view(np.uint64))
    h.close()


@pytest.mark.gpu
def test_two_gpus_projected(oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    rows = plant(c4_rows(20011), np.random.default_rng(6), 200)
    wi, wj, wd, _ = oracle.all_pairs(rows, THR)
    m = scema_b200.MultiCluster([0, 1])
    ne = m.compare_rows(rows, THR, scema_b200.PAIRS_TC)
    a, b, d = m.first.get_edges()
    assert ne == len(wi) and np.array_equal(a, wi) and np.array_equal(b, wj)
    assert np.array_equal(d.view(np.uint64), wd.view(np.uint64))
    assert m.first.tc_last_plan()["projected_chosen"]
    m.close()
