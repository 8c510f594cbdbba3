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


def c4_rows(n, seed=11, K=60):
    """config-4-shaped rows cut to K columns (ceil(K / 6) spline points, the first K of their columns)"""
    P = -(-K // 6)
    return synth.rows(seed, n, 16, P, 5e-3, synth.default_pert(THR, P))[:, :K].copy()


def c4s_rows(n, seed=12, K=60):
    P = -(-K // 6)
    return synth.rows(seed, n, 16, P, 2e-2, synth.default_pert(THR, P), model=1, spread=5e-3)[:, :K].copy()


# every row width the projection accepts at its ends, one chunk of widths the spline points give, odd widths in between
WIDTHS = (16, 17, 18, 24, 30, 42, 54, 59, 60)


def plant(rows, rng, count, scales=(1 - 4e-16, 1 - 2e-16, 1.0, 1 + 2e-16, 1 + 4e-16), thr=THR):
    """pairs planted a few ulp either side of the threshold: row 2q + 1 = row 2q + thr * f * u for a unit u"""
    out = rows.copy()
    for q in range(count):
        u = rng.standard_normal(rows.shape[1])
        u /= np.linalg.norm(u)
        out[2 * q + 1] = out[2 * q] + thr * scales[q % len(scales)] * u
    return out


# ------------------------------------------------------------------------------------------------ CPU


def width_cases(models):
    """(model, K) at every width; the 60-column cases keep the bare model as their id"""
    cases = [(m, K) for m in models for K in WIDTHS]
    return pytest.mark.parametrize("model,K", cases, ids=[m if K == 60 else f"{m}-K{K}" for m, K in cases])


@width_cases(["c4", "c4s"])
def test_projection_sound_on_workload_rows(model, K):
    rng = np.random.default_rng(1)
    n = 3000 if K == 60 else 2000
    rows = c4_rows(n, K=K) if model == "c4" else c4s_rows(n, K=K)
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
    sound_isotropic_offsets_and_nonfinite(60)


@pytest.mark.parametrize("K", [k for k in WIDTHS if k != 60])
def test_projection_sound_isotropic_offsets_and_nonfinite_at_width(K):
    sound_isotropic_offsets_and_nonfinite(K)


def sound_isotropic_offsets_and_nonfinite(K):
    rng = np.random.default_rng(3)
    n = 2500 if K == 60 else 1500
    iso = rng.standard_normal((n, K)) * 1e-3
    check_sound(plant(iso, rng, 100, scales=(1 - 1e-15, 1.0, 1 + 1e-15), thr=0.9e-3), 0.9e-3)
    shifted = c4_rows(n, seed=7, K=K) + 1e3            # large common offset: centring removes it
    check_sound(plant(shifted, rng, 100), THR)
    bad = plant(c4_rows(n, seed=8, K=K), rng, 100)
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


def test_basis_at_every_accepted_width():
    """16 <= K <= 60: the basis is the same bits for the same moments, orthonormal to 1e-14, every row signed so that its
    largest component is positive. 15 and 61 columns are refused (the 64-column filter takes those rows)."""
    for K in range(16, 61):
        rows = c4_rows(3000, seed=K, K=K)
        C = moments_of(rows, centre_of(rows))
        b1, d1 = binding.tc_basis(C)
        b2, d2 = binding.tc_basis(C.copy())
        assert np.array_equal(b1.view(np.uint64), b2.view(np.uint64)) and d1 == d2, K
        assert b1.shape == (R, K) and d1 <= 2.0 ** -32, (K, d1)
        assert np.abs(b1 @ b1.T - np.eye(R)).max() < 1e-14, K
        for k in range(R):
            assert b1[k, np.argmax(np.abs(b1[k]))] > 0, (K, k)
    for K in (15, 61):
        rows = c4_rows(3000, K=K)
        assert binding.tc_basis(moments_of(rows, centre_of(rows))) is None, K


@pytest.mark.parametrize("n", [2, 3, 5, 17])
def test_projection_sound_on_tiny_batches(n):
    """A handful of rows: the moments have rank n - 1 < 11, the basis is completed by the degenerate branch, and the
    image is still sound (each batch plants one pair at the threshold)."""
    for K in (16, 30, 60):
        rows = plant(c4_rows(n, seed=3, K=K), np.random.default_rng(n), 1)
        got = binding.tc_basis(moments_of(rows, centre_of(rows)))
        assert got is not None and got[1] <= 2.0 ** -32, (n, K)
        check_sound(rows, THR)


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


def scheduled_mask(n_pad, cg):
    """Accumulators k_filter_tc<CG> writes over the whole pair matrix: the items of tc_sched.h Sched<CG> (one unit, one
    shard, strips of one column tile, as tc_launch picks for n_pad <= 8192), a row tile being 128 * CG rows."""
    NT, RPC = n_pad // 256, 2 // cg
    mask = np.zeros((n_pad, n_pad), dtype=bool)
    for s in range(NT):                                   # strip s = column tile s
        for I in range(0, min(NT * RPC, (s + 1) * RPC)):  # rows of the strip: count(s) = min(R1, ce) - R0
            J0, J1 = max(I // RPC, s), s + 1
            mask[I * 128 * cg:(I + 1) * 128 * cg, J0 * 256:J1 * 256] = True
    return mask


def near_pairs(rows, thr):
    """(i, j), i < j, of every pair whose FP64 direct distance is below thr: Gram form of the centred rows to find the
    candidates within 2 thr (its cancellation error is far below thr^2 for finite rows of these magnitudes), then the
    direct differences."""
    n = rows.shape[0]
    a = rows - rows.mean(0)
    nrm = (a * a).sum(1)
    out_i, out_j = [], []
    for r0 in range(0, n, 1024):
        d2 = nrm[r0:r0 + 1024, None] + nrm[None, :] - 2.0 * (a[r0:r0 + 1024] @ a.T)
        i, j = np.nonzero(d2 < 4.0 * thr * thr)
        i = i + r0
        keep = i < j
        i, j = i[keep], j[keep]
        d = np.sqrt(((rows[i] - rows[j]) ** 2).sum(1))
        out_i.append(i[d < thr])
        out_j.append(j[d < thr])
    return np.concatenate(out_i), np.concatenate(out_j)


def check_projected_accumulators(hc, rows, thr, cg=2):
    """tc_debug of the projected filter: every accumulator the narrow kernel wrote equals the FP64 contraction of the
    operand image within a quarter of the guard band's tensor-core budget; exactly the scheduled tiles are written; the
    image is the numpy restatement's; padding rows can never survive; no true edge has its sign bit set."""
    n = rows.shape[0]
    hc.set_spline(rows)
    acc, ha, hb = hc.tc_debug(thr, n, 3)
    n_pad = acc.shape[0]
    assert n_pad == (n + 255) // 256 * 256
    A, B = unswizzle32(ha, n_pad), unswizzle32(hb, n_pad)
    must = scheduled_mask(n_pad, cg)
    for r0 in range(0, n_pad, 1024):
        a, m = acc[r0:r0 + 1024], must[r0:r0 + 1024]
        assert not np.any(np.isnan(a[m])) and np.all(np.isnan(a[~m])), r0
        want = A[r0:r0 + 1024] @ B.T
        budget = 2 * 2.0 ** -18 * (np.abs(A[r0:r0 + 1024]) @ np.abs(B).T)
        err = np.abs(a.astype(np.float64) - want)
        assert np.all(err[m] <= 0.25 * budget[m] + 1e-30), float(np.max(err[m] / np.maximum(budget[m], 1e-300)))
    # the image is the numpy restatement's (same centre, basis, scale and fold; FP64 sums in another order may move a
    # coordinate across an fp16 rounding boundary: one fp16 ulp)
    A_np, B_np, _ = projected_image(rows, thr)
    assert np.all(np.abs(A[:n, :12] - A_np[:, :12]) <= 2.0 ** -10 * np.abs(A_np[:, :12]) + 2.0 ** -24)
    assert np.array_equal(A[:, :12], B[:, :12])
    P, Q = 32768.0, 8.0
    fold, fold_np = P * A[:n, 12] + Q * A[:n, 13], P * A_np[:, 12] + Q * A_np[:, 13]
    assert np.all(np.abs(fold - fold_np) <= 2.0 ** -20 * np.abs(fold_np) + 2.0 ** -6)
    assert np.array_equal(A[:, 12:14], B[:, 14:16]) and np.all(A[:n, 14] == P) and np.all(B[:n, 12] == P)
    assert np.all(A[n:, 12] == -65504.0) and np.all(A[n:, :12] == 0)
    i, j = near_pairs(rows, thr)
    assert not np.any(np.signbit(acc[i, j])), "a true edge was rejected"
    return len(i)


def accumulator_rows(model, K, n, rng):
    thr = 1e-3 if model == "iso" else THR
    rows = {"c4": lambda: c4_rows(n, K=K), "c4s": lambda: c4s_rows(n, K=K), "iso": lambda: rng.standard_normal((n, K)) * 1e-3}[model]()
    return plant(rows, rng, min(100, n // 2), thr=thr), thr


ACC_CASES = [("c4", 60, 4000), ("c4s", 60, 4000), ("iso", 60, 4000)] + \
    [("c4", K, n) for K in (16, 18, 30, 59, 60) for n in (2, 255, 256, 257, 8192)]


@pytest.mark.gpu
@pytest.mark.parametrize("model,K,n", ACC_CASES, ids=[m if n == 4000 else f"K{K}-n{n}" for m, K, n in ACC_CASES])
def test_projected_accumulators_match_fp64(hc, model, K, n):
    """Rows of every width 16 .. 60 the projection takes, at one 256-row tile, either side of a tile boundary, a single
    pair and the largest matrix tc_debug returns (8192 rows: 32 column tiles)."""
    rng = np.random.default_rng(4)
    rows, thr = accumulator_rows(model, K, n, rng)
    assert check_projected_accumulators(hc, rows, thr) >= min(100, n // 2) // 5
    assert hc.tc_last_plan()["projected_chosen"]


_ACC_CG1 = (
    "import numpy as np, scema_b200\n"
    "import test_tc_projection as t\n"
    "hc = scema_b200.HistCluster(0)\n"
    "for model, K, n in (('c4', 60, 4000), ('iso', 60, 4000), ('c4', 18, 257), ('c4', 30, 2), ('c4', 16, 8192)):\n"
    "    rows, thr = t.accumulator_rows(model, K, n, np.random.default_rng(4))\n"
    "    print(model, K, n, t.check_projected_accumulators(hc, rows, thr, cg=1))\n"
    "    assert hc.tc_last_plan()['projected_chosen']\n"
    "print('ok')\n")


@pytest.mark.gpu
def test_projected_accumulators_single_cta_kernel():
    """SCEMA_TC_CG=1: the narrow single-CTA kernel (128-row tiles, 8 KB B stages from two 4 KB blocks) writes the tiles of
    its own schedule with the same accumulators."""
    _run(_ACC_CG1, [], SCEMA_TC_CG="1")


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


def bits_equal(got, want):
    return len(got[0]) == len(want[0]) and all(np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8))
                                               for x, y in zip(got, want))


def special_rows(K):
    """the special values of test_k2_special_values, cut to K columns"""
    rng = np.random.default_rng(5)
    P = -(-K // 6)
    rows = synth.rows(7, 600, 8, P, 5e-3, synth.default_pert(THR, P))[:, :K].copy()
    rows[10] = np.nan
    rows[20, 3] = np.inf
    rows[30] = rows[31]
    rows[40] = 1e200
    rows[41] = 1e200
    rows[50:60] = rows[50:60] * 0 + 3.0
    rows[60:70] = 1e-170 * rng.standard_normal((10, K))
    return rows


def dense_rows(n, K=60):
    """every pair an edge: 1e-3 plus 1e-9 of noise"""
    return 1e-3 + 1e-9 * np.random.default_rng(0).standard_normal((n, K))


def sample_missed_rows(n=131072, D=4000):
    """c4 rows with D of them replaced by one typical row plus 3e-6 of noise per column: mutual distances ~3e-5, far above
    THR and deep inside the projected band, so all D (D - 1) / 2 pairs survive the filter. The D rows are chosen among the
    rows that none of the survivor-density sample's pairs touches (k_tc_plan_sample: pair t = (mix(0x5ce3a0000 + 2t) % n,
    mix(0x5ce3a0001 + 2t) % n)) and outside the centre's sample (every n / 4096-th row), so the sample cannot see them."""
    mask = (1 << 64) - 1

    def mix(z):
        z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & mask
        z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & mask
        return z ^ (z >> 31)
    touched = np.zeros(n, dtype=bool)
    for t in range(8192):
        touched[mix(0x5ce3a0000 + 2 * t) % n] = touched[mix(0x5ce3a0001 + 2 * t) % n] = True
    free = np.flatnonzero(~touched & (np.arange(n) % (n // SAMPLE) != 0))
    rng = np.random.default_rng(7)
    block = np.sort(rng.choice(free, D, replace=False))
    rows = c4_rows(n)
    rows[block] = rows[1] + 3e-6 * rng.standard_normal((D, rows.shape[1]))
    return rows, block


def pinned_projection_cases(cg):
    """Run with SCEMA_TC_SLICES=3 (and SCEMA_AUDIT): the projected filter on every width, size and kind of row the suite
    knows, each edge list equal to the CPU oracle's (indices, order, distance bits) and the filter that ran asserted."""
    from oracle.pyoracle import Oracle
    o = Oracle()
    hc = scema_b200.HistCluster(0)
    rng = np.random.default_rng(10 + cg)

    def run(name, rows, thr, projected=True, passes=None):
        want = o.all_pairs(rows, thr)[:3]
        hc.set_spline(rows)
        ne = hc.compare(thr, scema_b200.PAIRS_TC)
        got = hc.get_edges()
        plan, c = hc.tc_last_plan(), hc.counters()
        assert plan["projected_chosen"] == projected and c["tc_slices"] == 1, (name, plan, c)
        assert passes is None or passes(c["passes"]), (name, c)
        assert ne == len(want[0]) and bits_equal(got, want), (name, ne, len(want[0]))
        assert hc.last_audit()[1] == 0, name
        print(name, ne, c["survivors"], c["passes"], flush=True)
        return ne

    for K in (16, 18, 30, 59, 60):
        for n in (2, 257, 3000, 8193):             # 8193 rows: 33 column tiles, one more than a strip
            run(f"K{K}-n{n}", plant(c4_rows(n, seed=K, K=K), rng, min(200, n // 2)), THR)
    for K in (60, 18):
        rows = special_rows(K)
        run(f"special-K{K}", rows, THR)
        hc.set_spline(rows)
        hc.compare(THR, scema_b200.PAIRS_TC)
        pairs = set(zip(*(x.tolist() for x in hc.get_edges()[:2])))
        assert (30, 31) in pairs and (40, 41) in pairs and (50, 59) in pairs and (60, 69) in pairs
        assert not any(10 in p for p in pairs)
    for scale in (1e-150, 1e140, 1e-300):
        n = 3000 if scale != 1e-300 else 1200
        rows = plant(c4_rows(n, seed=21) * scale, rng, 300, thr=THR * scale, scales=tuple(1 + q * 3e-16 for q in range(-5, 6)))
        ne = run(f"scale-{scale:g}", rows, THR * scale)
        assert scale != 1e-300 or ne == n * (n - 1) // 2   # every squared difference underflows in the reference
    rows = c4_rows(3000, seed=33)
    rows[[5, 700, 701, 1500, 2999]] *= 1e6        # left out of the scale: no image, survive against everybody
    rows[701] = rows[700] * (1 + 1e-12)
    run("outliers", rows, THR, passes=lambda p: p == 1)
    run("offset", plant(c4_rows(2500, seed=7) + 1e3, rng, 100), THR)
    rows = c4_rows(2500, seed=6)
    for thr in (THR, 0.3 * THR, 40 * THR, THR):    # the fold carries the threshold: rebuilt every time
        run(f"thr-{thr:g}", rows, thr)
    for K in (12, 66):                              # outside 16 .. 60: 64-column copies, one slice
        rows = plant(c4_rows(3000, seed=K, K=K), rng, 200)
        run(f"K{K}", rows, THR, projected=False)
        hc.set_spline(rows)
        try:
            hc.tc_debug(THR, 3000, 3)
            raise AssertionError(f"tc_debug took the projection at K = {K}")
        except scema_b200.ScemaError:
            pass
    run("dense", dense_rows(2200), THR, passes=lambda p: p >= 2)   # 2.4M survivors: the pinned filter grows the queue
    if cg == 2:
        rows, _ = sample_missed_rows()
        hc.set_spline(rows)
        ne = hc.compare(THR, scema_b200.PAIRS_TC)
        got, c, plan = hc.get_edges(), hc.counters(), hc.tc_last_plan()
        assert plan["projected_chosen"] and c["tc_slices"] == 1 and c["passes"] >= 2, (plan, c)
        assert hc.compare(THR, scema_b200.PAIRS_EXACT) == ne and bits_equal(got, hc.get_edges())
        print("sample-missed", ne, c, flush=True)
    for K in (60, 30):                              # full 32-tile strips, many items per CTA
        n = 80000
        sp = plant(c4_rows(n, seed=40 + K, K=K), rng, 2000)
        hc.set_spline(sp)
        ne = hc.compare(THR, scema_b200.PAIRS_TC)
        got, c, plan = hc.get_edges(), hc.counters(), hc.tc_last_plan()
        assert plan["projected_chosen"] and c["tc_slices"] == 1, (plan, c)
        assert hc.last_audit()[1] == 0
        assert hc.compare(THR, scema_b200.PAIRS_EXACT) == ne and bits_equal(got, hc.get_edges())
        a, b, d = got
        assert ne > n and o.check_edges(sp, THR, a, b, d) == 0
        for r in np.random.default_rng(K).choice(n - 1, size=200, replace=False).tolist():
            ei, ej, ed, _ = o.all_pairs(sp, THR, r, r + 1)
            lo, hi = np.searchsorted(a, r), np.searchsorted(a, r, side="right")
            assert np.array_equal(b[lo:hi], ej) and np.array_equal(d[lo:hi].view(np.uint64), ed.view(np.uint64)), r
        print(f"large-K{K}", ne, c, flush=True)
    hc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cg", ["2", "1"])
def test_pinned_projection_on_every_width_size_and_edge_case(cg):
    """SCEMA_TC_SLICES=3 with both CTA-group kernels: widths 16 .. 60 at 2 .. 8193 rows, special values, magnitudes down
    to 1e-300, outliers left out of the scale, a large offset, a threshold sweep, widths the projection refuses, a queue
    that must grow (all pairs edges; with cta_group::2 also 131072 rows whose survivors the sample cannot see), and
    80000 rows (32-tile strips) against the filter-free kernel, the oracle's edge check and 200 complete rows."""
    _run("import test_tc_projection as t, sys\nt.pinned_projection_cases(int(sys.argv[1]))\nprint('ok')\n", [cg],
         SCEMA_TC_SLICES="3", SCEMA_TC_CG=cg, SCEMA_AUDIT="200000")


@pytest.mark.gpu
def test_automatic_choice_overflows_on_a_block_the_sample_missed():
    """The sample sizes the queue for the c4 background; 4000 rows the sample cannot see bring 8e6 survivors, twice the
    queue. compare_panels must re-decide (a larger queue, or two 64-column slices instead of the projection) and still
    give the filter-free kernel's list."""
    rows, block = sample_missed_rows()
    n, D = rows.shape[0], len(block)
    h = scema_b200.HistCluster(0)                  # fresh context: the queue starts at the floor
    h.set_spline(rows)
    ne = h.compare(THR, scema_b200.PAIRS_TC)
    got, c, plan = h.get_edges(), h.counters(), h.tc_last_plan()
    # preconditions: the sample sized a queue too small for the block, so the overflow path really ran
    sized = plan["projected"] / plan["sample"] * n * (n - 1) / 2 * 1.25
    assert plan["projected"] < 4 or sized < D * (D - 1) / 2, plan
    assert c["passes"] >= 2 and c["survivors"] >= D * (D - 1) // 2, c
    # which way the re-decision went: a larger queue keeps the projection; two 64-column slices (or, should those
    # overflow as well, the DMMA filter: tc_slices 0) drop it
    assert plan["projected_chosen"] == (c["tc_slices"] == 1), (c, plan)
    print("re-decision", c, plan)
    assert h.compare(THR, scema_b200.PAIRS_EXACT) == ne and bits_equal(got, h.get_edges())
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
