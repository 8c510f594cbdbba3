"""Parity of the CUDA path (through the C ABI) with the CPU oracle and the golden fixtures.

Bit-exact everywhere: spline samples, the edge SET, the edge ORDER after canonical sort, and the
bits of every emitted distance. All tests need a GPU (-m gpu).
"""
import json
import os

import numpy as np
import pytest

import scema_b200
from scema_b200 import synth, PAIRS_DMMA, PAIRS_FMA, PAIRS_EXACT, PAIRS_TC

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
VARIANTS = [("tc", PAIRS_TC), ("dmma", PAIRS_DMMA), ("fma", PAIRS_FMA), ("exact", PAIRS_EXACT)]
THR = 1e-6


def unhex(lst):
    return np.array([float.fromhex(x) for x in lst], dtype=np.float64)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same_bits(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


def edges_equal(got, want):
    return (len(got[0]) == len(want[0]) and np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
            and same_bits(got[2], want[2]))


def plant_near_threshold(rows, thr, n_plant, rng, spread=1e-15):
    """Rewrite n_plant rows as partner + u*thr*(1 +- few ulp): pairs inside the guard band."""
    n, k = rows.shape
    for q in range(n_plant):
        a = int(rng.integers(0, n))
        b = int((a + n // 2) % n)
        if a == b:
            continue
        u = rng.standard_normal(k)
        u /= np.linalg.norm(u)
        rows[b] = rows[a] + u * thr * (1 + (q - n_plant / 2) * spread)
    return rows


# ------------------------------------------------------------------------------------------- synth
def test_synth_matches_numpy():
    import torch
    off = synth.device_offsets(3, 777, 16, 3, 90, first=1000)
    assert np.array_equal(off, synth.offsets(3, 777, 16, 3, 90, first=1000))
    d = synth.device_histories(3, 777, 16, 5e-3, 1.3e-7, off, first=1000).cpu().numpy()
    assert same_bits(d, synth.histories(3, 777, 16, 5e-3, 1.3e-7, off, first=1000))
    r = synth.device_rows(2, 501, 16, 10, 5e-3, 1.3e-7, first=64).cpu().numpy()
    assert same_bits(r, synth.rows(2, 501, 16, 10, 5e-3, 1.3e-7, first=64))
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------- K1
def test_k1_golden(hc):
    for kat in json.load(open(os.path.join(GOLD, "kat_spline.json"))):
        steps = unhex(kat["steps"]).reshape(kat["L"], 6)
        hc.set_histories(steps, np.array([0, kat["L"]], dtype=np.uint64))
        hc.resample(kat["P"])
        assert same_bits(hc.get_spline()[0], unhex(kat["spline"])), kat["name"]


@pytest.mark.parametrize("P", [1, 2, 10, 50])
def test_k1_ragged_vs_oracle(hc, oracle, P):
    n = 4003  # not a multiple of the 5-history warp group
    off = synth.offsets(3, n, 16, 3, 200)
    steps = synth.histories(3, n, 16, 5e-3, synth.default_pert(THR, max(P, 2)), off)
    rng = np.random.default_rng(1)
    steps[: off[40]] *= 10.0 ** rng.integers(-9, 3, size=(int(off[40]), 6))  # wild magnitudes
    steps[int(off[50]):int(off[60]), 2] = 0.0                                  # constant-zero component
    steps[int(off[60]):int(off[70]), 4] = -0.0
    hc.set_histories(steps, off)
    hc.resample(P)
    assert same_bits(hc.get_spline(), oracle.splinify_batch(steps, off, P))


def test_k1_long_and_equal_lengths(hc, oracle):
    # equal lengths (production: one sample per timestep, FE_problem.h:1091-1098) incl. the minimum 3
    for L in (3, 4, 17, 501):
        n = 257
        off = (np.arange(n + 1, dtype=np.uint64) * L)
        steps = np.random.default_rng(L).standard_normal((n * L, 6)) * 1e-3
        hc.set_histories(steps, off)
        hc.resample(10)
        assert same_bits(hc.get_spline(), oracle.splinify_batch(steps, off, 10)), L
    # lengths on both sides of every length class of the streamed kernel (64, 256, 2048, 16384,
    # 131072) incl. the global-scratch fallback beyond the last one, and of the staged kernel's slabs
    lens = np.array([3, 16, 17, 64, 65, 128, 129, 256, 257, 512, 513, 800, 801, 1500, 2048, 2049, 2500, 5, 5, 5, 801,
                     4, 4, 7, 16384, 16385, 131072, 131073], dtype=np.uint64)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    steps = np.random.default_rng(9).standard_normal((int(off[-1]), 6)) * 1e-2
    hc.set_histories(steps, off)
    hc.resample(10)
    assert same_bits(hc.get_spline(), oracle.splinify_batch(steps, off, 10))


def test_k1_special_magnitudes(hc, oracle):
    """Numerators outside the range where the reciprocal-based exact division applies (zeros,
    subnormals, 1e+-300, inf, NaN) must take the IEEE division and still match bit for bit."""
    n, L = 64, 37
    off = (np.arange(n + 1, dtype=np.uint64) * L)
    rng = np.random.default_rng(5)
    steps = rng.standard_normal((n * L, 6)) * 1e-3
    scale = np.array([1e-300, 1e-310, 5e-324, 1e300, 1e-280, 1e290, 2.0 ** -895, 2.0 ** 897])
    for q in range(8):
        steps[q * L:(q + 1) * L] *= scale[q]
    steps[8 * L + 3, 1] = np.inf
    steps[9 * L + 5, 2] = np.nan
    steps[10 * L:(11 * L), 0] = 0.0
    steps[11 * L:(12 * L), 3] = -0.0
    steps[12 * L + 7, 4] = 5e-324
    steps[13 * L:(14 * L), 5] = 1.7976931348623157e308
    hc.set_histories(steps, off)
    for P in (10, 50):  # P > L puts several samples into one interval
        hc.resample(P)
        with np.errstate(all="ignore"):
            want = oracle.splinify_batch(steps, off, P)
        assert same_bits(hc.get_spline(), want), P


def test_history_store_matches_batch_path(hc, oracle):
    """In-process pattern (FE_problem.h:1091-1103, :1167-1229): append one sample per point per
    timestep to the device-resident store, re-fit all points, compare the flagged subset."""
    n, P = 1237, 10
    ids = (np.arange(n, dtype=np.uint32) * 3 + 7)
    rng = np.random.default_rng(21)
    base = rng.standard_normal((n // 8 + 1, 6)) * 1e-3
    grow = np.repeat(base, 8, axis=0)[:n] * (1.0 + 2e-5 * rng.standard_normal((n, 1)))
    hc.store_reset(n, ids, capacity_steps=4)  # forces the store to grow several times
    with pytest.raises(scema_b200.ScemaError):
        hc.store_resample(P)  # no samples yet (strain2spline.h:142-148)
    hist = []
    for t in range(1, 41):
        sample = grow * t + 1e-9 * rng.standard_normal((n, 6))
        hist.append(sample)
        hc.store_append(sample)
        if t == 2:
            with pytest.raises(scema_b200.ScemaError) as e:
                hc.store_resample(P)
            assert "at least 3 points" in str(e.value)
        if t in (3, 4, 17, 40):
            hc.store_resample(P)
            steps = np.stack(hist, axis=1).reshape(n * t, 6)  # history-major [n][t][6]
            off = np.arange(n + 1, dtype=np.uint64) * t
            want = oracle.splinify_batch(steps, off, P)
            assert same_bits(hc.get_spline(), want), t
    assert hc.store_info()[:2] == (n, 40)
    # compare only the flagged points, as spline_comparison does
    flagged = np.sort(rng.choice(n, size=700, replace=False)).astype(np.uint32)
    thr = 2e-6
    hc.select_rows(flagged)
    ne = hc.compare(thr)
    got = hc.get_edges()
    wi, wj, wd, _ = oracle.all_pairs(np.ascontiguousarray(want[flagged]), thr)
    assert ne == len(wi) and ne > 50 and edges_equal(got, (wi, wj, wd))
    mapping, _, _ = hc.reduce_edges(int(ids.max()) + 1)  # IDs of the subset are carried along
    assert set(np.nonzero(mapping != np.arange(len(mapping)))[0]) <= set(ids[flagged].tolist())


def test_k1_too_short_history_is_an_error(hc):
    off = np.array([0, 5, 7, 12], dtype=np.uint64)  # middle history has 2 steps
    hc.set_histories(np.zeros((12, 6)), off)
    with pytest.raises(scema_b200.ScemaError) as e:
        hc.resample(10)
    assert e.value.code == 1 and "at least 3 points" in str(e.value)  # strain2spline.h:145-148
    with pytest.raises(scema_b200.ScemaError):
        hc.compare(THR)  # no spline: "Spline is not up to date." (strain2spline.h:216-219)


def test_empty_batch(hc):
    hc.set_histories(np.zeros((0, 6)), np.array([0], dtype=np.uint64))
    hc.resample(10)
    assert hc.compare(THR) == 0
    hc.set_spline(np.zeros((1, 60)))
    assert hc.compare(THR) == 0


# ---------------------------------------------------------------------------------------------- K2
@pytest.mark.parametrize("vname,variant", VARIANTS)
def test_k2_golden(hc, vname, variant):
    g = json.load(open(os.path.join(GOLD, "kat_pairs.json")))
    rows = unhex(g["rows"]).reshape(g["n"], g["K"])
    hc.set_spline(rows)
    hc.compare(g["thr"], variant)
    a, b, d = hc.get_edges()
    assert a.tolist() == g["edges"]["i"] and b.tolist() == g["edges"]["j"] and same_bits(d, unhex(g["edges"]["d"]))


@pytest.mark.parametrize("vname,variant", VARIANTS)
@pytest.mark.parametrize("n,P", [(2, 10), (127, 10), (128, 10), (129, 10), (1000, 1), (1500, 3), (3000, 10),
                                 (2100, 11), (1300, 50), (700, 21)])
def test_k2_vs_oracle(hc, oracle, vname, variant, n, P):
    rows = synth.rows(2, n, 16, max(P, 2), 5e-3, synth.default_pert(THR, max(P, 2)))[:, : 6 * P].copy()
    rng = np.random.default_rng(n + P)
    if n >= 100:
        plant_near_threshold(rows, THR, n // 10, rng)
    want = oracle.all_pairs(rows, THR)
    hc.set_spline(rows)
    ne = hc.compare(THR, variant)
    assert ne == len(want[0])
    assert edges_equal(hc.get_edges(), want)
    if n >= 1000 and P == 10:
        assert ne > n  # the case really has edges on both sides of the band


@pytest.mark.parametrize("vname,variant", VARIANTS)
def test_k2_special_values(hc, oracle, vname, variant):
    rng = np.random.default_rng(5)
    rows = synth.rows(7, 600, 8, 10, 5e-3, synth.default_pert(THR, 10))
    rows[10] = np.nan                         # NaN history: no edges (sqrt(NaN) < thr is false)
    rows[20, 3] = np.inf
    rows[30] = rows[31]                       # exact duplicate: distance 0 is an edge
    rows[40] = 1e200                          # norms overflow: filter must not reject the equal pair
    rows[41] = 1e200
    rows[50:60] = rows[50:60] * 0 + 3.0       # large common offset: wide guard band, all equal
    rows[60:70] = 1e-170 * rng.standard_normal((10, 60))  # squares underflow
    want = oracle.all_pairs(rows, THR)
    hc.set_spline(rows)
    hc.compare(THR, variant)
    got = hc.get_edges()
    assert edges_equal(got, want)
    pairs = set(zip(got[0].tolist(), got[1].tolist()))
    assert (30, 31) in pairs and (40, 41) in pairs and (50, 59) in pairs and (60, 69) in pairs
    assert not any(10 in p for p in pairs)


@pytest.mark.parametrize("thr", [0.0, -1.0, float("nan")])
def test_k2_nonpositive_threshold(hc, thr):
    hc.set_spline(np.zeros((300, 60)))
    assert hc.compare(thr) == 0               # diff >= 0 is never < thr


@pytest.mark.parametrize("vname,variant", VARIANTS)
def test_k2_dense_edges_grow_buffers(oracle, vname, variant):
    """Early in a run all histories are within 1e-6 of each other: O(N^2) edges (SURVEY §7).
    Exercises the overflow-and-retry path of the candidate queue and the edge buffers (fresh
    context, so the buffers start at their default capacity)."""
    hc = scema_b200.HistCluster(0)
    n = 2200
    rows = 1e-3 + 1e-9 * np.random.default_rng(0).standard_normal((n, 60))
    want = oracle.all_pairs(rows, THR)
    assert len(want[0]) == n * (n - 1) // 2
    hc.set_spline(rows)
    assert hc.compare(THR, variant) == n * (n - 1) // 2
    assert hc.counters()["passes"] >= 2
    assert edges_equal(hc.get_edges(), want)
    assert np.array_equal(hc.get_degrees(n), np.full(n, n - 1, dtype=np.uint32))
    hc.close()


def test_k2_huge_threshold_all_pairs(hc, oracle):
    rows = synth.rows(1, 700, 16, 10, 5e-3, 1e-7)
    want = oracle.all_pairs(rows, float("inf"))
    hc.set_spline(rows)
    assert hc.compare(float("inf")) == 700 * 699 // 2
    assert edges_equal(hc.get_edges(), want)


@pytest.mark.parametrize("vname,variant", VARIANTS)
def test_compare_stream_concatenates_to_compare(hc, vname, variant):
    """Edge streaming (config 5's mode): chunks of panels, delivered through the sink, concatenate
    to exactly the sorted list of the one-shot compare; also per shard."""
    n = 9000  # 5 panels of 2048 rows
    rows = synth.rows(12, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
    hc.set_spline(rows)
    ne = hc.compare(THR, variant)
    want = hc.get_edges()
    assert ne > 1000
    for ppc in (1, 2, 64):
        chunks = []
        tot = hc.compare_stream(THR, lambda a, b, d: chunks.append((a, b, d)), variant, panels_per_chunk=ppc)
        got = tuple(np.concatenate([c[k] for c in chunks]) for k in range(3))
        assert tot == ne and edges_equal(got, want), ppc
        if variant == PAIRS_TC:   # config-4-shaped rows: the streamed compare runs the projected filter
            assert hc.tc_last_plan()["projected_chosen"] and hc.counters()["tc_slices"] == 1, ppc
        if ppc == 1:
            assert len(chunks) >= 4
            assert all(chunks[i][0].max() < chunks[i + 1][0].min() for i in range(len(chunks) - 1))
    parts = []
    for shard in range(3):
        hc.compare_stream(THR, lambda a, b, d: parts.append((a, b, d)), variant, shard=shard, n_shards=3, panels_per_chunk=2)
        assert variant != PAIRS_TC or hc.tc_last_plan()["projected_chosen"], shard
    a = np.concatenate([c[0] for c in parts]); b = np.concatenate([c[1] for c in parts]); d = np.concatenate([c[2] for c in parts])
    o = np.lexsort((b, a))
    assert edges_equal((a[o], b[o], d[o]), want)
    with pytest.raises(scema_b200.ScemaError):
        hc.get_edges()  # nothing is retained after a streamed compare

    def bad_sink(a, b, d):
        raise RuntimeError("stop")
    with pytest.raises(RuntimeError):
        hc.compare_stream(THR, bad_sink, variant, panels_per_chunk=1)


def test_config2_full_oracle(hc, oracle):
    """BASELINE configs[1]: 16k histories x 6 x 10, full CPU oracle over all 1.34e8 pairs, with
    >= 1000 planted pairs within a few ulp of the threshold (SURVEY §8d C2)."""
    n = 16384
    rows = synth.rows(2, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
    plant_near_threshold(rows, THR, 1200, np.random.default_rng(2), spread=3e-16)
    want = oracle.all_pairs(rows, THR)
    for _, variant in VARIANTS:
        hc.set_spline(rows)
        hc.compare(THR, variant)
        assert edges_equal(hc.get_edges(), want)
    c = hc.counters()
    assert c["edges"] == len(want[0])


def test_sharded_compare_union(hc, oracle):
    """Tile-sharding: the union of the shards' edges is the whole edge list, no duplicates."""
    n = 5000
    rows = synth.rows(9, n, 16, 10, 5e-3, synth.default_pert(THR, 10))
    want = oracle.all_pairs(rows, THR)
    for _, variant in VARIANTS:
        for world in (2, 3, 8):
            parts = []
            for r in range(world):
                hc.set_spline(rows)
                hc.compare(THR, variant, shard=r, n_shards=world)
                parts.append(hc.get_edges())
                if variant == PAIRS_TC:   # every shard takes the projected filter on these rows
                    assert hc.tc_last_plan()["projected_chosen"] and hc.counters()["tc_slices"] == 1, (world, r)
            a = np.concatenate([p[0] for p in parts])
            b = np.concatenate([p[1] for p in parts])
            d = np.concatenate([p[2] for p in parts])
            o = np.lexsort((b, a))
            assert edges_equal((a[o], b[o], d[o]), want), (variant, world)
            # (the tcgen05 filter deals items out strip by strip; with every edge on the diagonal of this small
            # case one of three shards may legitimately get none)
            if variant not in (PAIRS_EXACT, PAIRS_TC) and world <= 3:
                assert all(len(p[0]) > 0 for p in parts)


# ------------------------------------------------------------------------------ pipeline and files
def test_pipeline_files_and_mapping(hc, oracle, tmp_path):
    """resample + compare + per-history files + native graph reduction vs the oracle on the
    config-1 golden case (576 histories, P=10, thr=1e-6) and its recorded reference outputs."""
    g = json.load(open(os.path.join(GOLD, "pipeline_c1", "reference_outputs.json")))
    n, P, L = g["n"], g["P"], g["L"]
    off = synth.offsets(g["seed"], n, g["cluster"], L, L)
    steps = synth.histories(g["seed"], n, g["cluster"], g["amp"], synth.default_pert(g["thr"], P), off)
    ids = np.arange(n, dtype=np.uint32)
    ne = hc.cluster(steps, off, ids, P, g["thr"])
    assert 2 * ne == sum(len(v.splitlines()) for v in g["results"].values())
    hc.write_similar_hist(str(tmp_path / "last.%u.similar_hist"))
    for i in range(n):
        got = open(tmp_path / f"last.{i}.similar_hist").read()
        assert sorted(got.splitlines()) == sorted(g["results"][str(i)].splitlines()), i
    # byte-for-byte against the oracle's writer (same batch order)
    a, b, d = hc.get_edges()
    (tmp_path / "o").mkdir()
    oracle.write_similar_files(ids, a, b, d, str(tmp_path / "o" / "last.%u.similar_hist"))
    for i in range(n):
        assert open(tmp_path / f"last.{i}.similar_hist").read() == open(tmp_path / "o" / f"last.{i}.similar_hist").read()
    # native reduction on these files == oracle restatement fed the same directory order
    it, nf, nr = scema_b200.reduce_dir(str(tmp_path), str(tmp_path / "mapping.csv"), n)
    assert nf == n
    eu, ev = [], []
    for nm in os.listdir(tmp_path):
        if nm.startswith("last.") and nm.endswith(".similar_hist"):
            for line in open(tmp_path / nm):
                x, y, _ = line.split()
                eu.append(int(x))
                ev.append(int(y))
    mp, it2, nr2 = oracle.reduce_graph(eu, ev, n)
    got = [int(l.split()[1]) for l in open(tmp_path / "mapping.csv")]
    assert got == mp.tolist() and (it, nr) == (it2, nr2)
    # in-memory reduction: batch-order call sequence
    mp3, it3, nr3 = hc.reduce_edges(n)
    eu, ev = [], []
    for i in range(n):
        for line in open(tmp_path / f"last.{i}.similar_hist"):
            x, y, _ = line.split()
            eu.append(int(x))
            ev.append(int(y))
    mp4, it4, nr4 = oracle.reduce_graph(eu, ev, n)
    assert mp3.tolist() == mp4.tolist() and (it3, nr3) == (it4, nr4)


def test_ids_are_carried(hc, oracle, tmp_path):
    n = 300
    rows = synth.rows(3, n, 8, 10, 5e-3, synth.default_pert(THR, 10))
    ids = (np.arange(n, dtype=np.uint32)[::-1] * 7 + 3).copy()
    hc.set_spline(rows, ids=ids)
    hc.compare(THR)
    a, b, d = hc.get_edges()
    hc.write_similar_hist(str(tmp_path / "ID_%u.txt"))
    (tmp_path / "o").mkdir()
    oracle.write_similar_files(ids, a, b, d, str(tmp_path / "o" / "ID_%u.txt"))
    for i in ids:
        assert open(tmp_path / f"ID_{i}.txt").read() == open(tmp_path / "o" / f"ID_{i}.txt").read()
    with pytest.raises(scema_b200.ScemaError) as e:
        hc.write_similar_hist(str(tmp_path / "missing_dir" / "ID_%u.txt"))
    assert e.value.code == 4  # the reference exits when the file cannot be opened (strain2spline.h:303-307)


# ------------------------------------------------------------------------- full-size properties
def test_config3_ragged_200k_properties(hc, oracle):
    """BASELINE configs[2] at full size: 200k ragged histories (6..200 steps), resample + all-pairs.
    Full oracle is infeasible (2e10 pairs); check (i) spline samples bit-exact on a 10k subset,
    (ii) every emitted edge re-derived on the CPU by direct differences (bits + threshold),
    (iii) completeness: 300 full rows recomputed on the CPU, (iv) DMMA and FMA edge lists equal."""
    n, P = 200000, 10
    off = synth.offsets(3, n, 16, 6, 200)
    steps = synth.histories(3, n, 16, 5e-3, synth.default_pert(THR, P), off)
    hc.set_histories(steps, off)
    hc.resample(P)
    sp = hc.get_spline()
    sub = np.random.default_rng(0).choice(n, size=10000, replace=False)
    sub.sort()
    sub_off = np.concatenate([[0], np.cumsum(off[sub + 1] - off[sub])]).astype(np.uint64)
    sub_steps = np.concatenate([steps[int(off[i]):int(off[i + 1])] for i in sub])
    assert same_bits(sp[sub], oracle.splinify_batch(sub_steps, sub_off, P))
    ne = hc.compare(THR, PAIRS_DMMA)
    a, b, d = hc.get_edges()
    assert ne > n and np.all(a < b) and np.all(np.diff(a.astype(np.int64) * n + b) > 0)  # sorted, unique
    assert oracle.check_edges(sp, THR, a, b, d) == 0
    rows_to_check = np.random.default_rng(1).choice(n - 1, size=300, replace=False)
    got = set(zip(a.tolist(), b.tolist()))
    for r in rows_to_check.tolist():
        ei, ej, ed, _ = oracle.all_pairs(sp, THR, r, r + 1)
        for i, j in zip(ei.tolist(), ej.tolist()):
            assert (i, j) in got
        assert len(ei) == int(np.count_nonzero(a == r))
    hc.compare(THR, PAIRS_FMA)
    assert edges_equal(hc.get_edges(), (a, b, d))
    hc.compare(THR, PAIRS_TC)
    assert edges_equal(hc.get_edges(), (a, b, d))


def test_config4_1M_properties(hc, oracle):
    """BASELINE configs[3] at full size on one GPU: 1M histories x 6 x 10 (5e11 pairs). Size-independent
    checks: (i) the filter-free exact kernel and the DMMA path emit the same edge list (ids, order, distance
    bits) over the WHOLE problem, (ii) every emitted edge re-derived on the CPU by direct differences,
    (iii) completeness of 200 full rows recomputed on the CPU, (iv) the streamed compare delivers the
    same list, (v) a 20k-history spline subset bit-exact against the oracle."""
    import torch
    n, P = 1000000, 10
    pert = synth.default_pert(THR, P)
    off = synth.device_offsets(4, n, 16, 8, 64)
    d_steps = synth.device_histories(4, n, 16, 5e-3, pert, off, device="cuda:0")
    torch.cuda.synchronize()
    hc.set_histories(None, off, device_ptr=d_steps.data_ptr())
    hc.resample(P)
    sp = hc.get_spline()
    sub = np.sort(np.random.default_rng(0).choice(n, size=20000, replace=False))
    sub_off = np.concatenate([[0], np.cumsum(off[sub + 1] - off[sub])]).astype(np.uint64)
    h_steps = d_steps.cpu().numpy()
    sub_steps = np.concatenate([h_steps[int(off[i]):int(off[i + 1])] for i in sub])
    assert same_bits(sp[sub], oracle.splinify_batch(sub_steps, sub_off, P))
    del h_steps, sub_steps
    ne = hc.compare(THR, PAIRS_DMMA)
    a, b, d = hc.get_edges()
    assert ne > n and np.all(a < b) and np.all(np.diff(a.astype(np.int64) * n + b) > 0)  # sorted, unique
    assert hc.counters()["survivors"] < ne + ne // 100  # the guard band stays a vanishing fraction
    assert oracle.check_edges(sp, THR, a, b, d) == 0
    for r in np.random.default_rng(1).choice(n - 1, size=200, replace=False).tolist():
        ei, ej, ed, _ = oracle.all_pairs(sp, THR, r, r + 1)
        lo, hi = np.searchsorted(a, r), np.searchsorted(a, r + 1)
        assert np.array_equal(b[lo:hi], ej) and same_bits(d[lo:hi], ed), r
    chunks = []
    tot = hc.compare_stream(THR, lambda x, y, z: chunks.append((x, y, z)), PAIRS_DMMA)
    assert tot == ne and len(chunks) > 4
    assert edges_equal(tuple(np.concatenate([c[k] for c in chunks]) for k in range(3)), (a, b, d))
    hc.compare(THR, PAIRS_EXACT)
    assert edges_equal(hc.get_edges(), (a, b, d))
    # the tcgen05 filter: same list over the whole problem, one-shot and streamed; its guard band is wider
    # (fp16 slices, fp32 accumulation) but still only keeps pairs of the same cluster
    assert hc.compare(THR, PAIRS_TC) == ne
    assert edges_equal(hc.get_edges(), (a, b, d))
    assert hc.counters()["survivors"] <= n * 15 // 2 + n // 100
    chunks = []
    tot = hc.compare_stream(THR, lambda x, y, z: chunks.append((x, y, z)), PAIRS_TC)
    assert tot == ne and edges_equal(tuple(np.concatenate([c[k] for c in chunks]) for k in range(3)), (a, b, d))
    del d_steps


def test_config5_shape_properties(hc, oracle):
    """BASELINE configs[4] shape (K = 300) at 60k histories (1.8e9 pairs): the chunked tcgen05 filter, the streamed
    compare and the filter-free exact kernel emit the same edge list; every edge re-derived on the CPU; 100 complete
    rows recomputed on the CPU."""
    import torch
    n, P = 60000, 50
    d_rows = synth.device_rows(5, n, 16, P, 5e-3, synth.default_pert(THR, P), device="cuda:0")
    torch.cuda.synchronize()
    hc.set_spline(device_ptr=d_rows.data_ptr(), n=n, k=6 * P)
    ne = hc.compare(THR, PAIRS_TC)
    a, b, d = hc.get_edges()
    assert hc.counters()["tc_slices"] == 1                      # the tcgen05 path really ran (5 chunks of 64 columns)
    assert ne > n and np.all(a < b) and np.all(np.diff(a.astype(np.int64) * n + b) > 0)
    sp = d_rows.cpu().numpy()
    assert oracle.check_edges(sp, THR, a, b, d) == 0
    for r in np.random.default_rng(3).choice(n - 1, size=100, replace=False).tolist():
        ei, ej, ed, _ = oracle.all_pairs(sp, THR, r, r + 1)
        lo, hi = np.searchsorted(a, r), np.searchsorted(a, r + 1)
        assert np.array_equal(b[lo:hi], ej) and same_bits(d[lo:hi], ed), r
    chunks = []
    tot = hc.compare_stream(THR, lambda x, y, z: chunks.append((x, y, z)), PAIRS_TC, panels_per_chunk=8)
    assert tot == ne and len(chunks) >= 3
    assert edges_equal(tuple(np.concatenate([c[k] for c in chunks]) for k in range(3)), (a, b, d))
    hc.compare(THR, PAIRS_EXACT)
    assert edges_equal(hc.get_edges(), (a, b, d))
    del d_rows


def test_select_rows_twice_and_with_duplicates(hc, oracle):
    """scema_select_rows on an already selected matrix (ADVICE r1: the gather must not run in place nor free its own
    source), with duplicates that make the second selection larger than the first."""
    rng = np.random.default_rng(5)
    rows = synth.rows(9, 3000, 16, 10, 5e-3, synth.default_pert(THR, 10))
    hc.set_spline(rows, ids=np.arange(3000, dtype=np.uint32) + 100)
    first = rng.choice(3000, size=700, replace=False).astype(np.uint32)
    hc.select_rows(first)
    assert same_bits(hc.get_spline(), rows[first])
    second = rng.integers(0, 700, size=2500).astype(np.uint32)      # duplicates, more rows than before
    hc.select_rows(second)
    want = rows[first][second]
    assert same_bits(hc.get_spline(), want)
    third = np.arange(0, 2500, 3, dtype=np.uint32)
    hc.select_rows(third)
    want = want[third]
    assert same_bits(hc.get_spline(), want)
    # distinct rows only for the compare (exact duplicates are at distance 0, still a valid edge)
    wi, wj, wd, _ = oracle.all_pairs(want, THR)
    assert hc.compare(THR, PAIRS_TC) == len(wi)
    assert edges_equal(hc.get_edges(), (wi, wj, wd))


def test_result_file_pattern_is_validated(hc, tmp_path):
    """The file name pattern of scema_write_similar_hist goes to snprintf: exactly one %u, nothing else (ADVICE r1)."""
    rows = synth.rows(2, 300, 16, 10, 5e-3, synth.default_pert(THR, 10))
    hc.set_spline(rows)
    hc.compare(THR, PAIRS_TC)
    for bad in ("%s", "a_%u_%u", "plain", "%u%n", "%d"):
        with pytest.raises(scema_b200.ScemaError) as e:
            hc.write_similar_hist(str(tmp_path / bad))
        assert e.value.code == 1
    hc.write_similar_hist(str(tmp_path / "100%%_ID_%u.txt"))
    assert len([f for f in os.listdir(tmp_path) if f.startswith("100%_ID_")]) == 300
