"""The oracle (oracle/hist_oracle.c) against the golden vectors and the reference.

The reference has no tests of its own (SURVEY.md §4); the fixtures in tests/golden/ were produced by
tests/golden/make_golden.py from the unmodified reference header. Bit-exact comparisons only. The
randomized comparisons run the reference live where oracle/_ref is built, and otherwise compare with
its recorded results (tests/golden/reference_runs.json: SHA-256 of the bit patterns, 64 bits of it
per history or file; written by tests/golden/make_golden_live.py).
"""
import hashlib
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def unhex(lst):
    return np.array([float.fromhex(x) for x in lst], dtype=np.float64)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same_bits(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    # NaN payload/sign is not specified by the reference either: treat all NaNs as one value
    return a.shape == b.shape and bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


def bits_sha(a):
    """SHA-256 of the bit patterns, every NaN as one value (as in same_bits)."""
    a = np.array(a, dtype=np.float64)
    a[np.isnan(a)] = np.nan
    return hashlib.sha256(np.ascontiguousarray(a).view(np.uint64).tobytes()).hexdigest()


def recorded(key):
    with open(os.path.join(GOLD, "reference_runs.json")) as f:
        return json.load(f)["oracle"][key]


def load_kats():
    return json.load(open(os.path.join(GOLD, "kat_spline.json")))


@pytest.mark.parametrize("kat", load_kats(), ids=lambda k: k["name"])
def test_oracle_spline_golden(oracle, kat):
    steps = unhex(kat["steps"]).reshape(kat["L"], 6)
    got = oracle.splinify(steps, kat["P"])
    assert same_bits(got, unhex(kat["spline"]))


def test_survey_kat_values():
    """Hex constants quoted in SURVEY.md §8c (KAT-1, KAT-4) are what the fixture holds."""
    kats = {k["name"]: k for k in load_kats()}
    k1 = kats["kat1_L5_P4"]["spline"]
    assert k1[6] == "0x1.cc7c5a8ba1e67p-10" and k1[20] == "0x1.0624dd2f1a9fep-11" and k1[1] == "-0x0.0p+0"
    k4 = kats["kat4_L3_P10"]["spline"]
    assert k4[6 * 1] == "0x1.04b4a3c8a7ff7p-12" and k4[6 * 9] == "0x1.89374bc6a7efap-10"


def test_oracle_pairs_golden(oracle):
    g = json.load(open(os.path.join(GOLD, "kat_pairs.json")))
    rows = unhex(g["rows"]).reshape(g["n"], g["K"])
    for e in g["l2"]:
        assert oracle.compare_l2(rows[e["a"]], rows[e["b"]]).hex() == e["d"]
    ei, ej, ed, pairs = oracle.all_pairs(rows, g["thr"])
    assert pairs == g["n"] * (g["n"] - 1) // 2
    assert ei.tolist() == g["edges"]["i"] and ej.tolist() == g["edges"]["j"]
    assert same_bits(ed, unhex(g["edges"]["d"]))
    # the planted pairs straddle the threshold: both outcomes occur among them
    planted = [(k, 48 + k) for k in range(12)]
    found = set(zip(ei.tolist(), ej.tolist()))
    hits = sum(p in found for p in planted)
    assert 0 < hits < 12


def test_oracle_min_steps(oracle):
    with pytest.raises(ValueError):
        oracle.splinify(np.zeros((2, 6)), 10)  # reference: exit(1), strain2spline.h:145-148


def test_oracle_files_golden(oracle, tmp_path):
    """Per-history file contents == the reference CLI's __results/ID_<id>.txt (as line sets; the
    line ORDER follows the directory enumeration of the generating run and is checked live in
    test_cli.py where oracle/_ref exists)."""
    from scema_b200 import synth
    g = json.load(open(os.path.join(GOLD, "pipeline_c1", "reference_outputs.json")))
    n, P, L, thr = g["n"], g["P"], g["L"], g["thr"]
    off = synth.offsets(g["seed"], n, g["cluster"], L, L)
    steps = synth.histories(g["seed"], n, g["cluster"], g["amp"], synth.default_pert(thr, P), off)
    # the CLI parsed repr()-printed text, which round-trips doubles exactly
    sp = oracle.splinify_batch(steps, off, P)
    ei, ej, ed, _ = oracle.all_pairs(sp, thr)
    ids = np.arange(n, dtype=np.uint32)
    assert oracle.write_similar_files(ids, ei, ej, ed, str(tmp_path / "ID_%u.txt")) == 0
    for i in range(n):
        got = open(tmp_path / f"ID_{i}.txt").read()
        assert sorted(got.splitlines()) == sorted(g["results"][str(i)].splitlines()), i
    assert 2 * len(ei) == sum(len(v.splitlines()) for v in g["results"].values())


FORMAT_VALUES = (1e-6, 0.0, 1.23456789e-7, 12345678.0, 1e-320, float("inf"), 9.9999995e-7, 100000.0, 999999.5, 1e22)


def random_record(lib):
    """splinify of 400 random histories, all_pairs of 400 rows of which 200 are near copies, format_double of a few
    values: what the oracle and the reference must agree on."""
    rng = np.random.default_rng(7)
    splines = []
    for trial in range(400):
        L = int(rng.integers(3, 260))
        P = int(rng.integers(1, 62))
        st = rng.standard_normal((L, 6)) * 10.0 ** rng.integers(-9, 1, size=6)
        if trial % 7 == 0:
            st[:, 2] = 0
        if trial % 11 == 0:
            st[:, 3] = st[0, 3]
        if trial % 13 == 0:
            st[:, 1] = -0.0
        splines.append(bits_sha(lib.splinify(st, P))[:16])
    rows = rng.standard_normal((400, 300)) * 1e-3
    rows[200:] = rows[:200] + rng.standard_normal((200, 300)) * 5.5e-8
    ei, ej, ed, _ = lib.all_pairs(rows, 1e-6)
    pairs = {"edges": len(ei), "i": hashlib.sha256(ei.tobytes()).hexdigest(), "j": hashlib.sha256(ej.tobytes()).hexdigest(),
             "d": bits_sha(ed)}
    return {"splines": splines, "pairs": pairs, "format": [lib.format_double(v) for v in FORMAT_VALUES]}


def test_oracle_vs_reference_random(oracle):
    from oracle.pyoracle import Reference, have_reference
    want = random_record(Reference()) if have_reference() else recorded("random")
    got = random_record(oracle)
    bad = [k for k, (a, b) in enumerate(zip(got["splines"], want["splines"])) if a != b]
    assert len(got["splines"]) == len(want["splines"]) and not bad, bad[:10]
    assert got["pairs"]["edges"] > 10 and got["pairs"] == want["pairs"]
    assert got["format"] == want["format"]


def pipeline_inputs():
    from scema_b200 import synth
    n, P, thr = 200, 10, 1e-6
    off = synth.offsets(5, n, 8, 4, 40)
    steps = synth.histories(5, n, 8, 1e-3, synth.default_pert(thr, P), off)
    ids = (np.arange(n, dtype=np.uint32) * 3 + 7)
    return steps, off, ids, P, thr


def pipeline_record(out_dir, ids, spline):
    """The resampled rows and every last.<id>.similar_hist file in out_dir."""
    files = {}
    for i in ids:
        with open(os.path.join(out_dir, f"last.{i}.similar_hist"), "rb") as f:
            files[str(i)] = hashlib.sha256(f.read()).hexdigest()[:16]
    return {"spline": bits_sha(spline), "files": files}


def reference_pipeline_record(reference, out_dir):
    """compare_histories_with_all_ranks + most_similar_histories_to_file of the reference header (the as-called path)."""
    steps, off, ids, P, thr = pipeline_inputs()
    sp = reference.pipeline(steps, off, ids, P, thr, os.path.join(out_dir, "last.%u.similar_hist"), want_spline=True)
    return pipeline_record(out_dir, ids, sp)


def oracle_pipeline_record(oracle, out_dir):
    steps, off, ids, P, thr = pipeline_inputs()
    mine = oracle.splinify_batch(steps, off, P)
    ei, ej, ed, _ = oracle.all_pairs(mine, thr)
    oracle.write_similar_files(ids, ei, ej, ed, os.path.join(out_dir, "last.%u.similar_hist"))
    return pipeline_record(out_dir, ids, mine)


def test_reference_pipeline_matches_oracle(oracle, tmp_path):
    """compare_histories_with_all_ranks + most_similar_histories_to_file (the as-called path)."""
    from oracle.pyoracle import Reference, have_reference
    (tmp_path / "r").mkdir()
    (tmp_path / "o").mkdir()
    want = reference_pipeline_record(Reference(), str(tmp_path / "r")) if have_reference() else recorded("pipeline")
    got = oracle_pipeline_record(oracle, str(tmp_path / "o"))
    assert got["spline"] == want["spline"]
    assert got["files"] == want["files"]
