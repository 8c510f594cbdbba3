"""Batch ingest (include/scema_ingest.h): the multi-threaded strain_<ID> reader and the
lhistory.csv converter, against the reference's own reader Strain6D::from_file
(headers/strain2spline.h:112-134) — through the committed golden cases (generated from the
unmodified reference by tests/golden/make_golden_ingest.py) and, where oracle/_ref is built, live."""
import json
import os

import numpy as np
import pytest

from scema_b200.binding import Batch, ScemaError

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def cases():
    return json.load(open(os.path.join(GOLD, "ingest_cases.json")))


def write_cases(d):
    names = []
    for k, c in enumerate(cases()):
        with open(os.path.join(d, f"strain_{k}"), "w", newline="") as f:
            f.write(c["text"])
        names.append(f"strain_{k}")
    with open(os.path.join(d, "notes.txt"), "w") as f:
        f.write("1 2 3 4 5 6\n")  # not a strain_ file: ignored (mpi_comparison_test.cc:74-77)
    return names


def test_reader_matches_golden_reference_outputs(tmp_path):
    d = str(tmp_path) + "/"
    write_cases(d)
    b = Batch.read_dir(d, n_threads=4)
    cs = cases()
    assert len(b) == len(cs)
    off, ids, steps = b.offsets, b.ids, b.steps
    seen = set()
    for q in range(len(b)):
        k = int(ids[q])
        assert b.name(q) == f"strain_{k}" and k not in seen
        seen.add(k)
        c = cs[k]
        got = steps[int(off[q]):int(off[q + 1])]
        want = np.array([float.fromhex(x) for x in c["steps"]]).reshape(-1, 6)
        assert got.shape == want.shape, (c["name"], got.shape, want.shape)
        assert np.array_equal(bits(got), bits(want)), c["name"]
    # batch order = readdir order, as the reference command lines enumerate the directory
    order = [e for e in os.listdir(d) if e.startswith("strain_")]
    assert [b.name(q) for q in range(len(b))] == order


def test_reader_matches_live_reference(tmp_path):
    """Random files in several number formats, read by the batch reader and by Strain6D::from_file where oracle/_ref is
    built. Elsewhere the reference's reading of these files is restated: whitespace-separated doubles, correctly
    rounded (libstdc++ `ifstream >> double`; every value here is a normal double), six per step."""
    from oracle.pyoracle import Reference, have_reference
    reference = Reference() if have_reference() else None
    d = str(tmp_path) + "/"
    rng = np.random.default_rng(3)
    n = 40
    for k in range(n):
        L = int(rng.integers(0, 60))
        v = rng.standard_normal((L, 6)) * 10.0 ** rng.integers(-14, 4, size=(L, 6))
        fmt = ["%r", "%.6g", "%.17g", "%.25f", "%.3e"][k % 5]
        with open(os.path.join(d, f"strain_{k}"), "w") as f:
            for row in v:
                f.write(" ".join((fmt % float(x)) for x in row) + "\n")
    paths = [os.path.join(d, f"strain_{k}") for k in range(n)]
    b = Batch.read_files(paths, n_threads=3)
    assert list(b.ids) == list(range(n))
    off, steps = b.offsets, b.steps
    for k in range(n):
        if reference is not None:
            want = reference.from_file(paths[k])
        else:
            want = np.array([float(x) for x in open(paths[k]).read().split()], dtype=np.float64).reshape(-1, 6)
        got = steps[int(off[k]):int(off[k + 1])]
        assert got.shape == want.shape and np.array_equal(bits(got), bits(want)), k


def test_missing_file_and_directory_are_io_errors(tmp_path):
    with pytest.raises(ScemaError) as e:
        Batch.read_files([str(tmp_path / "strain_404")])
    assert e.value.code == 4 and "Could not open" in str(e.value)  # strain2spline.h:117-120
    with pytest.raises(ScemaError) as e:
        Batch.read_dir(str(tmp_path / "nowhere") + "/")
    assert e.value.code == 4


def test_lhistory_converter_and_round_trip(tmp_path):
    """pr_<rank>.lhistory.csv (FE_problem.h:1985-2045) -> ragged batch -> strain_<ID> files -> batch."""
    rng = np.random.default_rng(11)
    hdr = "timestep,time,qpid,cell,qpoint,material"
    for pre in ("strain", "updstrain", "stress"):
        for k in range(3):
            for l in range(k, 3):
                hdr += f",{pre}_{k}{l}"
    qps = {0: [5, 2, 7], 1: [3, 11]}  # rank -> qpids
    truth = {}
    for rank, ids in qps.items():
        with open(tmp_path / f"pr_{rank}.lhistory.csv", "w") as f:
            f.write(hdr + "\n")
            for t in range(1, 7):
                for qp in ids:
                    if qp == 11 and t > 4:
                        continue  # ragged: this point stops early
                    vals = rng.standard_normal(18) * 1e-3
                    f.write(f"{t},{t * 0.5},{qp},{qp // 8},{qp % 8},g0," + ",".join("%.16g" % v for v in vals) + "\n")
                    s = [float("%.16g" % v) for v in vals[:6]]  # 00 01 02 11 12 22
                    truth.setdefault(qp, []).append([s[0], s[3], s[5], s[1], s[2], s[4]])
    files = [str(tmp_path / f"pr_{r}.lhistory.csv") for r in qps]
    b = Batch.from_lhistory(files, "strain")
    assert list(b.ids) == sorted(truth)
    off, steps = b.offsets, b.steps
    for q, qp in enumerate(b.ids):
        want = np.array(truth[int(qp)])
        assert np.array_equal(bits(steps[int(off[q]):int(off[q + 1])]), bits(want)), qp
    assert int(off[list(b.ids).index(11) + 1] - off[list(b.ids).index(11)]) == 4
    # other tensor of the log
    u = Batch.from_lhistory(files, "updstrain")
    assert u.steps.shape == steps.shape and not np.array_equal(u.steps, steps)
    # write as strain_<ID> files and read them back: every double survives (17 significant digits)
    out = tmp_path / "strains"
    out.mkdir()
    b.write_strain_files(str(out))
    back = Batch.read_files([str(out / f"strain_{qp}") for qp in b.ids])
    assert np.array_equal(back.offsets, off) and np.array_equal(bits(back.steps), bits(steps))
    with pytest.raises(ScemaError):
        Batch.from_lhistory(files, "nosuchtensor")


def test_lhistory_to_strain_command_line(tmp_path):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "scema_b200", "bin", "lhistory_to_strain")
    hdr = "timestep,time,qpid,cell,qpoint,material" + "".join(
        f",{p}_{k}{l}" for p in ("strain", "updstrain", "stress") for k in range(3) for l in range(k, 3))
    with open(tmp_path / "pr_0.lhistory.csv", "w") as f:
        f.write(hdr + "\n")
        for t in range(1, 5):
            for q in (4, 9):
                f.write(f"{t},{t * .1},{q},0,{q},g0," + ",".join(repr((t + q) * 1e-3 * (j + 1)) for j in range(18)) + "\n")
    out = tmp_path / "out"
    out.mkdir()
    r = subprocess.run([exe, str(out), str(tmp_path / "pr_0.lhistory.csv")], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout == "2 histories, 8 steps\n", r.stderr
    b = Batch.read_dir(str(out) + "/")
    assert sorted(b.ids.tolist()) == [4, 9]
    k = b.ids.tolist().index(9)
    first = b.steps[int(b.offsets[k])]
    s = [(1 + 9) * 1e-3 * (j + 1) for j in range(6)]  # 00 01 02 11 12 22
    assert first.tolist() == [s[0], s[3], s[5], s[1], s[2], s[4]]
    r = subprocess.run([exe, str(out)], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage" in r.stderr
