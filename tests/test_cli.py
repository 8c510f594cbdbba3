"""The C++ drop-in command lines (scema_b200/bin) against the reference's own binaries built from
the unmodified sources (oracle/_ref, run live on the same directory so that the directory
enumeration order — which fixes batch order and partner order — is the same for both).

Where oracle/_ref is not built, the reference runs recorded in tests/golden/reference_runs.json are
used instead (tests/golden/make_golden_live.py). Those came from another directory, whose
enumeration order may differ, so they are compared line set by line set: a SHA-256 of the sorted
lines of stdout and of every result file (its first 64 bits per file)."""
import hashlib
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from scema_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "scema_b200", "bin")
REF = os.path.join(ROOT, "oracle", "_ref")
THR = 1e-6


def write_strain_dir(path, n=150, seed=12, lmin=3, lmax=60):
    os.makedirs(path)
    off = synth.offsets(seed, n, 6, lmin, lmax)
    steps = synth.histories(seed, n, 6, 2e-3, synth.default_pert(THR, 10), off)
    ids = (np.arange(n) * 5 + 11).astype(np.uint32)
    for i in range(n):
        with open(os.path.join(path, f"strain_{ids[i]}"), "w") as f:
            for s in steps[int(off[i]):int(off[i + 1])]:
                f.write(" ".join(repr(float(v)) for v in s) + "\n")
    with open(os.path.join(path, "notes.txt"), "w") as f:
        f.write("not a strain file\n")
    return ids


def run(cmd, cwd):
    return subprocess.run(cmd, cwd=cwd, capture_output=True, text=True, timeout=600)


def sorted_lines_sha(text):
    return hashlib.sha256("\n".join(sorted(text.splitlines())).encode()).hexdigest()


def mpi_comparison_record(stdout, results_dir, ids):
    """A run of mpi_comparison_test as line sets: stdout and __results/ID_<id>.txt."""
    return {"stdout": sorted_lines_sha(stdout),
            "files": {str(i): sorted_lines_sha(open(os.path.join(results_dir, f"ID_{i}.txt")).read())[:16] for i in ids}}


def compare_all_record(stdout):
    """A run of compare_all_histories without its timing lines, as a line set."""
    strip = [ln for ln in stdout.splitlines() if not ln.startswith(("Read time", "Spline time", "Compare time"))]
    return {"stdout": sorted_lines_sha("\n".join(strip)), "lines": len(strip)}


def recorded(key):
    with open(os.path.join(ROOT, "tests", "golden", "reference_runs.json")) as f:
        return json.load(f)["cli"][key]


def test_mpi_comparison_test_matches_reference_binary(tmp_path):
    sdir = str(tmp_path / "strains") + "/"
    ids = write_strain_dir(sdir)
    ours = tmp_path / "ours"
    (ours / "__results").mkdir(parents=True)
    r = run([os.path.join(BIN, "mpi_comparison_test"), sdir, "10", repr(THR)], ours)
    assert r.returncode == 0, r.stderr
    assert "Ignoring: 'notes.txt'" in r.stdout
    assert len(os.listdir(ours / "__results")) == len(ids)
    n_lines = sum(len(open(ours / "__results" / f"ID_{i}.txt").read().splitlines()) for i in ids)
    assert n_lines > 50
    ref_bin = os.path.join(REF, "mpi_comparison_test")
    if os.path.exists(ref_bin):
        theirs = tmp_path / "theirs"
        (theirs / "__results").mkdir(parents=True)
        q = run([ref_bin, sdir, "10", repr(THR)], theirs)
        assert q.returncode == 0 and q.stdout == r.stdout
        for i in ids:
            assert open(ours / "__results" / f"ID_{i}.txt").read() == open(theirs / "__results" / f"ID_{i}.txt").read(), i
    else:
        assert mpi_comparison_record(r.stdout, ours / "__results", ids) == recorded("mpi_comparison_test")

    # downstream: the unchanged python consumer and the native reducer agree on these files
    macro = tmp_path / "macro"
    macro.mkdir()
    for i in ids:
        shutil.copy(ours / "__results" / f"ID_{i}.txt", macro / f"last.{i}.similar_hist")
    num_gps = int(ids.max()) + 1
    nat = run([os.path.join(BIN, "coarsegrain_dependency_network"), str(macro), str(tmp_path / "m_native.csv"), str(num_gps)], tmp_path)
    assert nat.returncode == 0, nat.stderr
    script = None
    for p in ("/root/reference/clustering/coarsegrain_dependency_network.py", os.path.join(REF, "coarsegrain_dependency_network.pyc")):
        if os.path.exists(p):
            script = p
            break
    if script:
        py = run([sys.executable, script, str(macro), str(tmp_path / "m_py.csv"), str(num_gps)], tmp_path)
        assert py.returncode == 0, py.stderr
        assert open(tmp_path / "m_py.csv").read() == open(tmp_path / "m_native.csv").read()
        assert py.stdout == nat.stdout


def test_compare_all_histories_matches_reference_binary(tmp_path):
    sdir = str(tmp_path / "strains") + "/"
    write_strain_dir(sdir, n=60, seed=5)
    r = run([os.path.join(BIN, "compare_all_histories"), sdir, "10"], tmp_path)
    assert r.returncode == 0, r.stderr
    vs = [ln for ln in r.stdout.splitlines() if " vs " in ln]
    assert len(vs) == 60 * 61 // 2
    assert r.stdout.splitlines()[-3].startswith("Read time: ") and r.stdout.splitlines()[-1].startswith("Compare time: ")
    ref_bin = os.path.join(REF, "compare_all_histories")
    if os.path.exists(ref_bin):
        q = run([ref_bin, sdir, "10"], tmp_path)
        assert q.returncode == 0
        strip = lambda out: [ln for ln in out.splitlines() if not ln.startswith(("Read time", "Spline time", "Compare time"))]
        assert strip(q.stdout) == strip(r.stdout)
    else:
        assert compare_all_record(r.stdout) == recorded("compare_all_histories")


def test_cli_error_behaviour(tmp_path):
    r = run([os.path.join(BIN, "mpi_comparison_test"), "x"], tmp_path)
    assert r.returncode == 1 and r.stderr == "Usage: ./mpi_comparison_test STRAIN_DIRECTORY NUM_SPLINE_POINTS THRESH\n"
    r = run([os.path.join(BIN, "compare_all_histories")], tmp_path)
    assert r.returncode == 1 and r.stderr == "Usage: ./compare_all_histories STRAIN_DIRECTORY NUM_SPLINE_POINTS\n"
    sdir = str(tmp_path / "strains") + "/"
    write_strain_dir(sdir, n=8)
    # no __results directory: the reference exits 1 with this message (strain2spline.h:303-307)
    r = run([os.path.join(BIN, "mpi_comparison_test"), sdir, "10", "1e-6"], tmp_path)
    assert r.returncode == 1 and "Could not open __results/ID_" in r.stderr
    # a history with two steps: splinify exits (strain2spline.h:145-148)
    with open(os.path.join(sdir, "strain_9999"), "w") as f:
        f.write("1 2 3 4 5 6\n1 2 3 4 5 6\n")
    (tmp_path / "__results").mkdir()
    r = run([os.path.join(BIN, "mpi_comparison_test"), sdir, "10", "1e-6"], tmp_path)
    assert r.returncode == 1 and "Need at least 3 points for splinify()" in r.stderr
