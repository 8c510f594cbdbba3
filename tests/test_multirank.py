"""Multi-rank semantics of compare_histories_with_all_ranks (reference headers/strain2spline.h:546-614): every history
ends up with the list of all others closer than the threshold, ordered own rank first, then the histories received from
rank-1, rank-2, ... each in its sender's order. The reference's real ring runs here with ranks as threads
(tests/helpers/mpi_threads/mpi.h); the drop-in header's gather-to-rank-0 branch runs through the same stand-in."""
import json
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = json.load(open(os.path.join(ROOT, "tests", "golden", "multirank_cases.json")))


def test_ring_order_host_logic(tmp_path):
    """b200::ring_sort == a literal simulation of the reference's ring loops, 1..5 ranks, random neighbour relations
    (host logic of the header only: compiled without the library)."""
    exe = str(tmp_path / "ring_check")
    subprocess.run(["g++", "-std=c++11", "-O1", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "scema_b200", "host"),
                    "-o", exe, os.path.join(ROOT, "tests", "helpers", "ring_order_check.cc")], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "ring order ok" in r.stdout, r.stdout + r.stderr


def test_golden_is_what_the_reference_ring_prints():
    """The committed golden outputs are reproduced by the reference header running its ring live (where oracle/_ref is built),
    and they show what the ring does with several ranks."""
    exe = os.path.join(ROOT, "oracle", "_ref", "multirank_driver_ref")
    if os.path.exists(exe):
        for c in CASES:
            r = subprocess.run([exe] + c["args"], capture_output=True, text=True, timeout=120)
            assert r.returncode == 0 and r.stdout == c["stdout"], c["args"]
    assert sum(c["stdout"].count("\n") for c in CASES) > 300
    # more than one rank really reorders the lists: same histories, different line order than the one-rank run
    one, three = CASES[0]["stdout"], CASES[2]["stdout"]
    assert sorted(l for l in one.splitlines() if not l.startswith("history")) == sorted(l for l in three.splitlines() if not l.startswith("history"))
    assert one != three


@pytest.mark.gpu
def test_dropin_header_multi_rank_branch_matches_the_reference_ring(tmp_path):
    """The same caller compiled against strain2spline_b200.h with MPI present (thread-backed): histories gathered on
    rank 0, one GPU batch, results scattered back — byte-identical to the reference ring for 1 to 4 ranks."""
    exe = str(tmp_path / "multirank_b200")
    subprocess.run(["g++", "-std=c++11", "-O2", "-ffp-contract=off", "-I" + os.path.join(ROOT, "tests", "helpers", "mpi_threads"),
                    "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "scema_b200", "host"), "-o", exe,
                    os.path.join(ROOT, "tests", "helpers", "multirank_driver.cc"), "-L" + os.path.join(ROOT, "scema_b200"),
                    "-lscema_hist", "-Wl,-rpath," + os.path.join(ROOT, "scema_b200"), "-lpthread"], check=True)
    for c in CASES:
        r = subprocess.run([exe] + c["args"], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        assert r.stdout == c["stdout"], c["args"]
