"""Graph reduction: oracle restatement and native C++ against the real script's recorded output
(tests/golden/graph_cases.json, pipeline_c1) and, where available, the script itself run live."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def script_cmd():
    for p in ("/root/reference/clustering/coarsegrain_dependency_network.py",
              os.path.join(ROOT, "oracle", "_ref", "coarsegrain_dependency_network.pyc")):
        if os.path.exists(p):
            return [sys.executable, p]
    return None


def native_calls(eu, ev, num_gps):
    import ctypes as C
    import scema_b200
    L = scema_b200.lib()
    eu = np.ascontiguousarray(eu, dtype=np.uint32)
    ev = np.ascontiguousarray(ev, dtype=np.uint32)
    mp = np.empty(num_gps, dtype=np.uint32)
    it, nr = C.c_uint64(0), C.c_uint64(0)
    rc = L.scema_reduce_calls(eu.ctypes.data, ev.ctypes.data, len(eu), num_gps, mp.ctypes.data, C.byref(it), C.byref(nr))
    assert rc == 0
    return mp, it.value, nr.value


@pytest.mark.parametrize("case", json.load(open(os.path.join(GOLD, "graph_cases.json"))), ids=lambda c: f"n{c['num_gps']}")
def test_reduce_golden(oracle, case):
    eu = [c[0] for c in case["calls"]]
    ev = [c[1] for c in case["calls"]]
    mp, it, nr = oracle.reduce_graph(eu, ev, case["num_gps"])
    assert mp.tolist() == case["mapping"]
    mp2, it2, nr2 = native_calls(eu, ev, case["num_gps"])
    assert mp2.tolist() == case["mapping"] and (it2, nr2) == (it, nr)


def test_reduce_pipeline_golden(oracle):
    g = json.load(open(os.path.join(GOLD, "pipeline_c1", "reference_outputs.json")))
    eu, ev = [], []
    for nm in g["glob_order"]:
        i = nm.split(".")[1]
        for line in g["results"][i].splitlines():
            a, b, _ = line.split()
            eu.append(int(a))
            ev.append(int(b))
    mp, it, nr = oracle.reduce_graph(eu, ev, g["n"])
    want = [int(l.split()[1]) for l in g["mapping_csv"].splitlines()]
    assert mp.tolist() == want
    assert f"Converged in {it} iterations" in g["python_stdout"]
    assert f"Number of simulations required:  {g['n'] - nr}" in g["python_stdout"]
    mp2, _, _ = native_calls(eu, ev, g["n"])
    assert mp2.tolist() == want


def test_reduce_errors(oracle):
    with pytest.raises(ValueError):
        oracle.reduce_graph([0, 5], [1, 2], 4)  # IndexError in the script
    with pytest.raises(ValueError):
        oracle.reduce_graph([0], [1], 4, dist=[0.0])  # ZeroDivisionError in the script


def test_reduce_dir_vs_script_live(oracle, tmp_path):
    """Native scema_reduce_dir and the real script on the same directory (same readdir order). Where the script is not
    available, the oracle's literal restatement of it (checked against the script's recorded outputs above) takes its
    place, fed the files in the script's glob order."""
    import glob
    import scema_b200
    rng = np.random.default_rng(3)
    n = 500
    files = {}
    for _ in range(1500):
        a, b = rng.integers(0, n, size=2)
        if a == b:
            continue
        files.setdefault(int(a), []).append((int(a), int(b)))
        files.setdefault(int(b), []).append((int(b), int(a)))
    d = tmp_path / "macro"
    d.mkdir()
    for a, lst in files.items():
        with open(d / f"last.{a}.similar_hist", "w") as f:
            for x, y in lst:
                f.write(f"{x} {y} 3.5e-07\n")
    (d / "last.7.all_similar_hist").write_text("7 8 1\n")  # must be ignored by the glob
    (d / "last.9999.similar_hist").write_text("")          # empty file: counted, no edges
    it, nf, nr = scema_b200.reduce_dir(str(d), str(tmp_path / "m_native.csv"), n)
    cmd = script_cmd()
    if cmd is not None:
        py = subprocess.run(cmd + [str(d), str(tmp_path / "m_py.csv"), str(n)], capture_output=True, text=True, check=True)
        assert open(tmp_path / "m_py.csv").read() == open(tmp_path / "m_native.csv").read()
        assert f"Converged in {it} iterations" in py.stdout
        assert f"udpated:  {nf}" in py.stdout
        assert f"required:  {nf - nr}" in py.stdout
    names = glob.glob(os.path.join(str(d), "last.*.similar_hist"))
    eu, ev = [], []
    for nm in names:
        for line in open(nm).read().splitlines():
            a, b, _ = line.split()
            eu.append(int(a))
            ev.append(int(b))
    mp, it_o, nr_o = oracle.reduce_graph(eu, ev, n)
    got = [tuple(int(x) for x in ln.split()) for ln in open(tmp_path / "m_native.csv").read().splitlines()]
    assert got == list(enumerate(mp.tolist()))
    assert (it, nf, nr) == (it_o, len(names), nr_o)


def _random_calls(rng, kind, n):
    """add_edge call sequences of several shapes: (eu, ev) with duplicates, both directions, self loops."""
    if kind == "clusters":          # the usual case: small cliques-with-holes, every edge listed from both endpoints
        cs = int(rng.integers(2, 24))
        eu, ev = [], []
        for b in range(0, n - cs, cs):
            for i in range(cs):
                for j in range(i + 1, cs):
                    if rng.random() < 0.5:
                        eu += [b + i, b + j]
                        ev += [b + j, b + i]
        o = rng.permutation(len(eu))
        return np.array(eu)[o], np.array(ev)[o]
    if kind == "giant":             # one big sparse component (> 96 nodes: the bucket path) plus debris
        m = int(n * rng.uniform(1.0, 3.0))
        return rng.integers(0, n, m), rng.integers(0, n, m)
    if kind == "hubs":              # a few nodes of very high degree, many ties among the rest
        hubs = rng.integers(0, n, 5)
        eu = rng.choice(hubs, 3 * n)
        ev = rng.integers(0, n, 3 * n)
        return np.concatenate([eu, ev[: n // 2]]), np.concatenate([ev, (ev[: n // 2] + 1) % n])
    if kind == "chains":            # paths and rings: all degrees 1 or 2, the tie-break decides everything
        a = np.arange(n - 1)
        keep = rng.random(n - 1) < 0.9
        eu, ev = a[keep], a[keep] + 1
        o = rng.permutation(len(eu))
        return eu[o], ev[o]
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["clusters", "giant", "hubs", "chains"])
def test_reduce_random_graphs_match_the_restated_script(oracle, kind):
    """The native reducer works connected component by connected component (a scan per pick up to 96 nodes, degree
    buckets above); the oracle restates the script literally (all nodes re-sorted every iteration,
    coarsegrain_dependency_network.py:6-21,59-94). Same mapping, iteration count and removed-neighbour count."""
    rng = np.random.default_rng({"clusters": 1, "giant": 2, "hubs": 3, "chains": 4}[kind])
    for trial in range(12):
        n = int(rng.integers(5, 1200))
        eu, ev = _random_calls(rng, kind, n)
        if trial % 3 == 0 and len(eu):   # self loops (networkx counts them twice in the degree) and repeated calls
            k = rng.integers(0, len(eu), max(1, len(eu) // 20))
            eu = np.concatenate([eu, eu[k], eu[k]])
            ev = np.concatenate([ev, eu[-len(k):], ev[k]])
        want = oracle.reduce_graph(eu, ev, n)
        got = native_calls(eu, ev, n)
        assert got[0].tolist() == want[0].tolist(), (kind, trial, n)
        assert (got[1], got[2]) == (want[1], want[2]), (kind, trial, n)
