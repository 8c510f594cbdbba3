"""Tile-sharded path on real GPUs (needs >= 2): one process per GPU under torchrun, NCCL
all-gather of the resampled rows and of the edge counts; union of the shards == oracle."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_gpu_sharded_pipeline():
    import torch
    ng = torch.cuda.device_count()
    if ng < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2 if ng < 4 else 4
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29611",
                        os.path.join(ROOT, "tools", "multigpu_check.py")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("multigpu_check ok") == 7   # DMMA, FMA, tcgen05 one-shot, tcgen05 streamed; overlapped x2, plain on aligned shares


def test_multi_gpu_behind_the_c_abi(oracle):
    """scema_multi_cluster / scema_multi_compare_rows (one process, one thread + context per GPU, NCCL inside the
    library): the merged list equals the oracle's (ids, order, distance bits) for the tcgen05 and the DMMA filter, the
    per-history files equal the single-GPU ones, and a shard that is too dense makes ALL shards switch filter."""
    import numpy as np
    import torch
    import scema_b200
    from scema_b200 import synth, PAIRS_TC, PAIRS_DMMA
    ng = torch.cuda.device_count()
    if ng < 2:
        pytest.skip("needs >= 2 GPUs")
    G = min(ng, 4)
    thr, P, n = 1e-6, 10, 20011
    off = synth.offsets(6, n, 16, 5, 70)
    steps = synth.histories(6, n, 16, 5e-3, synth.default_pert(thr, P), off)
    ids = (np.arange(n, dtype=np.uint32) * 3 + 7)
    want_rows = oracle.splinify_batch(steps, off, P)
    wi, wj, wd, _ = oracle.all_pairs(want_rows, thr)
    m = scema_b200.MultiCluster(list(range(G)))
    for variant in (PAIRS_TC, PAIRS_DMMA):
        ne = m.cluster(steps, off, ids, P, thr, variant)
        a, b, d = m.first.get_edges()
        assert ne == len(wi) and np.array_equal(a, wi) and np.array_equal(b, wj)
        assert np.array_equal(d.view(np.uint64), wd.view(np.uint64))
        cnt, offs = m.shard_edges()
        assert int(cnt.sum()) == ne and np.all(cnt > 0) and list(offs) == [int(cnt[:r].sum()) for r in range(G)]
        assert m.last_ms()["variant_used"] == variant
        sp = m.first.get_spline()
        assert np.array_equal(sp.view(np.uint64), want_rows.view(np.uint64))       # every GPU holds the full matrix
    ne = m.compare_rows(want_rows, thr, PAIRS_TC, ids)
    assert ne == len(wi)
    a, b, d = m.first.get_edges()
    assert np.array_equal(a, wi) and np.array_equal(b, wj) and np.array_equal(d.view(np.uint64), wd.view(np.uint64))
    # all pairs neighbours: the sample sends every shard to the filter-free kernel, consistently
    dense = 1e-3 + 1e-9 * np.random.default_rng(0).standard_normal((3000, 60))
    assert m.compare_rows(dense, thr, PAIRS_TC) == 3000 * 2999 // 2
    m.close()


def test_cli_on_several_gpus_matches_the_reference_binary(tmp_path):
    """bin/mpi_comparison_test with SCEMA_B200_DEVICES=0,1[,2,3]: byte-identical result files to the one-GPU run and, where
    oracle/_ref is built, to the reference binary (oracle/_ref/mpi_comparison_test)."""
    import filecmp
    import numpy as np
    import torch
    from scema_b200 import synth
    from oracle.pyoracle import ref_binary
    ng = torch.cuda.device_count()
    if ng < 2:
        pytest.skip("needs >= 2 GPUs")
    ref = ref_binary("mpi_comparison_test")
    n, P, thr = 3000, 10, 1e-6
    off = synth.offsets(9, n, 8, 6, 40)
    steps = synth.histories(9, n, 8, 5e-3, synth.default_pert(thr, P), off)
    sdir = tmp_path / "strain"
    sdir.mkdir()
    for i in range(n):
        with open(sdir / f"strain_{i * 2 + 1}", "w") as f:
            for row in steps[int(off[i]):int(off[i + 1])]:
                f.write(" ".join(repr(float(v)) for v in row) + "\n")
    ours = os.path.join(ROOT, "scema_b200", "bin", "mpi_comparison_test")
    runs = {"one": (ours, {}), "multi": (ours, {"SCEMA_B200_DEVICES": ",".join(str(d) for d in range(min(ng, 4)))})}
    if ref:
        runs["ref"] = (ref, {})
    for name, (exe, env) in runs.items():
        wd = tmp_path / name
        (wd / "__results").mkdir(parents=True)
        r = subprocess.run([exe, str(sdir) + "/", str(P), repr(thr)], cwd=wd, env=dict(os.environ, **env), capture_output=True, text=True,
                           timeout=600)
        assert r.returncode == 0, (name, r.stdout[-2000:], r.stderr[-2000:])
    base = "ref" if ref else "one"
    names = sorted(os.listdir(tmp_path / base / "__results"))
    assert len(names) == n
    for other in (k for k in runs if k != base):
        assert sorted(os.listdir(tmp_path / other / "__results")) == names
        match, mismatch, errors = filecmp.cmpfiles(tmp_path / base / "__results", tmp_path / other / "__results", names, shallow=False)
        assert not mismatch and not errors, (other, mismatch[:5], errors[:5])
    assert sum(os.path.getsize(tmp_path / base / "__results" / f) for f in names) > 10000
