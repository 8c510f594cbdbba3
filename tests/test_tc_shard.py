"""The sharded prepare of the tcgen05 filter (scema_tc_shard_{begin,stats,finish,check,commit}, include/scema_hist.h).

On one GPU, G contexts on the same device stand in for G ranks: every context borrows the same full FP64 row buffer,
`begin` and `stats` run on each rank's share, the harness plays the two all-gathers (rank 0's centre, the packets of all
ranks) and the exchange of the fp16 images with plain device copies, and `compare(thr, PAIRS_TC, shard=r, n_shards=G)`
runs on every context. The union of the shards must equal the CPU oracle in indices, order and distance bits.

Without a GPU: the plan by which ShardedCluster.run_overlapped all-gathers the images (image_exchange) and the gather
itself (gather_images, on gloo with CPU tensors of exactly the size the library promises).
"""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from scema_b200.distributed import CudaView, aligned_shard_bounds, gather_images, image_exchange

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THR = 1e-6
ERR_INVALID, ERR_STATE, ERR_DENSE = 1, 5, 7


# ------------------------------------------------------------------------------------------------ CPU: the gather plan
def test_image_exchange_plan():
    """For every (n, G): each non-empty share starts at a multiple of 128 and ends at a multiple of 128 or at n (what
    scema_tc_shard_begin accepts), the image rows the ranks build tile [0, n_pad) exactly, each fits the rank's slot of
    the gather, and an in-place gather is only planned when the slots fill exactly the n_pad rows of the image."""
    ns = [1, 2, 127, 128, 129, 255, 256, 257, 1000, 2047, 2048, 2049, 3000, 4096, 6143, 8192, 8193, 20011, 24576, 1000000,
          4000000]
    for n in ns:
        for G in range(1, 9):
            per, bounds, n_pad, own, staged = image_exchange(n, G)
            assert (per, bounds) == aligned_shard_bounds(n, G)
            assert n_pad % 256 == 0 and n <= n_pad < n + 256
            assert bounds[0][0] == 0 and bounds[-1][1] == n and all(bounds[i][1] == bounds[i + 1][0] for i in range(G - 1))
            for r, ((b, e), (ob, oe)) in enumerate(zip(bounds, own)):
                if e > b:
                    assert b % 128 == 0 and (e % 128 == 0 or e == n), (n, G, r)
                    assert ob == b == r * per and oe - ob <= per, (n, G, r)
                else:
                    assert ob == oe, (n, G, r)
            covered = [x for ob, oe in own for x in (ob, oe) if oe > ob]
            assert covered[0] == 0 and covered[-1] == n_pad and all(covered[i] == covered[i + 1] for i in range(1, len(covered) - 1, 2))
            if not staged:
                assert G * per == n_pad, (n, G)      # the in-place gather writes the image and nothing past it
            else:
                assert G * per > n_pad
    # the cases an in-place gather of G * per rows used to overrun (20011 only fitted into the [hi | lo] slack)
    assert image_exchange(2048, 4)[4] and image_exchange(20011, 4)[4] and image_exchange(3000, 1)[4]
    assert not image_exchange(8192, 4)[4]
    assert image_exchange(3000, 4)[1] == [(0, 2048), (2048, 3000), (3000, 3000), (3000, 3000)]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        for G in (1, 2, 3, 4, 8):
            group = dist.new_group(list(range(G)))
            if rank >= G:
                continue
            for n in (1, 300, 2048, 3000, 8192, 20011):
                for bpr in (128, 256):
                    per, bounds, n_pad, own, staged = image_exchange(n, G)
                    i = torch.arange(n_pad * bpr, dtype=torch.int64)
                    want = ((i // bpr) * 7 + i % bpr) % 251
                    want = want.to(torch.uint8)
                    img = torch.full((n_pad * bpr,), 0xEE, dtype=torch.uint8)    # exactly the bytes the library promises
                    b, e = own[rank]
                    img[b * bpr:e * bpr] = want[b * bpr:e * bpr]
                    stage = gather_images(img, n, G, rank, bpr, group)
                    assert torch.equal(img, want), (G, n, bpr, rank)
                    assert (stage is None) == (not staged)
                    if staged:      # a second step reuses the staging buffer
                        img[:] = 0xEE
                        img[b * bpr:e * bpr] = want[b * bpr:e * bpr]
                        assert gather_images(img, n, G, rank, bpr, group, stage) is stage and torch.equal(img, want)
        with pytest.raises(ValueError):
            gather_images(torch.zeros(2048 * 128 + 1, dtype=torch.uint8), 2048, 1, 0, 128)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_gather_images_gloo(tmp_path):
    """gather_images (run_overlapped's exchange of the fp16 images) on CPU tensors of exactly n_pad * bpr bytes: every
    rank ends with every rank's rows, for in-place and staged gathers, empty trailing shares included."""
    mp.spawn(_gather_worker, args=(8, _free_port(), str(tmp_path)), nprocs=8, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(8))


# ------------------------------------------------------------------------------------------------ GPU: the harness
def _view(ptr, count, typestr):
    return torch.as_tensor(CudaView(ptr, (count,), typestr), device="cuda")


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _edges_equal(got, want):
    return (len(got[0]) == len(want[0]) and np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
            and np.array_equal(_bits(got[2]), _bits(want[2])))


def _contexts(G, full, n, K):
    import scema_b200
    ctxs = [scema_b200.HistCluster(0) for _ in range(G)]
    for c in ctxs:
        c.set_spline(device_ptr=full.data_ptr(), n=n, k=K)
    return ctxs


def _close(ctxs):
    torch.cuda.synchronize()
    for c in ctxs:
        c.close()


def sharded_prepare(ctxs, n, K, thr, bounds, optimistic=False, before_commit=None):
    """One sharded prepare over the contexts (rank r = ctxs[r] owns bounds[r]), the exchanges played by device copies.
    before_commit() -> a recorded torch.cuda.Event (or None) that every commit passes as rows_ready_event.
    -> (choice, rank 0's centre as numpy)."""
    G = len(ctxs)
    torch.cuda.synchronize()
    cptr = [c.tc_shard_begin(thr, b, e) for c, (b, e) in zip(ctxs, bounds)]
    torch.cuda.synchronize()
    centre = _view(cptr[0], K, "<f8").clone()
    torch.cuda.synchronize()
    pk = [c.tc_shard_stats(centre.data_ptr()) for c in ctxs]
    torch.cuda.synchronize()
    words = pk[0][1]
    packets = torch.empty((G, words), dtype=torch.int64, device="cuda")
    for r, (p, w) in enumerate(pk):
        assert w == words
        packets[r].copy_(_view(p, w, "<i8"))
    torch.cuda.synchronize()
    fin = [c.tc_shard_finish(packets.data_ptr(), G, n * (n - 1) // 2 // G, optimistic) for c in ctxs]
    torch.cuda.synchronize()
    choice = fin[0][0]
    assert all(f[0] == choice for f in fin), fin           # every rank reduces the same packets
    if optimistic:
        assert choice == 1
    if choice == 1:
        bpr = fin[0][2]
        n_pad = (n + 255) // 256 * 256
        imgs = [_view(f[1], n_pad * bpr, "|u1") for f in fin]
        for q, (b, e) in enumerate(bounds):
            if e == b:
                continue
            lo, hi = b * bpr, (n_pad if e == n else e) * bpr    # the share that ends at n carries the padding rows
            for r in range(G):
                if r != q:
                    imgs[r][lo:hi].copy_(imgs[q][lo:hi])
        torch.cuda.synchronize()
        ev = before_commit() if before_commit else None
        for c in ctxs:
            c.tc_shard_commit(ev.cuda_event if ev is not None else None)
    return choice, centre.cpu().numpy()


def compare_shards(ctxs, thr, variant, allow_dense=False):
    """compare(shard=r, n_shards=G) on every context -> the union in canonical order, or None when a shard reported
    SCEMA_ERR_DENSE (allow_dense); the shards' lists are returned too."""
    from scema_b200 import ScemaError
    G, parts, dense = len(ctxs), [], False
    for r, c in enumerate(ctxs):
        try:
            c.compare(thr, variant, shard=r, n_shards=G)
            parts.append(c.get_edges())
        except ScemaError as e:
            if e.code != ERR_DENSE or not allow_dense:
                raise
            dense = True
    if dense:
        return None, parts
    a = np.concatenate([p[0] for p in parts])
    b = np.concatenate([p[1] for p in parts])
    d = np.concatenate([p[2] for p in parts])
    o = np.lexsort((b, a))
    return (a[o], b[o], d[o]), parts


def plant_across(rows, thr, bounds, n_plant, rng, spread=1e-16):
    """Rewrite n_plant rows as partner + u * thr * (1 +- a few ulp), the partner in another share wherever there are
    two non-empty shares: pairs inside the guard band that only the image exchange brings together."""
    shares = [(b, e) for b, e in bounds if e > b]
    for q in range(n_plant):
        sa = int(rng.integers(0, len(shares)))
        sb = (sa + 1 + int(rng.integers(0, len(shares) - 1))) % len(shares) if len(shares) > 1 else sa
        a = int(rng.integers(*shares[sa]))
        b = int(rng.integers(*shares[sb]))
        if a == b:
            continue
        u = rng.standard_normal(rows.shape[1])
        u /= np.linalg.norm(u)
        rows[b] = rows[a] + u * thr * (1 + (q - n_plant / 2) * spread)
    return rows


def workload(n, K, seed, bounds, n_plant=300):
    """Spline-like rows (synth.rows, clusters of 16) of K columns with pairs planted across the shares."""
    from scema_b200 import synth
    rng = np.random.default_rng(seed)
    if K % 6 == 0 and K >= 12:
        rows = synth.rows(seed, n, 16, K // 6, 5e-3, synth.default_pert(THR, K // 6))
    else:   # rows too short for a spline: clusters of 16 whose members lie about the threshold apart
        centres = 5e-3 * rng.uniform(-1, 1, size=((n + 15) // 16, K))
        scale = THR * rng.uniform(0.2, 0.8, size=(n, 1)) / np.sqrt(K)
        rows = centres[np.arange(n) // 16] + scale * rng.standard_normal((n, K))
    return plant_across(rows, THR, bounds, n_plant, rng)


def cross_share_edges(want, bounds):
    share = np.zeros(bounds[-1][1], dtype=np.int64)
    for r, (b, e) in enumerate(bounds):
        share[b:e] = r
    return int(np.count_nonzero(share[want[0]] != share[want[1]]))


def run_case(oracle, rows, bounds, optimistic=False, expect_choice_1=True):
    """Sharded prepare on rows + compare on every shard == oracle; on the one-slice path also the filter that ran and
    the centre every context used."""
    from scema_b200 import PAIRS_TC, PAIRS_DMMA
    n, K = rows.shape
    want = oracle.all_pairs(rows, THR)[:3]
    full = torch.from_numpy(np.ascontiguousarray(rows)).cuda()
    ctxs = _contexts(len(bounds), full, n, K)
    try:
        choice, centre = sharded_prepare(ctxs, n, K, THR, bounds, optimistic=optimistic)
        if expect_choice_1:
            assert choice == 1, choice
        got, _ = compare_shards(ctxs, THR, PAIRS_TC, allow_dense=True)
        if got is None:
            got, _ = compare_shards(ctxs, THR, PAIRS_DMMA)
        assert _edges_equal(got, want), (len(got[0]), len(want[0]))
        if choice == 1:
            for c in ctxs:
                assert c.counters()["tc_slices"] == 1
                assert np.array_equal(_bits(c.tc_centre()), _bits(centre))
        return choice, want
    finally:
        _close(ctxs)


# ---- ranks and shares
def _aligned(n, G):
    return aligned_shard_bounds(n, G)[1]


SHARES = [
    ("G1", 2500, [(0, 2500)]),
    ("G2_aligned", 9000, _aligned(9000, 2)),
    ("G3_aligned", 9000, _aligned(9000, 3)),
    ("G4_trailing_empty", 3000, _aligned(3000, 4)),             # (0,2048) (2048,3000) (3000,3000) (3000,3000)
    ("G4_three_empty_at_2048", 2048, _aligned(2048, 4)),       # an in-place image gather would overrun the image here
    ("G8_aligned", 20011, _aligned(20011, 8)),                 # five shares of 4096 rows or less, three empty
    ("G8_one_share_below_2048", 1000, _aligned(1000, 8)),      # seven empty shares at an unaligned row
    ("G3_unequal_128", 1000, [(0, 128), (128, 640), (640, 1000)]),
    ("G4_unequal_empty_middle", 5000, [(0, 384), (384, 384), (384, 2432), (2432, 5000)]),
    ("G2_unequal", 5000, [(0, 4736), (4736, 5000)]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,n,bounds", SHARES, ids=[s[0] for s in SHARES])
def test_shares(oracle, name, n, bounds):
    rows = workload(n, 60, 11, bounds)
    _, want = run_case(oracle, rows, bounds)
    if sum(e > b for b, e in bounds) > 1:
        assert cross_share_edges(want, bounds) >= 50


# ---- row widths: one chunk of 64 columns, two, ten (k_tc_derive_b swaps the fold columns of the last chunk only)
@pytest.mark.gpu
@pytest.mark.parametrize("K", [6, 30, 60, 66, 120, 636])
def test_row_widths(oracle, K):
    bounds = [(0, 896), (896, 1664), (1664, 2500)]
    rows = workload(2500, K, 20 + K, bounds)
    _, want = run_case(oracle, rows, bounds)
    assert cross_share_edges(want, bounds) >= 50


@pytest.mark.gpu
def test_rows_wider_than_ten_chunks_are_refused():
    import scema_b200
    n, K = 300, 642
    full = torch.zeros((n, K), dtype=torch.float64, device="cuda")
    ctxs = _contexts(1, full, n, K)
    try:
        with pytest.raises(scema_b200.ScemaError) as e:
            ctxs[0].tc_shard_begin(THR, 0, n)
        assert e.value.code == ERR_INVALID
    finally:
        _close(ctxs)


# ---- magnitudes: the shares must agree on one scale; special values outside rank 0's share
@pytest.mark.gpu
@pytest.mark.parametrize("optimistic", [False, True])
def test_shares_of_different_magnitude(oracle, optimistic):
    n = 3000
    bounds = [(0, 1024), (1024, 2048), (2048, 3000)]
    rng = np.random.default_rng(4)
    rows = workload(n, 60, 4, bounds, n_plant=0)
    rows[1024:2048] *= 2e5                           # share 1 near 1e3
    rows[2048:2148] *= 1e-147                        # part of share 2 near 1e-150: all of its pairs are edges
    plant_across(rows, THR, [(1024, 2048)], 60, rng)                       # near-threshold pairs at 1e3
    plant_across(rows, THR, [(0, 1024), (2148, 3000)], 120, rng)           # and across shares 0 and 2
    rows[1500] = np.nan
    rows[2100, 5] = np.inf
    rows[1100, 7] = -np.inf
    rows[1900] = rows[1901]                          # duplicates: in share 1, between shares 1 and 2, 0 and 2
    rows[2700] = rows[1800]
    rows[2650] = rows[100]
    _, want = run_case(oracle, rows, bounds, optimistic=optimistic, expect_choice_1=optimistic)
    pairs = set(zip(want[0].tolist(), want[1].tolist()))
    assert {(1900, 1901), (1800, 2700), (100, 2650), (2048, 2147)} <= pairs
    assert not any(1500 in p for p in pairs)


# ---- optimistic finish
@pytest.mark.gpu
def test_optimistic_finish_when_the_assumption_holds(oracle):
    from scema_b200 import PAIRS_TC
    n = 9000
    bounds = _aligned(n, 4)                          # the last share is empty
    rows = workload(n, 60, 8, bounds)
    want = oracle.all_pairs(rows, THR)[:3]
    full = torch.from_numpy(rows).cuda()
    ctxs = _contexts(4, full, n, 60)
    try:
        assert sharded_prepare(ctxs, n, 60, THR, bounds)[0] == 1
        assert _edges_equal(compare_shards(ctxs, THR, PAIRS_TC)[0], want)
        sharded_prepare(ctxs, n, 60, THR, bounds, optimistic=True)
        assert _edges_equal(compare_shards(ctxs, THR, PAIRS_TC)[0], want)
        assert [c.tc_shard_check() for c in ctxs] == [1] * 4
        assert all(c.counters()["tc_slices"] == 1 for c in ctxs)
    finally:
        _close(ctxs)


def _dense_rows(n):
    return 1e-3 + 1e-9 * np.random.default_rng(0).standard_normal((n, 60))


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 4])
def test_optimistic_finish_when_the_assumption_is_wrong(oracle, G):
    """All rows within the threshold of each other: the sample would not have chosen one slice. The optimistic image
    still gives the exact edges (or SCEMA_ERR_DENSE, and then every shard repeats with the DMMA filter); check() says
    so, and a single shard switches filter by itself."""
    from scema_b200 import PAIRS_TC, PAIRS_DMMA
    n = 3000
    bounds = _aligned(n, G)
    rows = _dense_rows(n)
    want = oracle.all_pairs(rows, THR)[:3]
    assert len(want[0]) == n * (n - 1) // 2
    full = torch.from_numpy(rows).cuda()
    ctxs = _contexts(G, full, n, 60)
    try:
        sharded_prepare(ctxs, n, 60, THR, bounds, optimistic=True)
        got, parts = compare_shards(ctxs, THR, PAIRS_TC, allow_dense=G > 1)
        keys = set(zip(want[0].tolist(), want[1].tolist()))
        for a, b, d in parts:                        # what a shard did return is right
            assert set(zip(a.tolist(), b.tolist())) <= keys and np.all(d < THR)
        checks = [c.tc_shard_check() for c in ctxs]
        assert len(set(checks)) == 1 and checks[0] != 1
        if got is not None:
            assert _edges_equal(got, want)
        if G > 1:
            got, _ = compare_shards(ctxs, THR, PAIRS_DMMA)
        assert _edges_equal(got, want)
    finally:
        _close(ctxs)


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 4])
def test_finish_choosing_another_filter(oracle, G):
    """A non-optimistic finish whose sample names another filter builds no image: commit is refused and the ordinary
    sharded compare is exact."""
    import scema_b200
    from scema_b200 import PAIRS_TC, PAIRS_DMMA
    n = 3000
    bounds = _aligned(n, G)
    rows = _dense_rows(n)
    want = oracle.all_pairs(rows, THR)[:3]
    full = torch.from_numpy(rows).cuda()
    ctxs = _contexts(G, full, n, 60)
    try:
        choice, _ = sharded_prepare(ctxs, n, 60, THR, bounds)
        assert choice != 1
        for c in ctxs:
            with pytest.raises(scema_b200.ScemaError) as e:
                c.tc_shard_commit()
            assert e.value.code == ERR_STATE
        got, _ = compare_shards(ctxs, THR, PAIRS_TC, allow_dense=True)
        if got is None:
            got, _ = compare_shards(ctxs, THR, PAIRS_DMMA)
        assert _edges_equal(got, want)
    finally:
        _close(ctxs)


# ---- after commit: a new threshold or new rows must not reuse the image
@pytest.mark.gpu
def test_changes_after_commit(oracle):
    from scema_b200 import PAIRS_TC
    n = 5000
    bounds = _aligned(n, 3)
    rows = workload(n, 60, 13, bounds)
    rows2 = workload(n, 60, 14, bounds)
    full = torch.from_numpy(rows).cuda()
    ctxs = _contexts(3, full, n, 60)
    try:
        assert sharded_prepare(ctxs, n, 60, THR, bounds)[0] == 1
        want2 = oracle.all_pairs(rows, 2 * THR)[:3]
        assert len(want2[0]) > len(oracle.all_pairs(rows, THR)[0])
        assert _edges_equal(compare_shards(ctxs, 2 * THR, PAIRS_TC)[0], want2)
        assert sharded_prepare(ctxs, n, 60, THR, bounds)[0] == 1
        full.copy_(torch.from_numpy(rows2))          # same buffer, new rows
        torch.cuda.synchronize()
        for c in ctxs:
            c.set_spline(device_ptr=full.data_ptr(), n=n, k=60)
        assert _edges_equal(compare_shards(ctxs, THR, PAIRS_TC)[0], oracle.all_pairs(rows2, THR)[:3])
    finally:
        _close(ctxs)


# ---- rows_ready_event: the filter runs on the images while the FP64 rows are still arriving
@pytest.mark.gpu
def test_rows_ready_event(oracle):
    from scema_b200 import PAIRS_TC
    n, K = 5000, 60
    bounds = _aligned(n, 3)
    rows = workload(n, K, 15, bounds)
    want = oracle.all_pairs(rows, THR)[:3]
    assert cross_share_edges(want, bounds) >= 50       # edges that need the other shares' rows
    src = torch.from_numpy(rows).cuda()
    bufs = []
    for b, e in bounds:                                # each context holds only its own rows, NaN elsewhere
        buf = torch.full((n, K), float("nan"), dtype=torch.float64, device="cuda")
        buf[b:e] = src[b:e]
        bufs.append(buf)
    import scema_b200
    ctxs = [scema_b200.HistCluster(0) for _ in bounds]
    side = torch.cuda.Stream()
    ev = torch.cuda.Event()
    try:
        for c, buf in zip(ctxs, bufs):
            c.set_spline(device_ptr=buf.data_ptr(), n=n, k=K)

        def rows_arrive():
            with torch.cuda.stream(side):
                torch.cuda._sleep(200_000_000)         # ~0.1 s: the compare is enqueued long before the rows are there
                for (b, e), buf in zip(bounds, bufs):
                    buf[:b].copy_(src[:b])
                    buf[e:].copy_(src[e:])
                ev.record()
            return ev

        assert sharded_prepare(ctxs, n, K, THR, bounds, before_commit=rows_arrive)[0] == 1
        assert not ev.query()
        got, _ = compare_shards(ctxs, THR, PAIRS_TC)
        assert _edges_equal(got, want)
    finally:
        _close(ctxs)


# ---- call order and arguments
@pytest.mark.gpu
def test_call_order_and_arguments():
    import scema_b200
    n, K = 1000, 60
    full = torch.from_numpy(workload(n, K, 3, [(0, n)])).cuda()
    packets = torch.zeros((1, 4096), dtype=torch.int64, device="cuda")

    def code(fn, *args):
        with pytest.raises(scema_b200.ScemaError) as e:
            fn(*args)
        return e.value.code

    ctxs = _contexts(1, full, n, K)
    c = ctxs[0]
    try:
        assert code(c.tc_shard_stats, 0) == ERR_STATE
        assert code(c.tc_shard_finish, packets.data_ptr(), 1, 1) == ERR_STATE
        assert code(c.tc_shard_commit) == ERR_STATE
        assert code(c.tc_shard_check) == ERR_STATE
        assert code(c.tc_shard_begin, THR, 64, n) == ERR_INVALID          # unaligned start of a non-empty share
        assert code(c.tc_shard_begin, THR, 0, n + 1) == ERR_INVALID       # past the end
        assert code(c.tc_shard_begin, THR, 0, 200) == ERR_INVALID         # ends inside a 128-row block before n
        assert code(c.tc_shard_begin, THR, 512, 256) == ERR_INVALID
        for r in (0, 640, n):                                           # empty shares at any row
            c.tc_shard_begin(THR, r, r)
        # out of turn after begin: commit before finish, finish before stats, stats twice
        c.tc_shard_begin(THR, 0, 512)
        assert code(c.tc_shard_commit) == ERR_STATE
        c.tc_shard_begin(THR, 0, 512)
        assert code(c.tc_shard_finish, packets.data_ptr(), 1, 1) == ERR_STATE
        c.tc_shard_begin(THR, 0, 512)
        c.tc_shard_stats(0)
        assert code(c.tc_shard_stats, 0) == ERR_STATE
        torch.cuda.synchronize()
    finally:
        _close(ctxs)


# ---- the driver itself on one rank
_DRIVER = r"""
import sys
import numpy as np
import torch
import torch.distributed as dist
sys.path.insert(0, sys.argv[1])
import scema_b200
from scema_b200 import synth
from scema_b200.distributed import ShardedCluster, aligned_shard_bounds, image_exchange
from oracle.pyoracle import Oracle

n, P, thr = 3000, 10, 1e-6
assert image_exchange(n, 1)[4]          # one rank: the slot (4096 rows) is larger than the image (3072): staged gather
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
dist.init_process_group("nccl", store=dist.FileStore(sys.argv[2], 1), rank=0, world_size=1, device_id=dev)
off = synth.offsets(6, n, 16, 5, 70)
steps = synth.histories(6, n, 16, 5e-3, synth.default_pert(thr, P), off)
o = Oracle()
want_rows = o.splinify_batch(steps, off, P)
wi, wj, wd, _ = o.all_pairs(want_rows, thr)
stream = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(stream)
hc = scema_b200.HistCluster(0, stream.cuda_stream)
hc.set_histories(steps, off)
sc = ShardedCluster(hc, side_group=dist.new_group(backend="nccl"), bounds=aligned_shard_bounds(n, 1)[1])
for step, mode in enumerate(("overlapped", "overlapped", "plain")):
    if mode == "overlapped":
        ne, counts, offs, full = sc.run_overlapped(n, P, thr)
        assert sc.path == "overlapped", sc.path
        assert sc._last_choice == 1, sc._last_choice     # the second step was optimistic and its sample agreed
    else:
        ne, counts, offs, full = sc.run(n, P, thr, 3)
    a, b, d = hc.get_edges()
    assert np.array_equal(full.cpu().numpy().view(np.uint64), want_rows.view(np.uint64))
    assert ne == len(wi) and np.array_equal(a, wi) and np.array_equal(b, wj) and np.array_equal(d.view(np.uint64), wd.view(np.uint64))
    assert hc.counters()["tc_slices"] == 1
    print("run_overlapped ok", step, mode, ne, flush=True)
hc.close()
dist.destroy_process_group()
"""


@pytest.mark.gpu
def test_run_overlapped_one_rank(tmp_path):
    """ShardedCluster.run_overlapped on a one-rank NCCL group: twice (the second step optimistic), then run(); all three
    give the oracle's edges."""
    r = subprocess.run([sys.executable, "-c", _DRIVER, ROOT, str(tmp_path / "store")], capture_output=True, text=True, timeout=600,
                       cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("run_overlapped ok") == 3, r.stdout
