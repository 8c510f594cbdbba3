"""Multi-GPU driver: one process per GPU, torch.distributed (NCCL over NVLink/NVSwitch) as plumbing.

Replaces the MPI ring of compare_histories_with_all_ranks (reference headers/strain2spline.h:567-599):
  1. every rank resamples its contiguous share of the histories (K1, independent units);
  2. ONE all-gather of the resampled row blocks gives every GPU the full N x K matrix (the only
     data-path exchange; 480 MB at 1M x 60);
  3. every rank filters/recomputes its share of the pair-matrix tile groups (K2+K3, no communication);
  4. one all-gather of the 8-byte edge counts gives every rank the exclusive offsets of its edge range.
The same class runs with the gloo backend on CPU tensors for the host-logic tests (sharding
arithmetic, gather of uneven shares); the kernels themselves only ever run on a GPU.
"""
import numpy as np
import torch
import torch.distributed as dist


class CudaView:
    """Zero-copy view of library-owned device memory for torch.as_tensor."""

    def __init__(self, ptr, shape, typestr="<f8"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2}


def shard_bounds(n, world):
    """Contiguous, balanced split of n histories over `world` ranks -> list of (begin, end)."""
    base, rem = divmod(n, world)
    out, b = [], 0
    for r in range(world):
        e = b + base + (1 if r < rem else 0)
        out.append((b, e))
        b = e
    return out


def aligned_shard_bounds(n, world, align=2048):
    """Equal shares of a multiple of `align` rows (the last ranks take what is left): rank r owns
    [r * per, min(n, (r + 1) * per)); ranks past the end get the empty share (n, n). Equal, aligned shares make every
    exchange of the sharded path one all-gather of equal slots (row blocks, fp16 operand images: image_exchange).
    -> (per, list of (begin, end))."""
    per = (n + world - 1) // world
    per = (per + align - 1) // align * align
    return per, [(min(n, r * per), min(n, (r + 1) * per)) for r in range(world)]


def image_exchange(n, world):
    """Shares and image rows of the overlapped tcgen05 path (scema_tc_shard_*, include/scema_hist.h). Rank r owns the
    rows bounds[r] of aligned_shard_bounds and builds the image rows own[r]: its share, and for the share that ends at n
    also the padding rows up to n_pad (n rounded up to 256); an empty share builds nothing. The all-gather moves `per`
    rows per rank (rank r's slot starts at row r * per). The library's image holds n_pad rows only, so when world * per
    exceeds n_pad (staged) the gather goes through a staging buffer. -> (per, bounds, n_pad, own, staged)"""
    per, bounds = aligned_shard_bounds(n, world)
    n_pad = (n + 255) // 256 * 256
    own = [(b, n_pad if e == n else e) if e > b else (b, b) for b, e in bounds]
    return per, bounds, n_pad, own, world * per > n_pad


def gather_images(img, n, world, rank, bpr, group=None, stage=None):
    """All-gather of the ranks' fp16 operand images into img (a byte tensor of exactly the n_pad * bpr bytes that
    scema_tc_shard_finish promises). In place when the equal slots fill the image exactly; otherwise every rank puts
    its rows into its slot of `stage` (world * per * bpr bytes, allocated when None or of another size), the slots are
    gathered there and the first n_pad rows copied into the image. -> the staging buffer (None when in place)."""
    per, _, n_pad, own, staged = image_exchange(n, world)
    if img.numel() != n_pad * bpr:
        raise ValueError(f"gather_images: image of {img.numel()} bytes, expected {n_pad} rows of {bpr}")
    slot = per * bpr
    if not staged:
        dist.all_gather_into_tensor(img, img[rank * slot:(rank + 1) * slot], group=group)
        return None
    if stage is None or stage.numel() != world * slot:
        stage = torch.empty(world * slot, dtype=torch.uint8, device=img.device)
    b, e = own[rank]
    mine = stage[rank * slot:(rank + 1) * slot]
    mine[:(e - b) * bpr].copy_(img[b * bpr:e * bpr])
    dist.all_gather_into_tensor(stage, mine, group=group)
    img.copy_(stage[:n_pad * bpr])
    return stage


def gather_rows(local_rows, n, world, group=None, bounds=None):
    """All-gather row blocks of possibly uneven height into the full [n, K] matrix (bounds: the ranks' row ranges,
    default shard_bounds(n, world))."""
    K = local_rows.shape[1]
    bounds = bounds or shard_bounds(n, world)
    h_max = max(e - b for b, e in bounds)
    if all(e - b == h_max for b, e in bounds):
        full = torch.empty((n, K), dtype=local_rows.dtype, device=local_rows.device)
        dist.all_gather_into_tensor(full, local_rows.contiguous(), group=group)
        return full
    pad = torch.zeros((h_max, K), dtype=local_rows.dtype, device=local_rows.device)
    pad[: local_rows.shape[0]] = local_rows
    buf = torch.empty((world * h_max, K), dtype=local_rows.dtype, device=local_rows.device)
    dist.all_gather_into_tensor(buf, pad, group=group)
    return torch.cat([buf[r * h_max: r * h_max + (e - b)] for r, (b, e) in enumerate(bounds)], dim=0)


def gather_counts(local_count, device, group=None, flag=0):
    """All-gather of the per-rank (edge count, flag) pairs -> (counts list, exclusive offsets list, max flag)."""
    world = dist.get_world_size(group)
    mine = torch.tensor([int(local_count), int(flag)], dtype=torch.int64, device=device)
    allc = torch.empty(2 * world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(allc, mine, group=group)
    both = allc.cpu().view(world, 2)
    counts = both[:, 0].tolist()
    offs = np.concatenate([[0], np.cumsum(counts)[:-1]]).tolist()
    return counts, offs, int(both[:, 1].max())


def gather_edges(a, b, d, n, counts, device, group=None):
    """All ranks' edge lists on every rank: (a, b, d) numpy arrays of this rank (counts[rank] entries) -> the union
    sorted by (a, b) as numpy arrays. Keys a * n + b travel as int64, distances as their bit patterns."""
    world = dist.get_world_size(group)
    m = max(max(counts), 1)
    mine = len(a)
    buf = torch.zeros((2, m), dtype=torch.int64)
    if mine:
        buf[0, :mine] = torch.from_numpy(a.astype(np.int64) * int(n) + b.astype(np.int64))
        buf[1, :mine] = torch.from_numpy(np.ascontiguousarray(d, dtype=np.float64).view(np.int64).copy())
    buf = buf.to(device).reshape(-1)
    allb = torch.empty(world * 2 * m, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(allb, buf, group=group)
    allb = allb.cpu().numpy().reshape(world, 2, m)
    keys = np.concatenate([allb[r, 0, :counts[r]] for r in range(world)])
    bits = np.concatenate([allb[r, 1, :counts[r]] for r in range(world)])
    order = np.argsort(keys, kind="stable")
    keys, bits = keys[order], bits[order]
    return (keys // int(n)).astype(np.uint32), (keys % int(n)).astype(np.uint32), bits.view(np.float64)


class ShardedCluster:
    """Tile-sharded all-pairs over the ranks of a process group (rank == GPU)."""

    def __init__(self, hc, group=None, side_group=None, bounds=None):
        """side_group: a second NCCL group over the same ranks (dist.new_group): the all-gather of the FP64 rows then
        runs on its own stream and overlaps the tcgen05 filter, which only needs the gathered fp16 operand images
        (run_overlapped). Without it run() is the plain sequence."""
        self.hc = hc
        self.group = group
        self.side_group = side_group
        self.bounds = bounds    # row ranges of the ranks for run() (default: shard_bounds); run_overlapped needs aligned_shard_bounds
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self._full = None
        self._side_stream = None
        self._main = None
        self._packets = None
        self._stage = None
        self._views = {}
        self._peers = None
        self._flag = None
        self._last_choice = None
        self.path = "plain"

    def stream(self):
        """The context's CUDA stream as a torch stream: the collectives and every torch op of run()
        are issued on it, so they are ordered with the library's kernels (the library may run on
        its own non-blocking stream, which does not synchronise with torch's default stream)."""
        ptr = self.hc.stream_ptr()
        if ptr == 0:
            return torch.cuda.default_stream()
        return torch.cuda.ExternalStream(ptr)

    def run(self, n, spline_points, threshold, variant=3, sink=None):
        """The local share of the histories must already be set on self.hc (set_histories).
        sink: callable(a, b, d) -> the shard's edges are streamed chunk by chunk
        (scema_compare_stream) instead of being kept on the device.
        -> (local_edge_count, counts, offsets, full_rows tensor)."""
        hc = self.hc
        with torch.cuda.stream(self.stream()):
            hc.resample(spline_points)
            n_local, K, ptr = hc.spline_info()
            local = torch.as_tensor(CudaView(ptr, (n_local, K)), device="cuda")
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            full = gather_rows(local, n, self.world, self.group, self.bounds)
            ev1.record()
            self.gather_events = (ev0, ev1)  # ev0.elapsed_time(ev1) after a synchronize = the all-gather alone
            hc.set_spline(device_ptr=full.data_ptr(), n=n, k=K)
            ne, counts, offs = self.compare_all_ranks(threshold, variant, sink, full.device)
        return ne, counts, offs, full

    def run_overlapped(self, n, spline_points, threshold, sink=None):
        """The tcgen05 path with the exchanges taken off the critical path (scema_tc_shard_*, include/scema_hist.h).
        Shares: aligned_shard_bounds(n, world) — set_histories must have installed exactly that share. Every rank
        resamples its rows into its slot of the full matrix; the all-gather of the FP64 rows (8 K bytes per row) goes to
        a side stream; meanwhile the ranks agree on centre and scale (two tiny all-gathers), build the fp16 image of their
        OWN rows and all-gather the images (128 bytes per row): the filter starts as soon as those are there, and only the
        exact recompute waits for the FP64 rows. Falls back to the plain sequence when the survivor sample prefers
        another filter. -> (local_edge_count, counts, offsets, full_rows tensor)."""
        hc, G = self.hc, self.world
        per, bounds, n_pad, _, _ = image_exchange(n, G)
        b, e = bounds[self.rank]
        if self._main is None:
            self._main = self.stream()
            self._side_stream = torch.cuda.Stream()
            self._events = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(), torch.cuda.Event()]
        main = self._main
        with torch.cuda.stream(main):
            hc.resample(spline_points)
            n_local, K, ptr = hc.spline_info()
            assert n_local == e - b, "set_histories must hold the rows of aligned_shard_bounds"
            if self._full is None or self._full.shape != (G * per, K):
                self._full = torch.empty((G * per, K), dtype=torch.float64, device="cuda")
                self._cents = torch.empty((G, K), dtype=torch.float64, device="cuda")
                self._views = {}
                self._peers = self._map_peers(self._full)
            full = self._full
            if n_local:
                full[b:e].copy_(self._view(ptr, (n_local, K), "<f8"))
            ev0, ev1, k1_done, rows_ready = self._events
            k1_done.record(main)
            hc.set_spline(device_ptr=full.data_ptr(), n=n, k=K)
            # FP64 rows on the side stream. An NCCL all-gather is an SM kernel and competes with the persistent filter
            # (one CTA per SM, static schedule) for SMs; COPY ENGINES do not: every rank maps its peers' buffers (CUDA IPC,
            # exchanged once) and PULLS their row blocks with peer-to-peer copies over NVLink, after a one-element
            # all-reduce on the side stream has established that every rank's K1 is done. (SCEMA_SHARD_PULL=0: NCCL.)
            with torch.cuda.stream(self._side_stream):
                self._side_stream.wait_event(k1_done)
                ev0.record()
                if self._peers is not None:
                    dist.all_reduce(self._flag, group=self.side_group)
                    for step in range(1, G):
                        q = (self.rank + step) % G
                        qb, qe = bounds[q]
                        if qe > qb:
                            full[qb:qe].copy_(self._peers[q][qb:qe], non_blocking=True)
                else:
                    dist.all_gather_into_tensor(full, full[self.rank * per:(self.rank + 1) * per], group=self.side_group)
                ev1.record()
                self.gather_events = (ev0, ev1)
                rows_ready.record()
            # centre: every rank's candidate, rank 0's is taken
            c_ptr = hc.tc_shard_begin(threshold, b, e)
            dist.all_gather_into_tensor(self._cents, self._view(c_ptr, (K,), "<f8"), group=self.group)
            p_ptr, words = hc.tc_shard_stats(self._cents[0].data_ptr())
            if self._packets is None or self._packets.shape != (G, words):
                self._packets = torch.empty((G, words), dtype=torch.int64, device="cuda")
            dist.all_gather_into_tensor(self._packets, self._view(p_ptr, (words,), "<i8"), group=self.group)
            # after a step whose sample said "one slice, centred copies" the next one does not wait for its own sample
            optimistic = self._last_choice == 1
            choice, img_ptr, bpr = hc.tc_shard_finish(self._packets.data_ptr(), G, n * (n - 1) // 2 // G, optimistic)
            if choice == 1:
                img = self._view(img_ptr, (n_pad * bpr,), "|u1")
                self._stage = gather_images(img, n, G, self.rank, bpr, self.group, self._stage)
                hc.tc_shard_commit(rows_ready.cuda_event)
                self.path = "overlapped"
            else:
                main.wait_event(rows_ready)   # another filter: it needs all rows first
                self.path = "plain (sample chose %d)" % choice
            ne, counts, offs = self.compare_all_ranks(threshold, 3, sink, full.device)
            if choice == 1 and optimistic:
                # what the sample really said; the edge list of this step is correct either way (every survivor is
                # recomputed exactly, an overflowing queue is handled inside the compare) — a different answer only means
                # the NEXT step waits for its sample again and takes the filter it names
                self._last_choice = hc.tc_shard_check()
            else:
                self._last_choice = choice
        return ne, counts, offs, full[:n]

    def _map_peers(self, full):
        """CUDA IPC: every rank's full-size row buffer mapped into every other rank (once per buffer). None when the
        environment asks for the NCCL all-gather or the mapping fails (then the all-gather is used)."""
        import os
        if os.environ.get("SCEMA_SHARD_PULL", "1") == "0":
            return None
        try:
            from torch.multiprocessing.reductions import reduce_tensor
            fn, args = reduce_tensor(full)
            handles = [None] * self.world
            dist.all_gather_object(handles, (fn, args), group=self.group)
            peers = [None if q == self.rank else handles[q][0](*handles[q][1]) for q in range(self.world)]
            self._flag = torch.zeros(1, dtype=torch.int32, device="cuda")
            ok = torch.ones(1, dtype=torch.int32, device="cuda")
        except Exception:  # noqa: BLE001 - no IPC (e.g. a container without it): every rank must take the same decision
            peers, ok = None, torch.zeros(1, dtype=torch.int32, device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
        return peers if int(ok.item()) == 1 else None

    def _view(self, ptr, shape, typestr):
        """Cached zero-copy tensor over library-owned device memory (the library keeps these buffers between steps)."""
        key = (int(ptr), tuple(shape), typestr)
        t = self._views.get(key)
        if t is None:
            t = torch.as_tensor(CudaView(ptr, shape, typestr=typestr), device="cuda")
            self._views[key] = t
        return t

    def compare_all_ranks(self, threshold, variant, sink, device):
        """This rank's share of the pair matrix, then ONE all-gather of (edge count, flag) per rank. The filters split
        the matrix between the shards differently, so a shard whose survivors are too dense for its queue does not
        change filter by itself (SCEMA_ERR_DENSE): it raises the flag and ALL ranks repeat with the next filter —
        tcgen05 -> DMMA -> filter-free kernel. -> (local edge count, counts, offsets)."""
        from .binding import ScemaError, PAIRS_DMMA, PAIRS_EXACT, PAIRS_TC, PAIRS_FMA
        ERR_DENSE = 7
        hc = self.hc
        chain = {PAIRS_TC: PAIRS_DMMA, PAIRS_DMMA: PAIRS_EXACT, PAIRS_FMA: PAIRS_EXACT}
        self.variant_used = variant
        while True:
            dense, ne = 0, 0
            try:
                if sink is not None:
                    ne = hc.compare_stream(threshold, sink, self.variant_used, shard=self.rank, n_shards=self.world)
                else:
                    ne = hc.compare(threshold, self.variant_used, shard=self.rank, n_shards=self.world)
            except ScemaError as e:
                if e.code != ERR_DENSE or self.variant_used not in chain:
                    raise
                dense = 1
            counts, offs, any_dense = gather_counts(ne, device, self.group, flag=dense)
            if not any_dense:
                return ne, counts, offs
            if sink is not None:
                raise ScemaError(ERR_DENSE, "a streamed shard ran out of queue after chunks had been delivered; rerun with variant DMMA")
            self.variant_used = chain[self.variant_used]
