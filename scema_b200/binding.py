"""ctypes binding of include/scema_hist.h and include/scema_synth.h (one function per entry point)."""
import ctypes as C
import os

import numpy as np

PAIRS_DMMA, PAIRS_FMA, PAIRS_EXACT, PAIRS_TC = 0, 1, 2, 3
T_NAMES = ("resample", "prep", "filter", "exact", "sort")

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


class ScemaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"scema error {code}: {msg}")
        self.code = code


def lib_path():
    # SCEMA_LIB: another build of the same library (A/B measurements of kernel changes on one box)
    return os.environ.get("SCEMA_LIB") or os.path.join(_HERE, "libscema_hist.so")


def lib():
    """Load libscema_hist.so. Fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    L = C.CDLL(path)
    vp, u64, u32, i32, dbl = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_double
    P = C.POINTER
    sig = {
        "scema_create": (i32, [P(vp), i32, vp]),
        "scema_destroy": (None, [vp]),
        "scema_last_error": (C.c_char_p, [vp]),
        "scema_version": (C.c_char_p, []),
        "scema_stream": (i32, [vp, P(vp)]),
        "scema_set_histories": (i32, [vp, vp, i32, vp, vp, u64]),
        "scema_resample": (i32, [vp, u32]),
        "scema_store_reset": (i32, [vp, u64, vp, u32]),
        "scema_store_append": (i32, [vp, vp, i32]),
        "scema_store_info": (i32, [vp, P(u64), P(u32), P(vp)]),
        "scema_store_resample": (i32, [vp, u32]),
        "scema_select_rows": (i32, [vp, vp, u64]),
        "scema_set_spline": (i32, [vp, vp, i32, u64, u32, vp]),
        "scema_get_spline": (i32, [vp, vp]),
        "scema_spline_info": (i32, [vp, P(u64), P(u32), P(vp)]),
        "scema_compare": (i32, [vp, dbl, i32, u32, u32, P(u64)]),
        "scema_compare_stream": (i32, [vp, dbl, i32, u32, u32, u32, vp, vp, P(u64)]),
        "scema_get_edges": (i32, [vp, vp, vp, vp, u64]),
        "scema_edges_device": (i32, [vp, P(vp), P(vp), P(u32), P(u64)]),
        "scema_get_degrees": (i32, [vp, vp]),
        "scema_cluster": (i32, [vp, vp, vp, vp, u64, u32, dbl, i32, P(u64)]),
        "scema_nearest": (i32, [vp, vp, vp]),
        "scema_knn": (i32, [vp, u32, i32, vp, vp]),
        "scema_knn_last_stats": (i32, [vp, vp, vp]),
        "scema_query_compare": (i32, [vp, vp, i32, u64, u32, dbl, i32, P(u64)]),
        "scema_query_get_edges": (i32, [vp, vp, vp, vp, u64]),
        "scema_query_knn": (i32, [vp, vp, i32, u64, u32, u32, i32, vp, vp]),
        "scema_query_last_stats": (i32, [vp, vp, vp, vp]),
        "scema_write_similar_hist": (i32, [vp, C.c_char_p]),
        "scema_reduce_edges": (i32, [vp, u32, vp, P(u64), P(u64)]),
        "scema_reduce_calls": (i32, [vp, vp, u64, u32, vp, P(u64), P(u64)]),
        "scema_reduce_dir": (i32, [C.c_char_p, C.c_char_p, u32, P(u64), P(u64), P(u64)]),
        "scema_last_timings": (i32, [vp, P(C.c_float)]),
        "scema_last_counters": (i32, [vp, P(u64)]),
        "scema_kernel_launches": (u64, [vp]),
        "scema_last_audit": (i32, [vp, vp]),
        "scema_fp64_peak": (i32, [vp, P(dbl)]),
        "scema_k1_tune": (i32, [C.c_int, C.c_int, C.c_int, C.c_int]),
        "scema_tc_debug": (i32, [vp, dbl, u32, vp, u64, vp, vp]),
        "scema_tc_plan": (i32, [u32, u32, u32, vp]),
        "scema_tc_shard_begin": (i32, [vp, dbl, u64, u64, P(vp)]),
        "scema_tc_shard_stats": (i32, [vp, vp, P(vp), P(u64)]),
        "scema_tc_shard_finish": (i32, [vp, vp, u32, u64, i32, P(i32), P(vp), P(u64)]),
        "scema_tc_shard_check": (i32, [vp, P(i32)]),
        "scema_tc_shard_commit": (i32, [vp, vp]),
        "scema_tc_centre": (i32, [vp, vp]),
        "scema_tc_last_plan": (i32, [vp, vp]),
        "scema_tc_choose": (i32, [u64, u32, vp, u64, u64, P(i32), P(i32), P(u64)]),
        "scema_tc_choose_projected": (i32, [u64, u32, vp, u64, u64, P(i32), P(i32), P(u64)]),
        "scema_tc_basis": (i32, [vp, u32, vp, P(dbl)]),
        "scema_tc_last_projection": (i32, [vp, vp]),
        "scema_pipeline_plan": (i32, [u64, vp, u32, P(u32)]),
        "scema_multi_create": (i32, [P(vp), vp, i32]),
        "scema_multi_destroy": (None, [vp]),
        "scema_multi_last_error": (C.c_char_p, [vp]),
        "scema_multi_devices": (i32, [vp]),
        "scema_multi_context": (vp, [vp, i32]),
        "scema_multi_cluster": (i32, [vp, vp, vp, vp, u64, u32, dbl, i32, P(u64)]),
        "scema_multi_compare_rows": (i32, [vp, vp, u64, u32, vp, dbl, i32, P(u64)]),
        "scema_multi_shard_edges": (i32, [vp, vp, vp]),
        "scema_multi_last_ms": (i32, [vp, P(dbl), P(i32)]),
        "scema_ingest_last_error": (C.c_char_p, []),
        "scema_batch_read_dir": (i32, [C.c_char_p, u32, P(vp)]),
        "scema_batch_read_files": (i32, [P(C.c_char_p), vp, u64, u32, P(vp)]),
        "scema_batch_from_lhistory": (i32, [P(C.c_char_p), u64, C.c_char_p, P(vp)]),
        "scema_batch_count": (u64, [vp]),
        "scema_batch_total_steps": (u64, [vp]),
        "scema_batch_steps": (vp, [vp]),
        "scema_batch_offsets": (vp, [vp]),
        "scema_batch_ids": (vp, [vp]),
        "scema_batch_name": (C.c_char_p, [vp, u64]),
        "scema_batch_write_strain_files": (i32, [vp, C.c_char_p]),
        "scema_set_histories_from_batch": (i32, [vp, vp]),
        "scema_batch_free": (None, [vp]),
        "scema_synth_offsets": (i32, [u64, u64, u64, u32, u32, u32, vp]),
        "scema_synth_histories_device": (i32, [u64, u64, u64, u32, dbl, dbl, vp, vp, vp]),
        "scema_synth_rows_device": (i32, [u64, u64, u64, u32, u32, dbl, dbl, vp, vp]),
        "scema_synth_histories_model_device": (i32, [i32, dbl, u64, u64, u64, u32, dbl, dbl, vp, vp, vp]),
        "scema_synth_rows_model_device": (i32, [i32, dbl, u64, u64, u64, u32, u32, dbl, dbl, vp, vp]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args
    _lib = L
    return L


EXPORTED = (
    "scema_create scema_destroy scema_last_error scema_version scema_stream scema_set_histories scema_resample "
    "scema_store_reset scema_store_append scema_store_info scema_store_resample scema_select_rows "
    "scema_set_spline scema_get_spline scema_spline_info scema_compare scema_compare_stream scema_get_edges scema_edges_device "
    "scema_get_degrees scema_cluster scema_nearest scema_knn scema_knn_last_stats "
    "scema_query_compare scema_query_get_edges scema_query_knn scema_query_last_stats scema_write_similar_hist scema_reduce_edges scema_reduce_calls scema_reduce_dir "
    "scema_last_timings scema_last_counters scema_kernel_launches scema_last_audit scema_fp64_peak scema_k1_tune scema_tc_debug scema_tc_plan scema_tc_shard_begin scema_tc_shard_stats scema_tc_shard_finish scema_tc_shard_check scema_tc_shard_commit scema_tc_centre scema_tc_last_plan scema_tc_choose scema_tc_choose_projected scema_tc_basis scema_tc_last_projection scema_pipeline_plan scema_synth_offsets "
    "scema_multi_create scema_multi_destroy scema_multi_last_error scema_multi_devices scema_multi_context scema_multi_cluster "
    "scema_multi_compare_rows scema_multi_shard_edges scema_multi_last_ms "
    "scema_synth_histories_device scema_synth_rows_device scema_synth_histories_model_device scema_synth_rows_model_device scema_ingest_last_error scema_batch_read_dir "
    "scema_batch_read_files scema_batch_from_lhistory scema_batch_count scema_batch_total_steps scema_batch_steps "
    "scema_batch_offsets scema_batch_ids scema_batch_name scema_batch_write_strain_files "
    "scema_set_histories_from_batch scema_batch_free").split()


def _ptr(a):
    """Host numpy array or raw integer (device pointer) -> c_void_p value."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return int(a)


def reduce_dir(input_folder, out_mapping_csv, num_gps):
    """Native coarsegrain_dependency_network.py. -> (iterations, files, neighbours_removed)."""
    it, nf, nr = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    rc = lib().scema_reduce_dir(os.fsencode(input_folder), os.fsencode(out_mapping_csv), num_gps,
                                C.byref(it), C.byref(nf), C.byref(nr))
    if rc:
        raise ScemaError(rc, "reduce_dir failed")
    return int(it.value), int(nf.value), int(nr.value)


class Batch:
    """Host-side ragged batch of strain histories read from files (include/scema_ingest.h)."""

    def __init__(self, handle):
        self._L = lib()
        self._h = handle

    @staticmethod
    def _take(rc, h):
        if rc:
            raise ScemaError(rc, lib().scema_ingest_last_error().decode())
        return Batch(h)

    @classmethod
    def read_dir(cls, strain_directory, n_threads=0):
        h = C.c_void_p(None)
        return cls._take(lib().scema_batch_read_dir(os.fsencode(strain_directory), int(n_threads), C.byref(h)), h)

    @classmethod
    def read_files(cls, paths, ids=None, n_threads=0):
        arr = (C.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint32)
        h = C.c_void_p(None)
        return cls._take(lib().scema_batch_read_files(arr, _ptr(ids_a), len(paths), int(n_threads), C.byref(h)), h)

    @classmethod
    def from_lhistory(cls, csv_paths, column_prefix="strain"):
        arr = (C.c_char_p * len(csv_paths))(*[os.fsencode(p) for p in csv_paths])
        h = C.c_void_p(None)
        return cls._take(lib().scema_batch_from_lhistory(arr, len(csv_paths), column_prefix.encode(), C.byref(h)), h)

    def __len__(self):
        return int(self._L.scema_batch_count(self._h))

    @property
    def offsets(self):
        n = len(self)
        return np.ctypeslib.as_array(C.cast(self._L.scema_batch_offsets(self._h), C.POINTER(C.c_uint64)), (n + 1,)).copy()

    @property
    def ids(self):
        n = len(self)
        if n == 0:
            return np.zeros(0, dtype=np.uint32)
        return np.ctypeslib.as_array(C.cast(self._L.scema_batch_ids(self._h), C.POINTER(C.c_uint32)), (n,)).copy()

    @property
    def steps(self):
        t = int(self._L.scema_batch_total_steps(self._h))
        if t == 0:
            return np.zeros((0, 6))
        return np.ctypeslib.as_array(C.cast(self._L.scema_batch_steps(self._h), C.POINTER(C.c_double)), (t, 6)).copy()

    def name(self, i):
        return self._L.scema_batch_name(self._h, int(i)).decode()

    def write_strain_files(self, out_directory):
        rc = self._L.scema_batch_write_strain_files(self._h, os.fsencode(out_directory))
        if rc:
            raise ScemaError(rc, self._L.scema_ingest_last_error().decode())

    def close(self):
        if getattr(self, "_h", None):
            self._L.scema_batch_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def tc_choose(pairs, k, counts, sample, mem_budget):
    """Host logic of the filter choice (scema_tc_choose); counts = survivors of the sample for (one slice, two slices)
    centred, (one slice, two slices) raw, DMMA and, when a sixth is given, the projected filter (choice 3).
    -> (choice, centred, estimated survivors)."""
    cnt = (C.c_uint64 * len(counts))(*[int(x) for x in counts])
    if len(counts) not in (5, 6):
        raise ValueError("tc_choose: five or six counts")
    fn = lib().scema_tc_choose_projected if len(counts) == 6 else lib().scema_tc_choose
    ch, cen, est = C.c_int(0), C.c_int(0), C.c_uint64(0)
    rc = fn(int(pairs), int(k), cnt, int(sample), int(mem_budget), C.byref(ch), C.byref(cen), C.byref(est))
    if rc:
        raise ScemaError(rc, "tc_choose")
    return int(ch.value), int(cen.value), int(est.value)


def tc_basis(moments):
    """Host logic of the projected filter's basis (scema_tc_basis): second moments [k, k] of the centred sample ->
    (basis [11, k], |B B^T - I|_F), or None when the library would keep the 64-column copies."""
    m = np.ascontiguousarray(moments, dtype=np.float64)
    k = m.shape[0]
    out = np.zeros((11, 60), dtype=np.float64)
    delta = C.c_double(0.0)
    if lib().scema_tc_basis(_ptr(m), int(k), _ptr(out), C.byref(delta)):
        return None
    return out[:, :k].copy(), float(delta.value)


class HistCluster:
    """One context = one GPU + one stream. Methods map 1:1 onto include/scema_hist.h."""

    def __init__(self, device=0, stream=None, _borrowed=None):
        self._L = lib()
        self._keep = []
        if _borrowed is not None:   # a context owned by a MultiCluster
            self._h = C.c_void_p(_borrowed)
            self._owned = False
            return
        self._owned = True
        self._h = C.c_void_p(None)
        rc = self._L.scema_create(C.byref(self._h), int(device), _ptr(stream) if stream else None)
        if rc:
            self._h = None
            raise ScemaError(rc, "scema_create failed (no CUDA device? there is no CPU fallback)")

    def close(self):
        if getattr(self, "_h", None):
            if getattr(self, "_owned", True):
                self._L.scema_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc:
            raise ScemaError(rc, self._L.scema_last_error(self._h).decode())

    def stream_ptr(self):
        """cudaStream_t (int) all work of this context is ordered on."""
        p = C.c_void_p(None)
        self._ck(self._L.scema_stream(self._h, C.byref(p)))
        return int(p.value or 0)

    # ---- ingest ----
    def set_histories(self, steps, offsets, ids=None, device_ptr=None):
        """steps: host ndarray [sumL,6] (or pass device_ptr=int for a device-resident buffer)."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint32)
        if device_ptr is not None:
            self._ck(self._L.scema_set_histories(self._h, int(device_ptr), 1, _ptr(offsets), _ptr(ids_a), n))
        else:
            steps = np.ascontiguousarray(steps, dtype=np.float64)
            self._ck(self._L.scema_set_histories(self._h, _ptr(steps), 0, _ptr(offsets), _ptr(ids_a), n))

    def set_histories_from_batch(self, batch):
        self._ck(self._L.scema_set_histories_from_batch(self._h, batch._h))

    # ---- incremental store ----
    def store_reset(self, n, ids=None, capacity_steps=64):
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint32)
        self._ck(self._L.scema_store_reset(self._h, int(n), _ptr(ids_a), int(capacity_steps)))

    def store_append(self, strain=None, device_ptr=None):
        """strain: host ndarray [n,6] (or device_ptr=int)."""
        if device_ptr is not None:
            self._ck(self._L.scema_store_append(self._h, int(device_ptr), 1))
        else:
            strain = np.ascontiguousarray(strain, dtype=np.float64)
            self._ck(self._L.scema_store_append(self._h, _ptr(strain), 0))

    def store_info(self):
        n, st, p = C.c_uint64(0), C.c_uint32(0), C.c_void_p(None)
        self._ck(self._L.scema_store_info(self._h, C.byref(n), C.byref(st), C.byref(p)))
        return int(n.value), int(st.value), p.value

    def store_resample(self, spline_points):
        self._ck(self._L.scema_store_resample(self._h, int(spline_points)))

    def select_rows(self, rows):
        rows = np.ascontiguousarray(rows, dtype=np.uint32)
        self._ck(self._L.scema_select_rows(self._h, _ptr(rows), len(rows)))

    def resample(self, spline_points):
        self._ck(self._L.scema_resample(self._h, int(spline_points)))

    def set_spline(self, rows=None, ids=None, device_ptr=None, n=None, k=None):
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint32)
        if device_ptr is not None:
            self._ck(self._L.scema_set_spline(self._h, int(device_ptr), 1, int(n), int(k), _ptr(ids_a)))
        else:
            rows = np.ascontiguousarray(rows, dtype=np.float64)
            self._ck(self._L.scema_set_spline(self._h, _ptr(rows), 0, rows.shape[0], rows.shape[1], _ptr(ids_a)))

    def spline_info(self):
        n, k, p = C.c_uint64(0), C.c_uint32(0), C.c_void_p(None)
        self._ck(self._L.scema_spline_info(self._h, C.byref(n), C.byref(k), C.byref(p)))
        return int(n.value), int(k.value), p.value

    def get_spline(self):
        n, k, _ = self.spline_info()
        out = np.empty((n, k), dtype=np.float64)
        self._ck(self._L.scema_get_spline(self._h, _ptr(out)))
        return out

    # ---- compare ----
    def compare(self, threshold, variant=PAIRS_TC, shard=0, n_shards=1):
        ne = C.c_uint64(0)
        self._ck(self._L.scema_compare(self._h, float(threshold), int(variant), int(shard), int(n_shards), C.byref(ne)))
        self.n_edges = int(ne.value)
        return self.n_edges

    def compare_stream(self, threshold, sink, variant=PAIRS_TC, shard=0, n_shards=1, panels_per_chunk=0):
        """Chunked compare; sink(a, b, d) is called with numpy copies of every chunk's sorted edges.
        -> total number of edges."""
        SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_double),
                           C.c_uint64)
        err = []

        def tramp(_user, pa, pb, pd, m):
            try:
                m = int(m)
                sink(np.ctypeslib.as_array(pa, (m,)).copy(), np.ctypeslib.as_array(pb, (m,)).copy(),
                     np.ctypeslib.as_array(pd, (m,)).copy())
                return 0
            except Exception as e:  # noqa: BLE001 - reported after the C call returns
                err.append(e)
                return 1

        cb = SINK(tramp)
        tot = C.c_uint64(0)
        rc = self._L.scema_compare_stream(self._h, float(threshold), int(variant), int(shard), int(n_shards),
                                          int(panels_per_chunk), C.cast(cb, C.c_void_p), None, C.byref(tot))
        if err:
            raise err[0]
        self._ck(rc)
        self.n_edges = 0
        return int(tot.value)

    def get_edges(self, out=None):
        """-> (index_a, index_b, diff). out = (a, b, d): caller-owned arrays of at least n_edges entries (uint32, uint32,
        float64; e.g. views of pinned memory that a caller reuses from call to call) that receive the edges; views
        of their first n_edges entries are returned."""
        m = self.n_edges
        if out is None:
            a = np.empty(m, dtype=np.uint32)
            b = np.empty(m, dtype=np.uint32)
            d = np.empty(m, dtype=np.float64)
        else:
            a, b, d = out
            if min(len(a), len(b), len(d)) < m or a.dtype != np.uint32 or b.dtype != np.uint32 or d.dtype != np.float64:
                raise ValueError("get_edges: out arrays too small or of the wrong type")
        self._ck(self._L.scema_get_edges(self._h, _ptr(a), _ptr(b), _ptr(d), m))
        return a[:m], b[:m], d[:m]

    def edges_device(self):
        keys, diff, sh, ne = C.c_void_p(None), C.c_void_p(None), C.c_uint32(0), C.c_uint64(0)
        self._ck(self._L.scema_edges_device(self._h, C.byref(keys), C.byref(diff), C.byref(sh), C.byref(ne)))
        return keys.value, diff.value, int(sh.value), int(ne.value)

    def get_degrees(self, n):
        out = np.empty(n, dtype=np.uint32)
        self._ck(self._L.scema_get_degrees(self._h, _ptr(out)))
        return out

    def nearest(self):
        """Legacy nearest neighbour of every history: (ids [n] uint32, diffs [n] float64)."""
        n, _, _ = self.spline_info()
        ids = np.empty(n, dtype=np.uint32)
        d = np.empty(n, dtype=np.float64)
        self._ck(self._L.scema_nearest(self._h, _ptr(ids), _ptr(d)))
        return ids, d

    def knn(self, k, variant=PAIRS_TC):
        """Exact k nearest neighbours of every history: (index [n, k] uint32, diff [n, k] float64), slots in order of
        (diff, ID, index); empty slots are (0xffffffff, inf)."""
        n, _, _ = self.spline_info()
        kk = max(int(k), 0)
        index = np.empty((n, kk), dtype=np.uint32)
        diff = np.empty((n, kk), dtype=np.float64)
        self._ck(self._L.scema_knn(self._h, int(k) & 0xffffffff, int(variant), _ptr(index), _ptr(diff)))
        return index, diff

    def knn_last_stats(self):
        """What the last knn did: filter rounds, rows finished per stage, exact pairs, survivors, edges, last filter
        variant and the radius of every round."""
        c = (C.c_uint64 * 8)()
        r = (C.c_double * 8)()
        self._ck(self._L.scema_knn_last_stats(self._h, c, r))
        return {"rounds": int(c[0]), "rows_round1": int(c[1]), "rows_later_rounds": int(c[2]), "rows_exact": int(c[3]),
                "exact_pairs": int(c[4]), "survivors": int(c[5]), "edges": int(c[6]), "variant": int(c[7]),
                "radii": [float(x) for x in r][:int(c[0])]}

    def _query_rows(self, rows, device_ptr, m, k_cols):
        """-> (pointer, on_device, m, k_cols, keep-alive) of the query rows: a host array [m, k_cols], or device_ptr with m
        and k_cols (k_cols defaults to the matrix's)."""
        if device_ptr is not None:
            if m is None:
                raise ValueError("query rows on the device: pass their number as m")
            if k_cols is None:
                k_cols = self.spline_info()[1]
            return int(device_ptr), 1, int(m), int(k_cols), None
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        if rows.ndim != 2:
            raise ValueError("query rows: a 2-d array [m, k]")
        return _ptr(rows) if rows.size else None, 0, rows.shape[0], rows.shape[1], rows

    def query_compare(self, rows, threshold, variant=PAIRS_TC, device_ptr=None, m=None, k_cols=None):
        """Every (query j, history i) with compare_L2_norm < threshold, sorted by (j, i): (query_index, row_index, diff).
        rows: host array [m, k]; or device_ptr=int with m (and k_cols) for device-resident rows."""
        p, dev, m, k_cols, keep = self._query_rows(rows, device_ptr, m, k_cols)
        ne = C.c_uint64(0)
        self._ck(self._L.scema_query_compare(self._h, p, dev, m, k_cols, float(threshold), int(variant), C.byref(ne)))
        del keep
        return self.query_edges(int(ne.value))

    def query_edges(self, count):
        """The first `count` cross edges of the last query_compare."""
        j = np.empty(count, dtype=np.uint32)
        i = np.empty(count, dtype=np.uint32)
        d = np.empty(count, dtype=np.float64)
        self._ck(self._L.scema_query_get_edges(self._h, _ptr(j), _ptr(i), _ptr(d), count))
        return j, i, d

    def query_knn(self, rows, k, variant=PAIRS_TC, device_ptr=None, m=None, k_cols=None):
        """The k nearest histories of every query row: (index [m, k] uint32, diff [m, k] float64), slots in order of
        (diff, ID, index); empty slots are (0xffffffff, inf)."""
        p, dev, m, k_cols, keep = self._query_rows(rows, device_ptr, m, k_cols)
        kk = max(int(k), 0)
        index = np.empty((m, kk), dtype=np.uint32)
        diff = np.empty((m, kk), dtype=np.float64)
        self._ck(self._L.scema_query_knn(self._h, p, dev, m, k_cols, int(k) & 0xffffffff, int(variant), _ptr(index), _ptr(diff)))
        del keep
        return index, diff

    def query_last_stats(self):
        """What the last query_compare / query_knn did: rounds, queries finished per stage, exact pairs, survivors, edges of
        the prefix compares, last filter variant, filter pairs, cross edges, compare passes, the radius of every round and the phase
        times (ms)."""
        c = (C.c_uint64 * 11)()
        r = (C.c_double * 8)()
        t = (C.c_float * 8)()
        self._ck(self._L.scema_query_last_stats(self._h, c, r, t))
        names = ("copy", "prep", "filter", "exact", "sort", "select", "topk")
        return {"rounds": int(c[0]), "rows_round1": int(c[1]), "rows_later_rounds": int(c[2]), "rows_exact": int(c[3]),
                "exact_pairs": int(c[4]), "survivors": int(c[5]), "edges": int(c[6]), "variant": int(c[7]),
                "filter_pairs": int(c[8]), "cross_edges": int(c[9]), "passes": int(c[10]), "radii": [float(x) for x in r][:max(int(c[0]), 1)],
                "ms": {names[w]: float(t[w]) for w in range(len(names))}}

    def cluster(self, steps, offsets, ids, spline_points, threshold, variant=PAIRS_TC):
        steps = np.ascontiguousarray(steps, dtype=np.float64)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint32)
        ne = C.c_uint64(0)
        self._ck(self._L.scema_cluster(self._h, _ptr(steps), _ptr(offsets), _ptr(ids_a), len(offsets) - 1,
                                       int(spline_points), float(threshold), int(variant), C.byref(ne)))
        self.n_edges = int(ne.value)
        return self.n_edges

    # ---- outputs ----
    def write_similar_hist(self, pattern):
        self._ck(self._L.scema_write_similar_hist(self._h, os.fsencode(pattern)))

    def reduce_edges(self, num_gps):
        mapping = np.empty(num_gps, dtype=np.uint32)
        it, nr = C.c_uint64(0), C.c_uint64(0)
        self._ck(self._L.scema_reduce_edges(self._h, int(num_gps), _ptr(mapping), C.byref(it), C.byref(nr)))
        return mapping, int(it.value), int(nr.value)

    # ---- instrumentation ----
    def timings(self):
        ms = (C.c_float * 8)()
        self._ck(self._L.scema_last_timings(self._h, ms))
        return {T_NAMES[i]: float(ms[i]) for i in range(len(T_NAMES))}

    def counters(self):
        c = (C.c_uint64 * 8)()
        self._ck(self._L.scema_last_counters(self._h, c))
        return {"pairs": int(c[0]), "survivors": int(c[1]), "edges": int(c[2]), "passes": int(c[3]), "tiles": int(c[4]),
                "tc_slices": int(c[5]), "pipeline_ranges": int(c[6]), "band_tiles": int(c[7])}

    def last_audit(self):
        """(sampled pairs that were reference edges, of those missing from the list) of the last SCEMA_AUDIT run."""
        out = (C.c_uint64 * 2)()
        self._ck(self._L.scema_last_audit(self._h, out))
        return int(out[0]), int(out[1])

    def kernel_launches(self):
        return int(self._L.scema_kernel_launches(self._h))

    def tc_debug(self, threshold, n, slices=2):
        """Accumulators and operand copies of the tcgen05 filter over the whole pair matrix (tests only); slices = 3:
        the projected filter (32-byte operand rows). Returns (acc [n_pad, n_pad] float32, A operand bytes, B operand bytes)."""
        n_pad = (n + 255) // 256 * 256
        acc = np.empty((n_pad, n_pad), dtype=np.float32)
        row_bytes = 32 if slices == 3 else 256
        ha = np.empty(n_pad * row_bytes, dtype=np.uint8)
        hb = np.empty(n_pad * row_bytes, dtype=np.uint8)
        self._ck(self._L.scema_tc_debug(self._h, float(threshold), int(slices), _ptr(acc), n_pad, _ptr(ha), _ptr(hb)))
        return acc, ha, hb

    # ---- sharded prepare of the tcgen05 filter (include/scema_hist.h) ----
    def tc_shard_begin(self, threshold, row0, row1):
        """-> device pointer of the K-double centre candidate of the own rows."""
        p = C.c_void_p(None)
        self._ck(self._L.scema_tc_shard_begin(self._h, float(threshold), int(row0), int(row1), C.byref(p)))
        return int(p.value)

    def tc_shard_stats(self, centre_ptr):
        """-> (device pointer of the statistics packet, its length in 8-byte words)."""
        p, w = C.c_void_p(None), C.c_uint64(0)
        self._ck(self._L.scema_tc_shard_stats(self._h, int(centre_ptr), C.byref(p), C.byref(w)))
        return int(p.value), int(w.value)

    def tc_shard_finish(self, packets_ptr, n_shards, pairs, optimistic=False):
        """-> (choice, device pointer of the operand image, bytes per row)."""
        ch, p, b = C.c_int(0), C.c_void_p(None), C.c_uint64(0)
        self._ck(self._L.scema_tc_shard_finish(self._h, int(packets_ptr), int(n_shards), int(pairs), int(bool(optimistic)), C.byref(ch),
                                               C.byref(p), C.byref(b)))
        return int(ch.value), int(p.value or 0), int(b.value)

    def tc_shard_check(self):
        """What the sample of the last optimistic tc_shard_finish really said (1 = the assumption held)."""
        ch = C.c_int(0)
        self._ck(self._L.scema_tc_shard_check(self._h, C.byref(ch)))
        return int(ch.value)

    def tc_shard_commit(self, rows_ready_event=None):
        self._ck(self._L.scema_tc_shard_commit(self._h, int(rows_ready_event) if rows_ready_event else None))

    def tc_centre(self):
        """Column means the tcgen05 filter subtracted from its operand copies."""
        _, k, _ = self.spline_info()
        out = np.empty(k, dtype=np.float64)
        self._ck(self._L.scema_tc_centre(self._h, _ptr(out)))
        return out

    def tc_last_plan(self):
        """-> dict: pairs of the last survivor-density sample that would survive 1 slice / 2 slices / DMMA / the projected
        filter, sample size, and whether the projected filter was taken."""
        p = (C.c_uint64 * 6)()
        self._ck(self._L.scema_tc_last_plan(self._h, p))
        q = (C.c_uint64 * 2)()
        self._ck(self._L.scema_tc_last_projection(self._h, q))
        return {"one_slice": int(p[0]), "two_slices": int(p[1]), "one_slice_raw": int(p[2]), "two_slices_raw": int(p[3]),
                "dmma": int(p[4]), "sample": int(p[5]), "projected": int(q[0]), "projected_chosen": bool(q[1])}

    def k1_tune(self, kernel=-1, wps_ragged=-1, wps_store=-1, flags=-1):
        """Measurement hook of K1 (process-wide): kernel 1 = two chains per lane / 0 = one, resident warps per SM, memory flags."""
        self._ck(self._L.scema_k1_tune(kernel, wps_ragged, wps_store, flags))

    def fp64_peak(self):
        out = (C.c_double * 2)()
        self._ck(self._L.scema_fp64_peak(self._h, out))
        return {"dfma_tflops": float(out[0]), "dmma_tflops": float(out[1])}


class MultiCluster:
    """Several GPUs of one box from one process (scema_multi_*): one context and host thread per GPU, NCCL inside the
    library. After cluster() / compare_rows() the result is served by .first (a HistCluster view of the first GPU's
    context): get_edges, write_similar_hist, reduce_edges ..."""

    def __init__(self, devices):
        self._L = lib()
        self._h = C.c_void_p(None)
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        rc = self._L.scema_multi_create(C.byref(self._h), devs, len(devices))
        if rc:
            self._h = None
            raise ScemaError(rc, "scema_multi_create failed (devices missing, listed twice, or NCCL unavailable)")
        self.n_devices = len(devices)
        self.contexts = [HistCluster(_borrowed=self._L.scema_multi_context(self._h, r)) for r in range(self.n_devices)]
        self.first = self.contexts[0]

    def close(self):
        if getattr(self, "_h", None):
            for c in self.contexts:
                c._h = None
            self._L.scema_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc:
            raise ScemaError(rc, self._L.scema_multi_last_error(self._h).decode())

    def cluster(self, steps, offsets, ids, spline_points, threshold, variant=PAIRS_TC):
        steps = np.ascontiguousarray(steps, dtype=np.float64)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint32)
        ne = C.c_uint64(0)
        self._ck(self._L.scema_multi_cluster(self._h, _ptr(steps), _ptr(offsets), _ptr(ids_a), len(offsets) - 1, int(spline_points),
                                             float(threshold), int(variant), C.byref(ne)))
        self.first.n_edges = int(ne.value)
        return int(ne.value)

    def compare_rows(self, rows, threshold, variant=PAIRS_TC, ids=None):
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint32)
        ne = C.c_uint64(0)
        self._ck(self._L.scema_multi_compare_rows(self._h, _ptr(rows), rows.shape[0], rows.shape[1], _ptr(ids_a), float(threshold),
                                                  int(variant), C.byref(ne)))
        self.first.n_edges = int(ne.value)
        return int(ne.value)

    def shard_edges(self):
        cnt = np.zeros(self.n_devices, dtype=np.uint64)
        off = np.zeros(self.n_devices, dtype=np.uint64)
        self._ck(self._L.scema_multi_shard_edges(self._h, _ptr(cnt), _ptr(off)))
        return cnt, off

    def last_ms(self):
        ms = (C.c_double * 4)()
        v = C.c_int(0)
        self._ck(self._L.scema_multi_last_ms(self._h, ms, C.byref(v)))
        return {"ingest_resample": ms[0], "allgather": ms[1], "compare": ms[2], "gather_sort": ms[3], "variant_used": int(v.value)}
