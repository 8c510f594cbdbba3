// C ABI of libscema_hist.so (include/scema_hist.h). Thin host glue: context, ingest, result access.
#include "common.cuh"
#include <new>
#include <algorithm>

using namespace scema;

extern "C" {

const char *scema_version(void) { return "scema-b200-histcluster 0.1 (sm_100a)"; }

int scema_create(scema_ctx **out, int device, void *stream)
{
    if (!out) return SCEMA_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return SCEMA_ERR_CUDA;  // no CPU fallback by design
    }
    scema_ctx *c = new (std::nothrow) scema_ctx();
    if (!c) return SCEMA_ERR_NOMEM;
    c->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete c; return SCEMA_ERR_CUDA; }
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, device) != cudaSuccess) { delete c; return SCEMA_ERR_CUDA; }
    c->sm_count = p.multiProcessorCount;
    c->smem_optin = p.sharedMemPerBlockOptin;
    {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); free_b = p.totalGlobalMem / 2; }
        c->mem_budget = free_b / 2;
    }
    if (stream) {
        c->stream = (cudaStream_t)stream;
    } else {
        if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return SCEMA_ERR_CUDA; }
        c->own_stream = true;
    }
    for (int i = 0; i < 2 * SCEMA_T_COUNT; i++)
        if (cudaEventCreate(&c->ev[i]) != cudaSuccess) { delete c; return SCEMA_ERR_CUDA; }
    *out = c;
    return SCEMA_OK;
}

void scema_destroy(scema_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    c->steps_own.release(); c->d_offsets.release(); c->d_tables.release(); c->d_table_index.release();
    c->zscratch.release(); c->d_order.release(); c->d_chunks.release(); c->d_chunk_counters.release(); c->spline_own.release(); c->spline_sel[0].release(); c->spline_sel[1].release(); c->d_select.release(); c->d_store.release(); c->d_filter.release(); c->d_halfnorm.release();
    c->d_blockmax.release(); c->d_panel_start.release(); c->d_cand.release(); c->d_counters.release();
    for (int b = 0; b < 2; b++) { c->d_edge_key[b].release(); c->d_edge_val[b].release(); }
    c->d_sort_tmp.release();
    c->d_tc_a.release(); c->d_tc_b.release(); c->d_tc_nrm.release(); c->d_tc_misc.release(); c->d_tc_centre.release();
    c->d_tc_perm.release(); c->d_tc_iota.release(); c->d_tc_snrm.release(); c->d_tc_band.release();
    c->d_tc_basis.release(); c->d_tc_cov.release();
    if (c->h_counters) cudaFreeHost(c->h_counters);
    if (c->h_plan) cudaFreeHost(c->h_plan);
    if (c->h_tc_cov) cudaFreeHost(c->h_tc_cov);
    for (int k = 0; k < 2; k++) {
        if (c->h_stage_key[k]) cudaFreeHost(c->h_stage_key[k]);
        if (c->h_stage_val[k]) cudaFreeHost(c->h_stage_val[k]);
        if (c->stage_ev[k]) cudaEventDestroy(c->stage_ev[k]);
    }
    for (int i = 0; i < 2 * SCEMA_T_COUNT; i++) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    for (cudaEvent_t e : c->copy_events) cudaEventDestroy(e);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->knn_child) scema_destroy(c->knn_child);
    for (scema::DevBuf &b : c->knn_buf) b.release();
    if (c->query_child) scema_destroy(c->query_child);
    c->query_j.release(); c->query_i.release(); c->query_d.release();
    for (cudaEvent_t e : c->query_ev) if (e) cudaEventDestroy(e);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char *scema_last_error(const scema_ctx *c) { return c ? c->err.c_str() : "null context"; }

int scema_stream(scema_ctx *c, void **stream)
{
    if (!c || !stream) return SCEMA_ERR_INVALID;
    *stream = (void *)c->stream;
    return SCEMA_OK;
}

static int enter(scema_ctx *c)
{
    if (!c) return SCEMA_ERR_INVALID;
    c->err.clear();
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, SCEMA_ERR_CUDA, "cudaSetDevice failed");
    return SCEMA_OK;
}

static void set_ids(std::vector<uint32_t> &dst, const uint32_t *ids, uint64_t n)
{
    dst.resize(n);
    if (ids) std::copy(ids, ids + n, dst.begin());
    else for (uint64_t i = 0; i < n; i++) dst[i] = (uint32_t)i;
}

// steps_mode: 0 = copy the host steps now, 1 = borrow the device pointer, 2 = only reserve the device buffer
// (the caller copies the steps itself, range by range: cluster_pipelined)
static int set_histories_impl(scema_ctx *c, const double *steps, int steps_mode, const uint64_t *offsets,
                              const uint32_t *ids, uint64_t n)
{
    const int steps_on_device = steps_mode == 1;
    int rc = enter(c);
    if (rc) return rc;
    if (n && (!offsets || !steps)) return fail(c, SCEMA_ERR_INVALID, "set_histories: null pointer");
    if (n >= (1ull << 32)) return fail(c, SCEMA_ERR_INVALID, "set_histories: more than 2^32-1 histories");
    c->have_histories = false;
    c->have_spline = false;  // as add_current_strain: up_to_date = false (strain2spline.h:77)
    c->have_edges = false;
    c->hn = n;
    if (offsets) c->h_offsets.assign(offsets, offsets + n + 1);
    else c->h_offsets.assign(1, 0);
    uint32_t mx = 0, mn = 0xffffffffu;
    for (uint64_t i = 0; i < n; i++) {
        if (offsets[i + 1] < offsets[i]) return fail(c, SCEMA_ERR_INVALID, "set_histories: offsets not monotone");
        uint64_t L = offsets[i + 1] - offsets[i];
        if (L > 0x7fffffffull / 64) return fail(c, SCEMA_ERR_INVALID, "set_histories: history too long");
        mx = std::max<uint32_t>(mx, (uint32_t)L);
        mn = std::min<uint32_t>(mn, (uint32_t)L);
    }
    c->max_len = mx;
    c->min_len = n ? mn : 0;
    c->total_steps = n ? offsets[n] : 0;  // offsets index `steps` absolutely
    c->hist_ids_lazy = ids == nullptr;
    if (ids) set_ids(c->hist_ids, ids, n);
    SCEMA_CUDA(c, c->d_offsets.reserve((n + 1) * sizeof(uint64_t)));
    SCEMA_CUDA(c, cudaMemcpyAsync(c->d_offsets.p, c->h_offsets.data(), (n + 1) * sizeof(uint64_t),
                                  cudaMemcpyHostToDevice, c->stream));
    if (steps_on_device) {
        c->d_steps = steps;
    } else {
        const uint64_t last = n ? offsets[n] : 0;
        SCEMA_CUDA(c, c->steps_own.reserve(std::max<uint64_t>(last, 1) * 6 * sizeof(double)));
        if (last && steps_mode == 0)
            SCEMA_CUDA(c, cudaMemcpyAsync(c->steps_own.p, steps, last * 6 * sizeof(double), cudaMemcpyHostToDevice,
                                          c->stream));
        c->d_steps = c->steps_own.as<double>();
    }
    SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));  // h_offsets / caller buffers may be pageable
    c->have_histories = true;
    c->histories_version++;
    return SCEMA_OK;
}

int scema_set_histories(scema_ctx *c, const double *steps, int steps_on_device, const uint64_t *offsets,
                        const uint32_t *ids, uint64_t n)
{
    return set_histories_impl(c, steps, steps_on_device ? 1 : 0, offsets, ids, n);
}

int scema_resample(scema_ctx *c, uint32_t spline_points)
{
    int rc = enter(c);
    if (rc) return rc;
    c->ev_used[SCEMA_T_RESAMPLE] = false;
    return resample_run(c, spline_points);
}

int scema_store_reset(scema_ctx *c, uint64_t n, const uint32_t *ids, uint32_t capacity_steps)
{
    int rc = enter(c);
    if (rc) return rc;
    return store_reset(c, n, ids, capacity_steps);
}

int scema_store_append(scema_ctx *c, const double *strain, int strain_on_device)
{
    int rc = enter(c);
    if (rc) return rc;
    return store_append(c, strain, strain_on_device);
}

int scema_store_info(scema_ctx *c, uint64_t *n, uint32_t *n_steps, const double **device_steps)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->have_store) return fail(c, SCEMA_ERR_STATE, "store_info: no store (call scema_store_reset)");
    if (n) *n = c->store_n;
    if (n_steps) *n_steps = c->store_steps;
    if (device_steps) *device_steps = c->d_store.as<double>();
    return SCEMA_OK;
}

int scema_store_resample(scema_ctx *c, uint32_t spline_points)
{
    int rc = enter(c);
    if (rc) return rc;
    return store_resample(c, spline_points);
}

int scema_select_rows(scema_ctx *c, const uint32_t *rows, uint64_t m)
{
    int rc = enter(c);
    if (rc) return rc;
    return select_rows(c, rows, m);
}

int scema_set_spline(scema_ctx *c, const double *rows, int rows_on_device, uint64_t n, uint32_t k, const uint32_t *ids)
{
    int rc = enter(c);
    if (rc) return rc;
    if (n && k && !rows) return fail(c, SCEMA_ERR_INVALID, "set_spline: null pointer");
    if (n >= (1ull << 32)) return fail(c, SCEMA_ERR_INVALID, "set_spline: more than 2^32-1 histories");
    c->have_spline = false;
    c->have_edges = false;
    c->n = n;
    c->K = k;
    c->ids_lazy = ids == nullptr;   // 0 .. n-1: filled on first use (ids_of)
    if (ids) set_ids(c->ids, ids, n);
    if (rows_on_device) {
        c->d_spline = rows;
    } else {
        SCEMA_CUDA(c, c->spline_own.reserve(std::max<uint64_t>(n * k, 1) * sizeof(double)));
        if (n * k != 0)
            SCEMA_CUDA(c, cudaMemcpyAsync(c->spline_own.p, rows, n * k * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));
        c->d_spline = c->spline_own.as<double>();
    }
    c->spline_version++;
    c->have_spline = true;
    return SCEMA_OK;
}

int scema_get_spline(scema_ctx *c, double *out_host)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->have_spline) return fail(c, SCEMA_ERR_STATE, "Spline is not up to date.");
    if (c->n * c->K == 0) return SCEMA_OK;
    if (!out_host) return fail(c, SCEMA_ERR_INVALID, "get_spline: null pointer");
    SCEMA_CUDA(c, cudaMemcpyAsync(out_host, c->d_spline, c->n * c->K * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));
    return SCEMA_OK;
}

int scema_spline_info(scema_ctx *c, uint64_t *n, uint32_t *k, const double **device_rows)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->have_spline) return fail(c, SCEMA_ERR_STATE, "Spline is not up to date.");
    if (n) *n = c->n;
    if (k) *k = c->K;
    if (device_rows) *device_rows = c->d_spline;
    return SCEMA_OK;
}

int scema_compare(scema_ctx *c, double threshold, int variant, uint32_t shard, uint32_t n_shards, uint64_t *n_edges)
{
    int rc = enter(c);
    if (rc) return rc;
    rc = compare_run(c, threshold, variant, shard, n_shards);
    if (rc) { c->have_edges = false; return rc; }
    if (n_edges) *n_edges = c->n_edges;
    return SCEMA_OK;
}

int scema_compare_stream(scema_ctx *c, double threshold, int variant, uint32_t shard, uint32_t n_shards,
                         uint32_t panels_per_chunk, scema_edge_sink sink, void *user, uint64_t *n_edges_total)
{
    int rc = enter(c);
    if (rc) return rc;
    for (int k = 0; k < 2; k++)
        if (!c->stage_ev[k]) SCEMA_CUDA(c, cudaEventCreateWithFlags(&c->stage_ev[k], cudaEventDisableTiming));
    rc = compare_stream_run(c, threshold, variant, shard, n_shards, panels_per_chunk, sink, user, n_edges_total);
    c->have_edges = false;
    return rc;
}

}  // extern "C"

// keys (a << shift | b) -> the two index arrays, on the device: the host then receives exactly the arrays it asked for
// (a host-side unpack of 4M keys plus the page faults of a temporary costs more than the copy)
static __global__ void k_unpack_keys(const uint64_t *__restrict__ keys, uint64_t m, uint32_t shift, uint32_t *__restrict__ a,
                              uint32_t *__restrict__ b)
{
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const uint64_t k = keys[e];
    a[e] = (uint32_t)(k >> shift);
    b[e] = (uint32_t)(k & ((1ull << shift) - 1));
}

extern "C" {

int scema_get_edges(scema_ctx *c, uint32_t *ia, uint32_t *ib, double *diff, uint64_t cap)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->have_edges) return fail(c, SCEMA_ERR_STATE, "get_edges: no compare result");
    const uint64_t m = std::min<uint64_t>(cap, c->n_edges);
    if (m == 0) return SCEMA_OK;
    if (diff) SCEMA_CUDA(c, cudaMemcpyAsync(diff, c->d_edge_val[c->edge_cur].p, m * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (ia || ib) {
        // the other half of the sort's double buffer is free after the sort: unpack there
        uint32_t *da = c->d_edge_key[c->edge_cur ^ 1].as<uint32_t>(), *db = da + m;
        k_unpack_keys<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(c->d_edge_key[c->edge_cur].as<uint64_t>(), m, c->key_shift, da, db);
        c->launches++;
        SCEMA_CUDA(c, cudaGetLastError());
        if (ia) SCEMA_CUDA(c, cudaMemcpyAsync(ia, da, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        if (ib) SCEMA_CUDA(c, cudaMemcpyAsync(ib, db, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    }
    SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));
    return SCEMA_OK;
}

int scema_edges_device(scema_ctx *c, const uint64_t **keys, const double **diff, uint32_t *key_shift, uint64_t *n_edges)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->have_edges) return fail(c, SCEMA_ERR_STATE, "edges_device: no compare result");
    if (keys) *keys = c->d_edge_key[c->edge_cur].as<uint64_t>();
    if (diff) *diff = c->d_edge_val[c->edge_cur].as<double>();
    if (key_shift) *key_shift = c->key_shift;
    if (n_edges) *n_edges = c->n_edges;
    return SCEMA_OK;
}

int scema_get_degrees(scema_ctx *c, uint32_t *degree_host)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->have_edges) return fail(c, SCEMA_ERR_STATE, "get_degrees: no compare result");
    std::vector<uint32_t> a(c->n_edges), b(c->n_edges);
    rc = scema_get_edges(c, a.data(), b.data(), nullptr, c->n_edges);
    if (rc) return rc;
    std::fill(degree_host, degree_host + c->n, 0u);
    for (uint64_t e = 0; e < c->n_edges; e++) { degree_host[a[e]]++; degree_host[b[e]]++; }
    return SCEMA_OK;
}

int scema_nearest(scema_ctx *c, uint32_t *nearest_id_host, double *nearest_diff_host)
{
    int rc = enter(c);
    if (rc) return rc;
    return nearest_run(c, nearest_id_host, nearest_diff_host);
}

int scema_knn(scema_ctx *c, uint32_t k, int variant, uint32_t *index_host, double *diff_host)
{
    int rc = enter(c);
    if (rc) return rc;
    return knn_run(c, k, variant, index_host, diff_host);
}

int scema_knn_last_stats(scema_ctx *c, uint64_t counts[8], double radii[8])
{
    if (!c) return SCEMA_ERR_INVALID;
    for (int i = 0; i < 8; i++) {
        if (counts) counts[i] = c->knn_counts[i];
        if (radii) radii[i] = c->knn_radii[i];
    }
    return SCEMA_OK;
}

int scema_query_compare(scema_ctx *c, const double *rows, int rows_on_device, uint64_t m, uint32_t k_cols, double threshold, int variant,
                        uint64_t *n_edges)
{
    int rc = enter(c);
    if (rc) return rc;
    return query_compare_run(c, rows, rows_on_device, m, k_cols, threshold, variant, n_edges);
}

int scema_query_get_edges(scema_ctx *c, uint32_t *query_index, uint32_t *row_index, double *diff, uint64_t cap)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->have_query) return fail(c, SCEMA_ERR_STATE, "query_get_edges: no scema_query_compare result");
    const uint64_t m = std::min<uint64_t>(cap, c->query_n);
    if (m == 0) return SCEMA_OK;
    if (query_index) SCEMA_CUDA(c, cudaMemcpyAsync(query_index, c->query_j.p, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    if (row_index) SCEMA_CUDA(c, cudaMemcpyAsync(row_index, c->query_i.p, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
    if (diff) SCEMA_CUDA(c, cudaMemcpyAsync(diff, c->query_d.p, m * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));
    return SCEMA_OK;
}

int scema_query_knn(scema_ctx *c, const double *rows, int rows_on_device, uint64_t m, uint32_t k_cols, uint32_t k, int variant,
                    uint32_t *index_host, double *diff_host)
{
    int rc = enter(c);
    if (rc) return rc;
    return query_knn_run(c, rows, rows_on_device, m, k_cols, k, variant, index_host, diff_host);
}

int scema_query_last_stats(scema_ctx *c, uint64_t counts[11], double radii[8], float ms[8])
{
    if (!c) return SCEMA_ERR_INVALID;
    for (int i = 0; i < 11; i++)
        if (counts) counts[i] = c->query_counts[i];
    for (int i = 0; i < 8; i++) {
        if (radii) radii[i] = c->query_radii[i];
        if (ms) ms[i] = c->query_ms[i];
    }
    return SCEMA_OK;
}

int scema_cluster(scema_ctx *c, const double *steps, const uint64_t *offsets, const uint32_t *ids, uint64_t n,
                  uint32_t spline_points, double threshold, int variant, uint64_t *n_edges)
{
    // Large host batches on the tcgen05 path are pipelined: the raw steps travel to the device range by range
    // and every range is resampled and compared against everything that arrived before it while the next one
    // is still on the bus (cluster_pipelined, pairs.cu). Same spline matrix, same edge list.
    if (c && steps && offsets && variant == SCEMA_PAIRS_TC && spline_points >= 1 && spline_points <= 10 && threshold > 0.0 &&
        pipeline_wanted(n)) {
        int rc = enter(c);
        if (rc) return rc;
        rc = pipeline_begin(c, steps, offsets, n);       // the first ranges are on the bus before anything else happens
        if (!rc) rc = set_histories_impl(c, steps, 2, offsets, ids, n);
        if (rc) {
            if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);  // the caller's buffer is the caller's again on return
            return rc;
        }
        bool done = false;
        rc = cluster_pipelined(c, steps, spline_points, threshold, &done);
        if (rc) { c->have_edges = false; return rc; }
        if (done) {
            if (n_edges) *n_edges = c->n_edges;
            return SCEMA_OK;
        }
        // not done (e.g. the survivors overflowed the queue): every step is on the device by now, carry on in order
        rc = scema_resample(c, spline_points);
        if (rc) return rc;
        return scema_compare(c, threshold, variant, 0, 1, n_edges);
    }
    int rc = scema_set_histories(c, steps, 0, offsets, ids, n);
    if (rc) return rc;
    rc = scema_resample(c, spline_points);
    if (rc) return rc;
    return scema_compare(c, threshold, variant, 0, 1, n_edges);
}

int scema_write_similar_hist(scema_ctx *c, const char *fname_pattern)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->have_edges) return fail(c, SCEMA_ERR_STATE, "write_similar_hist: no compare result");
    if (!fname_pattern) return fail(c, SCEMA_ERR_INVALID, "write_similar_hist: null pattern");
    return write_similar_hist(c, fname_pattern);
}

int scema_reduce_edges(scema_ctx *c, uint32_t num_gps, uint32_t *mapping_host, uint64_t *iterations,
                       uint64_t *neighbours_removed)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->have_edges) return fail(c, SCEMA_ERR_STATE, "reduce_edges: no compare result");
    const uint64_t m = c->n_edges;
    std::vector<uint32_t> a(m), b(m);
    std::vector<double> d(m);
    rc = scema_get_edges(c, a.data(), b.data(), d.data(), m);
    if (rc) return rc;
    // add_edge call sequence of the per-history files read in batch order: history k lists its
    // partners in ascending batch index (smaller ones first), see host_io.cc
    std::vector<uint64_t> start(c->n + 2, 0);
    for (uint64_t e = 0; e < m; e++) { start[a[e] + 1]++; start[b[e] + 1]++; }
    for (uint64_t i = 0; i < c->n; i++) start[i + 1] += start[i];
    std::vector<uint64_t> fill(start.begin(), start.begin() + c->n);
    std::vector<uint32_t> eu(2 * m), ev(2 * m);
    const std::vector<uint32_t> &idv = ids_of(c);
    for (uint64_t e = 0; e < m; e++) {
        if (d[e] == 0.0) return fail(c, SCEMA_ERR_MAPPING, "reduce: dist == 0 (the script raises ZeroDivisionError)");
        uint64_t q = fill[b[e]]++; eu[q] = idv[b[e]]; ev[q] = idv[a[e]];
    }
    for (uint64_t e = 0; e < m; e++) { uint64_t q = fill[a[e]]++; eu[q] = idv[a[e]]; ev[q] = idv[b[e]]; }
    rc = reduce_graph_calls(eu.data(), ev.data(), 2 * m, num_gps, mapping_host, iterations, neighbours_removed);
    if (rc) return fail(c, rc, "reduce: history ID >= num_gps (the script raises IndexError)");
    return SCEMA_OK;
}

int scema_last_timings(scema_ctx *c, float ms[SCEMA_T_COUNT])
{
    int rc = enter(c);
    if (rc) return rc;
    SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int w = 0; w < SCEMA_T_COUNT; w++) {
        ms[w] = c->acc_ms[w];
        if (c->ev_used[w]) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, c->ev[2 * w], c->ev[2 * w + 1]) == cudaSuccess) ms[w] += t;
            else cudaGetLastError();
        }
    }
    return SCEMA_OK;
}

int scema_last_counters(scema_ctx *c, uint64_t counters[8])
{
    if (!c) return SCEMA_ERR_INVALID;
    for (int i = 0; i < 8; i++) counters[i] = c->counters[i];
    return SCEMA_OK;
}

uint64_t scema_kernel_launches(const scema_ctx *c) { return c ? c->launches : 0; }

int scema_last_audit(scema_ctx *c, uint64_t out[2])
{
    if (!c || !out) return SCEMA_ERR_INVALID;
    out[0] = c->audit_edges;
    out[1] = c->audit_missing;
    return SCEMA_OK;
}

int scema_fp64_peak(scema_ctx *c, double out[2])
{
    int rc = enter(c);
    if (rc) return rc;
    return fp64_peak_run(c, out);
}

int scema_k1_tune(int kernel, int warps_per_sm_ragged, int warps_per_sm_store, int flags)
{
    return k1_tune(kernel, warps_per_sm_ragged, warps_per_sm_store, flags);
}

int scema_pipeline_plan(uint64_t n, uint64_t *bounds, uint32_t cap, uint32_t *n_ranges)
{
    if (!bounds || !n_ranges || n < 2) return SCEMA_ERR_INVALID;
    std::vector<uint64_t> b;
    pipeline_bounds(n, b);
    *n_ranges = (uint32_t)(b.size() - 1);
    if (b.size() > cap) return SCEMA_ERR_INVALID;
    std::copy(b.begin(), b.end(), bounds);
    return SCEMA_OK;
}

int scema_tc_plan(uint32_t k, uint32_t slices, uint32_t cta_group, uint32_t plan[6])
{
    if (!plan || k == 0 || (slices != 1 && slices != 2) || (cta_group != 1 && cta_group != 2)) return SCEMA_ERR_INVALID;
    plan[0] = tc_chunks_for(k);
    if (plan[0] > 10 || (plan[0] > 1 && slices != 1)) return SCEMA_ERR_INVALID;
    return tc_smem_plan(plan[0], slices, cta_group, &plan[1], &plan[2], &plan[3], &plan[4], &plan[5]) ? SCEMA_OK : SCEMA_ERR_INVALID;
}

int scema_tc_choose(uint64_t pairs, uint32_t k, const uint64_t counts[5], uint64_t sample, uint64_t mem_budget, int *choice,
                    int *centred, uint64_t *est_survivors)
{
    if (!counts || !choice || !centred || !est_survivors || sample == 0 || k == 0) return SCEMA_ERR_INVALID;
    const uint64_t c6[6] = {counts[0], counts[1], counts[2], counts[3], counts[4], 0};
    tc_choose(pairs, k, c6, sample, mem_budget, tc_chunks_for(k) <= 10, false, choice, centred, est_survivors);
    return SCEMA_OK;
}

int scema_tc_choose_projected(uint64_t pairs, uint32_t k, const uint64_t counts[6], uint64_t sample, uint64_t mem_budget, int *choice,
                              int *centred, uint64_t *est_survivors)
{
    if (!counts || !choice || !centred || !est_survivors || sample == 0 || k == 0) return SCEMA_ERR_INVALID;
    tc_choose(pairs, k, counts, sample, mem_budget, tc_chunks_for(k) <= 10, true, choice, centred, est_survivors);
    return SCEMA_OK;
}

int scema_tc_basis(const double *moments, uint32_t k, double *basis, double *delta)
{
    if (!moments || !basis || !delta) return SCEMA_ERR_INVALID;
    return tc_basis_from_moments(moments, k, basis, delta) ? SCEMA_OK : SCEMA_ERR_INVALID;
}

int scema_tc_last_projection(scema_ctx *c, uint64_t out[2])
{
    if (!c || !out) return SCEMA_ERR_INVALID;
    out[0] = c->tc_plan_counts[5];
    out[1] = c->tc_proj ? 1u : 0u;
    return SCEMA_OK;
}

int scema_tc_last_plan(scema_ctx *c, uint64_t plan[6])
{
    if (!c || !plan) return SCEMA_ERR_INVALID;
    for (int i = 0; i < 5; i++) plan[i] = c->tc_plan_counts[i];
    plan[5] = tc_plan_sample_size();
    return SCEMA_OK;
}

int scema_tc_centre(scema_ctx *c, double *centre_host)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!c->tc_valid || !centre_host) return fail(c, SCEMA_ERR_STATE, "tc_centre: no tensor-core operand copies");
    SCEMA_CUDA(c, cudaMemcpyAsync(centre_host, c->d_tc_centre.p, (size_t)c->tc_K * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));
    return SCEMA_OK;
}

int scema_tc_shard_begin(scema_ctx *c, double threshold, uint64_t row0, uint64_t row1, const double **centre_dev)
{
    int rc = enter(c);
    if (rc) return rc;
    return tc_shard_begin(c, threshold, row0, row1, centre_dev);
}

int scema_tc_shard_stats(scema_ctx *c, const double *centre_dev, const uint64_t **packet_dev, uint64_t *packet_words)
{
    int rc = enter(c);
    if (rc) return rc;
    const unsigned long long *p = nullptr;
    rc = tc_shard_stats(c, centre_dev, &p, packet_words);
    if (packet_dev) *packet_dev = reinterpret_cast<const uint64_t *>(p);
    return rc;
}

int scema_tc_shard_finish(scema_ctx *c, const uint64_t *packets_dev, uint32_t n_shards, uint64_t pairs, int optimistic, int *choice,
                          const void **image_dev, uint64_t *image_bytes_per_row)
{
    int rc = enter(c);
    if (rc) return rc;
    return tc_shard_finish(c, reinterpret_cast<const unsigned long long *>(packets_dev), n_shards, pairs, optimistic, choice, image_dev,
                           image_bytes_per_row);
}

int scema_tc_shard_check(scema_ctx *c, int *choice)
{
    int rc = enter(c);
    if (rc) return rc;
    if (!choice) return fail(c, SCEMA_ERR_INVALID, "tc_shard_check: null pointer");
    return tc_shard_check(c, choice, nullptr);
}

int scema_tc_shard_commit(scema_ctx *c, void *rows_ready_event)
{
    int rc = enter(c);
    if (rc) return rc;
    return tc_shard_commit(c, rows_ready_event);
}

int scema_tc_debug(scema_ctx *c, double threshold, uint32_t slices, float *acc_host, uint64_t ld, void *operand_a_host,
                   void *operand_b_host)
{
    int rc = enter(c);
    if (rc) return rc;
    return tc_debug_run(c, threshold, slices, acc_host, ld, (unsigned char *)operand_a_host, (unsigned char *)operand_b_host);
}

}  // extern "C"
