// Internal declarations shared by the translation units of libscema_hist.so.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>
#include <cuda_runtime.h>

#include "../../include/scema_hist.h"

namespace scema {

constexpr int TILE = 128;         // rows per pair-matrix tile side (K2)
// Measured rates on one B200 (DESIGN.md section 6) behind the up-front choice of the filter and the overflow
// decisions: pairs per second of the one-slice / two-slice tcgen05 filter (one chunk of 64 columns), the DMMA filter
// and the filter-free kernel at K = 60, survivors per second of the exact recompute.
constexpr double RATE_TC1 = 1.4e13, RATE_TC2 = 4.6e12, RATE_DMMA = 2.9e11, RATE_EXACT = 7.0e10, RATE_QUEUE = 1.0e10;
// the projected (16-column) tcgen05 filter, pairs per second (config 4: 26.9 ms for 5.0e11 pairs, one B200 at 1000 W)
constexpr double RATE_TCP = 1.86e13;
constexpr int PANEL_ROWBLOCKS = 16;  // row blocks per scheduling panel (L2 reuse of the B tiles)

// Growable device buffer.
struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
    cudaError_t reserve(size_t need)
    {
        if (need <= bytes) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        size_t want = need + need / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return e; }
        bytes = want;
        return cudaSuccess;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// Layout of the filter copy F of the spline matrix S (see DESIGN.md "K2 data layout"):
// F[chunk][row_padded][kc] with K zero-padded to n_chunks*kc, rows zero-padded to a multiple of
// TILE. kc % 8 == 4 makes the DMMA fragment loads (lane -> row g, column t) bank-conflict free
// when a TILE x kc block lands densely in shared memory.
struct FilterLayout {
    uint32_t K = 0, kc = 0, kt = 0, n_chunks = 0;  // kt: width of the last chunk (== kc unless the DMMA kernel runs)
    uint64_t n = 0, n_pad = 0, n_blocks = 0;
};

struct SplineTable {  // per distinct history length L: factorised tridiagonal system + sample map
    uint64_t offset;  // in doubles, into tables buffer
};

}  // namespace scema

struct scema_ctx {
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    size_t mem_budget = 0;  // half of the device memory that was free when the context was created: what a survivor queue may take
                            // (cudaMemGetInfo costs ~10 ms per call in a process that drives several GPUs through NCCL)
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    uint64_t launches = 0;

    // ---- raw histories
    uint64_t hn = 0;             // raw histories in the batch
    uint64_t total_steps = 0;
    uint32_t max_len = 0, min_len = 0;
    const double *d_steps = nullptr;  // borrowed or = steps_own
    scema::DevBuf steps_own, d_offsets;
    std::vector<uint64_t> h_offsets;
    std::vector<uint32_t> hist_ids;
    bool have_histories = false;

    // ---- K1 tables: one per (L) for the current P
    uint32_t table_P = 0;
    std::map<uint32_t, uint64_t> table_off;  // L -> offset (doubles) in d_tables
    scema::DevBuf d_tables, d_table_index;   // d_table_index: int64 [max_len+1] -> offset or -1
    uint64_t tables_used = 0;                // doubles
    uint64_t tables_for_version = ~0ull;     // histories_version the tables were last checked against
    uint32_t table_index_len = 0;
    scema::DevBuf zscratch, d_order, d_chunks, d_chunk_counters;  // K1 work plan: padded group order, chunk list
    std::vector<uint32_t> plan_chunk_begin;                        // [classes+1] into d_chunks
    std::vector<uint64_t> plan_groups, plan_first_slot;            // per range and class: groups, first group slot
    std::vector<uint64_t> plan_bounds, plan_steps;                 // history ranges the plan was built for; raw steps per range
    std::vector<uint32_t> plan_max_len;                            // per range
    uint64_t histories_version = 0, order_version = ~0ull;

    // ---- spline matrix S [n][K] (n == hn after a resample; set_spline may install any n)
    uint64_t n = 0;
    uint32_t K = 0;
    std::vector<uint32_t> ids;
    const double *d_spline = nullptr;  // borrowed or = spline_own
    scema::DevBuf spline_own;
    bool have_spline = false;
    scema::DevBuf spline_sel[2], d_select;  // scema_select_rows: compacted subset of the rows (ping-pong: a second
                                            // selection gathers out of the first one's buffer)

    // ---- incremental history store, time-major [step][store_n][6]
    scema::DevBuf d_store;
    uint64_t store_n = 0;
    uint32_t store_steps = 0, store_cap = 0;
    std::vector<uint32_t> store_ids;
    bool have_store = false;

    // ---- K2 filter copy
    scema::FilterLayout fl;
    scema::DevBuf d_filter, d_halfnorm, d_blockmax, d_panel_start;
    uint64_t filter_for_spline_version = 0, spline_version = 0;
    int filter_variant = -1;

    // ---- K2 tensor-core filter (SCEMA_PAIRS_TC): fp16 split operands, A- and B-flavoured
    scema::DevBuf d_tc_a, d_tc_b, d_tc_nrm, d_tc_misc, d_tc_centre;  // centre: [K] column means subtracted in the filter copies only
    uint64_t tc_plan_counts[6] = {0, 0, 0, 0, 0, 0};  // last survivor-density sample (of tc::PLAN_SAMPLE pairs): one / two slices centred, one / two slices raw, DMMA, projected
    scema::DevBuf d_tc_basis, d_tc_cov;  // projected filter: basis rows [11][60] (FP64), sample second moments [K][K]
    double *h_tc_cov = nullptr;          // pinned copy of the second moments
    bool tc_proj = false;                // operand copies are the projected 16-column image (k_tc_prep_proj)
    double tc_basis_h[11 * 60] = {};      // the basis on the host (tc::Basis layout), kernel argument of k_tc_prep_proj
    scema::DevBuf d_tc_perm, d_tc_iota, d_tc_snrm, d_tc_band;  // norm-band mode: permutation, sorted squared norms, band plan
    bool tc_band = false, tc_band_wanted = false, tc_band_allowed = false;
    uint64_t tc_for_version = 0, tc_n = 0;
    uint32_t tc_K = 0, tc_slices = 0;
    uint32_t tc_mode = 0;  // 1: the filter was chosen automatically and compare_panels may change it on overflow; 0: SCEMA_TC_SLICES pins it
    double tc_thr = 0.0, tc_T0 = 0.0, tc_cguard = 0.0;
    bool tc_valid = false;
    bool tc_compact = false;             // hi-only operand copies (sharded prepare)
    uint32_t shard_phase = 0;            // sharded prepare: 0 none, 1 begun, 2 statistics taken, 3 own image built (commit next)
    uint64_t shard_r0 = 0, shard_r1 = 0; // own rows of a sharded prepare
    uint64_t *h_plan = nullptr;          // pinned: survivor-density sample of a sharded prepare (read back asynchronously)
    bool plan_pending = false;
    uint64_t plan_pairs = 0;
    bool ids_lazy = false, hist_ids_lazy = false;  // the IDs are 0 .. n-1 and the vector has not been filled (a million-entry
                                                   // refill per call is a millisecond of host time on the per-timestep path)
    void *rows_ready_event = nullptr;    // cudaEvent_t the exact recompute of the next compare waits for (FP64 rows still arriving)

    // ---- candidate queue + edges
    scema::DevBuf d_cand, d_counters;  // counters: [0] candidates, [1] edges, [2] flags
    scema::DevBuf d_edge_key[2], d_edge_val[2], d_sort_tmp;
    uint64_t cand_cap = 0, edge_cap = 0;
    int edge_cur = 0;            // which of the double buffers holds the sorted result
    uint64_t n_edges = 0;
    uint32_t key_shift = 0;
    bool have_edges = false;
    uint64_t *h_counters = nullptr;  // pinned, 8 entries
    // streaming compare: pinned double-buffered staging of one chunk of edges
    uint64_t *h_stage_key[2] = {nullptr, nullptr};
    double *h_stage_val[2] = {nullptr, nullptr};
    uint64_t stage_cap[2] = {0, 0};
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};

    // ---- host-buffer pipeline of scema_cluster: copy stream + one event per range
    cudaStream_t copy_stream = nullptr;
    std::vector<cudaEvent_t> copy_events;
    std::vector<uint64_t> pipe_bounds;  // history ranges of the current pipelined batch
    uint64_t pipe_early = 0;            // ranges whose copy was queued by pipeline_begin

    // ---- instrumentation
    cudaEvent_t ev[2 * SCEMA_T_COUNT] = {};
    bool ev_used[SCEMA_T_COUNT] = {};
    float acc_ms[SCEMA_T_COUNT] = {};  // phases already folded in by earlier chunks of a streamed compare
    uint64_t counters[8] = {};
    uint64_t audit_edges = 0, audit_missing = 0;  // last SCEMA_AUDIT run: sampled pairs that are reference edges / of those, missing from the list

    // ---- scema_knn (knn.cu): the filter rounds run on a private child context (on the same device and stream) so that
    //      this context's compare results stay as they are; scratch buffers and the stats of the last call
    scema_ctx *knn_child = nullptr;
    scema::DevBuf knn_buf[16];  // scratch of scema_knn and the scema_query_* calls (nothing in it outlives a call)
    uint64_t knn_counts[8] = {};
    double knn_radii[8] = {};

    // ---- scema_query_compare / scema_query_knn (knn.cu): their own child context, so that a query leaves the state of
    //      scema_knn's child (queue sizes, filter decisions) as it was; the cross edges of the last scema_query_compare
    scema_ctx *query_child = nullptr;
    scema::DevBuf query_j, query_i, query_d;
    uint64_t query_n = 0;
    bool have_query = false;
    uint64_t query_counts[11] = {};
    double query_radii[8] = {};
    float query_ms[8] = {};
    cudaEvent_t query_ev[2] = {nullptr, nullptr};
};

namespace scema {

#define SCEMA_CUDA(ctx, call)                                                                   \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e__);                   \
            return e__ == cudaErrorMemoryAllocation ? SCEMA_ERR_NOMEM : SCEMA_ERR_CUDA;         \
        }                                                                                       \
    } while (0)

// exact pair distance: compare_L2_norm, strain2spline.h:476-483, operation for operation
__device__ __forceinline__ double exact_l2(const double *__restrict__ a, const double *__restrict__ b, uint32_t K)
{
    double sum = 0.0;
#pragma unroll 4
    for (uint32_t k = 0; k < K; k++) {
        double diff = __dsub_rn(__ldg(a + k), __ldg(b + k));
        sum = __dadd_rn(sum, __dmul_rn(diff, diff));
    }
    return __dsqrt_rn(sum);
}

// IDs of the current spline rows, filled on first use when they are the default 0 .. n-1
inline const std::vector<uint32_t> &ids_of(scema_ctx *c)
{
    if (c->ids_lazy) {
        c->ids.resize(c->n);
        for (uint64_t i = 0; i < c->n; i++) c->ids[i] = (uint32_t)i;
        c->ids_lazy = false;
    }
    return c->ids;
}

inline int fail(scema_ctx *ctx, int code, const std::string &msg)
{
    ctx->err = msg;
    return code;
}

inline void t_begin(scema_ctx *c, int which) { cudaEventRecord(c->ev[2 * which], c->stream); c->ev_used[which] = true; }
inline void t_end(scema_ctx *c, int which) { cudaEventRecord(c->ev[2 * which + 1], c->stream); }

// resample.cu
int resample_run(scema_ctx *ctx, uint32_t P);
int resample_prepare(scema_ctx *ctx, uint32_t P, const std::vector<uint64_t> &bounds);
int resample_launch_range(scema_ctx *ctx, uint32_t P, size_t r);
int store_reset(scema_ctx *ctx, uint64_t n, const uint32_t *ids, uint32_t capacity_steps);
int store_append(scema_ctx *ctx, const double *strain, int on_device);
int store_resample(scema_ctx *ctx, uint32_t P);
int k1_tune(int kernel, int wps_ragged, int wps_store, int flags);
int select_rows(scema_ctx *ctx, const uint32_t *rows, uint64_t m);
// pairs.cu
int compare_run(scema_ctx *ctx, double thr, int variant, uint32_t shard, uint32_t n_shards);
int wait_rows(scema_ctx *ctx);
int compare_stream_run(scema_ctx *ctx, double thr, int variant, uint32_t shard, uint32_t n_shards, uint32_t panels_per_chunk,
                       scema_edge_sink sink, void *user, uint64_t *n_total);
int fp64_peak_run(scema_ctx *ctx, double out[2]);
int nearest_run(scema_ctx *ctx, uint32_t *nearest_id_host, double *nearest_diff_host);
int compare_prefix_run(scema_ctx *ctx, double thr, int *variant, uint32_t p1, bool plan_prefix);
int edges_adopt(scema_ctx *ctx, const uint64_t *d_keys, const double *d_vals, uint64_t total);
bool pipeline_wanted(uint64_t n);
void pipeline_bounds(uint64_t n, std::vector<uint64_t> &bounds);
int pipeline_begin(scema_ctx *ctx, const double *steps_host, const uint64_t *offsets, uint64_t n);
int cluster_pipelined(scema_ctx *ctx, const double *steps_host, uint32_t P, double thr, bool *done);
// pairs_tc.cu
bool tc_supported(const scema_ctx *ctx);
bool tc_two_slices_possible(const scema_ctx *ctx);
bool tc_smem_plan(uint32_t nc, uint32_t slices, uint32_t cg, uint32_t *a_bytes, uint32_t *n_abuf, uint32_t *lg_nst,
                  uint32_t *stage_bytes, uint32_t *data_bytes);
uint32_t tc_chunks_for(uint32_t K);
int tc_prepare(scema_ctx *ctx, double thr, uint32_t slices, bool want_band, uint64_t pairs, int *choice, uint64_t *est_survivors);
void tc_choose(uint64_t pairs, uint32_t K, const uint64_t counts[6], uint64_t sample, uint64_t mem_budget, bool tc_ok, bool proj_ok, int *choice,
               int *centred, uint64_t *est_survivors);
int tc_centre_rows(scema_ctx *ctx, uint64_t r0, uint64_t r1);
int tc_plan_rows(scema_ctx *ctx, uint64_t r1, uint64_t counts[6], bool proj);
bool tc_basis_from_moments(const double *cov, uint32_t K, double *basis, double *delta);
bool tc_proj_possible(uint32_t K);
int tc_basis_range(scema_ctx *ctx, uint64_t r0, uint64_t r1, bool *ok);
uint32_t tc_plan_sample_size();
int tc_shard_begin(scema_ctx *ctx, double thr, uint64_t r0, uint64_t r1, const double **centre_dev);
int tc_shard_stats(scema_ctx *ctx, const double *centre_dev, const unsigned long long **packet_dev, uint64_t *packet_words);
int tc_shard_finish(scema_ctx *ctx, const unsigned long long *packets_dev, uint32_t G, uint64_t pairs, int optimistic, int *choice,
                    const void **image_dev, uint64_t *image_bytes_per_row);
int tc_shard_check(scema_ctx *ctx, int *choice, uint64_t *est_survivors);
int tc_shard_commit(scema_ctx *ctx, void *rows_ready_event);
int tc_prepare_begin(scema_ctx *ctx, double thr, uint32_t slices);
int tc_stats_rows(scema_ctx *ctx, uint64_t r0, uint64_t r1, bool into_scale);
int tc_fix_scale(scema_ctx *ctx, int headroom);
int tc_prep_rows(scema_ctx *ctx, uint64_t r0, uint64_t r1);
int tc_launch(scema_ctx *ctx, uint32_t I0, uint32_t I1, uint32_t C0, uint32_t C1, uint32_t shard, uint32_t n_shards,
              unsigned long long *cand_count, float *dbg, uint64_t dbg_ld);
int tc_debug_run(scema_ctx *ctx, double thr, uint32_t slices, float *acc_host, uint64_t ld, unsigned char *ha_host,
                 unsigned char *hb_host);
// knn.cu
int knn_run(scema_ctx *ctx, uint32_t k, int variant, uint32_t *index_host, double *diff_host);
int query_compare_run(scema_ctx *ctx, const double *rows, int rows_on_device, uint64_t m, uint32_t k_cols, double thr, int variant,
                      uint64_t *n_edges);
int query_knn_run(scema_ctx *ctx, const double *rows, int rows_on_device, uint64_t m, uint32_t k_cols, uint32_t k, int variant,
                  uint32_t *index_host, double *diff_host);
// host_io.cc
int write_similar_hist(scema_ctx *ctx, const char *pattern);
int reduce_graph_calls(const uint32_t *eu, const uint32_t *ev, uint64_t n_calls, uint32_t num_gps,
                       uint32_t *mapping, uint64_t *iterations, uint64_t *neighbours_removed);

}  // namespace scema
