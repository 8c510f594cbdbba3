/* scema_hist.h — C ABI of libscema_hist.so: SCEMa's MD-redundancy clustering hot path on B200.
 *
 * The reference (UCL-CCS/SCEMa) has no FFI layer for this path; its de-facto boundary is the
 * header API of namespace MatHistPredict (headers/strain2spline.h), two command lines
 * (clustering/compare_all_histories.cc, clustering/mpi_comparison_test.cc) and three file
 * formats. Each entry point below names the reference interface it replaces (file:line relative
 * to the reference root). scema_b200/host/strain2spline_b200.h re-creates the MatHistPredict
 * header API on top of this ABI, and INTEGRATION.md shows the binding a maintainer adds.
 *
 * Conventions: plain pointers and sizes only; every function returns SCEMA_OK or an error code
 * and never exits the process (the reference does fprintf(stderr)+exit(1) everywhere; the C++
 * shim maps non-zero codes back to that behaviour). A context is bound to one CUDA device and
 * one stream; calls on one context are not thread-safe; different contexts are independent.
 * There is NO CPU fallback: without a CUDA device scema_create fails with SCEMA_ERR_CUDA.
 */
#ifndef SCEMA_HIST_H
#define SCEMA_HIST_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCEMA_OK 0
#define SCEMA_ERR_INVALID 1 /* bad argument; includes a history with < 3 steps (strain2spline.h:142-148) */
#define SCEMA_ERR_CUDA 2    /* CUDA runtime failure, or no device */
#define SCEMA_ERR_NOMEM 3   /* host or device allocation failed */
#define SCEMA_ERR_IO 4      /* file could not be opened (strain2spline.h:117-120, :303-307) */
#define SCEMA_ERR_STATE 5   /* call order: e.g. compare before any spline matrix exists (strain2spline.h:214-221) */
#define SCEMA_ERR_MAPPING 6 /* graph reduction: ID >= num_gps or dist == 0 (coarsegrain_dependency_network.py:57,73) */
#define SCEMA_ERR_DENSE 7   /* sharded compare (n_shards > 1) only: this shard's survivors are too dense for its queue and the
                             * remedy — another filter — would change how the pair matrix is split between the shards; EVERY
                             * shard must repeat the compare with SCEMA_PAIRS_DMMA (and, if that fails too, SCEMA_PAIRS_EXACT).
                             * scema_cluster_multi and scema_b200/distributed.py do this; a single-shard compare switches by itself. */

/* Which kernel evaluates the all-pairs distance (north star: DMMA tensor path, CUDA-core FMA
 * variant kept for comparison, exact direct-difference kernel as the anchor). All three emit
 * the bit-identical edge list. */
#define SCEMA_PAIRS_DMMA 0  /* GEMM-form filter on FP64 mma.sync (DMMA) + exact recompute of survivors */
#define SCEMA_PAIRS_FMA 1   /* GEMM-form filter on CUDA-core DFMA + exact recompute of survivors */
#define SCEMA_PAIRS_EXACT 2 /* every pair by direct differences (compare_L2_norm order), no filter */
/* GEMM-form filter on the 5th-generation tensor cores: FP64 rows split into two fp16 slices, tcgen05.mma
 * kind::f16 with fp32 accumulators in tensor memory, row norms and threshold folded into spare operand
 * columns so that the sign of the accumulator decides; survivors (edges + a guard band covering the
 * slicing and accumulation error) take the same exact FP64 recompute. Same edge list, same distance
 * bits. Rows of up to 60 columns (10 spline points) start with the hi slices alone (a third of the
 * tensor work, guard band 2^-9 of the squared norms) and repeat with both slices (2^-13) when the
 * survivors overflow the candidate queue; SCEMA_TC_SLICES=1|2 in the environment pins the choice. Wider
 * rows (up to 636 columns = 106 spline points) are cut into 64-column chunks and run with the hi slices,
 * falling back to SCEMA_PAIRS_DMMA on overflow; beyond that SCEMA_PAIRS_DMMA is taken straight away.
 * SCEMA_NORM_BAND=1 (opt-in, scema_compare only, rows of up to 60 columns, all norms finite) additionally sorts
 * the rows by norm and skips every tile whose norm intervals lie farther apart than the threshold
 * (| |a| - |b| | <= d(a, b)): an exact shortcut whose gain depends entirely on how spread the norms are. */
#define SCEMA_PAIRS_TC 3

typedef struct scema_ctx scema_ctx;

/* ---- context ------------------------------------------------------------------------------ */
/* device: CUDA ordinal. stream: a cudaStream_t passed as void* (NULL = the library creates its
 * own non-blocking stream). */
int scema_create(scema_ctx **out, int device, void *stream);
void scema_destroy(scema_ctx *ctx);
const char *scema_last_error(const scema_ctx *ctx); /* "" when the last call succeeded */
const char *scema_version(void);
/* The cudaStream_t (as void*) every call of this context is ordered on: the caller's stream given
 * to scema_create, or the library's own non-blocking stream. Work that produces borrowed device
 * inputs or consumes device outputs (e.g. an NCCL all-gather of the spline rows) must be ordered
 * against this stream. */
int scema_stream(scema_ctx *ctx, void **stream);

/* ---- ingest: replaces Strain6D storage, add_current_strain (strain2spline.h:75-86) and the
 *      data half of from_file (:112-134) for a whole batch of quadrature points ---------------
 * steps:   [sum_i L_i][6] doubles, component order xx yy zz xy xz yz (as one line of strain_<ID>).
 * offsets: HOST array [n+1], offsets[i] = first step of history i (in steps, not doubles).
 * ids:     HOST array [n] of history IDs (set_ID, :68-72) or NULL for 0..n-1.
 * steps_on_device != 0: `steps` is a device pointer on the context's device; it is borrowed (not
 * copied) and must stay valid until the next scema_set_* call or scema_destroy. */
int scema_set_histories(scema_ctx *ctx, const double *steps, int steps_on_device,
                        const uint64_t *offsets, const uint32_t *ids, uint64_t n);

/* ---- K1 resample: replaces Strain6D::splinify for every history (strain2spline.h:140-180;
 *      tk::spline::set_points / operator(), spline.h:284-396). Result: device matrix
 *      [n][6*spline_points], row layout p*6+c exactly as Strain6D::spline. Bit-exact. ---------- */
int scema_resample(scema_ctx *ctx, uint32_t spline_points);

/* Already-resampled rows (what Strain6D::get_spline() returns, :214-221), row-major [n][k].
 * rows_on_device != 0: borrowed device pointer. ids as above. */
int scema_set_spline(scema_ctx *ctx, const double *rows, int rows_on_device, uint64_t n, uint32_t k,
                     const uint32_t *ids);

/* ---- device-resident incremental history store: the in-process caller's pattern. Every timestep
 *      FEProblem::update_strain_quadrature_point_history appends one sample per quadrature point
 *      (FE_problem.h:1091-1103 -> Strain6D::add_current_strain, strain2spline.h:75-86), then
 *      spline_building re-fits EVERY point (FE_problem.h:1167-1191) and spline_comparison compares
 *      only the points flagged for an MD update (FE_problem.h:1202-1229). The store keeps all
 *      histories on the device (time-major [step][n][6]), so a timestep costs one 48*n-byte copy
 *      instead of re-sending every history.
 *        scema_store_reset   n points with their IDs (NULL = 0..n-1), room for capacity_steps (grows)
 *        scema_store_append  one sample for every point: strain[n][6], xx yy zz xy xz yz
 *        scema_store_resample  splinify(spline_points) of all n points -> current spline matrix [n][6P]
 *        scema_select_rows   keep only the given rows of the current spline matrix (the flagged
 *                            points), IDs carried along; the following compare / get_edges /
 *                            write_similar_hist work on that subset. */
int scema_store_reset(scema_ctx *ctx, uint64_t n, const uint32_t *ids, uint32_t capacity_steps);
int scema_store_append(scema_ctx *ctx, const double *strain, int strain_on_device);
int scema_store_info(scema_ctx *ctx, uint64_t *n, uint32_t *n_steps, const double **device_steps);
int scema_store_resample(scema_ctx *ctx, uint32_t spline_points);
int scema_select_rows(scema_ctx *ctx, const uint32_t *rows, uint64_t m);

/* Copy the current spline matrix [n][k] to host memory / expose it on the device. */
int scema_get_spline(scema_ctx *ctx, double *out_host);
int scema_spline_info(scema_ctx *ctx, uint64_t *n, uint32_t *k, const double **device_rows);

/* ---- K2+K3 compare: replaces compare_histories_with_all_ranks (strain2spline.h:546-614) with
 *      compare_L2_norm (:469-484) and the strict threshold of choose_most_similar_history
 *      (:265-274). Produces the UNIQUE pairs a<b (indices into the batch) with
 *      diff = compare_L2_norm(a,b) < threshold, sorted by (a,b), diff bit-identical to the
 *      reference. shard/n_shards: this context evaluates only its share of the pair-matrix tiles
 *      (one context per GPU, shard = rank); shard=0,n_shards=1 is the whole problem. ---------- */
int scema_compare(scema_ctx *ctx, double threshold, int variant, uint32_t shard, uint32_t n_shards,
                  uint64_t *n_edges);

/* Streaming form of scema_compare for edge lists that should not be held on the device (or in one
 * host array) as a whole — BASELINE config 5, "sparse thresholded edge streaming". The pair matrix
 * is evaluated in chunks of panels_per_chunk panels (one panel = 2048 rows; 0 = default 64); each
 * chunk's edges, sorted by (a,b), are handed to `sink` from pinned host memory while the GPU works
 * on the next chunk. Index a of consecutive chunks is disjoint and increasing, so the calls
 * concatenate to exactly the list scema_compare would produce. The arrays are only valid during the
 * call; a non-zero return value of the sink aborts with SCEMA_ERR_STATE. Nothing is retained:
 * scema_get_edges / scema_write_similar_hist need a plain scema_compare. */
typedef int (*scema_edge_sink)(void *user, const uint32_t *index_a, const uint32_t *index_b, const double *diff,
                               uint64_t n_edges);
int scema_compare_stream(scema_ctx *ctx, double threshold, int variant, uint32_t shard, uint32_t n_shards,
                         uint32_t panels_per_chunk, scema_edge_sink sink, void *user, uint64_t *n_edges_total);

/* Edge list of the last scema_compare. Host copies (any pointer may be NULL): index_a/index_b are
 * batch indices, diff the distance. cap = array capacity in edges. */
int scema_get_edges(scema_ctx *ctx, uint32_t *index_a, uint32_t *index_b, double *diff, uint64_t cap);
/* Device views: keys[e] = (a << key_shift) | b sorted ascending, diff[e]. Valid until the next
 * compare. */
int scema_edges_device(scema_ctx *ctx, const uint64_t **keys, const double **diff, uint32_t *key_shift,
                       uint64_t *n_edges);
/* Per-history number of partners (size of most_similar_histories, strain2spline.h:429). */
int scema_get_degrees(scema_ctx *ctx, uint32_t *degree_host);

/* Legacy single nearest neighbour of every history of the current spline matrix (the most_similar_history the
 * reference keeps "for legacy reasons", strain2spline.h:277-289; get_most_similar_history_ID / _diff, :233-245): the
 * smallest compare_L2_norm to ANY other history — not only those below a threshold —, ties to the lowest ID, NaN
 * distances ignored; {UINT32_MAX, +inf} when there is no candidate. Every pair is evaluated exactly (two passes of the
 * filter-free tiles), nothing of size O(N^2) is stored. The full comparison lists (all_similar_histories, :271) are
 * what scema_compare(+inf, SCEMA_PAIRS_EXACT) returns. Host arrays [n]; either may be NULL. */
int scema_nearest(scema_ctx *ctx, uint32_t *nearest_id_host, double *nearest_diff_host);

/* k nearest neighbours of every history of the current spline matrix, exact (1 <= k <= 32, otherwise SCEMA_ERR_INVALID;
 * SCEMA_ERR_STATE without a spline matrix). Row i's k slots are [i*k, i*k + k) of both host arrays (either may be NULL):
 * index_host the batch indices (not IDs) of the partners, diff_host compare_L2_norm(i, j) with the reference's bits.
 * Slots in order of (diff, ids[j], j) ascending — the reference's tie-break to the lower ID, then the index, because IDs
 * may repeat after scema_select_rows. A history is never its own neighbour; partners at distance NaN are skipped (as in
 * scema_nearest), partners at +inf are listed; unused slots are {UINT32_MAX, +inf} (k > n - 1, rows with a NaN, n <= 1).
 * With k = 1, ids[index[i]] and the diff bits are what scema_nearest returns.
 * variant picks the filter of the rounds (SCEMA_PAIRS_TC with its fallbacks, _DMMA, _FMA): a thresholded compare at a radius
 * from a distance sample closes every row with at least k partners below it, later rounds repeat it for the open rows at a
 * larger radius, and the rows left over (all rows with SCEMA_PAIRS_EXACT or a small batch, and whenever a round would list
 * more than O(n k) edges) are evaluated against every history by an exact top-k kernel. The result is bit-identical for
 * every variant; memory is O(n k). The last compare's edges, degrees, timings, counters, audit and operand caches of this
 * context are left as they were, also when the call fails. */
int scema_knn(scema_ctx *ctx, uint32_t k, int variant, uint32_t *index_host, double *diff_host);
/* The last scema_knn: counts = {filter rounds run, rows finished in round 1, rows finished in later filter rounds, rows
 * finished by the exact kernel, pairs the exact kernel evaluated, filter survivors over all rounds, edges below the radius
 * over all rounds, filter variant of the last round (SCEMA_PAIRS_EXACT when none ran)}; radii = the radius of each round
 * (0 for rounds not run). Either pointer may be NULL. */
int scema_knn_last_stats(scema_ctx *ctx, uint64_t counts[8], double radii[8]);

/* ---- cross queries: a second set of m histories (the queries) against the current spline matrix (the retained
 *      histories), the question compare_histories_with_all_ranks (strain2spline.h:590-598) asks on every ring step after
 *      the first. rows = the queries [m][k_cols], already resampled (row layout p*6+c, as scema_get_spline), in host
 *      memory, or on the device with rows_on_device (borrowed for the duration of the call only; for raw histories,
 *      resample them on a second context and pass scema_spline_info's device pointer). Index i is the batch index of a
 *      retained history (also after scema_select_rows and on the store path), index j the position in the query array. A
 *      query is never "itself": a query equal to a retained row is listed at distance 0. (a - b)^2 and (b - a)^2 round
 *      identically, so every diff has the bits of compare_L2_norm(row i, query j). Every variant gives the identical
 *      result. SCEMA_ERR_INVALID: k_cols != the matrix's k, a bad variant, k outside [1, 32], m > 0 with rows == NULL,
 *      n + m >= 2^32; SCEMA_ERR_STATE without a spline matrix. m = 0 or n = 0 give an empty result. Both calls run on a
 *      private context: the last compare of this context (edges, degrees, timings, counters, audit, operand caches) and
 *      scema_knn_last_stats are left exactly as they were, also when the call fails. Memory: the scratch copy [Q; R] of
 *      (m + n) rows, plus the edges of its first ceil(m / 2048) row panels.
 *
 * scema_query_compare: every pair (query j, history i) with compare_L2_norm(i, j) < threshold (thresholds <= 0 or NaN:
 * none), sorted by (j, i). *n_edges = their number. scema_query_get_edges copies the first cap of them to host arrays (any
 * pointer may be NULL). They stay readable until the next scema_query_compare on this context, which replaces them (a
 * failed one leaves none: SCEMA_ERR_STATE); scema_compare, scema_knn, scema_query_knn and new spline matrices do not touch
 * them. */
int scema_query_compare(scema_ctx *ctx, const double *rows, int rows_on_device, uint64_t m, uint32_t k_cols, double threshold,
                        int variant, uint64_t *n_edges);
int scema_query_get_edges(scema_ctx *ctx, uint32_t *query_index, uint32_t *row_index, double *diff, uint64_t cap);
/* scema_query_knn: the k nearest retained histories of every query: slots [j*k, j*k + k) of both host arrays (either may
 * be NULL), ordered by (diff, ids[i], i) as scema_knn; NaN partners skipped, +inf listed, empty slots {UINT32_MAX, +inf}.
 * The rounds of scema_knn with the queries as the rows: a radius from the open queries sampled against a seeded subset
 * of the matrix, a compare of [open queries; matrix] that closes every query with k partners below it, and the exact
 * top-k kernel for what is left (all queries with SCEMA_PAIRS_EXACT, or when open queries * n <= 2^28). */
int scema_query_knn(scema_ctx *ctx, const double *rows, int rows_on_device, uint64_t m, uint32_t k_cols, uint32_t k, int variant,
                    uint32_t *index_host, double *diff_host);
/* The last scema_query_*: counts = {filter rounds run, queries finished in round 1, queries finished in later rounds,
 * queries finished by the exact kernel, pairs the exact kernel evaluated, filter survivors, edges of the [Q; R] prefix
 * compares (all of them: also query x query and the retained rows that share the last query panel), filter variant of
 * the last round (SCEMA_PAIRS_EXACT when none ran), pairs of the row panels the filter was launched on (at most
 * m n + m (m - 1) / 2 + 2048 n per round), cross edges (scema_query_compare), passes of the compares (more than one
 * per round: a queue or edge buffer overflowed and the compare grew it or re-decided its filter)}; radii = the threshold /
 * the radius of each round; ms = CUDA-event milliseconds of {scratch copy [Q; R] (with the upload of host queries),
 * operand prep, filter, exact recompute, sort, compaction / selection of the cross entries, exact top-k kernel, 0}. Any
 * pointer may be NULL. */
int scema_query_last_stats(scema_ctx *ctx, uint64_t counts[11], double radii[8], float ms[8]);

/* One call for a host caller: set_histories + resample + compare. With SCEMA_PAIRS_TC, 6 * spline_points <= 60
 * and a large batch (>= 65536 histories; SCEMA_PIPELINE=0 disables, SCEMA_PIPELINE_MIN_N moves the limit) the three
 * steps are pipelined range by range behind the host->device copy of the raw steps: range c is resampled and compared
 * with itself and all earlier ranges while range c+1 is still on the bus. Same spline matrix and edge list; the
 * per-phase timings then report the whole overlapped region as "filter". */
int scema_cluster(scema_ctx *ctx, const double *steps, const uint64_t *offsets, const uint32_t *ids,
                  uint64_t n, uint32_t spline_points, double threshold, int variant, uint64_t *n_edges);

/* ---- sharded prepare of the tcgen05 filter (one context per GPU, each owning the rows [row0, row1) of a spline matrix
 *      whose full-size buffer has been installed with scema_set_spline; the shares cover [0, n) without overlap, row0 is a
 *      multiple of 128 and row1 a multiple of 128 or n — except for an EMPTY share, row0 == row1 at any row <= n, which a
 *      GPU past the end of a split into equal shares gets: it takes part in every step, contributes no rows, no sample and
 *      no image): every GPU builds the fp16
 *      operand image of its own rows only and the caller all-gathers the images (128 bytes per row and 64-column chunk)
 *      instead of waiting for the FP64 rows of everybody (8 K bytes per row), which only the exact recompute needs:
 *        scema_tc_shard_begin   -> *centre_dev: K doubles on the device (centre candidate of the own rows); all-gather them
 *                                  and pass ONE of them (the same on every GPU) to
 *        scema_tc_shard_stats   -> *packet_dev: *packet_words 8-byte words (norm statistics and the survivor-density sample
 *                                  of the own rows); all-gather the packets of all n_shards GPUs and pass them to
 *        scema_tc_shard_finish  (optimistic = 0) -> *choice: 1 = one fp16 slice with centred copies: the own rows' image now sits at
 *                                  *image_dev + row0 * *image_bytes_per_row (hi-only layout; the share that ends at n also
 *                                  holds the padding rows up to n_pad = n rounded up to a multiple of 256). The image is
 *                                  n_pad * *image_bytes_per_row bytes and nothing may be written past that: copy every
 *                                  GPU's part into every other GPU's image, then scema_tc_shard_commit. Any other value (2: two slices, 3: raw copies,
 *                                  0: SCEMA_PAIRS_DMMA, -1: SCEMA_PAIRS_EXACT): nothing was built, take the ordinary
 *                                  scema_compare (every GPU gets the same value).
 *        scema_tc_shard_commit  derives the second operand flavour; rows_ready_event (a cudaEvent_t as void*, may be NULL)
 *                                  is what the exact recompute of the following scema_compare(threshold, SCEMA_PAIRS_TC,
 *                                  shard, n_shards) waits for — record it behind the all-gather of the FP64 rows, which may
 *                                  then overlap the filter. scema_b200/distributed.py drives this with torch.distributed.
 *      The calls must come in this order: stats, finish and commit out of turn return SCEMA_ERR_STATE, and so does commit
 *      after a finish that chose another filter. */
int scema_tc_shard_begin(scema_ctx *ctx, double threshold, uint64_t row0, uint64_t row1, const double **centre_dev);
int scema_tc_shard_stats(scema_ctx *ctx, const double *centre_dev, const uint64_t **packet_dev, uint64_t *packet_words);
int scema_tc_shard_finish(scema_ctx *ctx, const uint64_t *packets_dev, uint32_t n_shards, uint64_t pairs, int optimistic, int *choice,
                          const void **image_dev, uint64_t *image_bytes_per_row);
int scema_tc_shard_commit(scema_ctx *ctx, void *rows_ready_event);
/* optimistic != 0 in scema_tc_shard_finish: no host synchronisation in the middle of the step — the image is built on the
 * assumption that the sample again says "one slice, centred copies" (*choice = 1), and scema_tc_shard_check, called after
 * the following scema_compare (which synchronises anyway), returns what the sample really said; anything but 1 means the
 * step has to be repeated on the ordinary path (the optimistic result is still a correct edge list — every survivor is
 * recomputed exactly — it may just have cost more than necessary; overflowing queues are handled by the compare). */
int scema_tc_shard_check(scema_ctx *ctx, int *choice);

/* ---- several GPUs of one box behind the same boundary: replaces the collective of compare_histories_with_all_ranks
 *      (strain2spline.h:546-614: R - 1 ring steps of blocking messages per history, called at FE_problem.h:1229) with a
 *      tile-sharded all-pairs driven from ONE process. scema_multi_create(devices[n_devices]; NULL = 0..n-1) makes one
 *      context and one host thread per GPU and an NCCL communicator over them (NCCL is loaded at run time; one device
 *      needs none). scema_multi_cluster: host buffers as scema_cluster; every GPU receives its contiguous share of the
 *      histories over its own PCIe link and resamples it, ONE all-gather of the row blocks (NCCL over NVLink) gives every
 *      GPU the whole spline matrix, every GPU evaluates shard r of n_devices of the pair matrix (all shards switch filter
 *      together when one is too dense), an ncclAllGather of the edge counts yields the offsets at which the shards' lists
 *      are collected on the first GPU and put in canonical order. scema_multi_compare_rows: the same from already-
 *      resampled rows in host memory. Afterwards the FIRST context (scema_multi_context(m, 0)) serves the result through
 *      scema_get_edges / scema_get_degrees / scema_write_similar_hist / scema_reduce_edges exactly as after a one-GPU
 *      scema_compare (bit-identical list). The other contexts answer scema_last_timings / scema_last_counters for
 *      their shard. */
typedef struct scema_multi scema_multi;
int scema_multi_create(scema_multi **out, const int *devices, int n_devices);
void scema_multi_destroy(scema_multi *m);
const char *scema_multi_last_error(const scema_multi *m);
int scema_multi_devices(const scema_multi *m);
scema_ctx *scema_multi_context(scema_multi *m, int rank);
int scema_multi_cluster(scema_multi *m, const double *steps, const uint64_t *offsets, const uint32_t *ids, uint64_t n,
                        uint32_t spline_points, double threshold, int variant, uint64_t *n_edges);
int scema_multi_compare_rows(scema_multi *m, const double *rows, uint64_t n, uint32_t k, const uint32_t *ids, double threshold,
                             int variant, uint64_t *n_edges);
/* Edges every shard found and the offset of its block in the gathered list before the canonical sort (host arrays [n_devices]). */
int scema_multi_shard_edges(scema_multi *m, uint64_t *counts, uint64_t *offsets);
/* Wall-clock milliseconds of the last call's phases on the first GPU: {ingest + K1, all-gather of the rows, compare,
 * gather + sort of the edges}; *variant_used = the filter all shards ended up with. */
int scema_multi_last_ms(scema_multi *m, double ms[4], int *variant_used);

/* ---- result files: replaces most_similar_histories_to_file (strain2spline.h:301-314) as driven
 *      by FE_problem.h:1232-1235 ("<dir>/last.%u.similar_hist") and mpi_comparison_test.cc:99-103
 *      ("__results/ID_%u.txt"). One file per history of the batch (created even when empty), one
 *      line "<ID> <otherID> <diff>\n" per partner in the reference's single-rank order (partners in
 *      ascending batch index), diff in default ostream formatting (%g). fname_pattern has one %u. */
int scema_write_similar_hist(scema_ctx *ctx, const char *fname_pattern);

/* ---- graph reduction: native replacement of clustering/coarsegrain_dependency_network.py:24-94
 *      (greedy max-degree removal, ties to the node inserted last). mapping_host[num_gps].
 *      scema_reduce_edges uses the last compare's edges in the order the per-history files of
 *      scema_write_similar_hist would be globbed if the directory enumerated in batch order.
 *      scema_reduce_dir reads "<input_folder>/last.*.similar_hist" in readdir order exactly like the
 *      script's glob and writes out_mapping_csv ("<i> <m_i>\n", :88-90); no context needed. */
int scema_reduce_edges(scema_ctx *ctx, uint32_t num_gps, uint32_t *mapping_host, uint64_t *iterations,
                       uint64_t *neighbours_removed);
/* Same reduction for an explicit G.add_edge(cell1[k], cell2[k]) call sequence (:57); no context needed. */
int scema_reduce_calls(const uint32_t *cell1, const uint32_t *cell2, uint64_t n_calls, uint32_t num_gps,
                       uint32_t *mapping_host, uint64_t *iterations, uint64_t *neighbours_removed);
int scema_reduce_dir(const char *input_folder, const char *out_mapping_csv, uint32_t num_gps,
                     uint64_t *iterations, uint64_t *files_read, uint64_t *neighbours_removed);

/* ---- instrumentation ------------------------------------------------------------------------ */
#define SCEMA_T_RESAMPLE 0 /* K1 kernel(s) */
#define SCEMA_T_PREP 1     /* norms + filter-layout copy */
#define SCEMA_T_FILTER 2   /* K2 GEMM-form filter (tcgen05, DMMA or FMA) or the exact all-pairs kernel */
#define SCEMA_T_EXACT 3    /* exact recompute of survivors + K3 compaction */
#define SCEMA_T_SORT 4     /* canonical (a,b) ordering */
#define SCEMA_T_COUNT 8
/* CUDA-event durations (ms) of the phases of the last resample/compare on this context. */
int scema_last_timings(scema_ctx *ctx, float ms[SCEMA_T_COUNT]);
/* Counters of the last compare: [0] pairs evaluated by the filter, [1] survivors recomputed
 * exactly, [2] edges, [3] passes (>1 when a buffer had to grow), [4] tiles, [5] fp16 slices the
 * tcgen05 filter ended up using (SCEMA_PAIRS_TC only), [6] ranges of the host-buffer pipeline of
 * scema_cluster (0: the batch was not pipelined), [7] tiles (256 x 256 pairs; 128 x 256 with SCEMA_TC_CG=1) walked by the norm-band schedule
 * (0: dense schedule). */
int scema_last_counters(scema_ctx *ctx, uint64_t counters[8]);
/* Total kernels launched by this context so far. */
uint64_t scema_kernel_launches(const scema_ctx *ctx);
/* Run-time audit of the filters (environment SCEMA_AUDIT=<samples>, off by default; one-GPU compares): after the
 * compare, <samples> pairs (half random, half between histories of nearby index) are recomputed exactly and every one
 * the reference calls an edge must be in the emitted list, otherwise the compare fails with SCEMA_ERR_STATE.
 * out = {sampled pairs that were edges, of those missing from the list} of the last audited compare. */
int scema_last_audit(scema_ctx *ctx, uint64_t out[2]);
/* Validation hook of SCEMA_PAIRS_TC (tests only; n padded to 256 must be <= 8192): runs the instrumented
 * tcgen05 kernel over the whole pair matrix of the current spline rows. acc_host[row * ld + col] receives
 * every fp32 accumulator (a.b - h_row - h_col in the scaled units of the operands; slices = 2: all three
 * sliced products, slices = 1: a_hi.b_hi only, with the wider guard band folded in), operand_a_host /
 * operand_b_host (n_pad * 256 bytes each, may be NULL) the fp16 operand copies as they sit in memory:
 * blocks of 128 rows, each [hi slice | lo slice] of 128 rows x 128 bytes, 16-byte chunk c of row r
 * stored at chunk c ^ (r & 7). slices = 3: the projected filter (16 <= k <= 60); the operand copies are then
 * n_pad * 32 bytes each: blocks of 128 rows x 32 bytes, 16 fp16 per row (11 basis coordinates, the residual norm,
 * 4 fold columns), 16-byte chunk c of row r stored at chunk c ^ ((r >> 2) & 1). */
int scema_tc_debug(scema_ctx *ctx, double threshold, uint32_t slices, float *acc_host, uint64_t ld,
                   void *operand_a_host, void *operand_b_host);
/* The column means the tcgen05 filter subtracted from its operand copies (centre_host[k], k = columns of the rows;
 * the exact recompute never sees them). Valid after a compare / scema_tc_debug that built the copies. */
int scema_tc_centre(scema_ctx *ctx, double *centre_host);
/* Survivor-density sample behind the last automatic choice of the filter: plan = {pairs of the sample that would
 * survive the one-slice filter, the two-slice filter (centred copies), the same two with raw copies, the DMMA filter,
 * sample size}. */
int scema_tc_last_plan(scema_ctx *ctx, uint64_t plan[6]);
/* The choice itself as host logic (no device needed): given those five counts for `pairs` pairs of rows of k columns and
 * the bytes a survivor queue may take, *choice = 1 / 2 (tcgen05 filter with that many fp16 slices), 0 (SCEMA_PAIRS_DMMA)
 * or -1 (SCEMA_PAIRS_EXACT), *centred = whether the tcgen05 copies are centred, *est_survivors = queue entries expected. */
int scema_tc_choose(uint64_t pairs, uint32_t k, const uint64_t counts[5], uint64_t sample, uint64_t mem_budget, int *choice,
                    int *centred, uint64_t *est_survivors);
/* The same with a sixth count, the pairs of the sample that would survive the projected filter (16-column copies:
 * coordinates in a basis of the sample's leading principal directions plus the residual norm); *choice = 3 selects it. */
int scema_tc_choose_projected(uint64_t pairs, uint32_t k, const uint64_t counts[6], uint64_t sample, uint64_t mem_budget,
                              int *choice, int *centred, uint64_t *est_survivors);
/* The projected filter's basis as host logic: from the second moments moments[k * k] of the centred sample, 11 orthonormal
 * rows basis[11 * 60] (row-major, zero beyond k) and *delta = |B B^T - I|_F. SCEMA_ERR_INVALID when k is outside
 * [16, 60], the moments are not finite or delta exceeds 2^-32 (the filter then keeps its 64-column copies). */
int scema_tc_basis(const double *moments, uint32_t k, double *basis, double *delta);
/* The projected filter in the last automatic choice: out = {pairs of the survivor-density sample that would survive it,
 * 1 if the operand copies are the projected ones}. */
int scema_tc_last_projection(scema_ctx *ctx, uint64_t out[2]);
/* Ranges of histories the host-buffer pipeline of scema_cluster would use for a batch of n (host logic only):
 * bounds[0] = 0 < ... < bounds[*n_ranges] = n, at most 16 ranges, every inner boundary a multiple of 2048. */
int scema_pipeline_plan(uint64_t n, uint64_t *bounds, uint32_t cap, uint32_t *n_ranges);
/* Shared-memory plan the tcgen05 filter would use for rows of k columns (host logic only, no device needed):
 * plan = {chunks of 64 columns, bytes per A buffer, A buffers, log2(B stages), bytes per B stage, bytes used}.
 * SCEMA_ERR_INVALID when the variant does not take such rows (more than 10 chunks, or two slices on wide rows). */
int scema_tc_plan(uint32_t k, uint32_t slices, uint32_t cta_group, uint32_t plan[6]);
/* Measurement hook of K1 (process-wide, no device needed; the results never depend on it): which streamed resample kernel
 * runs (1 = two chains per lane, the default; 0 = one), the resident warps per SM its launches are sized for (ragged batch /
 * history store; 0 = the library's default) and the memory-behaviour flags of the two-chain kernel (y prefetch whole history /
 * none / windows = 0 / 1 / 2, +4 = evict_first on the y copies, +8 = evict_last on the z stores; -2 = chosen per launch, the
 * default). A negative argument (-1) leaves that setting as it is. The same settings come from SCEMA_K1_KERNEL=pair|stream,
 * SCEMA_K1_WPS and SCEMA_K1_FLAGS when the library is loaded. */
int scema_k1_tune(int kernel, int warps_per_sm_ragged, int warps_per_sm_store, int flags);
/* Measured FP64 issue rates on the context's device (TFLOP/s): out[0] DFMA, out[1] DMMA m8n8k4. */
int scema_fp64_peak(scema_ctx *ctx, double out[2]);

#ifdef __cplusplus
}
#endif
#endif /* SCEMA_HIST_H */
