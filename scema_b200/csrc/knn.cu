// scema_knn — exact k nearest neighbours of every history of the spline matrix (sm_100a), DESIGN.md "k-NN query".
//
// A row is final once a round has found every partner below a radius tau and at least k of them: every partner it did
// not see lies at tau or beyond (or at NaN), so its k best are among those found, ties at the k-th distance included.
// Round 1 runs the ordinary thresholded compare over all rows at a radius taken from a distance sample; rounds 2..
// KNN_MAX_ROUNDS re-run it only for the rows still open (gathered to the front of a scratch copy, so that the row panels
// [0, ceil(|U| / 2048)) hold every pair involving them) at a larger radius. The filter is conservative and every
// survivor is recomputed exactly, so the edge sets are exactly {d < tau}. Whatever is left — and every row when n is
// small, the variant is SCEMA_PAIRS_EXACT, or a round would produce too many edges — goes through k_knn_exact, which
// evaluates the open rows against all n rows. The rounds run on a private child context so that the caller's compare
// results, timings and operand caches stay untouched.
//
// scema_query_knn runs the same rounds for the rows of a second set (the queries) against the matrix: every round samples
// the open queries against the subset, stacks [open queries; matrix] on a private child context, and compares the prefix
// panels [0, ceil(|U| / 2048)), which hold every query x matrix pair; only those entries count. scema_query_compare is
// one such compare at the caller's threshold, with the cross edges compacted out of the prefix's list (DESIGN.md "Cross
// query").
//
// Order of the k slots: (diff, ID, index) ascending; non-negative doubles order as their bit patterns, so a slot is
// keyed by (bits, ID, index) and every kernel below keeps the k smallest keys under that total order — the result does
// not depend on the order in which candidates arrive.
#include "common.cuh"
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_partition.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#include <algorithm>
#include <cmath>

namespace scema {

// Constants of the query (DESIGN.md "k-NN query" gives the reasons).
constexpr uint32_t KNN_SAMPLE_ROWS = 8192;       // random subset whose pair distances set the radius of round 1
constexpr uint32_t KNN_SAMPLE_OPEN = 1024;       // open rows sampled against that subset for the radius of later rounds
constexpr double KNN_QUANTILE_C = 2.0;           // radius: the sampled fraction below it reaches C * k / (n - 1)
constexpr uint64_t KNN_QUANTILE_MIN = 16;        // ... and at least this many sampled distances lie below it
constexpr int KNN_MAX_ROUNDS = 4;                // filter rounds at most
constexpr double KNN_EXACT_PAIRS = 2147483648.0; // |U| * n at or below this: the open rows go to k_knn_exact
constexpr double KNN_QUERY_EXACT_PAIRS = 268435456.0;  // scema_query_knn: open queries * n at or below this go to k_knn_exact
constexpr double KNN_EDGE_BUDGET = 8.0;          // a round whose estimated edges exceed this * n * k (+ 2^20) is not run
constexpr uint64_t KNN_MIN_N = 2048;             // fewer rows (one panel): k_knn_exact for all of them
constexpr uint64_t KNN_SEED = 0x6b6e6e5eedull;   // seed of the subset

constexpr unsigned long long KNN_NONE = ~0ull;   // key of an empty slot (above +inf and every NaN bit pattern)

// ------------------------------------------------------------------------------------------------
// warp-wide top-k list (k <= 32): lane l holds the l-th smallest key so far; empty slots hold KNN_NONE
// ------------------------------------------------------------------------------------------------
struct TopK {
    unsigned long long b = KNN_NONE;  // distance bits
    uint32_t id = 0xffffffffu, ix = 0xffffffffu;
};

__device__ __forceinline__ bool key_less(unsigned long long b1, uint32_t id1, uint32_t ix1, unsigned long long b2, uint32_t id2,
                                         uint32_t ix2)
{
    if (b1 != b2) return b1 < b2;
    if (id1 != id2) return id1 < id2;
    return ix1 < ix2;
}

// Offer one candidate per lane (valid lanes only). A candidate is first compared with the current k-th key; the few that
// beat it are inserted one at a time (shift up behind the insertion point). All 32 lanes must call.
__device__ __forceinline__ void topk_offer(TopK &t, uint32_t k, bool valid, unsigned long long b, uint32_t id, uint32_t ix)
{
    const int lane = threadIdx.x & 31;
    unsigned long long wb = __shfl_sync(0xffffffffu, t.b, k - 1);
    uint32_t wid = __shfl_sync(0xffffffffu, t.id, k - 1), wix = __shfl_sync(0xffffffffu, t.ix, k - 1);
    unsigned m = __ballot_sync(0xffffffffu, valid && key_less(b, id, ix, wb, wid, wix));
    while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const unsigned long long cb = __shfl_sync(0xffffffffu, b, src);
        const uint32_t cid = __shfl_sync(0xffffffffu, id, src), cix = __shfl_sync(0xffffffffu, ix, src);
        if (!key_less(cb, cid, cix, wb, wid, wix)) continue;  // an earlier insertion raised the bar (warp-uniform)
        const unsigned before = __ballot_sync(0xffffffffu, (uint32_t)lane < k && key_less(t.b, t.id, t.ix, cb, cid, cix));
        const int pos = __popc(before);
        const unsigned long long ub = __shfl_up_sync(0xffffffffu, t.b, 1);
        const uint32_t uid = __shfl_up_sync(0xffffffffu, t.id, 1), uix = __shfl_up_sync(0xffffffffu, t.ix, 1);
        if (lane > pos && (uint32_t)lane < k) { t.b = ub; t.id = uid; t.ix = uix; }
        if (lane == pos) { t.b = cb; t.id = cid; t.ix = cix; }
        wb = __shfl_sync(0xffffffffu, t.b, k - 1);
        wid = __shfl_sync(0xffffffffu, t.id, k - 1);
        wix = __shfl_sync(0xffffffffu, t.ix, k - 1);
    }
}

// ------------------------------------------------------------------------------------------------
// k_knn_exact: the query rows Q[q_rows[0, nq)] against the columns S[0, n) of segment blockIdx.y, one query row per warp,
// tiles of 64 columns (two per lane) staged through shared memory in slices of 32 of the K entries, sums in the
// reference's order (k_exact_all's arithmetic; a - b and b - a round to the same magnitude). Writes each (query,
// segment)'s k best. self: Q == S and a query row is not its own neighbour (scema_knn); 0: a second set (scema_query_knn).
// ------------------------------------------------------------------------------------------------
constexpr int KQ = 8, KCOL = 64, KKC = 32;
__global__ void __launch_bounds__(256, 4) k_knn_exact(const double *__restrict__ S, uint64_t n, uint32_t K, const uint32_t *__restrict__ ids,
                                                   const double *__restrict__ Q, const uint32_t *__restrict__ q_rows, uint32_t nq, int self,
                                                   uint64_t seg_len, uint32_t k, unsigned long long *__restrict__ part_b,
                                                   uint32_t *__restrict__ part_ix)
{
    __shared__ double Qs[KQ][KKC];
    __shared__ double Cs[KCOL][KKC + 1];
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const uint32_t qp = blockIdx.x * KQ + w;
    const bool have_q = qp < nq;
    const uint32_t qrow = have_q && self ? q_rows[qp] : 0xffffffffu;  // n < 2^32 - 1: no column has this index
    const uint64_t c_begin = (uint64_t)blockIdx.y * seg_len, c_end = n < c_begin + seg_len ? n : c_begin + seg_len;
    TopK t;
    for (uint64_t c0 = c_begin; c0 < c_end; c0 += KCOL) {
        double s0 = 0.0, s1 = 0.0;
        for (uint32_t k0 = 0; k0 < K; k0 += KKC) {
            const uint32_t kn = K - k0 < (uint32_t)KKC ? K - k0 : (uint32_t)KKC;
            __syncthreads();
            {
                const int r = tid / KKC, kk = tid - r * KKC;  // KQ * KKC == 256: one entry per thread
                const uint32_t q = blockIdx.x * KQ + r;
                Qs[r][kk] = (q < nq && (uint32_t)kk < kn) ? Q[(uint64_t)q_rows[q] * K + k0 + kk] : 0.0;
            }
            for (int e = tid; e < KCOL * KKC; e += 256) {
                const int r = e / KKC, kk = e - r * KKC;
                Cs[r][kk] = (c0 + r < c_end && (uint32_t)kk < kn) ? S[(c0 + r) * K + k0 + kk] : 0.0;
            }
            __syncthreads();
            for (uint32_t kk = 0; kk < kn; kk++) {
                const double q = Qs[w][kk];
                const double d0 = __dsub_rn(q, Cs[lane][kk]), d1 = __dsub_rn(q, Cs[lane + 32][kk]);
                s0 = __dadd_rn(s0, __dmul_rn(d0, d0));
                s1 = __dadd_rn(s1, __dmul_rn(d1, d1));
            }
        }
        const double e0 = __dsqrt_rn(s0), e1 = __dsqrt_rn(s1);
        const uint64_t col0 = c0 + lane, col1 = col0 + 32;
        const bool v0 = have_q && col0 < c_end && (uint32_t)col0 != qrow && e0 == e0;  // NaN partners are skipped
        const bool v1 = have_q && col1 < c_end && (uint32_t)col1 != qrow && e1 == e1;
        topk_offer(t, k, v0, (unsigned long long)__double_as_longlong(e0), v0 ? ids[col0] : 0u, (uint32_t)col0);
        topk_offer(t, k, v1, (unsigned long long)__double_as_longlong(e1), v1 ? ids[col1] : 0u, (uint32_t)col1);
    }
    if (have_q && (uint32_t)lane < k) {
        const uint64_t o = ((uint64_t)qp * gridDim.y + blockIdx.y) * k + lane;
        part_b[o] = t.b;
        part_ix[o] = t.ix;
    }
}

// ------------------------------------------------------------------------------------------------
// k_knn_topk: the k best of candidate lists, one list per warp.
//   offs != nullptr (selection after a filter round): the list of open row `row` is the entries [offs[row], offs[row+1]);
//     rows with fewer than k entries stay open, the others are written and closed.
//   offs == nullptr (merge of k_knn_exact's segments): list p is [p * stride, (p + 1) * stride), always written.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_knn_topk(const unsigned long long *__restrict__ eb, const uint32_t *__restrict__ eix,
                                                  const uint32_t *__restrict__ ids, const uint32_t *__restrict__ rows, uint64_t n_lists,
                                                  const unsigned long long *__restrict__ offs, uint64_t stride, uint32_t k,
                                                  uint8_t *__restrict__ open, unsigned long long *__restrict__ closed,
                                                  uint32_t *__restrict__ out_ix, double *__restrict__ out_d)
{
    const uint64_t p = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (p >= n_lists) return;  // warp-uniform
    const uint64_t row = rows ? rows[p] : p;
    uint64_t beg, end;
    if (offs) {
        if (!open[row]) return;
        beg = offs[row];
        end = offs[row + 1];
        if (end - beg < k) return;
    } else {
        beg = p * stride;
        end = beg + stride;
    }
    TopK t;
    for (uint64_t e0 = beg; e0 < end; e0 += 32) {
        const uint64_t e = e0 + lane;
        const unsigned long long b = e < end ? eb[e] : KNN_NONE;
        const bool valid = b != KNN_NONE;
        const uint32_t ix = valid ? eix[e] : 0xffffffffu;
        topk_offer(t, k, valid, b, valid ? ids[ix] : 0u, ix);
    }
    if ((uint32_t)lane < k) {
        out_ix[row * k + lane] = t.ix;
        out_d[row * k + lane] = t.b == KNN_NONE ? __longlong_as_double(0x7ff0000000000000ll) : __longlong_as_double((long long)t.b);
    }
    if (offs && lane == 0) {
        open[row] = 0;
        atomicAdd(closed, 1ull);
    }
}

// Directed entries of a round's edges (a < b, indices into the round's matrix; perm maps them to rows of the caller's
// matrix, nullptr = identity) for the rows that are still open. PASS 0 counts per row, PASS 1 scatters (cursor = offsets).
// cross > 0 (scema_query_knn): the round's matrix is [open queries; retained rows] with `cross` queries in front; only the
// query -> retained entries (a < cross <= b) count, as (perm[a], b - cross).
template <int PASS>
__global__ void __launch_bounds__(256) k_knn_expand(const uint64_t *__restrict__ keys, const double *__restrict__ vals, uint64_t m,
                                                    uint32_t key_shift, const uint32_t *__restrict__ perm, uint64_t cross,
                                                    const uint8_t *__restrict__ open, unsigned long long *__restrict__ cnt_or_cursor,
                                                    unsigned long long *__restrict__ eb, uint32_t *__restrict__ eix)
{
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const uint64_t key = keys[e];
    uint32_t a = (uint32_t)(key >> key_shift), b = (uint32_t)(key & ((1ull << key_shift) - 1));
    const unsigned long long bits = (unsigned long long)__double_as_longlong(vals[e]);
    if (cross) {
        if (!(a < cross && b >= cross)) return;
        const uint32_t q = perm[a];
        if (open[q]) {
            const unsigned long long o = atomicAdd(cnt_or_cursor + q, 1ull);
            if (PASS == 1) { eb[o] = bits; eix[o] = b - (uint32_t)cross; }
        }
        return;
    }
    if (perm) { a = perm[a]; b = perm[b]; }
    if (open[a]) {
        const unsigned long long o = atomicAdd(cnt_or_cursor + a, 1ull);
        if (PASS == 1) { eb[o] = bits; eix[o] = b; }
    }
    if (open[b]) {
        const unsigned long long o = atomicAdd(cnt_or_cursor + b, 1ull);
        if (PASS == 1) { eb[o] = bits; eix[o] = a; }
    }
}

// Distance sample: rows A (SA[rows_a[a * a_span / na]], a < na) against rows B (S[rows_b[b]]); tri: only b > a (A == B).
// Same-row pairs (unless cross: A is another set than B) and NaN distances are left out. Bits appended with one atomic
// per warp.
__global__ void __launch_bounds__(256) k_knn_sample(const double *__restrict__ S, const double *__restrict__ SA, int cross, uint32_t K,
                                                    const uint32_t *__restrict__ rows_a, uint32_t na, uint64_t a_span,
                                                    const uint32_t *__restrict__ rows_b, uint32_t nb, int tri,
                                                    unsigned long long *__restrict__ out, unsigned long long *__restrict__ count)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t a = (uint32_t)(t / nb), b = (uint32_t)(t - (uint64_t)a * nb);
    bool keep = false;
    unsigned long long bits = 0;
    if (a < na && !(tri && b <= a)) {
        const uint32_t i = rows_a[(uint64_t)a * a_span / na], j = rows_b[b];
        if (cross || i != j) {
            const double d = exact_l2(SA + (uint64_t)i * K, S + (uint64_t)j * K, K);
            keep = d == d;
            bits = (unsigned long long)__double_as_longlong(d);
        }
    }
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (!m) return;
    const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(count, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (keep) out[base + __popc(m & ((1u << lane) - 1))] = bits;
}

// sorted[0, count): out[0] = entries below `bits`
__global__ void k_knn_count_below(const unsigned long long *__restrict__ sorted, uint64_t count, unsigned long long bits,
                                  unsigned long long *__restrict__ out)
{
    uint64_t lo = 0, hi = count;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (sorted[mid] < bits) lo = mid + 1; else hi = mid;
    }
    out[0] = lo;
}

// scratch copy of the rows in the order perm (open rows first)
__global__ void __launch_bounds__(256) k_knn_gather(const double *__restrict__ S, uint64_t n, uint32_t K, const uint32_t *__restrict__ perm,
                                                    double *__restrict__ out)
{
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * K) return;
    const uint64_t r = e / K, c = e - r * K;
    out[e] = S[(uint64_t)perm[r] * K + c];
}

// ------------------------------------------------------------------------------------------------
// scema_query_compare: the cross edges of a [Q; R] prefix compare. The child's sorted edges (a, b), a < b, of the stacked
// matrix are kept when a < m <= b (query a, retained row b - m), in order, so the list stays sorted by (j, i).
// flag[ne] = 0 so that the exclusive sum's last entry is the number kept.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_query_flag(const uint64_t *__restrict__ keys, uint64_t ne, uint32_t key_shift, uint64_t m,
                                                    unsigned long long *__restrict__ flag)
{
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e > ne) return;
    if (e == ne) { flag[e] = 0; return; }
    const uint64_t key = keys[e];
    const uint64_t a = key >> key_shift, b = key & ((1ull << key_shift) - 1);
    flag[e] = a < m && b >= m;
}

__global__ void __launch_bounds__(256) k_query_scatter(const uint64_t *__restrict__ keys, const double *__restrict__ vals, uint64_t ne,
                                                       uint32_t key_shift, uint64_t m, const unsigned long long *__restrict__ flag,
                                                       const unsigned long long *__restrict__ pos, uint32_t *__restrict__ out_j,
                                                       uint32_t *__restrict__ out_i, double *__restrict__ out_d)
{
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ne || !flag[e]) return;
    const uint64_t key = keys[e], o = pos[e];
    out_j[o] = (uint32_t)(key >> key_shift);
    out_i[o] = (uint32_t)((key & ((1ull << key_shift) - 1)) - m);
    out_d[o] = vals[e];
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
namespace {

enum { B_IDS, B_OPEN, B_PERM, B_OUT_IX, B_OUT_D, B_SUBSET, B_SAMPLE, B_TMP, B_MISC, B_CNT, B_EB, B_EIX, B_ROWS, B_PART_B, B_PART_IX, B_Q };

// Phases of the query calls, timed with the context's query events (the compare events belong to the last compare).
enum { QT_COPY, QT_PREP, QT_FILTER, QT_EXACT, QT_SORT, QT_SELECT, QT_TOPK };

// Events around a stretch of work on the caller's stream, folded into query_ms[which] (host-synchronising); on = false
// (scema_knn, which reports no phases) records nothing.
struct QTimer {
    scema_ctx *c;
    int which;
    bool on;
    QTimer(scema_ctx *ctx, int w, bool on_) : c(ctx), which(w), on(on_) { if (on) cudaEventRecord(c->query_ev[0], c->stream); }
    void stop()
    {
        if (!on) return;
        cudaEventRecord(c->query_ev[1], c->stream);
        float t = 0.f;
        if (cudaEventSynchronize(c->query_ev[1]) == cudaSuccess && cudaEventElapsedTime(&t, c->query_ev[0], c->query_ev[1]) == cudaSuccess)
            c->query_ms[which] += t;
        else
            cudaGetLastError();
    }
};

// Seeded stratified subset: one row from each of S equal slices of [0, n).
void make_subset(uint64_t n, std::vector<uint32_t> &out)
{
    const uint64_t s = std::min<uint64_t>(n, KNN_SAMPLE_ROWS);
    out.resize(s);
    for (uint64_t i = 0; i < s; i++) {
        uint64_t z = KNN_SEED + 0x9e3779b97f4a7c15ull * (i + 1);
        z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
        z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
        z ^= z >> 31;
        const uint64_t lo = i * n / s, hi = (i + 1) * n / s;
        out[i] = (uint32_t)(lo + z % (hi - lo));
    }
}

// The k nearest of `rows` listed rows among the n rows of the caller's matrix. scema_knn: the listed rows are the matrix
// itself (Q == nullptr) and a row is not its own neighbour. scema_query_knn: Q holds `rows` query rows of a second set,
// and every one of the n rows is a candidate.
struct Knn {
    scema_ctx *c;           // the caller's context: its stream, its rows, its scratch buffers
    uint64_t n;             // rows of the caller's matrix: the candidate partners
    uint64_t rows;          // rows whose neighbours are listed (n for scema_knn)
    const double *Q = nullptr;
    uint32_t K, k;
    uint64_t open_n;        // rows still open
    std::vector<uint32_t> subset;
    uint64_t stats[11] = {};
    double radii[8] = {};

    template <class T> T *buf(int b) { return c->knn_buf[b].as<T>(); }
    int reserve(int b, size_t bytes)
    {
        SCEMA_CUDA(c, c->knn_buf[b].reserve(std::max<size_t>(bytes, 256)));
        return SCEMA_OK;
    }
    unsigned long long *misc() { return buf<unsigned long long>(B_MISC); }
    int read_misc(uint64_t *out, int count)
    {
        SCEMA_CUDA(c, cudaMemcpyAsync(out, misc(), count * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
        SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));
        return SCEMA_OK;
    }
    uint64_t partners() const { return Q ? n : n - 1; }

    // buffers, IDs of the candidate rows, every listed row open
    int begin()
    {
        int rc;
        if ((rc = reserve(B_IDS, n * sizeof(uint32_t))) || (rc = reserve(B_OPEN, rows)) || (rc = reserve(B_PERM, rows * sizeof(uint32_t))) ||
            (rc = reserve(B_OUT_IX, rows * k * sizeof(uint32_t))) || (rc = reserve(B_OUT_D, rows * k * sizeof(double))) ||
            (rc = reserve(B_MISC, 8 * sizeof(uint64_t))))
            return rc;
        SCEMA_CUDA(c, cudaMemcpyAsync(buf<void>(B_IDS), ids_of(c).data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        SCEMA_CUDA(c, cudaMemsetAsync(buf<void>(B_OPEN), 1, rows, c->stream));
        open_n = rows;
        return SCEMA_OK;
    }

    // open rows first in B_PERM; returns their number in open_n
    int partition()
    {
        size_t tmp = 0;
        cub::CountingInputIterator<uint32_t> iota(0);
        SCEMA_CUDA(c, cub::DevicePartition::Flagged(nullptr, tmp, iota, buf<uint8_t>(B_OPEN), buf<uint32_t>(B_PERM), misc() + 1, (int64_t)rows,
                                                    c->stream));
        int rc = reserve(B_TMP, tmp);
        if (rc) return rc;
        SCEMA_CUDA(c, cub::DevicePartition::Flagged(buf<void>(B_TMP), tmp, iota, buf<uint8_t>(B_OPEN), buf<uint32_t>(B_PERM), misc() + 1,
                                                    (int64_t)rows, c->stream));
        c->launches += 2;
        uint64_t m[2];
        rc = read_misc(m, 2);
        if (rc) return rc;
        open_n = m[1];
        return SCEMA_OK;
    }

    // Radius from a distance sample: A rows against the subset (round 1 of scema_knn: the subset's own pairs). tau = the
    // smallest value with at least max(C * k / partners * count, KNN_QUANTILE_MIN) sampled distances strictly below it;
    // *frac_below = the sampled fraction below max(tau, floor). +inf (or 0 sampled distances) when no such value exists.
    int radius(const uint32_t *rows_a, uint32_t na, uint64_t a_span, bool tri, double floor_tau, double *tau, double *frac_below)
    {
        const uint32_t nb = (uint32_t)subset.size();
        const uint64_t total = (uint64_t)na * nb;
        int rc = reserve(B_SAMPLE, 2 * total * sizeof(unsigned long long));
        if (rc) return rc;
        unsigned long long *s0 = buf<unsigned long long>(B_SAMPLE), *s1 = s0 + total;
        SCEMA_CUDA(c, cudaMemsetAsync(misc(), 0, 4 * sizeof(uint64_t), c->stream));
        k_knn_sample<<<(unsigned)((total + 255) / 256), 256, 0, c->stream>>>(c->d_spline, Q ? Q : c->d_spline, Q ? 1 : 0, K, rows_a, na,
                                                                           a_span, buf<uint32_t>(B_SUBSET), nb, tri ? 1 : 0, s0, misc());
        c->launches++;
        SCEMA_CUDA(c, cudaGetLastError());
        uint64_t count = 0;
        rc = read_misc(&count, 1);
        if (rc) return rc;
        *tau = INFINITY;
        *frac_below = 1.0;
        if (count == 0) return SCEMA_OK;
        cub::DoubleBuffer<unsigned long long> db(s0, s1);
        size_t tmp = 0;
        SCEMA_CUDA(c, cub::DeviceRadixSort::SortKeys(nullptr, tmp, db, (int64_t)count, 0, 64, c->stream));
        rc = reserve(B_TMP, tmp);
        if (rc) return rc;
        SCEMA_CUDA(c, cub::DeviceRadixSort::SortKeys(buf<void>(B_TMP), tmp, db, (int64_t)count, 0, 64, c->stream));
        c->launches += 17;
        const double want = std::ceil(KNN_QUANTILE_C * k / (double)partners() * (double)count);
        const uint64_t m = std::max<uint64_t>(KNN_QUANTILE_MIN, (uint64_t)std::min<double>(want, 1e18));
        if (m > count) return SCEMA_OK;
        double v = 0.0;
        SCEMA_CUDA(c, cudaMemcpyAsync(&v, db.Current() + (m - 1), sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));
        double t = std::max(floor_tau, std::nextafter(v, INFINITY));
        if (!(t < INFINITY)) return SCEMA_OK;
        unsigned long long tb;
        memcpy(&tb, &t, sizeof tb);
        k_knn_count_below<<<1, 1, 0, c->stream>>>(db.Current(), count, tb, misc() + 2);
        c->launches++;
        SCEMA_CUDA(c, cudaGetLastError());
        uint64_t below[3];
        rc = read_misc(below, 3);
        if (rc) return rc;
        *tau = t;
        *frac_below = (double)below[2] / (double)count;
        return SCEMA_OK;
    }

    // Close every open row that has at least k entries among the edges the child context holds (its matrix is the
    // caller's rows in the order perm, nullptr = identity; with cross > 0 the first `cross` rows are the open queries in
    // the order perm, then the caller's rows). Returns the rows closed.
    int select(scema_ctx *child, const uint32_t *perm, uint64_t cross, uint64_t *closed)
    {
        const uint64_t m = child->n_edges;
        *closed = 0;
        if (m == 0) return SCEMA_OK;
        const uint64_t *keys = child->d_edge_key[child->edge_cur].as<uint64_t>();
        const double *vals = child->d_edge_val[child->edge_cur].as<double>();
        int rc = reserve(B_CNT, 2 * (rows + 1) * sizeof(unsigned long long));
        if (!rc) rc = reserve(B_EB, 2 * m * sizeof(unsigned long long));
        if (!rc) rc = reserve(B_EIX, 2 * m * sizeof(uint32_t));
        if (rc) return rc;
        unsigned long long *cnt = buf<unsigned long long>(B_CNT), *offs = cnt + (rows + 1);
        SCEMA_CUDA(c, cudaMemsetAsync(cnt, 0, (rows + 1) * sizeof(unsigned long long), c->stream));
        const unsigned g = (unsigned)((m + 255) / 256);
        k_knn_expand<0><<<g, 256, 0, c->stream>>>(keys, vals, m, child->key_shift, perm, cross, buf<uint8_t>(B_OPEN), cnt, nullptr, nullptr);
        size_t tmp = 0;
        SCEMA_CUDA(c, cub::DeviceScan::ExclusiveSum(nullptr, tmp, cnt, offs, (int64_t)(rows + 1), c->stream));
        rc = reserve(B_TMP, tmp);
        if (rc) return rc;
        SCEMA_CUDA(c, cub::DeviceScan::ExclusiveSum(buf<void>(B_TMP), tmp, cnt, offs, (int64_t)(rows + 1), c->stream));
        SCEMA_CUDA(c, cudaMemcpyAsync(cnt, offs, (rows + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
        k_knn_expand<1><<<g, 256, 0, c->stream>>>(keys, vals, m, child->key_shift, perm, cross, buf<uint8_t>(B_OPEN), cnt,
                                                 buf<unsigned long long>(B_EB), buf<uint32_t>(B_EIX));
        SCEMA_CUDA(c, cudaMemsetAsync(misc() + 3, 0, sizeof(uint64_t), c->stream));
        k_knn_topk<<<(unsigned)((rows + 7) / 8), 256, 0, c->stream>>>(buf<unsigned long long>(B_EB), buf<uint32_t>(B_EIX), buf<uint32_t>(B_IDS),
                                                                      nullptr, rows, offs, 0, k, buf<uint8_t>(B_OPEN), misc() + 3,
                                                                      buf<uint32_t>(B_OUT_IX), buf<double>(B_OUT_D));
        c->launches += 5;
        SCEMA_CUDA(c, cudaGetLastError());
        uint64_t got[4];
        rc = read_misc(got, 4);
        if (rc) return rc;
        *closed = got[3];
        return SCEMA_OK;
    }

    // k_knn_exact for the open rows (the first open_n entries of B_PERM after partition()), then the merge
    int exact()
    {
        const uint64_t nq = open_n;
        if (nq == 0) return SCEMA_OK;
        const uint64_t qblocks = (nq + KQ - 1) / KQ;
        // enough blocks to fill the GPU when few rows are left: the columns are cut into segments of >= 1024
        uint64_t nseg = std::max<uint64_t>(1, (4ull * c->sm_count + qblocks - 1) / qblocks);
        nseg = std::min<uint64_t>({nseg, std::max<uint64_t>(1, n / 1024), 65535});
        const uint64_t seg_len = ((n + nseg - 1) / nseg + KCOL - 1) / KCOL * KCOL;
        nseg = (n + seg_len - 1) / seg_len;
        int rc = reserve(B_PART_B, nq * nseg * k * sizeof(unsigned long long));
        if (!rc) rc = reserve(B_PART_IX, nq * nseg * k * sizeof(uint32_t));
        if (rc) return rc;
        k_knn_exact<<<dim3((unsigned)qblocks, (unsigned)nseg), 256, 0, c->stream>>>(c->d_spline, n, K, buf<uint32_t>(B_IDS), Q ? Q : c->d_spline,
                                                                                    buf<uint32_t>(B_PERM), (uint32_t)nq, Q ? 0 : 1, seg_len, k,
                                                                                    buf<unsigned long long>(B_PART_B), buf<uint32_t>(B_PART_IX));
        k_knn_topk<<<(unsigned)((nq + 7) / 8), 256, 0, c->stream>>>(buf<unsigned long long>(B_PART_B), buf<uint32_t>(B_PART_IX),
                                                                    buf<uint32_t>(B_IDS), buf<uint32_t>(B_PERM), nq, nullptr, nseg * k, k,
                                                                    nullptr, nullptr, buf<uint32_t>(B_OUT_IX), buf<double>(B_OUT_D));
        c->launches += 2;
        SCEMA_CUDA(c, cudaGetLastError());
        stats[3] += nq;
        stats[4] += nq * partners();
        return SCEMA_OK;
    }

    // Filter rounds on the private context `child`. Round 1 of scema_knn compares all rows at a radius from the subset's
    // own pairs. Every other round (all rounds of scema_query_knn) samples the open rows against the subset, gathers them
    // to the front of a scratch matrix — [open rows; the others] or [open queries; the caller's rows] — and compares the
    // prefix panels that hold every pair involving them.
    int rounds(scema_ctx *child, int variant)
    {
        make_subset(n, subset);
        int rc = reserve(B_SUBSET, subset.size() * sizeof(uint32_t));
        if (rc) return rc;
        SCEMA_CUDA(c, cudaMemcpyAsync(buf<void>(B_SUBSET), subset.data(), subset.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        if (Q && (rc = partition())) return rc;  // B_PERM = the queries in order
        const double budget = KNN_EDGE_BUDGET * (double)rows * k + 1048576.0;
        double tau_prev = 0.0;
        for (int round = 1; round <= KNN_MAX_ROUNDS && open_n > 0; round++) {
            if (Q ? (double)open_n * (double)n <= KNN_QUERY_EXACT_PAIRS : (round > 1 && (double)open_n * (double)n <= KNN_EXACT_PAIRS)) break;
            double tau = 0.0, frac = 1.0, pairs = 0.0;
            uint32_t p1 = 0;
            if (round == 1 && !Q) {
                rc = radius(buf<uint32_t>(B_SUBSET), (uint32_t)subset.size(), subset.size(), true, 0.0, &tau, &frac);
                pairs = 0.5 * (double)n * (double)(n - 1);
            } else {
                const uint32_t na = (uint32_t)std::min<uint64_t>(open_n, KNN_SAMPLE_OPEN);
                rc = radius(buf<uint32_t>(B_PERM), na, open_n, false, 2.0 * tau_prev, &tau, &frac);
                const uint32_t panel_rows = PANEL_ROWBLOCKS * TILE;
                p1 = (uint32_t)((open_n + panel_rows - 1) / panel_rows);
                const double N = Q ? (double)(open_n + n) : (double)n;
                const double r1 = std::min<double>(N, (double)p1 * panel_rows);
                pairs = r1 * N - 0.5 * r1 * (r1 + 1.0);
            }
            if (rc) return rc;
            if (!(tau < INFINITY) || pairs * frac > budget) break;  // too dense for an O(rows k) edge list: the exact kernel takes over
            const uint32_t *perm = nullptr;
            const uint64_t cross = Q ? open_n : 0;
            if (round == 1 && !Q) {
                rc = scema_set_spline(child, c->d_spline, 1, n, K, nullptr);
            } else {
                QTimer t(c, QT_COPY, Q != nullptr);
                const uint64_t lead = Q ? open_n : n;  // rows gathered through perm
                if ((rc = reserve(B_ROWS, (cross + n) * K * sizeof(double)))) return rc;
                k_knn_gather<<<(unsigned)((lead * K + 255) / 256), 256, 0, c->stream>>>(Q ? Q : c->d_spline, lead, K, buf<uint32_t>(B_PERM),
                                                                                      buf<double>(B_ROWS));
                c->launches++;
                SCEMA_CUDA(c, cudaGetLastError());
                if (Q)
                    SCEMA_CUDA(c, cudaMemcpyAsync(buf<double>(B_ROWS) + cross * K, c->d_spline, n * K * sizeof(double), cudaMemcpyDeviceToDevice,
                                                  c->stream));
                t.stop();
                rc = scema_set_spline(child, buf<double>(B_ROWS), 1, cross + n, K, nullptr);
                perm = buf<uint32_t>(B_PERM);
            }
            if (rc) return fail(c, rc, std::string(Q ? "query_knn: " : "knn: ") + scema_last_error(child));
            int v = variant;
            rc = compare_prefix_run(child, tau, &v, p1, Q != nullptr);
            if (rc) return fail(c, rc, std::string(Q ? "query_knn: " : "knn: ") + scema_last_error(child));
            stats[0]++;
            stats[5] += child->counters[1];
            stats[6] += child->n_edges;
            stats[7] = (uint64_t)v;
            stats[8] += child->counters[0];
            stats[10] += child->counters[3];
            radii[round - 1] = tau;
            tau_prev = tau;
            if (Q) child_timings(child);
            uint64_t closed = 0;
            {
                QTimer t(c, QT_SELECT, Q != nullptr);
                rc = select(child, perm, cross, &closed);
                if (rc) return rc;
                stats[round == 1 ? 1 : 2] += closed;
                rc = partition();  // the open rows to the front: sampled, gathered and queried by what follows
                if (rc) return rc;
                t.stop();
            }
        }
        return SCEMA_OK;
    }

    // the child's phase timings of its last compare, added to the query's
    void child_timings(scema_ctx *child)
    {
        float ms[SCEMA_T_COUNT];
        if (scema_last_timings(child, ms) == SCEMA_OK)
            for (int w = SCEMA_T_PREP; w <= SCEMA_T_SORT; w++) c->query_ms[QT_PREP + (w - SCEMA_T_PREP)] += ms[w];
    }

    // the open rows to the exact kernel, results to the host
    int finish(uint32_t *index_host, double *diff_host)
    {
        int rc = partition();
        if (rc) return rc;
        {
            QTimer t(c, QT_TOPK, Q != nullptr);
            rc = exact();
            if (rc) return rc;
            t.stop();
        }
        if (index_host)
            SCEMA_CUDA(c, cudaMemcpyAsync(index_host, buf<void>(B_OUT_IX), rows * k * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        if (diff_host)
            SCEMA_CUDA(c, cudaMemcpyAsync(diff_host, buf<void>(B_OUT_D), rows * k * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        SCEMA_CUDA(c, cudaStreamSynchronize(c->stream));
        return SCEMA_OK;
    }
};

// private context (same device and stream) for the compares of a query call
int child_of(scema_ctx *ctx, scema_ctx **slot, const char *what)
{
    if (!*slot) {
        scema_ctx *child = nullptr;
        const int rc = scema_create(&child, ctx->device, (void *)ctx->stream);
        if (rc) return fail(ctx, rc, std::string(what) + ": could not create the context of the filter rounds");
        *slot = child;
    }
    return SCEMA_OK;
}

// checks shared by scema_query_compare and scema_query_knn; resets the stats of the last query
int query_check(scema_ctx *ctx, const double *rows, uint64_t m, uint32_t k_cols, int variant, const char *what)
{
    for (int i = 0; i < 11; i++) ctx->query_counts[i] = 0;
    for (int i = 0; i < 8; i++) { ctx->query_radii[i] = 0.0; ctx->query_ms[i] = 0.f; }
    ctx->query_counts[7] = SCEMA_PAIRS_EXACT;
    if (!ctx->have_spline) return fail(ctx, SCEMA_ERR_STATE, "Spline is not up to date.");
    if (k_cols != ctx->K) return fail(ctx, SCEMA_ERR_INVALID, std::string(what) + ": query rows must have as many columns as the spline matrix");
    if (variant < 0 || variant > 3) return fail(ctx, SCEMA_ERR_INVALID, std::string(what) + ": bad variant");
    if (m > 0 && !rows) return fail(ctx, SCEMA_ERR_INVALID, std::string(what) + ": null pointer");
    if (m >= (1ull << 32) || ctx->n + m >= (1ull << 32)) return fail(ctx, SCEMA_ERR_INVALID, std::string(what) + ": n + m must stay below 2^32");
    if (!ctx->query_ev[0]) {
        for (int e = 0; e < 2; e++) SCEMA_CUDA(ctx, cudaEventCreate(&ctx->query_ev[e]));
    }
    return SCEMA_OK;
}

}  // namespace

int knn_run(scema_ctx *ctx, uint32_t k, int variant, uint32_t *index_host, double *diff_host)
{
    for (int i = 0; i < 8; i++) { ctx->knn_counts[i] = 0; ctx->knn_radii[i] = 0.0; }
    if (!ctx->have_spline) return fail(ctx, SCEMA_ERR_STATE, "Spline is not up to date.");
    if (k < 1 || k > 32) return fail(ctx, SCEMA_ERR_INVALID, "knn: k must be in [1, 32]");
    if (variant < 0 || variant > 3) return fail(ctx, SCEMA_ERR_INVALID, "knn: bad variant");
    if (ctx->n >= (1ull << 32)) return fail(ctx, SCEMA_ERR_INVALID, "knn: more than 2^32-1 histories");
    const uint64_t n = ctx->n;
    Knn q;
    q.c = ctx; q.n = n; q.rows = n; q.K = ctx->K; q.k = k;
    q.stats[7] = SCEMA_PAIRS_EXACT;
    if (n <= 1) {
        if (index_host) std::fill(index_host, index_host + n * k, 0xffffffffu);
        if (diff_host) std::fill(diff_host, diff_host + n * k, INFINITY);
        for (int i = 0; i < 8; i++) ctx->knn_counts[i] = q.stats[i];
        ctx->knn_counts[3] = n;
        return SCEMA_OK;
    }
    int rc = wait_rows(ctx);
    if (!rc) rc = q.begin();
    if (rc) return rc;
    if (variant != SCEMA_PAIRS_EXACT && n >= KNN_MIN_N) {
        if ((rc = child_of(ctx, &ctx->knn_child, "knn")) || (rc = q.rounds(ctx->knn_child, variant))) return rc;
    }
    if ((rc = q.finish(index_host, diff_host))) return rc;
    for (int i = 0; i < 8; i++) { ctx->knn_counts[i] = q.stats[i]; ctx->knn_radii[i] = q.radii[i]; }
    return SCEMA_OK;
}

int query_knn_run(scema_ctx *ctx, const double *rows, int rows_on_device, uint64_t m, uint32_t k_cols, uint32_t k, int variant,
                  uint32_t *index_host, double *diff_host)
{
    int rc = query_check(ctx, rows, m, k_cols, variant, "query_knn");
    if (rc) return rc;
    if (k < 1 || k > 32) return fail(ctx, SCEMA_ERR_INVALID, "query_knn: k must be in [1, 32]");
    const uint64_t n = ctx->n;
    if (m == 0) return SCEMA_OK;
    if (n == 0) {
        if (index_host) std::fill(index_host, index_host + m * k, 0xffffffffu);
        if (diff_host) std::fill(diff_host, diff_host + m * k, INFINITY);
        ctx->query_counts[3] = m;
        return SCEMA_OK;
    }
    Knn q;
    q.c = ctx; q.n = n; q.rows = m; q.K = ctx->K; q.k = k;
    q.stats[7] = SCEMA_PAIRS_EXACT;
    if ((rc = wait_rows(ctx))) return rc;
    q.Q = rows;
    if (!rows_on_device) {
        QTimer t(ctx, QT_COPY, true);  // the upload of host queries counts as scratch copy, as in scema_query_compare
        if ((rc = q.reserve(B_Q, m * q.K * sizeof(double)))) return rc;
        SCEMA_CUDA(ctx, cudaMemcpyAsync(q.buf<void>(B_Q), rows, m * q.K * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        t.stop();
        q.Q = q.buf<double>(B_Q);
    }
    if ((rc = q.begin())) return rc;
    if (variant != SCEMA_PAIRS_EXACT) {
        if ((rc = child_of(ctx, &ctx->query_child, "query_knn")) || (rc = q.rounds(ctx->query_child, variant))) return rc;
    }
    if ((rc = q.finish(index_host, diff_host))) return rc;
    for (int i = 0; i < 11; i++) ctx->query_counts[i] = q.stats[i];
    for (int i = 0; i < 8; i++) ctx->query_radii[i] = q.radii[i];
    return SCEMA_OK;
}

// scema_query_compare: [Q; R] on the private context, the prefix panels [0, ceil(m / 2048)) compared (they hold every
// query x retained pair), the cross edges compacted into the context's query buffers.
int query_compare_run(scema_ctx *ctx, const double *rows, int rows_on_device, uint64_t m, uint32_t k_cols, double thr, int variant,
                      uint64_t *n_edges)
{
    ctx->have_query = false;
    ctx->query_n = 0;
    if (n_edges) *n_edges = 0;
    int rc = query_check(ctx, rows, m, k_cols, variant, "query_compare");
    if (rc) return rc;
    ctx->query_radii[0] = thr;
    const uint64_t n = ctx->n, K = ctx->K, N = m + n;
    if (m == 0 || n == 0 || !(thr > 0.0)) {  // diff >= 0 or NaN: nothing passes a non-positive or NaN threshold
        ctx->have_query = true;
        return SCEMA_OK;
    }
    if ((rc = wait_rows(ctx)) || (rc = child_of(ctx, &ctx->query_child, "query_compare"))) return rc;
    scema_ctx *child = ctx->query_child;
    DevBuf &stack = ctx->knn_buf[B_ROWS];
    {
        QTimer t(ctx, QT_COPY, true);
        SCEMA_CUDA(ctx, stack.reserve(N * K * sizeof(double)));
        SCEMA_CUDA(ctx, cudaMemcpyAsync(stack.p, rows, m * K * sizeof(double), rows_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                                        ctx->stream));
        SCEMA_CUDA(ctx, cudaMemcpyAsync(stack.as<double>() + m * K, ctx->d_spline, n * K * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        t.stop();
    }
    rc = scema_set_spline(child, stack.as<double>(), 1, N, (uint32_t)K, nullptr);
    if (rc) return fail(ctx, rc, std::string("query_compare: ") + scema_last_error(child));
    const uint32_t panel_rows = PANEL_ROWBLOCKS * TILE;
    int v = variant;
    rc = compare_prefix_run(child, thr, &v, (uint32_t)((m + panel_rows - 1) / panel_rows), true);
    if (rc) return fail(ctx, rc, std::string("query_compare: ") + scema_last_error(child));
    Knn q;  // scratch buffers only
    q.c = ctx;
    const uint64_t ne = child->n_edges;
    uint64_t kept = 0;
    if (ne) {
        QTimer t(ctx, QT_SELECT, true);
        const uint64_t *keys = child->d_edge_key[child->edge_cur].as<uint64_t>();
        const double *vals = child->d_edge_val[child->edge_cur].as<double>();
        if ((rc = q.reserve(B_CNT, 2 * (ne + 1) * sizeof(unsigned long long)))) return rc;
        unsigned long long *flag = q.buf<unsigned long long>(B_CNT), *pos = flag + (ne + 1);
        k_query_flag<<<(unsigned)((ne + 1 + 255) / 256), 256, 0, ctx->stream>>>(keys, ne, child->key_shift, m, flag);
        size_t tmp = 0;
        SCEMA_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmp, flag, pos, (int64_t)(ne + 1), ctx->stream));
        if ((rc = q.reserve(B_TMP, tmp))) return rc;
        SCEMA_CUDA(ctx, cub::DeviceScan::ExclusiveSum(q.buf<void>(B_TMP), tmp, flag, pos, (int64_t)(ne + 1), ctx->stream));
        SCEMA_CUDA(ctx, cudaMemcpyAsync(&kept, pos + ne, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        SCEMA_CUDA(ctx, ctx->query_j.reserve(std::max<uint64_t>(kept, 1) * sizeof(uint32_t)));
        SCEMA_CUDA(ctx, ctx->query_i.reserve(std::max<uint64_t>(kept, 1) * sizeof(uint32_t)));
        SCEMA_CUDA(ctx, ctx->query_d.reserve(std::max<uint64_t>(kept, 1) * sizeof(double)));
        k_query_scatter<<<(unsigned)((ne + 255) / 256), 256, 0, ctx->stream>>>(keys, vals, ne, child->key_shift, m, flag, pos,
                                                                               ctx->query_j.as<uint32_t>(), ctx->query_i.as<uint32_t>(),
                                                                               ctx->query_d.as<double>());
        ctx->launches += 4;
        SCEMA_CUDA(ctx, cudaGetLastError());
        t.stop();
    }
    q.child_timings(child);
    uint64_t *st = ctx->query_counts;
    st[0] = 1;
    st[5] = child->counters[1];
    st[6] = ne;
    st[7] = (uint64_t)v;
    st[8] = child->counters[0];
    st[9] = kept;
    st[10] = child->counters[3];
    ctx->query_n = kept;
    ctx->have_query = true;
    if (n_edges) *n_edges = kept;
    return SCEMA_OK;
}

}  // namespace scema
