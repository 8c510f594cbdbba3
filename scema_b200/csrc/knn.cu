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
// k_knn_exact: the query rows q_rows[0, nq) against the columns of segment blockIdx.y, one query row per warp, tiles of
// 64 columns (two per lane) staged through shared memory in slices of 32 of the K entries, sums in the reference's
// order (k_exact_all's arithmetic; a - b and b - a round to the same magnitude). Writes each (query, segment)'s k best.
// ------------------------------------------------------------------------------------------------
constexpr int KQ = 8, KCOL = 64, KKC = 32;
__global__ void __launch_bounds__(256, 4) k_knn_exact(const double *__restrict__ S, uint64_t n, uint32_t K, const uint32_t *__restrict__ ids,
                                                   const uint32_t *__restrict__ q_rows, uint32_t nq, uint64_t seg_len, uint32_t k,
                                                   unsigned long long *__restrict__ part_b, uint32_t *__restrict__ part_ix)
{
    __shared__ double Qs[KQ][KKC];
    __shared__ double Cs[KCOL][KKC + 1];
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const uint32_t qp = blockIdx.x * KQ + w;
    const bool have_q = qp < nq;
    const uint32_t qrow = have_q ? q_rows[qp] : 0xffffffffu;  // n < 2^32: no column has this index
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
                Qs[r][kk] = (q < nq && (uint32_t)kk < kn) ? S[(uint64_t)q_rows[q] * K + k0 + kk] : 0.0;
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
template <int PASS>
__global__ void __launch_bounds__(256) k_knn_expand(const uint64_t *__restrict__ keys, const double *__restrict__ vals, uint64_t m,
                                                    uint32_t key_shift, const uint32_t *__restrict__ perm, const uint8_t *__restrict__ open,
                                                    unsigned long long *__restrict__ cnt_or_cursor, unsigned long long *__restrict__ eb,
                                                    uint32_t *__restrict__ eix)
{
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const uint64_t key = keys[e];
    uint32_t a = (uint32_t)(key >> key_shift), b = (uint32_t)(key & ((1ull << key_shift) - 1));
    if (perm) { a = perm[a]; b = perm[b]; }
    const unsigned long long bits = (unsigned long long)__double_as_longlong(vals[e]);
    if (open[a]) {
        const unsigned long long o = atomicAdd(cnt_or_cursor + a, 1ull);
        if (PASS == 1) { eb[o] = bits; eix[o] = b; }
    }
    if (open[b]) {
        const unsigned long long o = atomicAdd(cnt_or_cursor + b, 1ull);
        if (PASS == 1) { eb[o] = bits; eix[o] = a; }
    }
}

// Distance sample: rows A (rows_a[a * a_span / na], a < na) against rows B; tri: only b > a (A == B). Same-row pairs and
// NaN distances are left out. Bits appended with one atomic per warp.
__global__ void __launch_bounds__(256) k_knn_sample(const double *__restrict__ S, uint32_t K, const uint32_t *__restrict__ rows_a,
                                                    uint32_t na, uint64_t a_span, const uint32_t *__restrict__ rows_b, uint32_t nb, int tri,
                                                    unsigned long long *__restrict__ out, unsigned long long *__restrict__ count)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t a = (uint32_t)(t / nb), b = (uint32_t)(t - (uint64_t)a * nb);
    bool keep = false;
    unsigned long long bits = 0;
    if (a < na && !(tri && b <= a)) {
        const uint32_t i = rows_a[(uint64_t)a * a_span / na], j = rows_b[b];
        if (i != j) {
            const double d = exact_l2(S + (uint64_t)i * K, S + (uint64_t)j * K, K);
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
// host side
// ------------------------------------------------------------------------------------------------
namespace {

enum { B_IDS, B_OPEN, B_PERM, B_OUT_IX, B_OUT_D, B_SUBSET, B_SAMPLE, B_TMP, B_MISC, B_CNT, B_EB, B_EIX, B_ROWS, B_PART_B, B_PART_IX };

struct Knn {
    scema_ctx *c;           // the caller's context: its stream, its rows, its scratch buffers
    uint64_t n;
    uint32_t K, k;
    uint64_t open_n;        // rows still open
    std::vector<uint32_t> subset;
    uint64_t stats[8] = {};
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

    // open rows first in B_PERM; returns their number in open_n
    int partition()
    {
        size_t tmp = 0;
        cub::CountingInputIterator<uint32_t> iota(0);
        SCEMA_CUDA(c, cub::DevicePartition::Flagged(nullptr, tmp, iota, buf<uint8_t>(B_OPEN), buf<uint32_t>(B_PERM), misc() + 1, (int64_t)n,
                                                    c->stream));
        int rc = reserve(B_TMP, tmp);
        if (rc) return rc;
        SCEMA_CUDA(c, cub::DevicePartition::Flagged(buf<void>(B_TMP), tmp, iota, buf<uint8_t>(B_OPEN), buf<uint32_t>(B_PERM), misc() + 1,
                                                    (int64_t)n, c->stream));
        c->launches += 2;
        uint64_t m[2];
        rc = read_misc(m, 2);
        if (rc) return rc;
        open_n = m[1];
        return SCEMA_OK;
    }

    // Radius from a distance sample: A rows against the subset (round 1: the subset's own pairs). tau = the smallest
    // value with at least max(C * k / (n - 1) * count, KNN_QUANTILE_MIN) sampled distances strictly below it; *frac_below =
    // the sampled fraction below max(tau, floor). +inf (or 0 sampled distances) when no such value exists.
    int radius(const uint32_t *rows_a, uint32_t na, uint64_t a_span, bool tri, double floor_tau, double *tau, double *frac_below)
    {
        const uint32_t nb = (uint32_t)subset.size();
        const uint64_t total = (uint64_t)na * nb;
        int rc = reserve(B_SAMPLE, 2 * total * sizeof(unsigned long long));
        if (rc) return rc;
        unsigned long long *s0 = buf<unsigned long long>(B_SAMPLE), *s1 = s0 + total;
        SCEMA_CUDA(c, cudaMemsetAsync(misc(), 0, 4 * sizeof(uint64_t), c->stream));
        k_knn_sample<<<(unsigned)((total + 255) / 256), 256, 0, c->stream>>>(c->d_spline, K, rows_a, na, a_span, buf<uint32_t>(B_SUBSET), nb,
                                                                           tri ? 1 : 0, s0, misc());
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
        const double want = std::ceil(KNN_QUANTILE_C * k / (double)(n - 1) * (double)count);
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
    // caller's rows in the order perm, nullptr = identity). Returns the rows closed.
    int select(scema_ctx *child, const uint32_t *perm, uint64_t *closed)
    {
        const uint64_t m = child->n_edges;
        *closed = 0;
        if (m == 0) return SCEMA_OK;
        const uint64_t *keys = child->d_edge_key[child->edge_cur].as<uint64_t>();
        const double *vals = child->d_edge_val[child->edge_cur].as<double>();
        int rc = reserve(B_CNT, 2 * (n + 1) * sizeof(unsigned long long));
        if (!rc) rc = reserve(B_EB, 2 * m * sizeof(unsigned long long));
        if (!rc) rc = reserve(B_EIX, 2 * m * sizeof(uint32_t));
        if (rc) return rc;
        unsigned long long *cnt = buf<unsigned long long>(B_CNT), *offs = cnt + (n + 1);
        SCEMA_CUDA(c, cudaMemsetAsync(cnt, 0, (n + 1) * sizeof(unsigned long long), c->stream));
        const unsigned g = (unsigned)((m + 255) / 256);
        k_knn_expand<0><<<g, 256, 0, c->stream>>>(keys, vals, m, child->key_shift, perm, buf<uint8_t>(B_OPEN), cnt, nullptr, nullptr);
        size_t tmp = 0;
        SCEMA_CUDA(c, cub::DeviceScan::ExclusiveSum(nullptr, tmp, cnt, offs, (int64_t)(n + 1), c->stream));
        rc = reserve(B_TMP, tmp);
        if (rc) return rc;
        SCEMA_CUDA(c, cub::DeviceScan::ExclusiveSum(buf<void>(B_TMP), tmp, cnt, offs, (int64_t)(n + 1), c->stream));
        SCEMA_CUDA(c, cudaMemcpyAsync(cnt, offs, (n + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
        k_knn_expand<1><<<g, 256, 0, c->stream>>>(keys, vals, m, child->key_shift, perm, buf<uint8_t>(B_OPEN), cnt,
                                                 buf<unsigned long long>(B_EB), buf<uint32_t>(B_EIX));
        SCEMA_CUDA(c, cudaMemsetAsync(misc() + 3, 0, sizeof(uint64_t), c->stream));
        k_knn_topk<<<(unsigned)((n + 7) / 8), 256, 0, c->stream>>>(buf<unsigned long long>(B_EB), buf<uint32_t>(B_EIX), buf<uint32_t>(B_IDS),
                                                                   nullptr, n, offs, 0, k, buf<uint8_t>(B_OPEN), misc() + 3,
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
        k_knn_exact<<<dim3((unsigned)qblocks, (unsigned)nseg), 256, 0, c->stream>>>(c->d_spline, n, K, buf<uint32_t>(B_IDS), buf<uint32_t>(B_PERM),
                                                                                    (uint32_t)nq, seg_len, k, buf<unsigned long long>(B_PART_B),
                                                                                    buf<uint32_t>(B_PART_IX));
        k_knn_topk<<<(unsigned)((nq + 7) / 8), 256, 0, c->stream>>>(buf<unsigned long long>(B_PART_B), buf<uint32_t>(B_PART_IX),
                                                                    buf<uint32_t>(B_IDS), buf<uint32_t>(B_PERM), nq, nullptr, nseg * k, k,
                                                                    nullptr, nullptr, buf<uint32_t>(B_OUT_IX), buf<double>(B_OUT_D));
        c->launches += 2;
        SCEMA_CUDA(c, cudaGetLastError());
        stats[3] += nq;
        stats[4] += nq * (n - 1);
        return SCEMA_OK;
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
    q.c = ctx; q.n = n; q.K = ctx->K; q.k = k;
    q.stats[7] = SCEMA_PAIRS_EXACT;
    if (n <= 1) {
        if (index_host) std::fill(index_host, index_host + n * k, 0xffffffffu);
        if (diff_host) std::fill(diff_host, diff_host + n * k, INFINITY);
        for (int i = 0; i < 8; i++) ctx->knn_counts[i] = q.stats[i];
        ctx->knn_counts[3] = n;
        return SCEMA_OK;
    }
    int rc = wait_rows(ctx);
    if (rc) return rc;
    if ((rc = q.reserve(B_IDS, n * sizeof(uint32_t))) || (rc = q.reserve(B_OPEN, n)) || (rc = q.reserve(B_PERM, n * sizeof(uint32_t))) ||
        (rc = q.reserve(B_OUT_IX, n * k * sizeof(uint32_t))) || (rc = q.reserve(B_OUT_D, n * k * sizeof(double))) ||
        (rc = q.reserve(B_MISC, 8 * sizeof(uint64_t))))
        return rc;
    SCEMA_CUDA(ctx, cudaMemcpyAsync(q.buf<void>(B_IDS), ids_of(ctx).data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    SCEMA_CUDA(ctx, cudaMemsetAsync(q.buf<void>(B_OPEN), 1, n, ctx->stream));
    q.open_n = n;

    if (variant != SCEMA_PAIRS_EXACT && n >= KNN_MIN_N) {
        if (!ctx->knn_child) {
            scema_ctx *child = nullptr;
            rc = scema_create(&child, ctx->device, (void *)ctx->stream);
            if (rc) return fail(ctx, rc, "knn: could not create the context of the filter rounds");
            ctx->knn_child = child;
        }
        scema_ctx *child = ctx->knn_child;
        make_subset(n, q.subset);
        if ((rc = q.reserve(B_SUBSET, q.subset.size() * sizeof(uint32_t)))) return rc;
        SCEMA_CUDA(ctx, cudaMemcpyAsync(q.buf<void>(B_SUBSET), q.subset.data(), q.subset.size() * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                        ctx->stream));
        const double budget = KNN_EDGE_BUDGET * (double)n * k + 1048576.0;
        double tau_prev = 0.0;
        for (int round = 1; round <= KNN_MAX_ROUNDS && q.open_n > 0; round++) {
            if (round > 1 && (double)q.open_n * (double)n <= KNN_EXACT_PAIRS) break;
            double tau = 0.0, frac = 1.0, pairs = 0.0;
            uint32_t p1 = 0;
            if (round == 1) {
                rc = q.radius(q.buf<uint32_t>(B_SUBSET), (uint32_t)q.subset.size(), q.subset.size(), true, 0.0, &tau, &frac);
                pairs = 0.5 * (double)n * (double)(n - 1);
            } else {
                const uint32_t na = (uint32_t)std::min<uint64_t>(q.open_n, KNN_SAMPLE_OPEN);
                rc = q.radius(q.buf<uint32_t>(B_PERM), na, q.open_n, false, 2.0 * tau_prev, &tau, &frac);
                const uint32_t panel_rows = PANEL_ROWBLOCKS * TILE;
                p1 = (uint32_t)((q.open_n + panel_rows - 1) / panel_rows);
                const double r1 = std::min<double>((double)n, (double)p1 * panel_rows);
                pairs = r1 * (double)n - 0.5 * r1 * (r1 + 1.0);
            }
            if (rc) return rc;
            if (!(tau < INFINITY) || pairs * frac > budget) break;  // too dense for an O(n k) edge list: the exact kernel takes over
            const uint32_t *perm = nullptr;
            if (round == 1) {
                rc = scema_set_spline(child, ctx->d_spline, 1, n, q.K, nullptr);
            } else {
                if ((rc = q.reserve(B_ROWS, n * q.K * sizeof(double)))) return rc;
                k_knn_gather<<<(unsigned)((n * q.K + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_spline, n, q.K, q.buf<uint32_t>(B_PERM),
                                                                                        q.buf<double>(B_ROWS));
                ctx->launches++;
                SCEMA_CUDA(ctx, cudaGetLastError());
                rc = scema_set_spline(child, q.buf<double>(B_ROWS), 1, n, q.K, nullptr);
                perm = q.buf<uint32_t>(B_PERM);
            }
            if (rc) return fail(ctx, rc, std::string("knn: ") + scema_last_error(child));
            int v = variant;
            rc = compare_prefix_run(child, tau, &v, p1);
            if (rc) return fail(ctx, rc, std::string("knn: ") + scema_last_error(child));
            q.stats[0]++;
            q.stats[5] += child->counters[1];
            q.stats[6] += child->n_edges;
            q.stats[7] = (uint64_t)v;
            q.radii[round - 1] = tau;
            tau_prev = tau;
            uint64_t closed = 0;
            rc = q.select(child, perm, &closed);
            if (rc) return rc;
            q.stats[round == 1 ? 1 : 2] += closed;
            rc = q.partition();  // the open rows to the front: sampled, gathered and queried by what follows
            if (rc) return rc;
        }
    }
    rc = q.partition();
    if (!rc) rc = q.exact();
    if (rc) return rc;
    if (index_host)
        SCEMA_CUDA(ctx, cudaMemcpyAsync(index_host, q.buf<void>(B_OUT_IX), n * k * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (diff_host)
        SCEMA_CUDA(ctx, cudaMemcpyAsync(diff_host, q.buf<void>(B_OUT_D), n * k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SCEMA_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 8; i++) { ctx->knn_counts[i] = q.stats[i]; ctx->knn_radii[i] = q.radii[i]; }
    return SCEMA_OK;
}

}  // namespace scema
