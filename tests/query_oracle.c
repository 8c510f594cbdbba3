/* TEST INFRASTRUCTURE ONLY — CPU statement of scema_query_compare and scema_query_knn, on the oracle's compare_l2
 * (oracle/liboracle.so).
 *
 * R [n][K] are the retained rows (IDs ids[n]), Q [m][K] the queries. Every distance is compare_l2(R[i], Q[j]).
 *   query_radius_count: per_query[j] = #{i : d(i, j) < thr}; returns the sum.
 *   query_radius_fill:  the pairs in (j, i) order, query j's block starting at offsets[j].
 *   query_knn_oracle:   the k nearest retained rows of every query, slots ordered by (diff, ids[i], i) ascending; NaN
 *                       distances skipped, +inf listed, empty slots {UINT32_MAX, +inf}. No row is excluded.
 * tests/test_query.py compiles this file into a temporary directory, linked against oracle/liboracle.so
 * (gcc -O2 -ffp-contract=off -fopenmp, as the oracle). */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

double oracle_compare_l2(const double *a, const double *b, uint32_t K);

uint64_t query_radius_count(const double *R, uint64_t n, const double *Q, uint64_t m, uint32_t K, double thr, uint64_t *per_query)
{
    uint64_t total = 0;
#pragma omp parallel for schedule(dynamic, 4) reduction(+ : total)
    for (int64_t j = 0; j < (int64_t)m; j++) {
        uint64_t c = 0;
        for (uint64_t i = 0; i < n; i++)
            if (oracle_compare_l2(R + i * K, Q + (size_t)j * K, K) < thr) c++;
        per_query[j] = c;
        total += c;
    }
    return total;
}

void query_radius_fill(const double *R, uint64_t n, const double *Q, uint64_t m, uint32_t K, double thr, const uint64_t *offsets,
                       uint32_t *out_j, uint32_t *out_i, double *out_d)
{
#pragma omp parallel for schedule(dynamic, 4)
    for (int64_t j = 0; j < (int64_t)m; j++) {
        uint64_t o = offsets[j];
        for (uint64_t i = 0; i < n; i++) {
            const double d = oracle_compare_l2(R + i * K, Q + (size_t)j * K, K);
            if (d < thr) { out_j[o] = (uint32_t)j; out_i[o] = (uint32_t)i; out_d[o] = d; o++; }
        }
    }
}

static int knn_less(double d1, uint32_t id1, uint32_t i1, double d2, uint32_t id2, uint32_t i2)
{
    if (d1 != d2) return d1 < d2;
    if (id1 != id2) return id1 < id2;
    return i1 < i2;
}

void query_knn_oracle(const double *R, uint64_t n, const uint32_t *ids, const double *Q, uint64_t m, uint32_t K, uint32_t k,
                      uint32_t *out_index, double *out_diff)
{
#pragma omp parallel for schedule(dynamic, 4)
    for (int64_t j = 0; j < (int64_t)m; j++) {
        uint32_t *ix = out_index + (size_t)j * k;
        double *dv = out_diff + (size_t)j * k;
        uint32_t c = 0;
        for (uint32_t s = 0; s < k; s++) { ix[s] = UINT32_MAX; dv[s] = INFINITY; }
        for (uint64_t i = 0; i < n; i++) {
            const double d = oracle_compare_l2(R + i * K, Q + (size_t)j * K, K);
            if (d != d) continue;
            if (c == k && !knn_less(d, ids[i], (uint32_t)i, dv[k - 1], ids[ix[k - 1]], ix[k - 1])) continue;
            uint32_t p = c < k ? c : k - 1;
            while (p > 0 && knn_less(d, ids[i], (uint32_t)i, dv[p - 1], ids[ix[p - 1]], ix[p - 1])) {
                dv[p] = dv[p - 1]; ix[p] = ix[p - 1]; p--;
            }
            dv[p] = d; ix[p] = (uint32_t)i;
            if (c < k) c++;
        }
    }
}
