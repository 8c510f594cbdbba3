/* TEST INFRASTRUCTURE ONLY — CPU statement of scema_knn, on the oracle's compare_l2 (oracle/liboracle.so).
 *
 * k nearest neighbours of rows [row_begin, row_end) among all N rows: out_index / out_diff [(row_end - row_begin) * k],
 * slots ordered by (diff, ids[j], j) ascending; a row is not its own neighbour, NaN distances are skipped, +inf ones
 * listed, empty slots {UINT32_MAX, +inf}. Insertion into a sorted list of k. tests/test_knn.py compiles this file into a
 * temporary directory, linked against oracle/liboracle.so (gcc -O2 -ffp-contract=off -fopenmp, as the oracle). */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

double oracle_compare_l2(const double *a, const double *b, uint32_t K);

static int knn_less(double d1, uint32_t id1, uint32_t j1, double d2, uint32_t id2, uint32_t j2)
{
    if (d1 != d2) return d1 < d2;
    if (id1 != id2) return id1 < id2;
    return j1 < j2;
}

void knn_oracle(const double *rows, uint64_t N, uint32_t K, uint32_t k, const uint32_t *ids, uint64_t row_begin,
                uint64_t row_end, uint32_t *out_index, double *out_diff)
{
    if (row_end > N) row_end = N;
    if (row_begin > row_end) row_begin = row_end;
#pragma omp parallel for schedule(dynamic, 4)
    for (int64_t i = (int64_t)row_begin; i < (int64_t)row_end; i++) {
        uint32_t *ix = out_index + (size_t)(i - (int64_t)row_begin) * k;
        double *dv = out_diff + (size_t)(i - (int64_t)row_begin) * k;
        uint32_t m = 0;
        for (uint32_t s = 0; s < k; s++) { ix[s] = UINT32_MAX; dv[s] = INFINITY; }
        for (uint64_t j = 0; j < N; j++) {
            if (j == (uint64_t)i) continue;
            const double d = oracle_compare_l2(rows + (size_t)i * K, rows + (size_t)j * K, K);
            if (d != d) continue;
            if (m == k && !knn_less(d, ids[j], (uint32_t)j, dv[k - 1], ids[ix[k - 1]], ix[k - 1])) continue;
            uint32_t p = m < k ? m : k - 1;
            while (p > 0 && knn_less(d, ids[j], (uint32_t)j, dv[p - 1], ids[ix[p - 1]], ix[p - 1])) {
                dv[p] = dv[p - 1]; ix[p] = ix[p - 1]; p--;
            }
            dv[p] = d; ix[p] = (uint32_t)j;
            if (m < k) m++;
        }
    }
}
