// TEST INFRASTRUCTURE ONLY -- never part of the product library.
//
// A plain sequential host implementation of the k-NN entry points of the C ABI (irt_nnset_*, include/irt_b200.h),
// following the contract stated there: the compound-space distance summed left to right, the k nearest by
// (distance, index), excluded items skipped, only finite distances <= bound.  The C++ host mirror includes it when
// it is built over the test-only stand-in of the C ABI (tests/cpp/abi_standin_over_oracle.cpp, -DIRT_TEST_OVER_STANDIN),
// so that the mirror's device-k-NN code paths -- batched connection, mask words, device-copy bookkeeping, the
// temporary vertex of ikNearest -- run and are checked where there is no GPU.
#pragma once

#include <algorithm>
#include <cmath>
#include <utility>
#include <vector>

#include "../../include/irt_b200.h"

struct irt_nnset {
  int dim;
  irt_metric m;
  std::vector<double> rows;
};

extern "C" {

inline int irt_nnset_create(irt_ctx *, int dim, const irt_metric *m, irt_nnset **out) {
  if (dim < 1 || dim > 16 || !m || m->n_euclid < 1 || m->n_euclid > dim) return IRT_ERR_INVALID_ARGUMENT;
  *out = new irt_nnset{dim, *m, {}};
  return IRT_OK;
}
inline void irt_nnset_destroy(irt_nnset *s) { delete s; }
inline int64_t irt_nnset_size(const irt_nnset *s) { return (int64_t)(s->rows.size() / s->dim); }
inline int irt_nnset_append(irt_ctx *, irt_nnset *s, const double *rows, int64_t n) {
  s->rows.insert(s->rows.end(), rows, rows + n * s->dim);
  return IRT_OK;
}
inline int irt_nnset_clear(irt_ctx *, irt_nnset *s) {
  s->rows.clear();
  return IRT_OK;
}
inline int irt_nnset_knn(irt_ctx *, const irt_nnset *s, const double *queries, int64_t m, int k, double bound,
                         const uint32_t *exclude_words, int64_t *idx, double *dist) {
  if (k < 1 || k > IRT_KNN_MAX_K) return IRT_ERR_INVALID_ARGUMENT;
  const int64_t n = irt_nnset_size(s);
  const irt_metric &mt = s->m;
  for (int64_t q = 0; q < m; q++) {
    const double *a = queries + q * s->dim;
    std::vector<std::pair<double, int64_t>> d;
    for (int64_t i = 0; i < n; i++) {
      if (exclude_words && ((exclude_words[i >> 5] >> (i & 31)) & 1u)) continue;
      const double *b = s->rows.data() + i * s->dim;
      double e = 0.0;
      for (int j = 0; j < mt.n_euclid; j++) e += (a[j] - b[j]) * (a[j] - b[j]);
      double v = std::sqrt(e);
      if (mt.so2_col >= 0) {
        double dr = std::fabs(a[mt.so2_col] - b[mt.so2_col]);
        if (dr > M_PI) dr = 2.0 * M_PI - dr;
        v += mt.w_so2 * dr;
      }
      if (mt.lin_col >= 0) v += mt.w_lin * std::fabs(a[mt.lin_col] - b[mt.lin_col]);
      if (std::isfinite(v) && v <= bound) d.emplace_back(v, i);
    }
    const size_t kk = std::min<size_t>(k, d.size());
    std::partial_sort(d.begin(), d.begin() + kk, d.end());
    for (int j = 0; j < k; j++) {
      idx[q * k + j] = (size_t)j < kk ? d[j].second : -1;
      if (dist) dist[q * k + j] = (size_t)j < kk ? d[j].first : INFINITY;
    }
  }
  return IRT_OK;
}

}  // extern "C"
