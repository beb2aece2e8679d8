// knn.cu -- exact k-nearest neighbours over a device-resident point set (irt_nnset_*, include/irt_b200.h).
//
// Two brute-force kernels, chosen from the number of queries m (KNN_SMALL_M):
//   * small m (single queries of roadmapIk / addMilestone, latency-bound): the database is split over many CTAs per
//     query; every lane takes one item, a warp offers its surviving candidates to a top-k list that the warp holds
//     in registers (rank r at lane r % 32, register r / 32);
//   * large m (the connection batch of createRoadmap): one query per thread, database tiles staged through shared
//     memory and read as broadcasts, a private top-k list per thread in shared memory.
// Both write sorted partial lists that knn_merge_kernel reduces with the same warp list, so the two give the same
// bits: every candidate's distance is computed by the one function knn_dist, and the lists are ordered by the
// total order (distance, index).
//
// The current k-th distance theta stays in a register and rejects almost every pair before its square root:
// d >= fl(w_so2 s + w_lin l) exactly (rounding is monotone and every part is >= 0), and the tension part is
// rejected when its square exceeds (theta - rest + theta 2^-40)^2 (1 + 2^-40), a margin that covers the rounding of
// the bound and of the exact distance (DESIGN.md, the k-NN section).
#include <algorithm>
#include <cmath>
#include <vector>

#include "common.cuh"

namespace {

constexpr int KNN_SMALL_M = 64;       // m below this: the item-parallel kernel
constexpr int KNN_MAX_DIM = 16;
constexpr int LARGE_THREADS = 128;    // queries per CTA of the large-m kernel
constexpr int LARGE_TILE = 256;       // items per shared-memory tile
constexpr int SMALL_THREADS = 256;
constexpr int NO_IDX = 0x7fffffff;    // index of an empty list entry; sorts after every real item

struct KnnMetric {
  int ne, so2, lin;                   // so2 / lin: 1 if the term is present
  int W;                              // stored width: ne + so2 + lin, canonical column order e..., s, l
  int dim;
  int col[KNN_MAX_DIM];               // canonical column -> column of a caller's row
  double w_so2, w_lin;
};

}  // namespace

struct irt_nnset {
  irt_ctx *ctx = nullptr;
  int dim = 0;
  irt_metric metric;
  KnnMetric km;
  int64_t n = 0, cap = 0;
  double *d_rows = nullptr;           // [cap][W], canonical column order
};

namespace {

__device__ __forceinline__ bool knn_less(double da, int ia, double db, int ib) {
  return da < db || (da == db && ia < ib);
}

// the rest of the distance (SO(2) and retraction parts) and the tension sum of squares, operation by operation as in
// the contract; knn_dist finishes it.  q: the query in canonical order, r: one stored row.
template <int NE>
__device__ __forceinline__ double knn_rest(const KnnMetric &mt, const double *q, const double *r, double &a,
                                           double &b) {
  a = 0.0;
  b = 0.0;
  double rest = 0.0;
  if (mt.so2) {
    double dr = fabs(__dsub_rn(q[NE], r[NE]));
    if (dr > M_PI) dr = __dsub_rn(2.0 * M_PI, dr);
    a = __dmul_rn(mt.w_so2, dr);
    rest = a;
  }
  if (mt.lin) {
    const double ql = mt.so2 ? q[NE + 1] : q[NE], rl = mt.so2 ? r[NE + 1] : r[NE];   // no dynamic register index
    b = __dmul_rn(mt.w_lin, fabs(__dsub_rn(ql, rl)));
    rest = mt.so2 ? __dadd_rn(a, b) : b;
  }
  return rest;
}

template <int NE>
__device__ __forceinline__ double knn_sum2(const double *q, const double *r) {
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < NE; j++) {
    const double t = __dsub_rn(q[j], r[j]);
    s = __dadd_rn(s, __dmul_rn(t, t));
  }
  return s;
}

// exact distance, or +inf when it is certainly > theta (theta: the current k-th distance, or the bound)
template <int NE>
__device__ __forceinline__ double knn_dist(const KnnMetric &mt, const double *q, const double *r, double theta) {
  double a, b;
  const double rest = knn_rest<NE>(mt, q, r, a, b);
  if (rest > theta) return INFINITY;
  const double s2 = knn_sum2<NE>(q, r);
  const double u = __dadd_rn(__dsub_rn(theta, rest), __dmul_rn(theta, 0x1p-40));
  if (u >= 0.0 && s2 > __dmul_rn(__dmul_rn(u, u), 1.0 + 0x1p-40)) return INFINITY;
  double d = __dsqrt_rn(s2);
  if (mt.so2) d = __dadd_rn(d, a);
  if (mt.lin) d = __dadd_rn(d, b);
  return d;
}

__device__ __forceinline__ bool excluded(const uint32_t *words, int i) {
  return words && ((__ldg(words + (i >> 5)) >> (i & 31)) & 1u);
}

// a sorted top-k list held by one warp: rank lane in (d0, i0), rank lane + 32 in (d1, i1)
struct WarpList {
  double d0, d1;
  int i0, i1;
  __device__ void init() { d0 = d1 = INFINITY; i0 = i1 = NO_IDX; }
  // the k-th entry (k - 1 = rank), warp-uniform
  __device__ void kth(int k, double &d, int &i) const {
    const int r = k - 1;
    d = __shfl_sync(0xffffffffu, r < 32 ? d0 : d1, r & 31);
    i = __shfl_sync(0xffffffffu, r < 32 ? i0 : i1, r & 31);
  }
  // insert (cd, ci), warp-uniform, known to be < the k-th entry
  __device__ void insert(double cd, int ci, int lane) {
    const unsigned lt0 = __ballot_sync(0xffffffffu, knn_less(d0, i0, cd, ci));
    const unsigned lt1 = __ballot_sync(0xffffffffu, knn_less(d1, i1, cd, ci));
    const int pos = __popc(lt0) + __popc(lt1);
    double ud0 = __shfl_up_sync(0xffffffffu, d0, 1), ud1 = __shfl_up_sync(0xffffffffu, d1, 1);
    int ui0 = __shfl_up_sync(0xffffffffu, i0, 1), ui1 = __shfl_up_sync(0xffffffffu, i1, 1);
    const double last_d = __shfl_sync(0xffffffffu, d0, 31);
    const int last_i = __shfl_sync(0xffffffffu, i0, 31);
    if (lane == 0) { ud1 = last_d; ui1 = last_i; }
    if (lane > pos) { d0 = ud0; i0 = ui0; } else if (lane == pos) { d0 = cd; i0 = ci; }
    if (lane + 32 > pos) { d1 = ud1; i1 = ui1; } else if (lane + 32 == pos) { d1 = cd; i1 = ci; }
  }
  // offer one candidate per lane (ok = lane has one); lanes are walked in order, each re-checked against the list
  __device__ void offer(bool ok, double d, int i, int k, int lane) {
    unsigned bits = __ballot_sync(0xffffffffu, ok);
    while (bits) {
      const int src = __ffs(bits) - 1;
      bits &= bits - 1;
      const double cd = __shfl_sync(0xffffffffu, d, src);
      const int ci = __shfl_sync(0xffffffffu, i, src);
      double td;
      int ti;
      kth(k, td, ti);
      if (knn_less(cd, ci, td, ti)) insert(cd, ci, lane);
    }
  }
  __device__ void store(int k, int lane, double *pd, int *pi) const {
    if (lane < k) { pd[lane] = d0; pi[lane] = i0; }
    if (lane + 32 < k) { pd[lane + 32] = d1; pi[lane + 32] = i1; }
  }
};

__device__ __forceinline__ bool accept(double d, double bound) { return d <= bound && d < INFINITY; }

// rows -> canonical stored layout
__global__ void knn_gather_kernel(const double *src, int64_t n, KnnMetric mt, double *dst) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n * mt.W) return;
  const int64_t i = t / mt.W;
  const int c = (int)(t - i * mt.W);
  dst[t] = src[i * mt.dim + mt.col[c]];
}

template <int NE>
__device__ __forceinline__ void load_query(const KnnMetric &mt, const double *queries, int64_t qi, double *q) {
#pragma unroll
  for (int c = 0; c < NE + 2; c++)
    q[c] = (c < mt.W) ? queries[qi * mt.dim + mt.col[c]] : 0.0;
}

// small m: grid (slices, m), SMALL_THREADS threads; every warp writes one partial list
template <int NE>
__global__ void __launch_bounds__(SMALL_THREADS) knn_small_kernel(const double *__restrict__ rows, int n, KnnMetric mt,
                                                                  const double *__restrict__ queries, int k,
                                                                  double bound, const uint32_t *__restrict__ excl,
                                                                  int per_slice, double *pd, int *pi) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t qi = blockIdx.y;
  double q[NE + 2];
  load_query<NE>(mt, queries, qi, q);
  WarpList L;
  L.init();
  const int lo = blockIdx.x * per_slice, hi = min(n, lo + per_slice);
  for (int base = lo; base < hi; base += SMALL_THREADS) {
    const int i = base + threadIdx.x;
    double td;
    int ti;
    L.kth(k, td, ti);
    const double theta = fmin(td, bound);
    double d = INFINITY;
    bool ok = false;
    if (i < hi && !excluded(excl, i)) {
      double r[NE + 2];
#pragma unroll
      for (int c = 0; c < NE + 2; c++) r[c] = (c < mt.W) ? rows[(int64_t)i * mt.W + c] : 0.0;
      d = knn_dist<NE>(mt, q, r, theta);
      ok = accept(d, bound) && knn_less(d, i, td, ti);
    }
    L.offer(ok, d, i, k, lane);
  }
  const int64_t slot = (qi * gridDim.x + blockIdx.x) * (SMALL_THREADS / 32) + warp;
  L.store(k, lane, pd + slot * k, pi + slot * k);
}

// large m: grid (slices, ceil(m / LARGE_THREADS)), one query per thread; dynamic shared memory: the tile, then the
// per-thread lists (rank r of thread t at [r * LARGE_THREADS + t])
template <int NE>
__global__ void __launch_bounds__(LARGE_THREADS) knn_large_kernel(const double *__restrict__ rows, int n, KnnMetric mt,
                                                                  const double *__restrict__ queries, int64_t m, int k,
                                                                  double bound, const uint32_t *__restrict__ excl,
                                                                  int per_slice, double *pd, int *pi) {
  extern __shared__ double smem[];
  double *tile = smem;                                             // [LARGE_TILE][W]
  uint32_t *tex = (uint32_t *)(tile + LARGE_TILE * mt.W);          // [LARGE_TILE / 32] exclude words of the tile
  double *ld = (double *)(tex + LARGE_TILE / 32);                  // [k][LARGE_THREADS]
  int *li = (int *)(ld + (size_t)k * LARGE_THREADS);
  const int t = threadIdx.x;
  const int64_t qi = (int64_t)blockIdx.y * LARGE_THREADS + t;
  const bool active = qi < m;
  double q[NE + 2];
  load_query<NE>(mt, queries, active ? qi : 0, q);
  for (int r = 0; r < k; r++) { ld[r * LARGE_THREADS + t] = INFINITY; li[r * LARGE_THREADS + t] = NO_IDX; }
  double td = INFINITY;
  int ti = NO_IDX;
  const int lo = blockIdx.x * per_slice, hi = min(n, lo + per_slice);
  for (int base = lo; base < hi; base += LARGE_TILE) {
    const int cnt = min(LARGE_TILE, hi - base);
    __syncthreads();
    for (int e = t; e < cnt * mt.W; e += LARGE_THREADS) tile[e] = rows[(int64_t)base * mt.W + e];
    if (t < LARGE_TILE / 32) {
      uint32_t w = 0;
      if (excl)
        for (int b = 0; b < 32; b++) {
          const int i = base + t * 32 + b;
          if (t * 32 + b < cnt && excluded(excl, i)) w |= 1u << b;
        }
      tex[t] = w;
    }
    __syncthreads();
    if (!active) continue;
    for (int j = 0; j < cnt; j++) {
      if ((tex[j >> 5] >> (j & 31)) & 1u) continue;
      double r[NE + 2];
#pragma unroll
      for (int c = 0; c < NE + 2; c++) r[c] = (c < mt.W) ? tile[j * mt.W + c] : 0.0;
      const double d = knn_dist<NE>(mt, q, r, fmin(td, bound));
      const int i = base + j;
      if (!(accept(d, bound) && knn_less(d, i, td, ti))) continue;
      int p = k - 1;                                               // rare: about k ln(n / k) times per query
      while (p > 0 && knn_less(d, i, ld[(p - 1) * LARGE_THREADS + t], li[(p - 1) * LARGE_THREADS + t])) {
        ld[p * LARGE_THREADS + t] = ld[(p - 1) * LARGE_THREADS + t];
        li[p * LARGE_THREADS + t] = li[(p - 1) * LARGE_THREADS + t];
        p--;
      }
      ld[p * LARGE_THREADS + t] = d;
      li[p * LARGE_THREADS + t] = i;
      td = ld[(k - 1) * LARGE_THREADS + t];
      ti = li[(k - 1) * LARGE_THREADS + t];
    }
  }
  if (!active) return;
  const int64_t slot = qi * gridDim.x + blockIdx.x;
  for (int r = 0; r < k; r++) {
    pd[slot * k + r] = ld[r * LARGE_THREADS + t];
    pi[slot * k + r] = li[r * LARGE_THREADS + t];
  }
}

// one warp per query: the k smallest of its `parts` sorted partial lists
__global__ void knn_merge_kernel(const double *pd, const int *pi, int64_t m, int parts, int k, int64_t *idx,
                                 double *dist) {
  const int lane = threadIdx.x & 31;
  const int64_t q = blockIdx.x * (int64_t)(blockDim.x / 32) + (threadIdx.x >> 5);
  if (q >= m) return;
  WarpList L;
  L.init();
  const int64_t total = (int64_t)parts * k;
  const double *qd = pd + q * total;
  const int *qix = pi + q * total;
  for (int64_t base = 0; base < total; base += 32) {
    double td;
    int ti;
    L.kth(k, td, ti);
    const int64_t e = base + lane;
    double d = INFINITY;
    int i = NO_IDX;
    if (e < total) { d = qd[e]; i = qix[e]; }
    L.offer(i != NO_IDX && knn_less(d, i, td, ti), d, i, k, lane);
  }
  for (int r = lane; r < 64; r += 32) {
    if (r >= k) break;
    const double d = r < 32 ? L.d0 : L.d1;
    const int i = r < 32 ? L.i0 : L.i1;
    idx[q * k + r] = (i == NO_IDX) ? -1 : (int64_t)i;
    dist[q * k + r] = (i == NO_IDX) ? INFINITY : d;
  }
}

template <int NE>
void launch_small(dim3 g, cudaStream_t st, const double *rows, int n, const KnnMetric &mt, const double *qs, int k,
                  double bound, const uint32_t *ex, int per, double *pd, int *pi) {
  knn_small_kernel<NE><<<g, SMALL_THREADS, 0, st>>>(rows, n, mt, qs, k, bound, ex, per, pd, pi);
}
template <int NE>
cudaError_t launch_large(dim3 g, size_t sm, cudaStream_t st, const double *rows, int n, const KnnMetric &mt,
                         const double *qs, int64_t m, int k, double bound, const uint32_t *ex, int per, double *pd,
                         int *pi) {
  cudaError_t e = cudaFuncSetAttribute(knn_large_kernel<NE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  if (e != cudaSuccess) return e;
  knn_large_kernel<NE><<<g, LARGE_THREADS, sm, st>>>(rows, n, mt, qs, m, k, bound, ex, per, pd, pi);
  return cudaSuccess;
}

#define KNN_NE_CASES(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16)

int metric_check(irt_ctx *ctx, int dim, const irt_metric *m, KnnMetric *out) {
  if (dim < 1 || dim > KNN_MAX_DIM) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "nnset dim %d outside [1, 16]", dim);
  if (!m) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "null metric");
  if (m->n_euclid < 1 || m->n_euclid > dim)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "n_euclid %d outside [1, dim]", m->n_euclid);
  for (int c : {m->so2_col, m->lin_col})
    if (c != -1 && (c < m->n_euclid || c >= dim))
      return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "metric column %d outside [n_euclid, dim) and not -1", c);
  if (m->so2_col != -1 && m->so2_col == m->lin_col)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "so2_col and lin_col coincide");
  if ((m->so2_col != -1 && !(m->w_so2 >= 0.0 && m->w_so2 < INFINITY)) ||
      (m->lin_col != -1 && !(m->w_lin >= 0.0 && m->w_lin < INFINITY)))
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "metric weights must be finite and >= 0");
  KnnMetric k{};
  k.ne = m->n_euclid;
  k.so2 = m->so2_col != -1;
  k.lin = m->lin_col != -1;
  k.W = k.ne + k.so2 + k.lin;
  k.dim = dim;
  for (int c = 0; c < k.ne; c++) k.col[c] = c;
  if (k.so2) k.col[k.ne] = m->so2_col;
  if (k.lin) k.col[k.ne + k.so2] = m->lin_col;
  k.w_so2 = m->w_so2;
  k.w_lin = m->w_lin;
  *out = k;
  return IRT_OK;
}

}  // namespace

extern "C" {

int irt_nnset_create(irt_ctx *ctx, int dim, const irt_metric *m, irt_nnset **out) {
  if (!ctx || !out) return IRT_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  KnnMetric km;
  int rc = metric_check(ctx, dim, m, &km);
  if (rc != IRT_OK) return rc;
  irt_nnset *s = new irt_nnset();
  s->ctx = ctx;
  s->dim = dim;
  s->metric = *m;
  s->km = km;
  *out = s;
  return IRT_OK;
}

void irt_nnset_destroy(irt_nnset *s) {
  if (!s) return;
  cudaSetDevice(s->ctx->device);
  if (s->d_rows) cudaFree(s->d_rows);
  delete s;
}

int64_t irt_nnset_size(const irt_nnset *s) { return s ? s->n : 0; }

int irt_nnset_clear(irt_ctx *ctx, irt_nnset *s) {
  if (!ctx || !s) return IRT_ERR_INVALID_ARGUMENT;
  s->n = 0;
  return IRT_OK;
}

int irt_nnset_append(irt_ctx *ctx, irt_nnset *s, const double *rows, int64_t n) {
  if (!ctx || !s || n < 0 || (n > 0 && !rows)) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "nnset_append: bad args");
  if (n == 0) return IRT_OK;
  if (s->n + n > (int64_t)NO_IDX - 1) return irt_fail(ctx, IRT_ERR_CAPACITY, "nnset holds at most 2^31 - 2 items");
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int W = s->km.W;
  if (s->n + n > s->cap) {                 // grow geometrically: appends of one row stay amortised O(1)
    int64_t cap = std::max<int64_t>(s->n + n, s->cap + s->cap / 2);
    cap = std::max<int64_t>(cap, 1024);
    double *nr = nullptr;
    IRT_CUDA(ctx, cudaMalloc(&nr, (size_t)cap * W * sizeof(double)));
    if (s->n) {
      cudaError_t e = cudaMemcpyAsync(nr, s->d_rows, (size_t)s->n * W * sizeof(double), cudaMemcpyDeviceToDevice, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) {
        cudaFree(nr);
        return irt_fail(ctx, IRT_ERR_CUDA, "nnset grow: %s", cudaGetErrorString(e));
      }
    }
    if (s->d_rows) cudaFree(s->d_rows);
    s->d_rows = nr;
    s->cap = cap;
  }
  double *raw = (double *)ctx_scratch(ctx, (size_t)n * s->dim * sizeof(double));
  if (!raw) return irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc failed");
  IRT_CUDA(ctx, cudaMemcpyAsync(raw, rows, (size_t)n * s->dim * sizeof(double), cudaMemcpyHostToDevice, st));
  const int64_t total = n * W;
  knn_gather_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(raw, n, s->km, s->d_rows + s->n * W);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  IRT_CUDA(ctx, cudaStreamSynchronize(st));
  s->n += n;
  return IRT_OK;
}

int irt_nnset_knn(irt_ctx *ctx, const irt_nnset *s, const double *queries, int64_t m, int k, double bound,
                  const uint32_t *exclude_words, int64_t *idx, double *dist) {
  if (!ctx || !s) return IRT_ERR_INVALID_ARGUMENT;
  if (k < 1 || k > IRT_KNN_MAX_K) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "k=%d outside [1, %d]", k, IRT_KNN_MAX_K);
  if (m < 0 || (m > 0 && (!queries || !idx))) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "nnset_knn: bad args");
  if (m == 0) return IRT_OK;
  const int n = (int)s->n;
  if (n == 0) {
    for (int64_t e = 0; e < m * k; e++) {
      idx[e] = -1;
      if (dist) dist[e] = INFINITY;
    }
    return IRT_OK;
  }
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const KnnMetric &mt = s->km;
  const int sms = ctx->sm_count > 0 ? ctx->sm_count : 148;
  const bool small = m < KNN_SMALL_M;
  // slices per query: about four CTAs per SM over the whole grid
  int64_t groups = small ? m : (m + LARGE_THREADS - 1) / LARGE_THREADS;
  const int64_t min_items = small ? SMALL_THREADS : LARGE_TILE;
  int64_t slices = std::max<int64_t>(1, (4 * sms + groups - 1) / groups);
  slices = std::min<int64_t>(slices, std::max<int64_t>(1, n / min_items));
  const int per = (int)((n + slices - 1) / slices);
  slices = (n + per - 1) / per;
  const int64_t parts = small ? slices * (SMALL_THREADS / 32) : slices;
  const size_t nw = exclude_words ? (size_t)(n + 31) / 32 : 0;
  // scratch: queries, exclude words, partial lists (dist, index), final lists
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t bq = al((size_t)m * s->dim * 8), bx = al(nw * 4), bpd = al((size_t)m * parts * k * 8),
               bpi = al((size_t)m * parts * k * 4), bo = al((size_t)m * k * 8);
  char *base = (char *)ctx_scratch(ctx, bq + bx + bpd + bpi + 2 * bo);
  if (!base) return irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc failed");
  double *d_q = (double *)base;
  uint32_t *d_x = nw ? (uint32_t *)(base + bq) : nullptr;
  double *d_pd = (double *)(base + bq + bx);
  int *d_pi = (int *)(base + bq + bx + bpd);
  int64_t *d_idx = (int64_t *)(base + bq + bx + bpd + bpi);
  double *d_dist = (double *)(base + bq + bx + bpd + bpi + bo);
  IRT_CUDA(ctx, cudaMemcpyAsync(d_q, queries, (size_t)m * s->dim * 8, cudaMemcpyHostToDevice, st));
  if (nw) IRT_CUDA(ctx, cudaMemcpyAsync(d_x, exclude_words, nw * 4, cudaMemcpyHostToDevice, st));
  if (small) {
    dim3 g((unsigned)slices, (unsigned)m);
    switch (mt.ne) {
#define X(NE) case NE: launch_small<NE>(g, st, s->d_rows, n, mt, d_q, k, bound, d_x, per, d_pd, d_pi); break;
      KNN_NE_CASES(X)
#undef X
    }
  } else {
    dim3 g((unsigned)slices, (unsigned)groups);
    const size_t sm = (size_t)LARGE_TILE * mt.W * 8 + LARGE_TILE / 32 * 4 + (size_t)k * LARGE_THREADS * 12;
    cudaError_t e = cudaSuccess;
    switch (mt.ne) {
#define X(NE) case NE: e = launch_large<NE>(g, sm, st, s->d_rows, n, mt, d_q, m, k, bound, d_x, per, d_pd, d_pi); break;
      KNN_NE_CASES(X)
#undef X
    }
    IRT_CUDA(ctx, e);
  }
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  knn_merge_kernel<<<(unsigned)((m + 3) / 4), 128, 0, st>>>(d_pd, d_pi, m, (int)parts, k, d_idx, d_dist);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  IRT_CUDA(ctx, cudaMemcpyAsync(idx, d_idx, (size_t)m * k * 8, cudaMemcpyDeviceToHost, st));
  if (dist) IRT_CUDA(ctx, cudaMemcpyAsync(dist, d_dist, (size_t)m * k * 8, cudaMemcpyDeviceToHost, st));
  IRT_CUDA(ctx, cudaStreamSynchronize(st));
  return IRT_OK;
}

}  // extern "C"
