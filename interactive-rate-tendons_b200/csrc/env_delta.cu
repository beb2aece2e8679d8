// env_delta.cu -- incremental revalidation of a set store after an environment change.
//
// The replanning loop changes the environment a little and asks which roadmap items changed validity.  A set's
// verdict `any(bits & env[key])` over its leaves can only change at a leaf whose bits overlap the changed voxels:
// for a leaf with bits & (old ^ new) == 0, bits & new == bits & old.  So the work of a tick can follow the change
// instead of the roadmap:
//
//   index    an inverted index of the store, built once: per leaf-block key the (set, leaf bits) of every set that
//            has a leaf there, as CSR over the Nb^3 keys (offsets u64[Nb^3+1], set u32[], bits u64[]: SoA, 12 B per
//            leaf).  Built by counting sort: a count per key, one CUB scan, a scatter.
//   changes  one pass over both grids' Nb^3 blocks collects (key, old ^ new) of the changed blocks and sums the
//            lengths of their index lists; one read-back gives the host those counts.
//   select   when the summed list length (plus the leaves of the unindexed tail) is above a fixed share of the range's
//            leaves, streaming the lists costs more than one K3 sweep of the range: the range is swept into scratch
//            words and XOR-ed with the old ones.  Otherwise:
//   mark     every entry of a changed key's list whose bits overlap the change marks its set in a candidate bitmap
//            (atomicOr); the lane that set the bit appends the set to the candidate list.  Filtering on the bits,
//            not on the key alone, matters: every backbone starts at the robot base, so the base block is in
//            essentially every set, and a change near the base would otherwise re-check the whole roadmap.
//   recheck  a warp per candidate (and per tail set) tests its leaves against the new grid the way K3 does
//            (occupancy bitmap, then predicated env[key] loads); the ballot is the new bit, which is compared with the
//            old one.  The candidate bit is cleared on the way out, so the bitmap needs no memset before the next call.
//
// Flips are sorted (CUB radix sort) before they go back.  Kernels read their sizes from device counters; every
// buffer of a call is laid out in the context's scratch before the first kernel runs.
#include <algorithm>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

struct irt_setindex {
  irt_ctx *ctx = nullptr;
  const irt_setstore *store = nullptr;
  uint64_t generation = 0;                      // the store's generation at the build
  int64_t n_sets = 0, n_entries = 0, n_keys = 0;
  unsigned long long *d_key_off = nullptr;      // [n_keys + 1]
  uint32_t *d_set = nullptr;                    // [n_entries]
  uint64_t *d_bits = nullptr;                   // [n_entries]
  uint32_t *d_cand = nullptr;                   // [(n_sets + 31) / 32], all clear between calls
};

namespace {

constexpr int ED_THREADS = 256;
// Above this share of the range's leaves, the delta path (index entries of the changed keys streamed with atomics
// and scattered reads, candidates re-checked) is taken to cost more than one in-order K3 sweep of the range plus the
// XOR.  An estimate from the bytes each path reads; tools/time_env_delta.py measures the crossover (DESIGN.md
// section 3, "Incremental revalidation").
constexpr double ENV_DELTA_SWEEP_FRACTION = 0.25;

struct DeltaCounters {
  unsigned long long n_changed, sum_len, range_leaves, tail_leaves, n_cand, n_flips;
};

__device__ __forceinline__ uint64_t ld_env_if(const uint64_t *p, uint32_t pred) {
  uint64_t v;
  asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\tmov.u64 %0, 0;\n\t@p ld.global.nc.u64 %0, [%2];\n\t}"
      : "=l"(v) : "r"(pred), "l"(p));
  return v;
}

// leaves per key; lanes with equal keys add once
__global__ void ix_count_kernel(const uint32_t *__restrict__ keys, int64_t n, unsigned long long *__restrict__ cnt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool ok = i < n;
  const uint32_t key = ok ? keys[i] : 0xffffffffu;
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  if (ok && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&cnt[key], (unsigned long long)__popc(peers));
}

// a warp per set: each leaf goes to the next free slot of its key's list
__global__ void __launch_bounds__(ED_THREADS)
ix_fill_kernel(const uint64_t *__restrict__ offsets, const uint32_t *__restrict__ keys,
               const uint64_t *__restrict__ bits, int64_t n_sets, unsigned long long *__restrict__ cursor,
               uint32_t *__restrict__ ix_set, uint64_t *__restrict__ ix_bits) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (ED_THREADS / 32);
  for (int64_t s = (int64_t)blockIdx.x * (ED_THREADS / 32) + (threadIdx.x >> 5); s < n_sets; s += warps) {
    const uint64_t lo = offsets[s], hi = offsets[s + 1];
    for (uint64_t j = lo + lane; j < hi; j += 32) {
      const unsigned long long pos = atomicAdd(&cursor[keys[j]], 1ull);
      ix_set[pos] = (uint32_t)s;
      ix_bits[pos] = bits[j];
    }
  }
}

// changed blocks of the two grids, the summed index-list length of their keys, and the leaf counts of the range and
// of its unindexed tail [tail_lo, end)
__global__ void ed_changes_kernel(const uint64_t *__restrict__ env_old, const uint64_t *__restrict__ env_new,
                                  int64_t n_keys, const unsigned long long *__restrict__ key_off,
                                  const uint64_t *__restrict__ offsets, int64_t begin, int64_t tail_lo, int64_t end,
                                  uint32_t *__restrict__ chg_key, uint64_t *__restrict__ chg_diff,
                                  unsigned long long *__restrict__ chg_len, DeltaCounters *__restrict__ c) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k == 0) {
    c->range_leaves = offsets[end] - offsets[begin];
    c->tail_leaves = offsets[end] - offsets[tail_lo];
  }
  if (k >= n_keys) return;
  const uint64_t d = env_old[k] ^ env_new[k];
  if (d == 0) return;
  const unsigned long long pos = atomicAdd(&c->n_changed, 1ull);
  const unsigned long long len = key_off[k + 1] - key_off[k];
  chg_key[pos] = (uint32_t)k;
  chg_diff[pos] = d;
  chg_len[pos] = len;
  atomicAdd(&c->sum_len, len);
}

// entry e of the concatenated lists of the changed keys (chg_pre = exclusive scan of their lengths) marks its set
// when its leaf bits overlap the change and the set lies in [begin, end_ix)
__global__ void __launch_bounds__(ED_THREADS)
ed_mark_kernel(const uint32_t *__restrict__ chg_key, const uint64_t *__restrict__ chg_diff,
               const unsigned long long *__restrict__ chg_pre, DeltaCounters *c,
               const unsigned long long *__restrict__ key_off, const uint32_t *__restrict__ ix_set,
               const uint64_t *__restrict__ ix_bits, int64_t begin, int64_t end_ix, uint32_t *__restrict__ cand_bm,
               uint32_t *__restrict__ cand) {
  const unsigned long long total = c->sum_len;
  const int64_t nch = (int64_t)c->n_changed;
  for (unsigned long long e = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (unsigned long long)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = nch - 1;   // last change whose list starts at or before e
    while (lo < hi) {
      const int64_t mid = (lo + hi + 1) >> 1;
      if (chg_pre[mid] <= e) lo = mid; else hi = mid - 1;
    }
    const unsigned long long ent = key_off[chg_key[lo]] + (e - chg_pre[lo]);
    const int64_t s = ix_set[ent];
    if (s < begin || s >= end_ix || (ix_bits[ent] & chg_diff[lo]) == 0) continue;
    const uint32_t bit = 1u << (s & 31);
    if (!(atomicOr(&cand_bm[s >> 5], bit) & bit)) cand[atomicAdd(&c->n_cand, 1ull)] = (uint32_t)s;
  }
}

// a warp per candidate, then per tail set [tail_lo, end): the new verdict against env_new, compared with the old bit
__global__ void __launch_bounds__(ED_THREADS)
ed_recheck_kernel(const uint32_t *__restrict__ cand, DeltaCounters *c, int64_t tail_lo, int64_t n_tail,
                  const uint64_t *__restrict__ offsets, const uint32_t *__restrict__ keys,
                  const uint64_t *__restrict__ bits, const uint64_t *__restrict__ env,
                  const uint32_t *__restrict__ occ, int64_t begin, int64_t n_ix, const uint32_t *__restrict__ old_words,
                  uint32_t *__restrict__ cand_bm, unsigned long long *__restrict__ flips) {
  const int lane = threadIdx.x & 31;
  const int64_t n_cand = (int64_t)c->n_cand;
  const int64_t total = n_cand + n_tail;
  const int64_t warps = (int64_t)gridDim.x * (ED_THREADS / 32);
  for (int64_t w = (int64_t)blockIdx.x * (ED_THREADS / 32) + (threadIdx.x >> 5); w < total; w += warps) {
    const int64_t s = w < n_cand ? (int64_t)cand[w] : tail_lo + (w - n_cand);
    const uint64_t lo = offsets[s], hi = offsets[s + 1];
    bool hit = false;
    for (uint64_t j = lo + lane; j < hi; j += 32) {
      const uint32_t k = keys[j];
      const uint32_t o = (__ldg(occ + (k >> 5)) >> (k & 31)) & 1u;
      hit |= (bits[j] & ld_env_if(env + k, o)) != 0ull;
    }
    const bool now = __any_sync(0xffffffffu, hit);
    if (lane == 0) {
      const int64_t r = s - begin;
      const bool was = (old_words[r >> 5] >> (r & 31)) & 1u;
      if (now != was) flips[atomicAdd(&c->n_flips, 1ull)] = (unsigned long long)s;
      if (s < n_ix) atomicAnd(&cand_bm[s >> 5], ~(1u << (s & 31)));
    }
  }
}

// full-sweep path: the sets whose old and new bits differ
__global__ void ed_xor_kernel(const uint32_t *__restrict__ old_words, const uint32_t *__restrict__ new_words,
                              int64_t n, int64_t begin, DeltaCounters *__restrict__ c,
                              unsigned long long *__restrict__ flips) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= (n + 31) / 32) return;
  uint32_t x = old_words[w] ^ new_words[w];
  if (w == (n - 1) / 32 && (n & 31)) x &= (1u << (n & 31)) - 1u;
  if (!x) return;
  unsigned long long p = atomicAdd(&c->n_flips, (unsigned long long)__popc(x));
  for (; x; x &= x - 1) flips[p++] = (unsigned long long)(begin + w * 32 + __ffs(x) - 1);
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

extern "C" {

int irt_setindex_create(irt_ctx *ctx, const irt_setstore *store, irt_setindex **out) {
  if (!ctx || !store || !out) return IRT_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  if (store->ctx->device != ctx->device) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "a store of another device");
  if (store->n_sets >= ((int64_t)1 << 32))
    return irt_fail(ctx, IRT_ERR_CAPACITY, "the index holds set numbers as u32: %lld sets", (long long)store->n_sets);
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  irt_setindex *ix = new irt_setindex();
  ix->ctx = ctx;
  ix->store = store;
  ix->generation = store->generation;
  ix->n_sets = store->n_sets;
  ix->n_entries = store->n_blocks;
  ix->n_keys = (int64_t)store->gd.Nb * store->gd.Nb * store->gd.Nb;
  const int64_t nk = ix->n_keys, ne = ix->n_entries;
  if (cudaMalloc(&ix->d_key_off, (size_t)(nk + 1) * 8) != cudaSuccess ||
      cudaMalloc(&ix->d_set, (size_t)std::max<int64_t>(ne, 1) * 4) != cudaSuccess ||
      cudaMalloc(&ix->d_bits, (size_t)std::max<int64_t>(ne, 1) * 8) != cudaSuccess ||
      cudaMalloc(&ix->d_cand, (size_t)std::max<int64_t>((ix->n_sets + 31) / 32, 1) * 4) != cudaSuccess) {
    irt_setindex_destroy(ix);
    return irt_fail(ctx, IRT_ERR_CUDA, "set index allocation failed (%lld leaves)", (long long)ne);
  }
  auto fail = [&](int rc) { irt_setindex_destroy(ix); return rc; };
#define IX_CUDA(call)                                                                                \
  do {                                                                                               \
    cudaError_t _e = (call);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return fail(irt_fail(ctx, IRT_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e)));      \
  } while (0)
  IX_CUDA(cudaMemsetAsync(ix->d_key_off, 0, (size_t)(nk + 1) * 8, st));
  IX_CUDA(cudaMemsetAsync(ix->d_cand, 0, (size_t)std::max<int64_t>((ix->n_sets + 31) / 32, 1) * 4, st));
  if (ne > 0) {
    size_t cub_bytes = 0;
    IX_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, ix->d_key_off, ix->d_key_off, nk + 1, st));
    char *scr = (char *)ctx_scratch(ctx, align256((size_t)nk * 8) + cub_bytes + 64);
    if (!scr) return fail(irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc failed"));
    unsigned long long *cursor = (unsigned long long *)scr;
    ix_count_kernel<<<(unsigned)((ne + ED_THREADS - 1) / ED_THREADS), ED_THREADS, 0, st>>>(store->d_keys, ne,
                                                                                         ix->d_key_off);
    IRT_LAUNCHED(ctx);
    IX_CUDA(cudaGetLastError());
    IX_CUDA(cub::DeviceScan::ExclusiveSum(scr + align256((size_t)nk * 8), cub_bytes, ix->d_key_off, ix->d_key_off,
                                          nk + 1, st));
    IRT_LAUNCHED(ctx);
    IX_CUDA(cudaMemcpyAsync(cursor, ix->d_key_off, (size_t)nk * 8, cudaMemcpyDeviceToDevice, st));
    int64_t blocks = (ix->n_sets + ED_THREADS / 32 - 1) / (ED_THREADS / 32);
    blocks = std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)ctx->sm_count * 16));
    ix_fill_kernel<<<(unsigned)blocks, ED_THREADS, 0, st>>>(store->d_offsets, store->d_keys, store->d_bits,
                                                            ix->n_sets, cursor, ix->d_set, ix->d_bits);
    IRT_LAUNCHED(ctx);
    IX_CUDA(cudaGetLastError());
  }
  IX_CUDA(cudaStreamSynchronize(st));
#undef IX_CUDA
  *out = ix;
  return IRT_OK;
}

void irt_setindex_destroy(irt_setindex *ix) {
  if (!ix) return;
  cudaSetDevice(ix->ctx->device);
  if (ix->d_key_off) cudaFree(ix->d_key_off);
  if (ix->d_set) cudaFree(ix->d_set);
  if (ix->d_bits) cudaFree(ix->d_bits);
  if (ix->d_cand) cudaFree(ix->d_cand);
  delete ix;
}

int64_t irt_setindex_num_sets(const irt_setindex *ix) { return ix ? ix->n_sets : -1; }

int irt_check_sets_changed(irt_ctx *ctx, const irt_setstore *store, const irt_setindex *ix,
                           const irt_env *env_old, const irt_env *env_new, int64_t begin, int64_t end,
                           uint32_t *verdict_words, int64_t *flipped, int64_t cap_flipped, int64_t *n_flipped,
                           int64_t *stats) {
  // ---- every argument first: nothing runs, and verdict_words stays as it is, on any error
  if (!ctx || !store || !ix || !env_old || !env_new) return IRT_ERR_INVALID_ARGUMENT;
  if (store->ctx->device != ctx->device || ix->ctx->device != ctx->device || env_old->ctx->device != ctx->device ||
      env_new->ctx->device != ctx->device)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "handles of another device");
  if (!same_grid(env_old->grid, env_new->grid))
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "the two environments' grids differ");
  if (store->grid.Ng != env_new->grid.Ng)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "voxel dimension mismatch (%d != %d)", store->grid.Ng,
                    env_new->grid.Ng);
  if (begin < 0 || end < begin || end > store->n_sets)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "set range [%lld,%lld) outside [0,%lld]", (long long)begin,
                    (long long)end, (long long)store->n_sets);
  if (ix->store != store) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "the index belongs to another store");
  if (ix->generation != store->generation)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "stale index: the store's content was replaced after the build");
  if (cap_flipped < 0) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "cap_flipped < 0");
  const int64_t n = end - begin;
  if (n > 0 && !verdict_words) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "verdict_words is NULL");
  if (n_flipped) *n_flipped = 0;
  if (stats) stats[0] = stats[1] = stats[2] = 0;
  if (n == 0 || env_old == env_new) return IRT_OK;

  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t nk = ix->n_keys, W = (n + 31) / 32;
  const int64_t end_ix = std::min(end, ix->n_sets), tail_lo = std::max(begin, end_ix), n_tail = end - tail_lo;
  const int64_t n_ix_range = std::max<int64_t>(0, end_ix - begin);
  const int end_bit = 64 - __builtin_clzll((unsigned long long)end);

  // ---- scratch: one layout for either path, sized by the bounds known now (flips <= n, candidates <= n)
  size_t scan_bytes = 0, sort_bytes = 0;
  IRT_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (unsigned long long *)nullptr,
                                              (unsigned long long *)nullptr, nk, st));
  IRT_CUDA(ctx, cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, (unsigned long long *)nullptr,
                                               (unsigned long long *)nullptr, n, 0, end_bit, st));
  size_t off = 0;
  auto carve = [&](size_t bytes) { const size_t o = off; off += align256(bytes); return o; };
  const size_t o_cnt = carve(sizeof(DeltaCounters)), o_old = carve((size_t)W * 4), o_new = carve((size_t)W * 4);
  const size_t o_key = carve((size_t)nk * 4), o_diff = carve((size_t)nk * 8), o_len = carve((size_t)nk * 8);
  const size_t o_cand = carve((size_t)std::max<int64_t>(n_ix_range, 1) * 4);
  const size_t o_fl = carve((size_t)n * 8), o_fs = carve((size_t)n * 8);
  const size_t o_tmp = carve(std::max(scan_bytes, sort_bytes));
  char *scr = (char *)ctx_scratch(ctx, off + 64);
  if (!scr) return irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc failed");
  DeltaCounters *d_c = (DeltaCounters *)(scr + o_cnt);
  uint32_t *d_old = (uint32_t *)(scr + o_old), *d_new = (uint32_t *)(scr + o_new);
  uint32_t *d_key = (uint32_t *)(scr + o_key), *d_cand = (uint32_t *)(scr + o_cand);
  uint64_t *d_diff = (uint64_t *)(scr + o_diff);
  unsigned long long *d_len = (unsigned long long *)(scr + o_len);
  unsigned long long *d_fl = (unsigned long long *)(scr + o_fl), *d_fs = (unsigned long long *)(scr + o_fs);
  void *d_tmp = scr + o_tmp;

  // ---- the change list and its counts: one read-back
  IRT_CUDA(ctx, cudaMemsetAsync(d_c, 0, sizeof(DeltaCounters), st));
  IRT_CUDA(ctx, cudaMemcpyAsync(d_old, verdict_words, (size_t)W * 4, cudaMemcpyHostToDevice, st));
  ed_changes_kernel<<<(unsigned)((nk + ED_THREADS - 1) / ED_THREADS), ED_THREADS, 0, st>>>(
      env_old->d_blocks, env_new->d_blocks, nk, ix->d_key_off, store->d_offsets, begin, tail_lo, end, d_key, d_diff,
      d_len, d_c);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  DeltaCounters h;
  IRT_CUDA(ctx, cudaMemcpyAsync(&h, d_c, sizeof(h), cudaMemcpyDeviceToHost, st));
  IRT_CUDA(ctx, cudaStreamSynchronize(st));
  if (stats) stats[0] = (int64_t)h.n_changed;
  if (h.n_changed == 0) return IRT_OK;   // equal grids: no verdict can change

  const bool sweep = (double)(h.sum_len + h.tail_leaves) > ENV_DELTA_SWEEP_FRACTION * (double)h.range_leaves;
  int64_t rechecked = n;
  if (sweep) {
    int rc = check_sets_launch(ctx, store, env_new, begin, end, d_new, st);
    if (rc) return rc;
    ed_xor_kernel<<<(unsigned)((W + ED_THREADS - 1) / ED_THREADS), ED_THREADS, 0, st>>>(d_old, d_new, n, begin, d_c,
                                                                                       d_fl);
    IRT_LAUNCHED(ctx);
    IRT_CUDA(ctx, cudaGetLastError());
  } else {
    if (h.sum_len > 0) {
      IRT_CUDA(ctx, cub::DeviceScan::ExclusiveSum(d_tmp, scan_bytes, d_len, d_len, (int64_t)h.n_changed, st));
      IRT_LAUNCHED(ctx);
      const int64_t blocks = std::min<int64_t>(((int64_t)h.sum_len + ED_THREADS - 1) / ED_THREADS,
                                               (int64_t)ctx->sm_count * 16);
      ed_mark_kernel<<<(unsigned)blocks, ED_THREADS, 0, st>>>(d_key, d_diff, d_len, d_c, ix->d_key_off, ix->d_set,
                                                              ix->d_bits, begin, end_ix, ix->d_cand, d_cand);
      IRT_LAUNCHED(ctx);
      IRT_CUDA(ctx, cudaGetLastError());
    }
    // warps for the candidates (at most min(entries scanned, indexed sets in range)) and the tail
    const int64_t bound = std::min<int64_t>((int64_t)h.sum_len, n_ix_range) + n_tail;
    if (bound > 0) {
      int64_t blocks = (bound + ED_THREADS / 32 - 1) / (ED_THREADS / 32);
      blocks = std::min<int64_t>(blocks, (int64_t)ctx->sm_count * 8);
      ed_recheck_kernel<<<(unsigned)blocks, ED_THREADS, 0, st>>>(
          d_cand, d_c, tail_lo, n_tail, store->d_offsets, store->d_keys, store->d_bits, env_new->d_blocks,
          env_new->d_occ, begin, ix->n_sets, d_old, ix->d_cand, d_fl);
      IRT_LAUNCHED(ctx);
      IRT_CUDA(ctx, cudaGetLastError());
    }
  }
  IRT_CUDA(ctx, cudaMemcpyAsync(&h, d_c, sizeof(h), cudaMemcpyDeviceToHost, st));
  IRT_CUDA(ctx, cudaStreamSynchronize(st));
  if (!sweep) rechecked = (int64_t)h.n_cand + n_tail;
  const int64_t nf = (int64_t)h.n_flips;
  if (stats) {
    stats[1] = rechecked;
    stats[2] = sweep ? 1 : 0;
  }
  if (n_flipped) *n_flipped = nf;
  if (flipped && nf > cap_flipped)
    return irt_fail(ctx, IRT_ERR_CAPACITY, "%lld sets flipped, room for %lld", (long long)nf, (long long)cap_flipped);

  // ---- results: sorted flips; the new words (sweep) or the old ones with the flipped bits toggled (delta)
  const unsigned long long *d_sorted = d_fl;
  if (flipped && nf > 1) {
    IRT_CUDA(ctx, cub::DeviceRadixSort::SortKeys(d_tmp, sort_bytes, d_fl, d_fs, nf, 0, end_bit, st));
    IRT_LAUNCHED(ctx);
    d_sorted = d_fs;
  }
  std::vector<int64_t> own;
  int64_t *fl_host = flipped;
  if (!sweep && !flipped) {
    own.resize((size_t)nf);
    fl_host = own.data();
  }
  if (fl_host && nf > 0)
    IRT_CUDA(ctx, cudaMemcpyAsync(fl_host, d_sorted, (size_t)nf * 8, cudaMemcpyDeviceToHost, st));
  if (sweep) IRT_CUDA(ctx, cudaMemcpyAsync(verdict_words, d_new, (size_t)W * 4, cudaMemcpyDeviceToHost, st));
  IRT_CUDA(ctx, cudaStreamSynchronize(st));
  if (!sweep)
    for (int64_t i = 0; i < nf; i++) {
      const int64_t r = fl_host[i] - begin;
      verdict_words[r >> 5] ^= 1u << (r & 31);
    }
  return IRT_OK;
}

}  // extern "C"
