// TEST INFRASTRUCTURE ONLY -- never part of the product library.
//
// irt_setindex_* and irt_check_sets_changed (include/irt_b200.h) for the test-only stand-in of the C ABI
// (tests/cpp/abi_standin_over_oracle.cpp), by export + host comparison: the "index" is an exported copy of the sets it
// covers (a store whose first sets no longer match it is stale), and a call re-checks the whole range against the new
// environment with irt_check_sets and compares the words.  The C++ host mirror includes it when it is built over the
// stand-in (-DIRT_TEST_OVER_STANDIN), so that updateEnvironment's bookkeeping runs and is checked where there is no
// GPU.  stats[0] (changed blocks) is not computed here.
#pragma once

#include <cstdint>
#include <vector>

#include "../../include/irt_b200.h"

struct irt_setindex {
  const irt_setstore *store;
  std::vector<uint64_t> off;
  std::vector<uint32_t> keys;
  std::vector<uint64_t> bits;
};

namespace irt_standin {
// the first n sets of a store as CSR (offsets of n + 1 entries)
inline int export_sets(irt_ctx *ctx, const irt_setstore *s, int64_t n, std::vector<uint64_t> &off,
                       std::vector<uint32_t> &keys, std::vector<uint64_t> &bits) {
  const int64_t ns = irt_setstore_num_sets(s);
  std::vector<uint64_t> o(ns + 1);
  std::vector<uint32_t> k(irt_setstore_num_blocks(s) + 1);
  std::vector<uint64_t> b(k.size());
  const int rc = irt_setstore_export(ctx, s, o.data(), k.data(), b.data());
  if (rc != IRT_OK) return rc;
  off.assign(o.begin(), o.begin() + n + 1);
  keys.assign(k.begin(), k.begin() + o[n]);
  bits.assign(b.begin(), b.begin() + o[n]);
  return IRT_OK;
}
}  // namespace irt_standin

extern "C" {

inline int irt_setindex_create(irt_ctx *ctx, const irt_setstore *store, irt_setindex **out) {
  if (!ctx || !store || !out) return IRT_ERR_INVALID_ARGUMENT;
  irt_setindex *ix = new irt_setindex{store, {}, {}, {}};
  const int rc = irt_standin::export_sets(ctx, store, irt_setstore_num_sets(store), ix->off, ix->keys, ix->bits);
  if (rc != IRT_OK) {
    delete ix;
    return rc;
  }
  *out = ix;
  return IRT_OK;
}

inline void irt_setindex_destroy(irt_setindex *ix) { delete ix; }

inline int64_t irt_setindex_num_sets(const irt_setindex *ix) { return ix ? (int64_t)ix->off.size() - 1 : -1; }

inline int irt_check_sets_changed(irt_ctx *ctx, const irt_setstore *store, const irt_setindex *ix,
                                  const irt_env *env_old, const irt_env *env_new, int64_t begin, int64_t end,
                                  uint32_t *verdict_words, int64_t *flipped, int64_t cap_flipped, int64_t *n_flipped,
                                  int64_t *stats) {
  if (!ctx || !store || !ix || !env_old || !env_new || ix->store != store || cap_flipped < 0)
    return IRT_ERR_INVALID_ARGUMENT;
  if (begin < 0 || end < begin || end > irt_setstore_num_sets(store)) return IRT_ERR_INVALID_ARGUMENT;
  const int64_t n_ix = irt_setindex_num_sets(ix);
  if (irt_setstore_num_sets(store) < n_ix) return IRT_ERR_INVALID_ARGUMENT;
  std::vector<uint64_t> off;
  std::vector<uint32_t> keys;
  std::vector<uint64_t> bits;
  int rc = irt_standin::export_sets(ctx, store, n_ix, off, keys, bits);
  if (rc != IRT_OK) return rc;
  if (off != ix->off || keys != ix->keys || bits != ix->bits) return IRT_ERR_INVALID_ARGUMENT;   // stale
  const int64_t n = end - begin, W = (n + 31) / 32;
  if (n_flipped) *n_flipped = 0;
  if (stats) stats[0] = stats[1] = stats[2] = 0;
  if (n == 0 || env_old == env_new) return IRT_OK;
  std::vector<uint32_t> now(W + 1, 0);
  rc = irt_check_sets(ctx, store, env_new, begin, end, now.data());
  if (rc != IRT_OK) return rc;
  std::vector<int64_t> fl;
  for (int64_t i = 0; i < n; i++)
    if (((verdict_words[i >> 5] ^ now[i >> 5]) >> (i & 31)) & 1u) fl.push_back(begin + i);
  if (n_flipped) *n_flipped = (int64_t)fl.size();
  if (stats) {
    stats[1] = n;
    stats[2] = 1;
  }
  if (flipped && (int64_t)fl.size() > cap_flipped) return IRT_ERR_CAPACITY;
  for (size_t k = 0; flipped && k < fl.size(); k++) flipped[k] = fl[k];
  for (int64_t w = 0; w < W; w++) verdict_words[w] = now[w];
  return IRT_OK;
}

}  // extern "C"
