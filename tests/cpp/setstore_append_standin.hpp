// TEST INFRASTRUCTURE ONLY -- never part of the product library.
//
// irt_setstore_append (include/irt_b200.h) for the test-only stand-in of the C ABI
// (tests/cpp/abi_standin_over_oracle.cpp): both stores are exported, the kept sets of the range are concatenated on
// the host and the result is imported into dst -- which is what the contract says the device append equals.  The
// C++ host mirror includes it when it is built over the stand-in (-DIRT_TEST_OVER_STANDIN), so that
// extendVoxelCache's bookkeeping runs and is checked where there is no GPU.
#pragma once

#include <cstdint>
#include <vector>

#include "../../include/irt_b200.h"

extern "C" {

inline int irt_setstore_append(irt_ctx *ctx, irt_setstore *dst, const irt_setstore *src, int64_t begin, int64_t end,
                               const uint32_t *keep_words) {
  if (!ctx || !dst || !src || dst == src) return IRT_ERR_INVALID_ARGUMENT;
  const int64_t ns = irt_setstore_num_sets(src), nd = irt_setstore_num_sets(dst);
  if (begin < 0 || begin > end || end > ns) return IRT_ERR_INVALID_ARGUMENT;
  std::vector<uint64_t> so(ns + 1), off(nd + 1);
  std::vector<uint32_t> sk(irt_setstore_num_blocks(src) + 1), keys(irt_setstore_num_blocks(dst) + 1);
  std::vector<uint64_t> sb(sk.size()), bits(keys.size());
  int rc = irt_setstore_export(ctx, src, so.data(), sk.data(), sb.data());
  if (rc == IRT_OK) rc = irt_setstore_export(ctx, dst, off.data(), keys.data(), bits.data());
  if (rc != IRT_OK) return rc;
  keys.resize(off[nd]);
  bits.resize(off[nd]);
  for (int64_t i = 0; i < end - begin; i++) {
    if (keep_words && !((keep_words[i >> 5] >> (i & 31)) & 1u)) continue;
    const int64_t s = begin + i;
    keys.insert(keys.end(), sk.begin() + so[s], sk.begin() + so[s + 1]);
    bits.insert(bits.end(), sb.begin() + so[s], sb.begin() + so[s + 1]);
    off.push_back(keys.size());
  }
  keys.push_back(0);
  bits.push_back(0);
  return irt_setstore_import(ctx, dst, (int64_t)off.size() - 1, off.data(), keys.data(), bits.data());
}

}  // extern "C"
