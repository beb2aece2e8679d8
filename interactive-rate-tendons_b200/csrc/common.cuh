// common.cuh -- shared declarations of the sm_100a hot-path library (libirt_b200.so).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdio>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/irt_b200.h"

#define IRT_CAP_PTS_MAX 512  // upper bound on backbone points per shape (L/dL + 2)
// doubles per tendon in a row of the constant-memory routing table: rx, ry, rdx, rdy, rddx, rddy and the
// state-independent products rx^2, ry^2, rx ry, |r|^2 (= rx^2 + ry^2) of the RK4 stage's accumulations
#define IRT_CT_WIDTH 10

struct irt_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;  // D2H of finished chunks overlaps the next chunk's kernels
  int sm_count = 148;
  std::string last_error;
  std::atomic<int64_t> launches{0};
  std::mutex mu;
  // growable device scratch owned by the context (never shrinks)
  void *scratch = nullptr;
  size_t scratch_bytes = 0;
  // second grow-only arena for the K2 pipelines (sample pools, raster slots); kept across calls so
  // repeated roadmap builds do not pay cudaMalloc/cudaFree of multi-GB pools
  void *arena = nullptr;
  size_t arena_bytes = 0;
  // staging for the host-pointer FK entry point (two pipeline stages), also grow-only
  void *io = nullptr;
  size_t io_bytes = 0;
  cudaEvent_t ev_computed[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
  // packed FK outputs: per-stage "row offsets are on the host" events and a small pinned host buffer
  cudaEvent_t ev_offsets[2] = {nullptr, nullptr};
  void *pinned = nullptr;
  size_t pinned_bytes = 0;
  bool debug_sync = false;   // IRT_B200_DEBUG_SYNC=1
};

// device-resident robot constants (passed to kernels by value)
struct RobotDev {
  double Kse[3], Kbt[3], KseInv[3], KbtInv[3];
  double L, dL, r, residual_threshold;
  double C[IRT_MAX_TENDONS * IRT_MAX_COEF];
  double D[IRT_MAX_TENDONS * IRT_MAX_COEF];
  double home_factor[IRT_MAX_TENDONS];  // L_i^home = (L - s) * home_factor  (TendonRobot.cpp:281-310)
  double min_length[IRT_MAX_TENDONS], max_length[IRT_MAX_TENDONS];
  int n_tendons, n_c, n_d, enable_rotation, enable_retraction;
  int Kfull;          // number of grid nodes for s = 0, excluding the start point
  int n_table;        // 2*Kfull - 1 entries: idx(node i) = 2i, idx(mid of step i -> i-1) = 2i - 1
  int n_head;         // no-retraction robots: tabulated first-gap stages (<= 4 entries)
  double head_h[2];   // no-retraction robots: first-gap step sizes (h[1] = 0 if one step)
  double tau_bin_scale;  // FK bucket key: tension bin = (int)(sum(tau) * tau_bin_scale)
  int simple_routing;    // every tendon is straight or helical with constant rho (n_c <= 2, n_d == 1)
  int c1_uniform;        // ... and all tendons wind at the same rate |C1| (or not at all)
  double c1_abs;         // that rate
  double c1_sign[IRT_MAX_TENDONS];                        // C1_j = c1_sign_j * c1_abs (0 for a straight tendon)
  double sin_c0[IRT_MAX_TENDONS], cos_c0[IRT_MAX_TENDONS];  // sin / cos of C0_j (host libm)
  const double *table;  // device: [n_table][N][6] = rx, ry, rdx, rdy, rddx, rddy
  const double *head;   // device: [4][N][6]
  const double *node_t; // device: [Kfull] canonical node times L - i*dL
};

struct irt_robot {
  irt_ctx *ctx = nullptr;
  unsigned long long uid = 0;   // process-unique (the constant-memory copy of the routing table is tagged with it)
  irt_robot_desc desc;
  RobotDev dev;
  int state_size = 0;
  int max_points = 0;
  double *d_table = nullptr;
  double *d_ctab = nullptr;     // [n_table][N][IRT_CT_WIDTH]: source of the constant-memory copy
  double *d_head = nullptr;
  double *d_node_t = nullptr;
  std::vector<double> node_t;
};

struct GridDev {
  int Ng, Nb, levels;       // Nb = Ng/4, levels = log2(Nb)
  double lo[3], hi[3], d[3], inv_d[3];
  double inv_rot[9];
  int identity_rot;
};

struct irt_env {
  irt_ctx *ctx = nullptr;
  irt_grid grid;
  GridDev gd;
  uint64_t *d_blocks = nullptr;  // [Nb^3] Morton-ordered dense leaf blocks
  uint32_t *d_occ = nullptr;     // [Nb^3/32] leaf-occupancy bitmap (bit = block non-empty)
  int64_t n_blocks_total = 0;
};

struct irt_setstore {
  irt_ctx *ctx = nullptr;
  irt_grid grid;
  GridDev gd;
  int64_t n_sets = 0, n_blocks = 0;
  uint64_t *d_offsets = nullptr;  // [n_sets + 1]
  uint32_t *d_keys = nullptr;     // [n_blocks]
  uint64_t *d_bits = nullptr;     // [n_blocks]
  size_t cap_sets = 0, cap_blocks = 0;
  // bumped whenever the content is replaced (import, irt_voxelize_*), not by an append: an irt_setindex built at
  // another generation describes sets that are no longer there
  uint64_t generation = 0;
};

// Ng, limits and rotation all equal: voxel sets and grids of the two are comparable block by block
inline bool same_grid(const irt_grid &a, const irt_grid &b) {
  if (a.Ng != b.Ng) return false;
  for (int i = 0; i < 6; i++)
    if (a.lim[i] != b.lim[i]) return false;
  for (int i = 0; i < 9; i++)
    if (a.inv_rot[i] != b.inv_rot[i]) return false;
  return true;
}

int irt_fail(irt_ctx *ctx, int status, const char *fmt, ...);
GridDev make_grid_dev(const irt_grid &g);
int grid_check(irt_ctx *ctx, const irt_grid *g);
void *ctx_scratch(irt_ctx *ctx, size_t bytes);  // nullptr on failure
void *ctx_arena(irt_ctx *ctx, size_t bytes);    // nullptr on failure
void *ctx_io(irt_ctx *ctx, size_t bytes);       // nullptr on failure
void *ctx_pinned(irt_ctx *ctx, size_t bytes);   // page-locked HOST memory, nullptr on failure
int setstore_grow_blocks(irt_ctx *ctx, irt_setstore *s, int64_t need_blocks, int64_t keep_blocks,
                         cudaStream_t st);

#define IRT_CUDA(ctx, call)                                                             \
  do {                                                                                  \
    cudaError_t _e = (call);                                                            \
    if (_e != cudaSuccess)                                                              \
      return irt_fail((ctx), IRT_ERR_CUDA, "%s failed: %s (%s:%d)", #call,              \
                      cudaGetErrorString(_e), __FILE__, __LINE__);                      \
  } while (0)

// counts a kernel launch; with IRT_B200_DEBUG_SYNC=1 in the environment (read at context creation) it also
// synchronises the device and reports the first kernel that failed with its source line
void irt_launched(irt_ctx *ctx, const char *file, int line);
#define IRT_LAUNCHED(ctx) irt_launched((ctx), __FILE__, __LINE__)

// internal cross-file entry points
int env_rebuild_occ(irt_ctx *ctx, irt_env *env, cudaStream_t st);
int setstore_reserve(irt_ctx *ctx, irt_setstore *s, int64_t n_sets, int64_t n_blocks);
int setstore_finalize(irt_ctx *ctx, irt_setstore *s, int64_t n_sets, int64_t n_blocks,
                      cudaStream_t st);
// K3 over sets [begin, end) into device words, stream-ordered; the same argument checks as irt_check_sets_dev
int check_sets_launch(irt_ctx *ctx, const irt_setstore *store, const irt_env *env, int64_t begin, int64_t end,
                      uint32_t *d_verdict, cudaStream_t st);
// d_row_off == nullptr: dense outputs p/R/t[n][cap_pts]; else packed rows, configuration i at row d_row_off[i].
// d_range != nullptr: the batch is rows [lo, hi) of d_states and of the outputs, {lo, hi} read from device memory
// when the kernels run (n = upper bound of hi - lo); work = fk_work_bytes(rb, n) bytes of device scratch private
// to this launch (nullptr: the context's scratch buffer, one launch in flight per context).
size_t fk_work_bytes(const irt_robot *rb, int64_t n);
int fk_launch(irt_ctx *ctx, const irt_robot *rb, const double *d_states, int64_t n, int cap_pts,
              const irt_fk_outputs &o, cudaStream_t st, const int64_t *d_row_off = nullptr,
              const int32_t *d_range = nullptr, void *work = nullptr);
int fk_row_counts(irt_ctx *ctx, const irt_robot *rb, const double *d_states, int64_t n,
                  int64_t *d_counts, cudaStream_t st);
// same conventions for d_range / work (selfcol_work_bytes(n) bytes)
size_t selfcol_work_bytes(int64_t n);
int self_collision_launch(irt_ctx *ctx, const irt_robot *rb, const double *d_p,
                          const int32_t *d_npts, int64_t n, int cap_pts, uint32_t *d_flags,
                          cudaStream_t st, const int64_t *d_row_off = nullptr,
                          const int32_t *d_range = nullptr, void *work = nullptr);
