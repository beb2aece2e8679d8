// voxel_raster.cu -- K2 `swept_voxel_raster`: backbone polyline -> sparse voxel block sets,
// for roadmap vertices (one FK sample per set) and edges (adaptive swept volume).
//
// Replaces, behind the same results:
//   VoxelOctree::add_line / add_piecewise_line      collision/VoxelOctree.cpp:325-432
//   segment_aabox_intersect                         collision/collision_primitives.h:62-85
//   VoxelBackboneValidityChecker::voxelize_impl     motion-planning/VoxelBackboneValidityChecker.h:49-57
//   VoxelEnvironment::voxelize_valid_backbone_motion motion-planning/VoxelEnvironment.cpp:207-444
//   VoxelBackboneMotionValidator::generic_voxelize  motion-planning/VoxelBackboneMotionValidator.cpp:41-74
//
// B200-first structure (not a translation of the reference's per-edge LIFO loop):
//   * the bisection of ALL edges of a chunk runs level-synchronously: every round interpolates the
//     midpoints of all open intervals, runs ONE batched K1 launch (+ validity epilogue) over them,
//     then one warp per interval evaluates should_subdivide (VoxelEnvironment.cpp:304-341).  The
//     sample set this produces below the first invalid t equals the reference's depth-first
//     order exactly (DESIGN.md "level-synchronous bisection" has the argument).
//   * rasterisation: one warp per set; lanes take polyline segments, run the reference's voxel
//     traversal literally (same operation order, this file is compiled with -fmad=false so no
//     contraction changes a cell index) and OR cell bits into a shared-memory hash keyed by the
//     Morton block key; the table is then rank-sorted by key, which is the reference's
//     visit_leaves order, and written as {u32 key, u64 bits} records (8 consecutive keys = one
//     512-bit 2x2x2 super-block).  Two passes (count, exclusive scan, emit) give an exact CSR
//     without per-set capacity slots.
#include <cmath>
#include <cstring>
#include <vector>

#include <chrono>
#include <thread>

#include "common.cuh"

namespace {

#include "raster_line.h"   // D3, segment_aabox_intersect, add_line: shared with the host harness tests/cpp/test_raster_line_host.cpp

// IRT_B200_TRACE=1: per-phase wall-clock of the K2 host pipeline (synchronising; debugging only)
struct Trace {
  bool on;
  cudaStream_t st;
  std::chrono::steady_clock::time_point t0;
  explicit Trace(cudaStream_t s) : on(getenv("IRT_B200_TRACE") && getenv("IRT_B200_TRACE")[0] == '1'), st(s), t0(std::chrono::steady_clock::now()) {}
  void point(const char *name, long long count = -1) {
    if (!on) return;
    cudaStreamSynchronize(st);
    auto t1 = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[irt trace] %-28s %9.3f ms", name, std::chrono::duration<double, std::milli>(t1 - t0).count());
    if (count >= 0) std::fprintf(stderr, "  (%lld)", count);
    std::fprintf(stderr, "\n");
    t0 = std::chrono::steady_clock::now();
  }
};

// IRT_B200_TRACE=2: device timeline of the K2 pipeline -- timing events recorded on the lanes' streams (nothing
// synchronises until the call is over), printed relative to the first mark (debugging / profiling only)
struct Timeline {
  struct Mark { cudaEvent_t ev; const char *label; int lane; long long v; };
  bool on;
  std::vector<Mark> marks;
  std::chrono::steady_clock::time_point h0 = std::chrono::steady_clock::now();
  Timeline() { const char *e = getenv("IRT_B200_TRACE"); on = e && e[0] == '2'; }
  void host(const char *label) {   // host wall-clock since the timeline was created
    if (!on) return;
    std::fprintf(stderr, "[irt timeline host] %9.3f ms  %s\n",
                 std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count(), label);
  }
  void mark(cudaStream_t st, const char *label, int lane, long long v = -1) {
    if (!on) return;
    cudaEvent_t ev;
    if (cudaEventCreate(&ev) != cudaSuccess) return;
    cudaEventRecord(ev, st);
    marks.push_back({ev, label, lane, v});
  }
  void print() {
    if (!on || marks.empty()) return;
    cudaDeviceSynchronize();
    for (auto &m : marks) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, marks[0].ev, m.ev);
      std::fprintf(stderr, "[irt timeline] %9.3f ms  lane %d  %-18s %lld\n", ms, m.lane, m.label, m.v);
    }
    for (auto &m : marks) cudaEventDestroy(m.ev);
    marks.clear();
  }
};

constexpr int RS_WARPS = 4;
constexpr int ES_MINB = 4;   // resident CTAs per SM of the subdivision test
constexpr int RS_MINB = 6;   // resident CTAs per SM the main raster pass is compiled for (80 registers; 5 -> 6: -10 %, 7 and 8: no further gain)
constexpr int RS_HLOG_SMALL = 8;     // main pass: 256 hash entries per warp (a set rarely exceeds ~150 blocks)
constexpr int RS_HLOG_BIG = 12;      // fallback pass for the sets that overflow it: 4096 entries, 1 warp per CTA
constexpr int RS_SLOT = 1 << RS_HLOG_SMALL;   // slot capacity of the main pass
constexpr int RS_BIGSLOT = 1 << RS_HLOG_BIG;  // slot capacity of the fallback pass
constexpr int RS_MAX_OVF = 2048;     // fallback slots per raster launch
constexpr uint32_t RS_EMPTY = 0xffffffffu;
constexpr int RS_MAXS = 128;          // samples of one set handled by the flat segment walk
constexpr int rs_warp_bytes(int hlog) { return (1 << hlog) * 18 + 16 + RS_MAXS * 12; }
constexpr uint32_t INVALID_MASK = IRT_FLAG_NONCONVERGED | IRT_FLAG_LENGTH_LIMIT |
                                  IRT_FLAG_SELF_COLLISION | IRT_FLAG_BAD_STATE | IRT_FLAG_ENV_COLLISION;

__device__ __forceinline__ uint32_t spread3(uint32_t x) {
  x = (x | (x << 16)) & 0x030000FFu;
  x = (x | (x << 8)) & 0x0300F00Fu;
  x = (x | (x << 4)) & 0x030C30C3u;
  x = (x | (x << 2)) & 0x09249249u;
  return x;
}
// x is the most significant bit of each 3-bit group: child index 4*x + 2*y + z (TreeNode.h:66-68)
__device__ __forceinline__ uint32_t morton_key(uint32_t bx, uint32_t by, uint32_t bz) {
  return (spread3(bx) << 2) | (spread3(by) << 1) | spread3(bz);
}

__device__ __forceinline__ D3 rotate_pt(const GridDev &g, const double *p) {
  if (g.identity_rot) return {p[0], p[1], p[2]};
  // Eigen 3x3 * 3x1: (m0*b0 + m1*b1) + m2*b2
  return {(g.inv_rot[0] * p[0] + g.inv_rot[1] * p[1]) + g.inv_rot[2] * p[2],
          (g.inv_rot[3] * p[0] + g.inv_rot[4] * p[1]) + g.inv_rot[5] * p[2],
          (g.inv_rot[6] * p[0] + g.inv_rot[7] * p[1]) + g.inv_rot[8] * p[2]};
}

struct WarpHash {
  uint32_t *keys;   // [H]
  unsigned long long *bits;  // [H]
  uint16_t *list;   // [H] slots in insertion order (dense list of the occupied entries)
  uint32_t *count;  // number of occupied entries
  uint32_t *overflow;
  int hlog;         // H = 1 << hlog
};

__device__ __forceinline__ void hash_insert(const WarpHash &h, uint32_t key, unsigned long long mask) {
  const uint32_t H = 1u << h.hlog;
  if (*h.overflow) return;  // this set will be redone with the big table
  uint32_t slot = (key * 2654435761u) >> (32 - h.hlog);
  for (uint32_t probe = 0; probe < H; probe++) {
    const uint32_t old = atomicCAS(&h.keys[slot], RS_EMPTY, key);
    if (old == RS_EMPTY) {
      const uint32_t idx = atomicAdd(h.count, 1u);
      h.list[idx] = (uint16_t)slot;
      if (idx >= (H >> 2) * 3) *h.overflow = 1u;  // keep the load factor below 3/4
    }
    if (old == RS_EMPTY || old == key) {
      // bits are only ever OR-ed: two native 32-bit shared-memory ORs instead of a 64-bit CAS loop
      uint32_t *w = reinterpret_cast<uint32_t *>(&h.bits[slot]);
      if ((uint32_t)mask) atomicOr(w, (uint32_t)mask);
      if ((uint32_t)(mask >> 32)) atomicOr(w + 1, (uint32_t)(mask >> 32));
      return;
    }
    slot = (slot + 1) & (H - 1);
  }
  *h.overflow = 1u;
}

// VoxelOctree::set_cell(ix,iy,iz,true) -- collision/VoxelOctree.cpp:262-272,1501-1503.
// Consecutive cells of a segment mostly fall into the same 4x4x4 block: bits are collected in
// registers and flushed to the shared hash (one Morton key + one atomicOr) when the block changes.
struct BlockAcc {
  int bx = -1, by = 0, bz = 0;
  unsigned long long mask = 0ull;
};
// Inside the hash a block is keyed by its packed coordinates (two shifts); the Morton key (36 bit operations)
// is only formed for the occupied blocks of a finished set, ~23 per set instead of ~2 per segment.
__device__ __forceinline__ uint32_t linear_key(int bx, int by, int bz) {
  return ((uint32_t)bx << 16) | ((uint32_t)by << 8) | (uint32_t)bz;
}
__device__ __forceinline__ uint32_t morton_of_linear(uint32_t k) {
  return morton_key(k >> 16, (k >> 8) & 0xffu, k & 0xffu);
}
__device__ __forceinline__ void flush_block(const WarpHash &h, BlockAcc &acc) {
  if (acc.mask) hash_insert(h, linear_key(acc.bx, acc.by, acc.bz), acc.mask);
  acc.mask = 0ull;
}
__device__ __forceinline__ void set_cell(const WarpHash &h, BlockAcc &acc, int ix, int iy, int iz) {
  const int bx = ix >> 2, by = iy >> 2, bz = iz >> 2;
  if (bx != acc.bx || by != acc.by || bz != acc.bz) {
    flush_block(h, acc);
    acc.bx = bx; acc.by = by; acc.bz = bz;
  }
  acc.mask |= 1ull << ((ix & 3) * 16 + (iy & 3) * 4 + (iz & 3));
}

// cell sinks of the voxel traversal: HashSink builds a voxel set, EnvSink only asks whether any
// traversed cell is occupied in the environment (AbstractVoxelValidityChecker::collides of a shape)
struct HashSink {
  const WarpHash &h;
  BlockAcc acc;
  __device__ __forceinline__ explicit HashSink(const WarpHash &hh) : h(hh) {}
  __device__ __forceinline__ void cell(int ix, int iy, int iz) { set_cell(h, acc, ix, iy, iz); }
  __device__ __forceinline__ void finish() { flush_block(h, acc); }
};
// Collects the {block key, bit mask} pairs of ONE segment in registers (a backbone segment is shorter than a
// voxel: it touches one or two 4x4x4 blocks, three at a corner).  The warp then inserts the pairs of its 32
// segments together (warp_insert_pairs): consecutive segments of a backbone mostly fall into the same block, so
// lanes with equal keys merge their masks with a shuffle reduction and ONE lane per distinct key touches the
// hash -- instead of 4-8 lanes contending for the same shared-memory word with atomicCAS / atomicOr.
constexpr int RS_PAIRS = 3;
constexpr int RS_SEGS = 2;   // consecutive segments a lane handles per warp iteration
struct PairSink {
  const WarpHash &h;
  BlockAcc acc;
  uint32_t key[RS_PAIRS];
  unsigned long long mask[RS_PAIRS];
  int n = 0;
  __device__ __forceinline__ explicit PairSink(const WarpHash &hh) : h(hh) {
#pragma unroll
    for (int i = 0; i < RS_PAIRS; i++) { key[i] = RS_EMPTY; mask[i] = 0ull; }
  }
  __device__ __forceinline__ void push() {
    const unsigned long long m = acc.mask;
    if (!m) return;
    acc.mask = 0ull;
    const uint32_t k = linear_key(acc.bx, acc.by, acc.bz);
    bool placed = false;
#pragma unroll
    for (int i = 0; i < RS_PAIRS; i++) {   // selects, not branches: lanes change blocks at different times
      const bool hit = !placed && (key[i] == k || key[i] == RS_EMPTY);
      key[i] = hit ? k : key[i];
      mask[i] |= hit ? m : 0ull;
      placed = placed || hit;
    }
    if (!placed) hash_insert(h, k, m);   // more blocks than slots (a long segment): straight to the hash
  }
  __device__ __forceinline__ void cell(int ix, int iy, int iz) {
    const int bx = ix >> 2, by = iy >> 2, bz = iz >> 2;
    if (bx != acc.bx || by != acc.by || bz != acc.bz) {
      push();
      acc.bx = bx; acc.by = by; acc.bz = bz;
    }
    acc.mask |= 1ull << ((ix & 3) * 16 + (iy & 3) * 4 + (iz & 3));
  }
  __device__ __forceinline__ void finish() { push(); }
};
// all 32 lanes (converged): insert every lane's pairs.  Lanes hold consecutive segments, so equal keys sit in
// adjacent lanes: a segmented OR scan over the lanes (5 shuffle steps) leaves the union of a run of equal keys in
// its last lane, and only that lane touches the hash.
__device__ __forceinline__ void warp_insert_pairs(const WarpHash &h, const PairSink &ps) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int r = 0; r < RS_PAIRS; r++) {
    const uint32_t k = ps.key[r];
    if (!__any_sync(0xffffffffu, k != RS_EMPTY)) break;
    uint32_t lo = (uint32_t)ps.mask[r], hi = (uint32_t)(ps.mask[r] >> 32);
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t ok = __shfl_up_sync(0xffffffffu, k, d);
      const uint32_t olo = __shfl_up_sync(0xffffffffu, lo, d), ohi = __shfl_up_sync(0xffffffffu, hi, d);
      if (lane >= d && ok == k) { lo |= olo; hi |= ohi; }
    }
    const uint32_t nk = __shfl_down_sync(0xffffffffu, k, 1);
    if (k != RS_EMPTY && (lane == 31 || nk != k)) hash_insert(h, k, ((unsigned long long)hi << 32) | lo);
  }
}
struct EnvSink {
  const uint64_t *env;
  const uint32_t *occ;
  bool hit = false;
  __device__ __forceinline__ EnvSink(const uint64_t *e, const uint32_t *o) : env(e), occ(o) {}
  __device__ __forceinline__ void cell(int ix, int iy, int iz) {
    const uint32_t key = morton_key((uint32_t)ix >> 2, (uint32_t)iy >> 2, (uint32_t)iz >> 2);
    if ((occ[key >> 5] >> (key & 31)) & 1u)
      if ((env[key] >> ((ix & 3) * 16 + (iy & 3) * 4 + (iz & 3))) & 1ull) hit = true;
  }
  __device__ __forceinline__ void finish() {}
};

// ---- sample pools ---------------------------------------------------------------------------------
// Vertex pool: FK results of the edge endpoints (roadmap vertices), computed once and shared by all incident
// edges.  Mid pool: the samples the bisection creates.  A sample is named, relative to its edge, by an int32
// reference: >= 0 = index into the mid pool, -1 = endpoint a (t = 0), -2 = endpoint b (t = 1).
struct EdgePool {
  const double *v_state;    // [nv][S]
  const double *v_p;        // [nv][cap_pts][3]
  const int32_t *v_npts;    // [nv]
  const uint32_t *v_flags;  // [nv]
  int64_t nv;
  int64_t *pairs;           // [E][2] endpoint vertices of this chunk's edges
  double *thr;              // [E] rel_threshold
  unsigned long long *first_invalid;  // [E] double bits (positive -> uint order == double order)
  int32_t *head;            // [E] newest mid sample of the edge (linked through m_next) or -1
  uint32_t *eflags;         // [E]
  int32_t *m_edge, *m_next, *m_npts;
  uint32_t *m_flags;
  double *m_t, *m_state, *m_p;
  int32_t cap_mid, cap_q, E;
  int S, N, enable_rotation, enable_retraction, cap_pts;
};
__device__ __forceinline__ int64_t end_vertex(const EdgePool &P, int32_t edge, int32_t ref) {
  return P.pairs[2 * (int64_t)edge + (-1 - ref)];
}
__device__ __forceinline__ const double *smp_pts(const EdgePool &P, int32_t edge, int32_t ref) {
  return ref >= 0 ? P.m_p + (int64_t)ref * P.cap_pts * 3 : P.v_p + end_vertex(P, edge, ref) * P.cap_pts * 3;
}
__device__ __forceinline__ int smp_npts(const EdgePool &P, int32_t edge, int32_t ref) {
  return ref >= 0 ? P.m_npts[ref] : P.v_npts[end_vertex(P, edge, ref)];
}
__device__ __forceinline__ double smp_t(const EdgePool &P, int32_t ref) {
  return ref >= 0 ? P.m_t[ref] : (ref == -1 ? 0.0 : 1.0);
}

// device-side counters of one in-flight chunk (int32 words): the host never reads them between rounds
enum { C_NMID = 0, C_NPEND = 1, C_NQ0 = 2, C_NQ1 = 3, C_LO = 4, C_HI = 5, C_ERR = 6, C_WORDS = 16 };

// what a raster launch reads its sets from
struct SetSrc {
  int edge_mode;
  // vertex mode: set i = the single shape i (heads[i] < 0: invalid shape, empty set)
  const double *pts;
  const int32_t *npts;
  const int32_t *heads;
  int cap_pts;
  // edge mode: set e = endpoints + mid samples of edge e with t < tlimit[e] (VoxelEnvironment.cpp:406-422)
  EdgePool P;
  const double *tlimit;
};

// One warp per set.  Output: the set's occupied leaf blocks, key-sorted, in its slot (slot_keys / slot_bits),
// counts[set], optional t_last / nsamples.  A gather kernel then packs the slots into the CSR at
// the scanned offsets.  Per-set cost is proportional to the number of occupied blocks: occupied
// hash slots are kept in an append list, so neither the sort nor the clean-up scans the table.
// HLOG = RS_HLOG_SMALL: main pass over sets [set0, set0 + nsets); a set that outgrows the small table is
// appended to ovf_list and left for the HLOG = RS_HLOG_BIG pass, which works through that list (count on
// the device) with one warp per CTA and writes into the big slots.  Per-set arrays (counts, t_last,
// nsamples, set_flags, ovf_slot) are indexed relative to set0.
template <int HLOG, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, WARPS == 1 ? 1 : RS_MINB)
swept_voxel_raster_kernel(const GridDev g, const SetSrc src, int64_t set0, int64_t nsets,
                          uint32_t *__restrict__ counts, double *__restrict__ t_last,
                          int32_t *__restrict__ nsamples, uint32_t *__restrict__ slot_keys,
                          uint64_t *__restrict__ slot_bits, uint32_t *__restrict__ set_flags,
                          int32_t *__restrict__ ovf_list, int32_t *__restrict__ ovf_count,
                          int32_t *__restrict__ ovf_slot) {
  constexpr int H = 1 << HLOG;
  constexpr bool BIG = (HLOG == RS_HLOG_BIG);
  extern __shared__ unsigned long long rs_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // per warp: bits u64[H] | keys u32[H] | dense keys u32[H] | list u16[H] | count, overflow | sample list
  unsigned char *wbase = reinterpret_cast<unsigned char *>(rs_smem) + (size_t)warp * rs_warp_bytes(HLOG);
  WarpHash h;
  h.hlog = HLOG;
  h.bits = reinterpret_cast<unsigned long long *>(wbase);
  h.keys = reinterpret_cast<uint32_t *>(wbase + H * 8);
  uint32_t *dk = reinterpret_cast<uint32_t *>(wbase + H * 12);
  h.list = reinterpret_cast<uint16_t *>(wbase + H * 16);
  h.count = reinterpret_cast<uint32_t *>(wbase + H * 18);
  h.overflow = h.count + 1;
  const double **lp = reinterpret_cast<const double **>(wbase + H * 18 + 16);   // sample point arrays
  int32_t *lc = reinterpret_cast<int32_t *>(wbase + H * 18 + 16 + RS_MAXS * 8);  // first flat segment index
  for (int i = lane; i < H; i += 32) { h.keys[i] = RS_EMPTY; h.bits[i] = 0ull; }
  if (lane == 0) { *h.count = 0u; *h.overflow = 0u; }
  __syncwarp();

  const int64_t n_work = BIG ? (int64_t)min(*ovf_count, RS_MAX_OVF) : nsets;
  for (int64_t w = (int64_t)blockIdx.x * WARPS + warp; w < n_work; w += (int64_t)gridDim.x * WARPS) {
    const int64_t rel = BIG ? (int64_t)ovf_list[w] : w;
    const int64_t set = set0 + rel;
    double tl = 0.0;
    int ns = 0, nsm = 0, total = 0;
    // pass 1: list the included samples with their cumulative segment counts (flat work list)
    auto take = [&](const double *sp, int P) {
      if (P < 2) return;             // add_piecewise_line of fewer than 2 points adds nothing
      if (nsm < RS_MAXS) {
        if (lane == 0) { lp[nsm] = sp; lc[nsm] = total; }
        nsm++;
        total += P - 1;
      } else {  // very long sample lists: the remainder goes sample by sample
        for (int i = 1 + lane; i < P; i += 32) {
          HashSink sink(h);
          add_line(g, sink, rotate_pt(g, sp + 3 * (i - 1)), rotate_pt(g, sp + 3 * i));
        }
      }
    };
    if (!src.edge_mode) {
      const int32_t smp = src.heads[set];
      if (smp >= 0) {
        ns = 1;
        take(src.pts + (int64_t)smp * src.cap_pts * 3, src.npts[smp]);
      }
    } else {
      const EdgePool &P = src.P;
      const int32_t e = (int32_t)set;
      const double lim = src.tlimit[e];
      ns = 2;
      if (0.0 < lim) take(smp_pts(P, e, -1), smp_npts(P, e, -1));   // VoxelEnvironment.cpp:409: t < first_invalid_t
      if (1.0 < lim) { tl = 1.0; take(smp_pts(P, e, -2), smp_npts(P, e, -2)); }
      for (int32_t m = P.head[e]; m >= 0; m = P.m_next[m]) {
        ns++;
        const double t = P.m_t[m];
        if (!(t < lim)) continue;
        if (tl < t) tl = t;          // :419-422 last valid t
        take(P.m_p + (int64_t)m * P.cap_pts * 3, P.m_npts[m]);
      }
    }
    __syncwarp();
    // pass 2: a lane takes RS_SEGS consecutive segments of the concatenated polylines per iteration (the point
    // two segments of one sample share is transformed once; the block accumulator runs across both), then the
    // warp inserts the blocks of its 32 * RS_SEGS segments together
    {
      int k = 0;   // sample cursor: f only grows, so the sample a lane's segment belongs to only moves forward
      for (int f0 = 0; f0 < total; f0 += 32 * RS_SEGS) {
        PairSink sink(h);
        D3 prev = {0.0, 0.0, 0.0};
        bool have_prev = false;
#pragma unroll 1
        for (int sgm = 0; sgm < RS_SEGS; sgm++) {
          const int f = f0 + RS_SEGS * lane + sgm;
          if (f < total) {
            while (k + 1 < nsm && lc[k + 1] <= f) { k++; have_prev = false; }
            const int i = f - lc[k] + 1;  // segment (i-1, i) of sample k
            const double *sp = lp[k];
            const D3 a = have_prev ? prev : rotate_pt(g, sp + 3 * (i - 1));
            const D3 b = rotate_pt(g, sp + 3 * i);
            add_line(g, sink, a, b);
            prev = b;
            have_prev = true;
          }
        }
        warp_insert_pairs(h, sink);
      }
    }
    __syncwarp();
    const bool over = *h.overflow != 0u;
    const int used = (int)min(*h.count, (uint32_t)H);
    int cnt = used;
    int64_t slot_id = rel;
    if (!BIG && over) {
      // defer to the big-table pass (or give up with a flag when its slots are exhausted)
      cnt = 0;
      if (lane == 0) {
        const int32_t idx = atomicAdd(ovf_count, 1);
        if (idx < RS_MAX_OVF) ovf_list[idx] = (int32_t)rel;
        else if (set_flags) set_flags[rel] |= IRT_FLAG_CAPACITY;
      }
    } else {
      if (BIG) {
        slot_id = w;
        if (over && lane == 0 && set_flags) set_flags[rel] |= IRT_FLAG_CAPACITY;
      }
      for (int i = lane; i < cnt; i += 32) dk[i] = morton_of_linear(h.keys[h.list[i]]);
      __syncwarp();
      // rank sort by key == the reference's visit_leaves order
      uint32_t *sk = slot_keys + slot_id * H;
      uint64_t *sb = slot_bits + slot_id * H;
      for (int i = lane; i < cnt; i += 32) {
        const uint32_t k = dk[i];
        int rank = 0;
        for (int j = 0; j < cnt; j++) rank += (dk[j] < k);
        sk[rank] = k;
        sb[rank] = h.bits[h.list[i]];
      }
    }
    if (lane == 0) {
      counts[rel] = (uint32_t)cnt;
      if (BIG) ovf_slot[rel] = (int32_t)w + 1;
      if (t_last) t_last[rel] = tl;
      if (nsamples) nsamples[rel] = ns;
    }
    __syncwarp();
    for (int i = lane; i < used; i += 32) {  // clean only what was used
      const int sl = h.list[i];
      h.keys[sl] = RS_EMPTY;
      h.bits[sl] = 0ull;
    }
    __syncwarp();
    if (lane == 0) { *h.count = 0u; *h.overflow = 0u; }
    __syncwarp();
  }
}

// voxelize_until_invalid: a sample is also invalid when its own backbone voxels hit the
// environment (_vc->collides(shape), VoxelBackboneMotionValidator.cpp:83-91).  One warp per
// sample of rows [lo, hi) (device range, or [0, n)); no set is built, the traversal just probes the grid.
__global__ void sample_env_collision_kernel(const GridDev g, const double *__restrict__ pts,
                                            const int32_t *__restrict__ npts, int cap_pts, int64_t n_host,
                                            const int32_t *__restrict__ range,
                                            const uint64_t *__restrict__ env, const uint32_t *__restrict__ occ,
                                            uint32_t *__restrict__ flags) {
  const int lane = threadIdx.x & 31;
  int64_t lo = 0, n = n_host;
  if (range) { lo = range[0]; n = (int64_t)range[1] - lo; }
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n; w += nwarps) {
    const int64_t smp = lo + w;
    if (flags[smp] & INVALID_MASK) continue;  // is_valid_shape short-circuits the collision check
    const int P = npts[smp];
    const double *sp = pts + smp * (int64_t)cap_pts * 3;
    EnvSink sink(env, occ);
    for (int i = 1 + lane; i < P; i += 32) add_line(g, sink, rotate_pt(g, sp + 3 * (i - 1)), rotate_pt(g, sp + 3 * i));
    if (__any_sync(0xffffffffu, sink.hit) && lane == 0) flags[smp] |= IRT_FLAG_ENV_COLLISION;
  }
}

// pack the slots into the CSR: one warp per set, coalesced copies.  A store that is too small for the
// leaves raises *overflow and leaves the set out (the caller re-runs with the measured size).
__global__ void raster_gather_kernel(const uint32_t *__restrict__ slot_keys, const uint64_t *__restrict__ slot_bits,
                                     const uint32_t *__restrict__ big_keys, const uint64_t *__restrict__ big_bits,
                                     const int32_t *__restrict__ ovf_slot,
                                     const uint32_t *__restrict__ counts, const uint64_t *__restrict__ offsets,
                                     int64_t nsets, uint32_t *__restrict__ out_keys, uint64_t *__restrict__ out_bits,
                                     uint64_t cap_blocks, int32_t *__restrict__ overflow) {
  const int lane = threadIdx.x & 31;
  const int64_t set = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (set >= nsets) return;
  const uint32_t n = counts[set];
  const uint64_t base = offsets[set];
  if (base + n > cap_blocks) {
    if (lane == 0 && n) *overflow = 1;
    return;
  }
  const int32_t ov = ovf_slot[set];
  const uint32_t *sk = ov ? big_keys + (int64_t)(ov - 1) * RS_BIGSLOT : slot_keys + set * RS_SLOT;
  const uint64_t *sb = ov ? big_bits + (int64_t)(ov - 1) * RS_BIGSLOT : slot_bits + set * RS_SLOT;
  for (uint32_t i = lane; i < n; i += 32) {
    out_keys[base + i] = sk[i];
    out_bits[base + i] = sb[i];
  }
}

// ---- exclusive scan: uint32 counts -> uint64 offsets (n+1 entries) ------------------------
constexpr int SCAN_T = 256, SCAN_ITEMS = 8, SCAN_TILE = SCAN_T * SCAN_ITEMS;

__global__ void scan_tile_sums_kernel(const uint32_t *__restrict__ in, int64_t n,
                                      uint64_t *__restrict__ tile_sums) {
  __shared__ uint64_t sh[SCAN_T / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
  uint64_t s = 0;
  for (int k = 0; k < SCAN_ITEMS; k++) {
    const int64_t i = base + (int64_t)k * SCAN_T + threadIdx.x;
    if (i < n) s += in[i];
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint64_t t = 0;
    for (int w = 0; w < SCAN_T / 32; w++) t += sh[w];
    tile_sums[blockIdx.x] = t;
  }
}

// tile_sums[i] <- running + exclusive prefix; running += total  (running: leaves appended to the store so far;
// chained on the device from raster launch to raster launch, the host only reads it at the very end)
__global__ void scan_tile_offsets_kernel(uint64_t *tile_sums, int64_t ntiles, uint64_t *running) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    uint64_t acc = *running;
    for (int64_t i = 0; i < ntiles; i++) {
      const uint64_t c = tile_sums[i];
      tile_sums[i] = acc;
      acc += c;
    }
    *running = acc;
  }
}

__global__ void scan_apply_kernel(const uint32_t *__restrict__ in, int64_t n,
                                  const uint64_t *__restrict__ tile_sums,
                                  const uint64_t *__restrict__ running,
                                  uint64_t *__restrict__ out) {
  // thread t owns SCAN_ITEMS consecutive items of the tile
  __shared__ uint64_t sh[SCAN_T];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS];
  uint64_t s = 0;
  for (int k = 0; k < SCAN_ITEMS; k++) {
    v[k] = (base + k < n) ? in[base + k] : 0u;
    s += v[k];
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < SCAN_T; o <<= 1) {  // Hillis-Steele inclusive scan of the thread sums
    uint64_t add = (threadIdx.x >= o) ? sh[threadIdx.x - o] : 0;
    __syncthreads();
    sh[threadIdx.x] += add;
    __syncthreads();
  }
  uint64_t acc = tile_sums[blockIdx.x] + sh[threadIdx.x] - s;
  for (int k = 0; k < SCAN_ITEMS; k++) {
    if (base + k < n) out[base + k] = acc;
    acc += v[k];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = *running;
}

// offsets[0..n] = *d_running + exclusive scan of counts[0..n); *d_running += sum(counts).  No host sync.
int exclusive_scan_chained(irt_ctx *ctx, const uint32_t *d_counts, int64_t n, uint64_t *d_running,
                           uint64_t *d_offsets, uint64_t *d_tmp /* ntiles + 1 */, cudaStream_t st) {
  const int64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  scan_tile_sums_kernel<<<(unsigned)ntiles, SCAN_T, 0, st>>>(d_counts, n, d_tmp);
  IRT_LAUNCHED(ctx);
  scan_tile_offsets_kernel<<<1, 32, 0, st>>>(d_tmp, ntiles, d_running);
  IRT_LAUNCHED(ctx);
  scan_apply_kernel<<<(unsigned)ntiles, SCAN_T, 0, st>>>(d_counts, n, d_tmp, d_running, d_offsets);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  return IRT_OK;
}

// ---- vertex mode helpers --------------------------------------------------------------------
__global__ void vertex_heads_kernel(const uint32_t *__restrict__ flags, int64_t n,
                                    int32_t *__restrict__ heads) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) heads[i] = (flags[i] & INVALID_MASK) ? -1 : (int32_t)i;
}

// ---- edge mode: level-synchronous bisection, driven from the device ----------------------------
struct Interval {
  int32_t edge, ia, ib;   // ia / ib: sample references (see EdgePool)
};
struct Pending {
  int32_t edge, ia, im, ib;
};

// OMPL compound interpolate restated (RealVector linear, SO2 shortest arc + wrap), the `interp`
// lambda of VoxelBackboneMotionValidator.cpp:58-66
__device__ void interpolate_state(const EdgePool &P, const double *a, const double *b, double t,
                                  double *out) {
  const double pi = 3.14159265358979323846;
  for (int i = 0; i < P.N; i++) out[i] = a[i] + (b[i] - a[i]) * t;
  int idx = P.N;
  if (P.enable_rotation) {
    double diff = b[idx] - a[idx];
    if (fabs(diff) <= pi) {
      out[idx] = a[idx] + diff * t;
    } else {
      if (diff > 0.0) diff = 2.0 * pi - diff;
      else diff = -2.0 * pi - diff;
      double v = a[idx] - diff * t;
      if (v > pi) v -= 2.0 * pi;
      else if (v < -pi) v += 2.0 * pi;
      out[idx] = v;
    }
    idx++;
  }
  if (P.enable_retraction) out[idx] = a[idx] + (b[idx] - a[idx]) * t;
}

// one thread per edge of the chunk: validates / clamps the endpoint indices, rel_threshold =
// 1 / validSegmentCount(a, b) (VoxelBackboneMotionValidator.cpp:55-56, the same arithmetic as
// irt_valid_segment_count: this file is compiled without FMA contraction), first_invalid_t from the endpoint
// validity (VoxelEnvironment.cpp:261-268), empty sample list
__global__ void edge_init_kernel(EdgePool P, int32_t *__restrict__ C, double len_t, double len_r, double len_s) {
  const int32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P.E) return;
  int64_t va = P.pairs[2 * (int64_t)e], vb = P.pairs[2 * (int64_t)e + 1];
  if (va < 0 || va >= P.nv || vb < 0 || vb >= P.nv) {   // reported as IRT_ERR_OUT_OF_RANGE by the host
    atomicOr(&C[C_ERR], 1);
    va = (va < 0 || va >= P.nv) ? 0 : va;
    vb = (vb < 0 || vb >= P.nv) ? 0 : vb;
    P.pairs[2 * (int64_t)e] = va;
    P.pairs[2 * (int64_t)e + 1] = vb;
  }
  const double pi = 3.14159265358979323846;
  const double *ea = P.v_state + va * P.S, *eb = P.v_state + vb * P.S;
  double d2 = 0;
  for (int i = 0; i < P.N; i++) d2 += (ea[i] - eb[i]) * (ea[i] - eb[i]);
  unsigned sc = (unsigned)ceil(sqrt(d2) / len_t);
  int idx = P.N;
  if (P.enable_rotation) {
    double d = fabs(ea[idx] - eb[idx]);
    d = (d > pi) ? 2.0 * pi - d : d;
    const unsigned c = (unsigned)ceil(d / len_r);
    if (c > sc) sc = c;
    idx++;
  }
  if (P.enable_retraction) {
    const double d = sqrt((ea[idx] - eb[idx]) * (ea[idx] - eb[idx]));
    const unsigned c = (unsigned)ceil(d / len_s);
    if (c > sc) sc = c;
  }
  P.thr[e] = 1.0 / double(sc);
  double fi = 10.0;                                       // VoxelEnvironment.cpp:261
  if (P.v_flags[va] & INVALID_MASK) fi = 0.0;             // :266-268: the smallest invalid t
  else if (P.v_flags[vb] & INVALID_MASK) fi = 1.0;
  P.first_invalid[e] = (unsigned long long)__double_as_longlong(fi);
  P.head[e] = -1;
  P.eflags[e] = 0u;
}

// non-indexed entry points: the endpoints of edge e are vertices 2e and 2e+1 of the chunk's own vertex pool
__global__ void edge_identity_pairs_kernel(int64_t *__restrict__ pairs, int32_t E) {
  const int32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E) { pairs[2 * (int64_t)e] = 2 * (int64_t)e; pairs[2 * (int64_t)e + 1] = 2 * (int64_t)e + 1; }
}

// start of a round: the samples created from here on are [lo, ...); the queue this round fills is empty
__global__ void round_begin_kernel(int32_t *__restrict__ C, int32_t cap_mid, int q_next) {
  if (threadIdx.x == 0) {
    C[C_LO] = min(C[C_NMID], cap_mid);
    C[C_NPEND] = 0;
    C[C_NQ0 + q_next] = 0;
  }
}
__global__ void round_mid_kernel(int32_t *__restrict__ C, int32_t cap_mid) {
  if (threadIdx.x == 0) C[C_HI] = min(C[C_NMID], cap_mid);
}

// one thread per open interval: VoxelEnvironment.cpp:369-384
__global__ void edge_split_kernel(EdgePool P, const Interval *__restrict__ cur, int32_t *__restrict__ C, int q_cur,
                                  Pending *__restrict__ pend) {
  const int32_t ncur = min(C[C_NQ0 + q_cur], P.cap_q);
  for (int32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < ncur; q += gridDim.x * blockDim.x) {
    const Interval iv = cur[q];
    const double ta = smp_t(P, iv.ia), tb = smp_t(P, iv.ib);
    if ((tb - ta) <= P.thr[iv.edge]) continue;
    const double fi = __longlong_as_double((long long)P.first_invalid[iv.edge]);
    if (fi <= ta) continue;
    const int32_t m = atomicAdd(&C[C_NMID], 1);
    if (m >= P.cap_mid) {   // pool full: the host sees C_NMID > cap_mid and redoes the chunk in two halves
      atomicOr(&P.eflags[iv.edge], IRT_FLAG_CAPACITY);
      continue;
    }
    const double tm = (ta + tb) / 2;
    P.m_edge[m] = iv.edge;
    P.m_t[m] = tm;
    interpolate_state(P, P.v_state + end_vertex(P, iv.edge, -1) * P.S, P.v_state + end_vertex(P, iv.edge, -2) * P.S,
                      tm, P.m_state + (int64_t)m * P.S);
    P.m_next[m] = atomicExch(&P.head[iv.edge], m);
    const int32_t k = atomicAdd(&C[C_NPEND], 1);
    pend[k] = Pending{iv.edge, iv.ia, m, iv.ib};
  }
}

// after FK: invalid samples lower first_invalid_t of their edge (VoxelEnvironment.cpp:266-268)
__global__ void edge_mark_kernel(EdgePool P, const int32_t *__restrict__ C) {
  const int32_t lo = C[C_LO], hi = C[C_HI];
  for (int32_t i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x)
    if (P.m_flags[i] & INVALID_MASK)
      atomicMin(&P.first_invalid[P.m_edge[i]], (unsigned long long)__double_as_longlong(P.m_t[i]));
}

// should_subdivide(a, b) -- VoxelEnvironment.cpp:304-341, warp-cooperative: lanes over points, scanned from the
// tip like the reference so the first event found is the same one.  A bisected interval needs TWO such tests
// (a, m) and (m, b) (VoxelEnvironment.cpp:350-353, 386-397); the kernel is bound by memory latency (a chain of
// sample header -> points of the top 32 nodes -> next 32 ...), so both tests of an interval run in ONE loop with
// all their loads issued together: 3 dependent rounds per interval instead of 6.
struct SmpView {
  const double *p;
  int n;
  uint32_t flags;
};
__device__ __forceinline__ SmpView smp_view(const EdgePool &P, int32_t edge, int32_t ref) {
  SmpView s;
  if (ref >= 0) {
    s.p = P.m_p + (int64_t)ref * P.cap_pts * 3; s.n = P.m_npts[ref]; s.flags = P.m_flags[ref];
  } else {
    const int64_t v = end_vertex(P, edge, ref);
    s.p = P.v_p + v * P.cap_pts * 3; s.n = P.v_npts[v]; s.flags = P.v_flags[v];
  }
  return s;
}
// event of one point pair: 0 = cells at most 1 apart, 1 = far apart, 2 = domain error (a point outside the grid)
__device__ __forceinline__ int pair_event(const GridDev &g, const D3 &ra, const D3 &rb) {
  const double pa[3] = {ra.x, ra.y, ra.z}, pb[3] = {rb.x, rb.y, rb.z};
  return pair_event_core(g, rotate_pt(g, pa), rotate_pt(g, pb));   // raster_line.h
}
// up to two tests at once: test 0 = (x0, y0), test 1 = (x1, y1); run[t] selects; res[t] = should_subdivide
__device__ __forceinline__ void should_subdivide2(const GridDev &g, const EdgePool &P, int32_t edge, const SmpView &x0,
                                                  const SmpView &y0, const SmpView &x1, const SmpView &y1, bool run0,
                                                  bool run1, int lane, bool &res0, bool &res1) {
  res0 = res1 = false;
  bool live0 = run0 && !(x0.flags & INVALID_MASK), live1 = run1 && !(x1.flags & INVALID_MASK);
  if (live0 && (x0.n + 1 < y0.n || x0.n > y0.n + 1)) { res0 = true; live0 = false; }
  if (live1 && (x1.n + 1 < y1.n || x1.n > y1.n + 1)) { res1 = true; live1 = false; }
  int top0 = min(x0.n, y0.n) - 1, top1 = min(x1.n, y1.n) - 1;
  if (top0 < 0) live0 = false;
  if (top1 < 0) live1 = false;
  while (live0 || live1) {   // warp-uniform
    const int i0 = top0 - lane, i1 = top1 - lane;
    // all twelve coordinates of this round are requested before any of them is looked at
    const bool act0 = live0 && i0 >= 0, act1 = live1 && i1 >= 0;
    const D3 zero = {0.0, 0.0, 0.0};
    D3 xa = zero, ya = zero, xb = zero, yb = zero;
    if (act0) {
      const double *px = x0.p + 3 * i0, *py = y0.p + 3 * i0;
      xa = {px[0], px[1], px[2]}; ya = {py[0], py[1], py[2]};
    }
    if (act1) {
      const double *px = x1.p + 3 * i1, *py = y1.p + 3 * i1;
      xb = {px[0], px[1], px[2]}; yb = {py[0], py[1], py[2]};
    }
    const int ev0 = act0 ? pair_event(g, xa, ya) : 0;
    const int ev1 = act1 ? pair_event(g, xb, yb) : 0;
    const unsigned m0 = __ballot_sync(0xffffffffu, ev0 != 0), m1 = __ballot_sync(0xffffffffu, ev1 != 0);
    if (live0) {
      if (m0) {
        const int fev = __shfl_sync(0xffffffffu, ev0, __ffs(m0) - 1);   // lane 0 holds the highest index
        if (fev == 2) { if (lane == 0) atomicOr(&P.eflags[edge], IRT_FLAG_OUT_OF_DOMAIN); }
        else res0 = true;
        live0 = false;
      } else if ((top0 -= 32) < 0) live0 = false;
    }
    if (live1) {
      if (m1) {
        const int fev = __shfl_sync(0xffffffffu, ev1, __ffs(m1) - 1);
        if (fev == 2) { if (lane == 0) atomicOr(&P.eflags[edge], IRT_FLAG_OUT_OF_DOMAIN); }
        else res1 = true;
        live1 = false;
      } else if ((top1 -= 32) < 0) live1 = false;
    }
  }
}

// one warp per candidate: round 0 tests the whole edge (a, b); later rounds test both halves of a bisected
// interval (VoxelEnvironment.cpp:350-353,386-397)
__global__ void __launch_bounds__(256, ES_MINB)
edge_subdivide_kernel(const GridDev g, EdgePool P, const Pending *__restrict__ pend,
                      int32_t *__restrict__ C, Interval *__restrict__ next, int q_next) {
  const int lane = threadIdx.x & 31;
  const int32_t total = pend ? min(C[C_NPEND], P.cap_mid) : P.E;
  const int32_t nwarps = (gridDim.x * blockDim.x) >> 5;
  int32_t *n_next = &C[C_NQ0 + q_next];
  for (int32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < total; w += nwarps) {
    if (!pend) {
      const int32_t e = w;
      const SmpView a = smp_view(P, e, -1), b = smp_view(P, e, -2);
      bool whole, unused;
      should_subdivide2(g, P, e, a, b, a, b, true, false, lane, whole, unused);
      if (whole && lane == 0) {
        const int32_t k = atomicAdd(n_next, 1);
        if (k < P.cap_q) next[k] = Interval{e, -1, -2};
        else atomicOr(&P.eflags[e], IRT_FLAG_CAPACITY);
      }
      continue;
    }
    const Pending pd = pend[w];
    const SmpView a = smp_view(P, pd.edge, pd.ia), m = smp_view(P, pd.edge, pd.im), b = smp_view(P, pd.edge, pd.ib);
    bool distal, proximal;
    should_subdivide2(g, P, pd.edge, m, b, a, m, true, true, lane, distal, proximal);
    if (lane == 0) {
      if (distal) {
        const int32_t k = atomicAdd(n_next, 1);
        if (k < P.cap_q) next[k] = Interval{pd.edge, pd.im, pd.ib};
        else atomicOr(&P.eflags[pd.edge], IRT_FLAG_CAPACITY);
      }
      if (proximal) {
        const int32_t k = atomicAdd(n_next, 1);
        if (k < P.cap_q) next[k] = Interval{pd.edge, pd.ia, pd.im};
        else atomicOr(&P.eflags[pd.edge], IRT_FLAG_CAPACITY);
      }
    }
  }
}

__global__ void edge_finish_kernel(EdgePool P, double *__restrict__ tlimit, uint32_t *__restrict__ flags_out) {
  const int32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P.E) return;
  const double fi = __longlong_as_double((long long)P.first_invalid[e]);
  tlimit[e] = fi;
  uint32_t f = P.eflags[e];
  if (!(5.0 < fi)) f |= IRT_FLAG_PARTIAL;  // VoxelEnvironment.cpp:438
  flags_out[e] = f;
}

// bump allocator over the context's grow-only K2 arena.  Layouts are described once by a
// lambda and run twice: a dry run to size the arena, then the real carve-up.
struct Arena {
  char *base = nullptr;
  size_t cap = 0, used = 0;
  bool dry = true;
  template <typename T>
  bool alloc(T **out, size_t count) {
    const size_t bytes = ((count ? count : 1) * sizeof(T) + 255) & ~(size_t)255;
    if (dry) { *out = nullptr; used += bytes; return true; }
    if (used + bytes > cap) return false;
    *out = reinterpret_cast<T *>(base + used);
    used += bytes;
    return true;
  }
};
template <typename F>
int arena_layout(irt_ctx *ctx, const F &layout) {
  Arena dry;
  layout(dry);
  char *base = (char *)ctx_arena(ctx, dry.used);
  if (!base) return irt_fail(ctx, IRT_ERR_CUDA, "K2 arena allocation of %zu bytes failed", dry.used);
  Arena real;
  real.base = base; real.cap = dry.used; real.dry = false;
  if (!layout(real)) return irt_fail(ctx, IRT_ERR_CUDA, "K2 arena layout failed");
  return IRT_OK;
}

constexpr int64_t RS_CHUNK_SETS = 524288;  // sets rasterised per launch (slot scratch = 3 KiB per set)

struct RasterScratch {
  uint32_t *slot_keys = nullptr, *big_keys = nullptr;
  uint64_t *slot_bits = nullptr, *big_bits = nullptr;
  uint32_t *counts = nullptr;
  uint64_t *scan_tmp = nullptr;
  int32_t *ovf_list = nullptr, *ovf_count = nullptr, *ovf_slot = nullptr;
  int64_t chunk = 0;
  template <typename A>
  bool layout(A &a, int64_t chunk_sets) {
    chunk = chunk_sets;
    const int64_t ntiles = (chunk + SCAN_TILE - 1) / SCAN_TILE;
    return a.alloc(&slot_keys, (size_t)chunk * RS_SLOT) && a.alloc(&slot_bits, (size_t)chunk * RS_SLOT) &&
           a.alloc(&big_keys, (size_t)RS_MAX_OVF * RS_BIGSLOT) && a.alloc(&big_bits, (size_t)RS_MAX_OVF * RS_BIGSLOT) &&
           a.alloc(&counts, (size_t)chunk) && a.alloc(&scan_tmp, (size_t)ntiles + 2) &&
           a.alloc(&ovf_list, (size_t)RS_MAX_OVF) && a.alloc(&ovf_count, 64) && a.alloc(&ovf_slot, (size_t)chunk);
  }
};

// Rasterise sets [0, nsets) of `src` and APPEND them to the store: they become store sets
// [set_base, set_base + nsets), their leaves follow the *d_running leaves already there (device-chained:
// no host synchronisation; *d_running advances).  A store too small for the leaves raises *d_overflow.
// Per-set outputs (d_tlast, d_nsamples, d_setflags) are indexed like the sets of `src`.
int raster_append(irt_ctx *ctx, const GridDev &g, const SetSrc &src, int64_t nsets, double *d_tlast,
                  int32_t *d_nsamples, uint32_t *d_setflags, RasterScratch &rs, irt_setstore *store,
                  int64_t set_base, uint64_t *d_running, int32_t *d_overflow, cudaStream_t st) {
  auto k_small = swept_voxel_raster_kernel<RS_HLOG_SMALL, RS_WARPS>;
  auto k_big = swept_voxel_raster_kernel<RS_HLOG_BIG, 1>;
  const int smem_small = RS_WARPS * rs_warp_bytes(RS_HLOG_SMALL), smem_big = rs_warp_bytes(RS_HLOG_BIG);
  IRT_CUDA(ctx, cudaFuncSetAttribute(k_big, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_big));
  for (int64_t c0 = 0; c0 < nsets; c0 += rs.chunk) {
    const int64_t m = (nsets - c0 < rs.chunk) ? (nsets - c0) : rs.chunk;
    int64_t blocks = (m + RS_WARPS - 1) / RS_WARPS;
    const int64_t max_blocks = (int64_t)ctx->sm_count * 16;
    if (blocks > max_blocks) blocks = max_blocks;
    IRT_CUDA(ctx, cudaMemsetAsync(rs.ovf_count, 0, 4, st));
    IRT_CUDA(ctx, cudaMemsetAsync(rs.ovf_slot, 0, (size_t)m * 4, st));
    k_small<<<(unsigned)blocks, RS_WARPS * 32, smem_small, st>>>(
        g, src, c0, m, rs.counts, d_tlast ? d_tlast + c0 : nullptr, d_nsamples ? d_nsamples + c0 : nullptr,
        rs.slot_keys, rs.slot_bits, d_setflags ? d_setflags + c0 : nullptr, rs.ovf_list, rs.ovf_count, rs.ovf_slot);
    IRT_LAUNCHED(ctx);
    // sets that outgrew the small table (normally none): big-table pass over the device-side list
    k_big<<<(unsigned)ctx->sm_count, 32, smem_big, st>>>(
        g, src, c0, m, rs.counts, d_tlast ? d_tlast + c0 : nullptr, d_nsamples ? d_nsamples + c0 : nullptr,
        rs.big_keys, rs.big_bits, d_setflags ? d_setflags + c0 : nullptr, rs.ovf_list, rs.ovf_count, rs.ovf_slot);
    IRT_LAUNCHED(ctx);
    IRT_CUDA(ctx, cudaGetLastError());
    int rc = exclusive_scan_chained(ctx, rs.counts, m, d_running, store->d_offsets + set_base + c0, rs.scan_tmp, st);
    if (rc) return rc;
    const int T = 256;
    raster_gather_kernel<<<(unsigned)((m * 32 + T - 1) / T), T, 0, st>>>(
        rs.slot_keys, rs.slot_bits, rs.big_keys, rs.big_bits, rs.ovf_slot, rs.counts,
        store->d_offsets + set_base + c0, m, store->d_keys, store->d_bits, (uint64_t)store->cap_blocks - 4,
        d_overflow);
    IRT_LAUNCHED(ctx);
    IRT_CUDA(ctx, cudaGetLastError());
  }
  return IRT_OK;
}

// device words shared by the raster launches of one call: [0] running leaf total (u64), [1] overflow flag
struct RasterTotals {
  uint64_t *d_running = nullptr;
  int32_t *d_overflow = nullptr;
  template <typename A>
  bool layout(A &a) {
    uint64_t *w = nullptr;
    if (!a.alloc(&w, 4)) return false;
    d_running = w;
    d_overflow = reinterpret_cast<int32_t *>(w + 1);
    return true;
  }
  int reset(irt_ctx *ctx, cudaStream_t st) {
    IRT_CUDA(ctx, cudaMemsetAsync(d_running, 0, 16, st));
    return IRT_OK;
  }
  // total leaves / overflow flag after everything on `st` has run
  int read(irt_ctx *ctx, cudaStream_t st, uint64_t *total, bool *overflow) {
    uint64_t h[2] = {0, 0};
    IRT_CUDA(ctx, cudaMemcpyAsync(h, d_running, 16, cudaMemcpyDeviceToHost, st));
    IRT_CUDA(ctx, cudaStreamSynchronize(st));
    *total = h[0];
    *overflow = (h[1] & 0xffffffffull) != 0;
    return IRT_OK;
  }
};

}  // namespace

// ===============================================================================================
// C ABI
// ===============================================================================================
extern "C" {

uint32_t irt_valid_segment_count(const irt_robot_desc *rb, const irt_space *sp, const double *a,
                                 const double *b) {
  // OMPL 1.5 documented behaviour: StateSpace::validSegmentCount = ceil(distance /
  // longestValidSegment), longestValidSegment = maximumExtent * fraction (fractions set in
  // motion-planning/Problem.cpp:118-144); CompoundStateSpace takes the max over subspaces.
  const int N = rb->n_tendons;
  double ext2 = 0;
  for (int i = 0; i < N; i++) ext2 += rb->max_tension[i] * rb->max_tension[i];
  const double tendon_extent = std::sqrt(ext2);
  const double len_t = tendon_extent * (sp->min_tension_change / tendon_extent);
  double d2 = 0;
  for (int i = 0; i < N; i++) d2 += (a[i] - b[i]) * (a[i] - b[i]);
  unsigned sc = (unsigned)std::ceil(std::sqrt(d2) / len_t);
  int idx = N;
  if (rb->enable_rotation) {
    const double len_r = M_PI * (sp->min_rotation_change / (2 * M_PI));
    double d = std::fabs(a[idx] - b[idx]);
    d = (d > M_PI) ? 2.0 * M_PI - d : d;
    unsigned c = (unsigned)std::ceil(d / len_r);
    if (c > sc) sc = c;
    idx++;
  }
  if (rb->enable_retraction) {
    const double len_s = rb->L * std::fmin(0.01, sp->min_retraction_change / rb->L);
    double d = std::sqrt((a[idx] - b[idx]) * (a[idx] - b[idx]));
    unsigned c = (unsigned)std::ceil(d / len_s);
    if (c > sc) sc = c;
  }
  return sc;
}

}  // extern "C"

static int store_begin(irt_ctx *ctx, irt_setstore *store, int64_t n, int64_t est_blocks, cudaStream_t st) {
  int rc = setstore_reserve(ctx, store, n, est_blocks);
  if (rc) return rc;
  if (n == 0) IRT_CUDA(ctx, cudaMemsetAsync(store->d_offsets, 0, 8, st));
  return IRT_OK;
}

static int check_dl_vs_grid(irt_ctx *ctx, const irt_robot *rb, const GridDev &g) {
  // VoxelBackboneValidityChecker ctor: dL must not exceed the largest voxel side (.h:37-45)
  const double dmax = std::fmax(g.d[0], std::fmax(g.d[1], g.d[2]));
  if (rb->desc.dL > dmax)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT,
                    "robot.specs.dL is larger than expected by VoxelBackboneValidityChecker (%g > %g)",
                    rb->desc.dL, dmax);
  return IRT_OK;
}

// vertex sets: FK + validity + raster, chunk by chunk; the leaf offsets chain on the device, so the only host
// synchronisation is the one at the end (and per chunk when the caller wants flags / tips on the host).
// A store that turns out too small is grown to the measured size and the call repeated (once).
static int voxelize_vertices_impl(irt_ctx *ctx, const irt_robot *rb, const double *states, const double *p_in,
                                  const int32_t *npts_in, int cap, int state_size, int64_t n, irt_setstore *store,
                                  uint32_t *flags, double *tips, int64_t est_blocks) {
  const GridDev &g = store->gd;
  cudaStream_t st = ctx->stream;
  int rc = store_begin(ctx, store, n, est_blocks, st);
  if (rc) return rc;
  if (n == 0) return setstore_finalize(ctx, store, 0, 0, st);
  const int S = state_size;
  const int64_t chunk = std::min<int64_t>(n, 262144);
  double *d_states = nullptr, *d_p = nullptr, *d_tip = nullptr;
  int32_t *d_npts = nullptr, *d_heads = nullptr;
  uint32_t *d_flags = nullptr;
  RasterScratch rs;
  RasterTotals tot;
  rc = arena_layout(ctx, [&](Arena &a) {
    return a.alloc(&d_states, (size_t)chunk * (states ? S : 1)) && a.alloc(&d_p, (size_t)chunk * cap * 3) &&
           a.alloc(&d_tip, (size_t)chunk * 3) && a.alloc(&d_npts, (size_t)chunk) &&
           a.alloc(&d_heads, (size_t)chunk) && a.alloc(&d_flags, (size_t)chunk) && tot.layout(a) &&
           rs.layout(a, std::min<int64_t>(chunk, RS_CHUNK_SETS));
  });
  if (rc) return rc;
  rc = tot.reset(ctx, st);
  if (rc) return rc;
  const int T = 256;
  for (int64_t off = 0; off < n; off += chunk) {
    const int64_t m = std::min<int64_t>(chunk, n - off);
    if (states) {
      IRT_CUDA(ctx, cudaMemcpyAsync(d_states, states + off * S, (size_t)m * S * 8, cudaMemcpyHostToDevice, st));
      irt_fk_outputs o;
      std::memset(&o, 0, sizeof(o));
      o.p = d_p; o.npts = d_npts; o.flags = d_flags; o.tip = d_tip;
      rc = fk_launch(ctx, rb, d_states, m, cap, o, st);
      if (rc) return rc;
      rc = self_collision_launch(ctx, rb, d_p, d_npts, m, cap, d_flags, st);
      if (rc) return rc;
    } else {   // shapes given by the caller
      IRT_CUDA(ctx, cudaMemcpyAsync(d_p, p_in + off * cap * 3, (size_t)m * cap * 24, cudaMemcpyHostToDevice, st));
      IRT_CUDA(ctx, cudaMemcpyAsync(d_npts, npts_in + off, (size_t)m * 4, cudaMemcpyHostToDevice, st));
      IRT_CUDA(ctx, cudaMemsetAsync(d_flags, 0, (size_t)m * 4, st));
    }
    vertex_heads_kernel<<<(unsigned)((m + T - 1) / T), T, 0, st>>>(d_flags, m, d_heads);
    IRT_LAUNCHED(ctx);
    SetSrc src;
    std::memset(&src, 0, sizeof(src));
    src.edge_mode = 0; src.pts = d_p; src.npts = d_npts; src.heads = d_heads; src.cap_pts = cap;
    rc = raster_append(ctx, g, src, m, nullptr, nullptr, d_flags, rs, store, off, tot.d_running, tot.d_overflow, st);
    if (rc) return rc;
    if (flags) IRT_CUDA(ctx, cudaMemcpyAsync(flags + off, d_flags, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
    if (tips) IRT_CUDA(ctx, cudaMemcpyAsync(tips + off * 3, d_tip, (size_t)m * 24, cudaMemcpyDeviceToHost, st));
    if ((flags || tips || !states) && off + chunk < n) IRT_CUDA(ctx, cudaStreamSynchronize(st));  // staging reused
  }
  uint64_t total = 0;
  bool overflow = false;
  rc = tot.read(ctx, st, &total, &overflow);
  if (rc) return rc;
  if (overflow) {
    if ((int64_t)total <= est_blocks) return irt_fail(ctx, IRT_ERR_CAPACITY, "set store overflow");
    return voxelize_vertices_impl(ctx, rb, states, p_in, npts_in, cap, state_size, n, store, flags, tips,
                                  (int64_t)total);
  }
  return setstore_finalize(ctx, store, n, (int64_t)total, st);
}

extern "C" {

int irt_voxelize_vertices(irt_ctx *ctx, const irt_robot *rb, const double *states, int state_size,
                          int64_t n, irt_setstore *store, uint32_t *flags, double *tips) {
  if (!ctx || !rb || !store || n < 0 || (n > 0 && !states)) return IRT_ERR_INVALID_ARGUMENT;
  if (state_size != rb->state_size)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "State is not the right size (%d != %d)",
                    state_size, rb->state_size);
  int rc = check_dl_vs_grid(ctx, rb, store->gd);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  return voxelize_vertices_impl(ctx, rb, states, nullptr, nullptr, rb->max_points, state_size, n, store, flags, tips,
                                n * 24);
}

int irt_voxelize_shapes(irt_ctx *ctx, const double *p, const int32_t *npts, int cap_pts, int64_t n,
                        irt_setstore *store) {
  if (!ctx || !store || n < 0 || cap_pts < 1 || (n > 0 && (!p || !npts))) return IRT_ERR_INVALID_ARGUMENT;
  for (int64_t i = 0; i < n; i++)
    if (npts[i] < 0 || npts[i] > cap_pts)
      return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "npts[%lld] out of range", (long long)i);
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  return voxelize_vertices_impl(ctx, nullptr, nullptr, p, npts, cap_pts, 0, n, store, nullptr, nullptr, n * 24);
}

}  // extern "C"

// ---- edges ------------------------------------------------------------------------------------------
namespace {

// host-side copy between pageable user arrays and the context's pinned staging, on a few threads (one core
// moves ~8-10 GB/s; the roadmap's index pairs and per-edge outputs are 160 MB each at 10M edges)
void par_memcpy(void *dst, const void *src, size_t bytes) {
  const int nt = bytes >= ((size_t)16 << 20) ? 4 : 1;
  if (nt == 1) { std::memcpy(dst, src, bytes); return; }
  std::thread th[3];
  const size_t part = ((bytes / nt) + 4095) & ~(size_t)4095;
  for (int t = 1; t < nt; t++) {
    const size_t b = (size_t)t * part, e = std::min(bytes, b + part);
    if (b < e) th[t - 1] = std::thread([=] { std::memcpy((char *)dst + b, (const char *)src + b, e - b); });
  }
  std::memcpy(dst, src, std::min(bytes, part));
  for (int t = 1; t < nt; t++)
    if (th[t - 1].joinable()) th[t - 1].join();
}

// per-edge outputs of a finished chunk on their way to the caller's arrays: device -> pinned staging (async, on
// the chunk's stream) -> caller memory (host copy, done while the GPU works on later chunks)
struct OutJob {
  int64_t off;
  int32_t E;
  cudaEvent_t ev;
  bool done;
};

// one in-flight chunk of edges: its stream, its share of the arena, its device counters
struct Lane {
  cudaStream_t st = nullptr;
  cudaEvent_t ev_bisect = nullptr;
  EdgePool P{};
  int32_t *C = nullptr;            // device counters
  int32_t *h_C = nullptr;          // pinned host copy
  Interval *q[2] = {nullptr, nullptr};
  Pending *pend = nullptr;
  double *tlimit = nullptr;
  void *fk_work = nullptr, *sc_work = nullptr;
  // non-indexed mode: this chunk's own vertex pool (2 endpoints per edge)
  double *v_state = nullptr, *v_p = nullptr;
  int32_t *v_npts = nullptr;
  uint32_t *v_flags = nullptr;
  RasterScratch rs;
  int64_t off = 0;
  int32_t E = 0;
  int q_cur = 0;
  int rounds = 0;
  int id = 0;
};

struct EdgeJob {
  irt_ctx *ctx;
  const irt_robot *rb;
  const irt_env *env;
  irt_setstore *store;
  GridDev g;
  int S, cap;
  bool indexed;
  const double *a, *b;          // host, non-indexed
  const int64_t *pairs;         // host, indexed
  int64_t *d_pairs_all = nullptr;   // device copy of all index pairs (indexed)
  double len_t, len_r, len_s;
  int static_rounds;
  // whole-call device outputs (indexed by edge)
  uint32_t *d_flags = nullptr;
  double *d_tlast = nullptr;
  int32_t *d_nsamp = nullptr;
  RasterTotals tot;
  cudaEvent_t ev_raster = nullptr;   // raster phases run in chunk order: each waits for the previous one
  bool raster_pending = false;
  int64_t mids_total = 0;
  // caller's output arrays (may be null) and their pinned staging
  uint32_t *u_flags = nullptr, *h_flags = nullptr;
  double *u_tlast = nullptr, *h_tlast = nullptr;
  int32_t *u_nsamp = nullptr, *h_nsamp = nullptr;
  std::vector<OutJob> outs;
  Timeline tl;
};

// copies finished chunks' outputs from the staging to the caller's arrays; block = wait for all of them
int drain_outputs(EdgeJob &J, bool block) {
  for (auto &o : J.outs) {
    if (o.done) continue;
    if (block) IRT_CUDA(J.ctx, cudaEventSynchronize(o.ev));
    else if (cudaEventQuery(o.ev) != cudaSuccess) {
      (void)cudaGetLastError();   // cudaErrorNotReady is recorded as the thread's last error: clear it
      continue;
    }
    if (J.u_flags) std::memcpy(J.u_flags + o.off, J.h_flags + o.off, (size_t)o.E * 4);
    if (J.u_tlast) std::memcpy(J.u_tlast + o.off, J.h_tlast + o.off, (size_t)o.E * 8);
    if (J.u_nsamp) std::memcpy(J.u_nsamp + o.off, J.h_nsamp + o.off, (size_t)o.E * 4);
    o.done = true;
  }
  return IRT_OK;
}


const int K2_T = 256;


int issue_round(EdgeJob &J, Lane &L) {
  irt_ctx *ctx = J.ctx;
  cudaStream_t st = L.st;
  const int qc = L.q_cur, qn = qc ^ 1;
  const int G = ctx->sm_count * 4;
  round_begin_kernel<<<1, 32, 0, st>>>(L.C, L.P.cap_mid, qn);
  IRT_LAUNCHED(ctx);
  edge_split_kernel<<<G, K2_T, 0, st>>>(L.P, L.q[qc], L.C, qc, L.pend);
  IRT_LAUNCHED(ctx);
  round_mid_kernel<<<1, 32, 0, st>>>(L.C, L.P.cap_mid);
  IRT_LAUNCHED(ctx);
  irt_fk_outputs o;
  std::memset(&o, 0, sizeof(o));
  o.p = L.P.m_p; o.npts = L.P.m_npts; o.flags = L.P.m_flags;
  int rc = fk_launch(ctx, J.rb, L.P.m_state, L.P.cap_mid, J.cap, o, st, nullptr, L.C + C_LO, L.fk_work);
  if (rc) return rc;
  rc = self_collision_launch(ctx, J.rb, o.p, o.npts, L.P.cap_mid, J.cap, o.flags, st, nullptr, L.C + C_LO, L.sc_work);
  if (rc) return rc;
  if (J.env) {
    sample_env_collision_kernel<<<G, K2_T, 0, st>>>(J.g, o.p, o.npts, J.cap, 0, L.C + C_LO, J.env->d_blocks,
                                                    J.env->d_occ, o.flags);
    IRT_LAUNCHED(ctx);
  }
  edge_mark_kernel<<<G, K2_T, 0, st>>>(L.P, L.C);
  IRT_LAUNCHED(ctx);
  edge_subdivide_kernel<<<G * 2, K2_T, 0, st>>>(J.g, L.P, L.pend, L.C, L.q[qn], qn);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  L.q_cur = qn;
  L.rounds++;
  J.tl.mark(st, "round end", L.id, L.rounds);
  return IRT_OK;
}

// everything of a chunk up to (not including) the raster: uploads, endpoint FK (non-indexed), init, all rounds
int issue_bisection(EdgeJob &J, Lane &L, int64_t off, int32_t E) {
  irt_ctx *ctx = J.ctx;
  cudaStream_t st = L.st;
  L.off = off; L.E = E; L.P.E = E; L.q_cur = 0; L.rounds = 0;
  J.tl.mark(st, "bisection begin", L.id, off);
  IRT_CUDA(ctx, cudaMemsetAsync(L.C, 0, C_WORDS * 4, st));
  if (J.indexed) {
    L.P.pairs = J.d_pairs_all + 2 * off;
  } else {
    // this chunk's vertex pool: endpoint a of edge e = vertex 2e, endpoint b = vertex 2e + 1
    const size_t row = (size_t)J.S * 8;
    IRT_CUDA(ctx, cudaMemcpy2DAsync(L.v_state, 2 * row, J.a + off * J.S, row, row, E, cudaMemcpyHostToDevice, st));
    IRT_CUDA(ctx, cudaMemcpy2DAsync(L.v_state + J.S, 2 * row, J.b + off * J.S, row, row, E, cudaMemcpyHostToDevice, st));
    edge_identity_pairs_kernel<<<(E + K2_T - 1) / K2_T, K2_T, 0, st>>>(L.P.pairs, E);
    IRT_LAUNCHED(ctx);
    irt_fk_outputs o;
    std::memset(&o, 0, sizeof(o));
    o.p = L.v_p; o.npts = L.v_npts; o.flags = L.v_flags;
    int rc = fk_launch(ctx, J.rb, L.v_state, 2 * (int64_t)E, J.cap, o, st, nullptr, nullptr, L.fk_work);
    if (rc) return rc;
    rc = self_collision_launch(ctx, J.rb, o.p, o.npts, 2 * (int64_t)E, J.cap, o.flags, st, nullptr, nullptr, L.sc_work);
    if (rc) return rc;
    if (J.env) {
      sample_env_collision_kernel<<<ctx->sm_count * 4, K2_T, 0, st>>>(J.g, o.p, o.npts, J.cap, 2 * (int64_t)E, nullptr,
                                                                      J.env->d_blocks, J.env->d_occ, o.flags);
      IRT_LAUNCHED(ctx);
    }
    L.P.nv = 2 * (int64_t)E;
  }
  edge_init_kernel<<<(E + K2_T - 1) / K2_T, K2_T, 0, st>>>(L.P, L.C, J.len_t, J.len_r, J.len_s);
  IRT_LAUNCHED(ctx);
  edge_subdivide_kernel<<<ctx->sm_count * 8, K2_T, 0, st>>>(J.g, L.P, nullptr, L.C, L.q[0], 0);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  for (int r = 0; r < J.static_rounds; r++) {
    int rc = issue_round(J, L);
    if (rc) return rc;
  }
  IRT_CUDA(ctx, cudaMemcpyAsync(L.h_C, L.C, C_WORDS * 4, cudaMemcpyDeviceToHost, st));
  IRT_CUDA(ctx, cudaEventRecord(L.ev_bisect, st));
  return IRT_OK;
}

// waits for the chunk's bisection; runs extra rounds while intervals are still open.
// *overflow: the mid pool was too small (the chunk has to be redone in smaller pieces)
int finish_bisection(EdgeJob &J, Lane &L, bool *overflow) {
  irt_ctx *ctx = J.ctx;
  for (;;) {
    IRT_CUDA(ctx, cudaEventSynchronize(L.ev_bisect));
    if (L.h_C[C_ERR] & 1)
      return irt_fail(ctx, IRT_ERR_OUT_OF_RANGE, "edge endpoint index outside [0,%lld)", (long long)L.P.nv);
    *overflow = L.h_C[C_NMID] > L.P.cap_mid;
    const int32_t open = L.h_C[C_NQ0 + L.q_cur];
    if (open > L.P.cap_q) *overflow = true;
    if (*overflow || open == 0 || L.rounds >= 64) return IRT_OK;
    for (int r = 0; r < 2; r++) {   // deeper than the static bound (states outside the space bounds): keep going
      int rc = issue_round(J, L);
      if (rc) return rc;
    }
    IRT_CUDA(ctx, cudaMemcpyAsync(L.h_C, L.C, C_WORDS * 4, cudaMemcpyDeviceToHost, L.st));
    IRT_CUDA(ctx, cudaEventRecord(L.ev_bisect, L.st));
  }
}

int issue_raster(EdgeJob &J, Lane &L) {
  irt_ctx *ctx = J.ctx;
  cudaStream_t st = L.st;
  edge_finish_kernel<<<(L.E + K2_T - 1) / K2_T, K2_T, 0, st>>>(L.P, L.tlimit, J.d_flags + L.off);
  IRT_LAUNCHED(ctx);
  // the leaf offsets chain through *d_running: raster phases run in chunk order
  if (J.raster_pending) IRT_CUDA(ctx, cudaStreamWaitEvent(st, J.ev_raster, 0));
  J.tl.mark(st, "raster begin", L.id, L.off);
  SetSrc src;
  std::memset(&src, 0, sizeof(src));
  src.edge_mode = 1; src.P = L.P; src.tlimit = L.tlimit; src.cap_pts = J.cap;
  // rasterise every sample below the first invalid t (VoxelEnvironment.cpp:406-422)
  int rc = raster_append(ctx, J.g, src, L.E, J.d_tlast + L.off, J.d_nsamp + L.off, J.d_flags + L.off, L.rs, J.store,
                         L.off, J.tot.d_running, J.tot.d_overflow, st);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaEventRecord(J.ev_raster, st));
  J.tl.mark(st, "raster end", L.id, L.h_C[C_NMID]);
  J.raster_pending = true;
  J.mids_total += std::min(L.h_C[C_NMID], L.P.cap_mid);
  if (J.u_flags || J.u_tlast || J.u_nsamp) {
    if (J.u_flags) IRT_CUDA(ctx, cudaMemcpyAsync(J.h_flags + L.off, J.d_flags + L.off, (size_t)L.E * 4, cudaMemcpyDeviceToHost, st));
    if (J.u_tlast) IRT_CUDA(ctx, cudaMemcpyAsync(J.h_tlast + L.off, J.d_tlast + L.off, (size_t)L.E * 8, cudaMemcpyDeviceToHost, st));
    if (J.u_nsamp) IRT_CUDA(ctx, cudaMemcpyAsync(J.h_nsamp + L.off, J.d_nsamp + L.off, (size_t)L.E * 4, cudaMemcpyDeviceToHost, st));
    OutJob o{L.off, L.E, nullptr, false};
    IRT_CUDA(ctx, cudaEventCreateWithFlags(&o.ev, cudaEventDisableTiming));
    IRT_CUDA(ctx, cudaEventRecord(o.ev, st));
    J.outs.push_back(o);
  }
  return IRT_OK;
}

}  // namespace

// a, b: per-edge endpoint states (host) -- or, indexed form: vstates[nv][S] + pairs[n][2]
static int voxelize_edges_core(irt_ctx *ctx, const irt_robot *rb, const irt_space *space, const double *a,
                               const double *b, const double *vstates, int64_t nv, const int64_t *pairs,
                               int state_size, int64_t n, const irt_env *env, irt_setstore *store,
                               uint32_t *flags, double *t_last, int32_t *nsamples, int64_t est_blocks = -1) {
  const bool indexed = pairs != nullptr;
  if (env && store && env->grid.Ng != store->grid.Ng)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "voxel dimension mismatch (%d != %d)", env->grid.Ng,
                    store->grid.Ng);
  if (!ctx || !rb || !space || !store || n < 0) return IRT_ERR_INVALID_ARGUMENT;
  if (!indexed && n > 0 && (!a || !b)) return IRT_ERR_INVALID_ARGUMENT;
  if (indexed && (nv < 0 || (nv > 0 && !vstates))) return IRT_ERR_INVALID_ARGUMENT;
  if (indexed && n > 0 && nv == 0) return irt_fail(ctx, IRT_ERR_OUT_OF_RANGE, "edges over an empty vertex list");
  if (state_size != rb->state_size)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "State is not the right size (%d != %d)",
                    state_size, rb->state_size);
  const GridDev &g = store->gd;
  int rc = check_dl_vs_grid(ctx, rb, g);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  const int S = state_size, cap = rb->max_points;
  if (n > (int64_t)0x3fffffff) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "too many edges");
  if (est_blocks < 0) est_blocks = n * 32;
  rc = store_begin(ctx, store, n, est_blocks, ctx->stream);
  if (rc) return rc;
  if (n == 0) return setstore_finalize(ctx, store, 0, 0, ctx->stream);
  Trace tr(ctx->stream);

  EdgeJob J;
  J.ctx = ctx; J.rb = rb; J.env = env; J.store = store; J.g = g; J.S = S; J.cap = cap;
  J.indexed = indexed; J.a = a; J.b = b; J.pairs = pairs;
  {
    // longest valid segment lengths of the three subspaces (Problem.cpp:118-144), as in
    // irt_valid_segment_count; the per-edge count itself is evaluated on the device.  The deepest
    // bisection any edge inside the space bounds can need gives the number of rounds launched blind.
    double ext2 = 0;
    for (int i = 0; i < rb->desc.n_tendons; i++) ext2 += rb->desc.max_tension[i] * rb->desc.max_tension[i];
    const double tendon_extent = std::sqrt(ext2);
    J.len_t = tendon_extent * (space->min_tension_change / tendon_extent);
    J.len_r = M_PI * (space->min_rotation_change / (2 * M_PI));
    J.len_s = rb->desc.L * std::fmin(0.01, space->min_retraction_change / rb->desc.L);
    double nmax = std::ceil(tendon_extent / J.len_t);
    if (rb->desc.enable_rotation) nmax = std::fmax(nmax, std::ceil(M_PI / J.len_r));
    if (rb->desc.enable_retraction) nmax = std::fmax(nmax, std::ceil(rb->desc.L / J.len_s));
    int depth = 1;
    while (depth < 40 && std::ldexp(1.0, depth) < nmax) depth++;
    J.static_rounds = depth + 1;
  }

  // ---- sizing: two lanes (chunks in flight) share the budget ------------------------------------
  size_t free_b = 0, total_b = 0;
  IRT_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
  free_b += ctx->arena_bytes;  // the arena is ours to reuse
  size_t budget = (size_t)24 << 30;
  if (budget > free_b * 2 / 5) budget = free_b * 2 / 5;
  const size_t per_mid = (size_t)cap * 24 + (size_t)S * 8 + 24 /* edge, next, npts, flags, t */ +
                         2 * 2 * sizeof(Interval) + sizeof(Pending) + 8 /* fk keys + perm */ + 12 /* selfcol lists */;
  const size_t per_vertex = (size_t)cap * 24 + (size_t)S * 8 + 8;
  const int64_t rs_sets = std::min<int64_t>(n, RS_CHUNK_SETS);
  const size_t raster_fixed = (size_t)rs_sets * RS_SLOT * 12 + (size_t)RS_MAX_OVF * RS_BIGSLOT * 12 + ((size_t)8 << 20);
  const size_t fixed = (size_t)n * 32 + (indexed ? (size_t)nv * (per_vertex + 12) : 0) + 2 * raster_fixed + ((size_t)64 << 20);
  const size_t avail = (budget > fixed) ? budget - fixed : 0;
  const int mids_per_edge = 3;   // roadmap edges need 2-3 mid samples on average; a chunk whose pool overflows is split
  const size_t per_edge = mids_per_edge * per_mid + 64 + (indexed ? 0 : 2 * (per_vertex + 20));
  int64_t chunk = (int64_t)(avail / 2 / per_edge);
  if (chunk < 256) chunk = 256;
  int64_t nchunks = (n + chunk - 1) / chunk;
  if (nchunks > 1 && (nchunks & 1)) nchunks++;   // an even number of chunks keeps both lanes busy to the end
  chunk = (n + nchunks - 1) / nchunks;
  const int nlanes = nchunks > 1 ? 2 : 1;
  int64_t cap_mid = chunk * mids_per_edge;
  {
    // calls that do not need the whole budget take more room per edge: up to 8 mid samples per edge (sparse
    // roadmaps have long edges), 64 for small calls (single long edges need dozens of samples)
    const int64_t room = (int64_t)((avail - std::min(avail, (size_t)nlanes * chunk * per_edge)) / nlanes / per_mid) + cap_mid;
    const int64_t want = (n <= 65536) ? std::max<int64_t>(chunk * 64, 4096) : chunk * 8;
    cap_mid = std::max<int64_t>(cap_mid, std::min<int64_t>(want, room));
  }
  if (cap_mid > 0x3fffffff) cap_mid = 0x3fffffff;
  const int64_t cap_q = std::max<int64_t>(chunk, 2 * cap_mid);
  const int64_t fkn = std::max<int64_t>(cap_mid, indexed ? 0 : 2 * chunk);

  Lane lanes[2];
  double *d_vstates = nullptr, *d_vp = nullptr;
  int32_t *d_vnpts = nullptr;
  uint32_t *d_vflags = nullptr;
  int64_t *d_pairs_all = nullptr;
  void *v_fk_work = nullptr, *v_sc_work = nullptr;
  const int64_t vchunk = std::min<int64_t>(nv, 1048576);
  rc = arena_layout(ctx, [&](Arena &A) {
    if (!(A.alloc(&J.d_flags, (size_t)n) && A.alloc(&J.d_tlast, (size_t)n) && A.alloc(&J.d_nsamp, (size_t)n) &&
          J.tot.layout(A)))
      return false;
    if (indexed) {
      char *w1 = nullptr, *w2 = nullptr;
      if (!(A.alloc(&d_pairs_all, (size_t)n * 2) && A.alloc(&d_vstates, (size_t)nv * S) && A.alloc(&d_vp, (size_t)nv * cap * 3) &&
            A.alloc(&d_vnpts, (size_t)nv) && A.alloc(&d_vflags, (size_t)nv) &&
            A.alloc(&w1, fk_work_bytes(rb, vchunk)) && A.alloc(&w2, selfcol_work_bytes(vchunk))))
        return false;
      v_fk_work = w1; v_sc_work = w2;
    }
    for (int l = 0; l < nlanes; l++) {
      Lane &L = lanes[l];
      EdgePool &P = L.P;
      char *w1 = nullptr, *w2 = nullptr;
      if (!((indexed || A.alloc(&P.pairs, (size_t)chunk * 2)) && A.alloc(&P.thr, (size_t)chunk) &&
            A.alloc(&P.first_invalid, (size_t)chunk) && A.alloc(&P.head, (size_t)chunk) &&
            A.alloc(&P.eflags, (size_t)chunk) && A.alloc(&L.tlimit, (size_t)chunk) &&
            A.alloc(&P.m_edge, (size_t)cap_mid) && A.alloc(&P.m_next, (size_t)cap_mid) &&
            A.alloc(&P.m_npts, (size_t)cap_mid) && A.alloc(&P.m_flags, (size_t)cap_mid) &&
            A.alloc(&P.m_t, (size_t)cap_mid) && A.alloc(&P.m_state, (size_t)cap_mid * S) &&
            A.alloc(&P.m_p, (size_t)cap_mid * cap * 3) && A.alloc(&L.q[0], (size_t)cap_q) &&
            A.alloc(&L.q[1], (size_t)cap_q) && A.alloc(&L.pend, (size_t)cap_mid) && A.alloc(&L.C, (size_t)C_WORDS) &&
            A.alloc(&w1, fk_work_bytes(rb, fkn)) && A.alloc(&w2, selfcol_work_bytes(fkn)) &&
            L.rs.layout(A, std::min<int64_t>(chunk, RS_CHUNK_SETS))))
        return false;
      L.fk_work = w1; L.sc_work = w2;
      if (!indexed &&
          !(A.alloc(&L.v_state, (size_t)chunk * 2 * S) && A.alloc(&L.v_p, (size_t)chunk * 2 * cap * 3) &&
            A.alloc(&L.v_npts, (size_t)chunk * 2) && A.alloc(&L.v_flags, (size_t)chunk * 2)))
        return false;
    }
    return true;
  });
  if (rc) return rc;
  // pinned host staging (grow-only, owned by the context): chunk counters, the caller's per-edge outputs, and
  // (indexed form) the vertex states and index pairs -- so every transfer is a real asynchronous DMA
  const size_t pin_c = 256, pin_out = ((size_t)n * 16 + 255) & ~(size_t)255;
  const size_t pin_pairs = indexed ? (((size_t)n * 16 + 255) & ~(size_t)255) : 0;
  const size_t pin_vs = indexed ? (((size_t)nv * S * 8 + 255) & ~(size_t)255) : 0;
  char *pin = (char *)ctx_pinned(ctx, pin_c + pin_out + pin_pairs + pin_vs);
  if (!pin) return irt_fail(ctx, IRT_ERR_CUDA, "pinned staging allocation failed");
  int32_t *h_C = (int32_t *)pin;
  J.u_flags = flags; J.u_tlast = t_last; J.u_nsamp = nsamples;
  J.h_tlast = (double *)(pin + pin_c);
  J.h_flags = (uint32_t *)(pin + pin_c + (size_t)n * 8);
  J.h_nsamp = (int32_t *)(pin + pin_c + (size_t)n * 12);
  int64_t *h_pairs = (int64_t *)(pin + pin_c + pin_out);
  double *h_vstates = (double *)(pin + pin_c + pin_out + pin_pairs);
  for (int l = 0; l < nlanes; l++) {
    Lane &L = lanes[l];
    L.id = l;
    L.st = l == 0 ? ctx->stream : ctx->copy_stream;
    L.ev_bisect = ctx->ev_computed[l];
    L.h_C = h_C + l * C_WORDS;
    EdgePool &P = L.P;
    P.cap_mid = (int32_t)cap_mid; P.cap_q = (int32_t)cap_q;
    P.S = S; P.N = rb->desc.n_tendons; P.cap_pts = cap;
    P.enable_rotation = rb->desc.enable_rotation ? 1 : 0;
    P.enable_retraction = rb->desc.enable_retraction ? 1 : 0;
    if (indexed) { P.v_state = d_vstates; P.v_p = d_vp; P.v_npts = d_vnpts; P.v_flags = d_vflags; P.nv = nv; }
    else { P.v_state = L.v_state; P.v_p = L.v_p; P.v_npts = L.v_npts; P.v_flags = L.v_flags; P.nv = 0; }
  }
  J.ev_raster = ctx->ev_copied[0];
  J.d_pairs_all = d_pairs_all;
  cudaStream_t s0 = ctx->stream;
  rc = J.tot.reset(ctx, s0);
  if (rc) return rc;
  tr.point("layout", cap_mid);
  J.tl.host("layout done");
  J.tl.mark(s0, "start", 0, n);

  // ---- indexed form: FK of every roadmap vertex once; edges read their endpoint shapes from it ------
  if (indexed) {
    par_memcpy(h_vstates, vstates, (size_t)nv * S * 8);
    IRT_CUDA(ctx, cudaMemcpyAsync(d_vstates, h_vstates, (size_t)nv * S * 8, cudaMemcpyHostToDevice, s0));
    for (int64_t v0 = 0; v0 < nv; v0 += vchunk) {
      const int64_t m = std::min<int64_t>(vchunk, nv - v0);
      irt_fk_outputs o;
      std::memset(&o, 0, sizeof(o));
      o.p = d_vp + v0 * cap * 3; o.npts = d_vnpts + v0; o.flags = d_vflags + v0;
      rc = fk_launch(ctx, rb, d_vstates + v0 * S, m, cap, o, s0, nullptr, nullptr, v_fk_work);
      if (rc) return rc;
      rc = self_collision_launch(ctx, rb, o.p, o.npts, m, cap, o.flags, s0, nullptr, nullptr, v_sc_work);
      if (rc) return rc;
      if (env) {
        sample_env_collision_kernel<<<ctx->sm_count * 4, K2_T, 0, s0>>>(g, o.p, o.npts, cap, m, nullptr, env->d_blocks,
                                                                        env->d_occ, o.flags);
        IRT_LAUNCHED(ctx);
      }
    }
    // all index pairs in ONE upload on the second stream; the host-side copy into the staging runs while the
    // GPU computes the vertex shapes
    cudaStream_t sp = lanes[nlanes - 1].st;
    par_memcpy(h_pairs, pairs, (size_t)n * 16);
    IRT_CUDA(ctx, cudaMemcpyAsync(d_pairs_all, h_pairs, (size_t)n * 16, cudaMemcpyHostToDevice, sp));
    IRT_CUDA(ctx, cudaEventRecord(ctx->ev_copied[1], sp));
    IRT_CUDA(ctx, cudaStreamWaitEvent(s0, ctx->ev_copied[1], 0));
  }
  // the second lane starts after the vertex pool and the resets above
  IRT_CUDA(ctx, cudaEventRecord(ctx->ev_offsets[0], s0));
  if (nlanes > 1) IRT_CUDA(ctx, cudaStreamWaitEvent(lanes[1].st, ctx->ev_offsets[0], 0));
  tr.point("vertex fk issued", nv);
  J.tl.mark(s0, "vertex fk end", 0, nv);
  J.tl.host("vertex fk + pair upload issued");

  // ---- chunks: up to two in flight, rastered in index order ----------------------------------------
  std::vector<std::pair<int64_t, int64_t>> todo;   // (offset, count), lowest offset LAST (a stack)
  for (int64_t off = n - ((n - 1) % chunk + 1); off >= 0; off -= chunk)
    todo.emplace_back(off, std::min<int64_t>(chunk, n - off));
  std::vector<Lane *> inflight;                    // sorted by offset
  std::vector<Lane *> idle;
  for (int l = nlanes - 1; l >= 0; l--) idle.push_back(&lanes[l]);
  auto fail = [&](int code) {
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->copy_stream);
    for (auto &o : J.outs) cudaEventDestroy(o.ev);
    return code;
  };
  // Chunks are sized by the sample pool: est_mpe = mid samples an edge needs (3 to begin with, then what the
  // finished chunks needed); a chunk whose pool overflows anyway is re-cut by what it turned out to need.
  double est_mpe = (double)mids_per_edge;
  for (;;) {
    rc = drain_outputs(J, false);   // finished chunks' outputs go to the caller while the GPU works on
    if (rc) return fail(rc);
    while (!idle.empty() && !todo.empty()) {
      Lane *L = idle.back();
      idle.pop_back();
      auto w = todo.back();
      todo.pop_back();
      const int64_t fit = std::max<int64_t>(256, (int64_t)((double)cap_mid / (est_mpe * 1.1)));
      if (w.second > fit && w.second > 256) {   // more edges than the pool is expected to hold: take a part
        todo.emplace_back(w.first + fit, w.second - fit);
        w.second = fit;
      }
      rc = issue_bisection(J, *L, w.first, (int32_t)w.second);
      if (rc) return fail(rc);
      auto it = inflight.begin();
      while (it != inflight.end() && (*it)->off < L->off) ++it;
      inflight.insert(it, L);
    }
    if (inflight.empty()) break;
    Lane *L = inflight.front();
    inflight.erase(inflight.begin());
    bool overflow = false;
    rc = finish_bisection(J, *L, &overflow);
    if (rc) return fail(rc);
    tr.point("bisection done", L->h_C[C_NMID]);
    {
      // C_NMID keeps counting past the pool size, so an overflowed chunk still tells (a lower bound of) its need
      const double seen = (double)L->h_C[C_NMID] / (double)std::max<int32_t>(L->E, 1);
      est_mpe = overflow ? std::max(est_mpe, seen) * 1.3 : std::max(0.5 * est_mpe, seen);
      if (est_mpe < 0.25) est_mpe = 0.25;
    }
    if (overflow && L->E > 256) {   // redo this range (the issue loop re-cuts it), before anything that follows it
      todo.emplace_back(L->off, L->E);
      idle.push_back(L);
      continue;
    }
    rc = issue_raster(J, *L);
    if (rc) return fail(rc);
    idle.push_back(L);
  }
  // everything is issued; the lanes' streams join on the context stream
  if (nlanes > 1) {
    IRT_CUDA(ctx, cudaEventRecord(ctx->ev_offsets[1], lanes[1].st));
    IRT_CUDA(ctx, cudaStreamWaitEvent(s0, ctx->ev_offsets[1], 0));
  }
  J.tl.host("everything issued");
  rc = drain_outputs(J, true);
  if (rc) return fail(rc);
  J.tl.host("outputs drained");
  for (auto &o : J.outs) cudaEventDestroy(o.ev);
  J.outs.clear();
  uint64_t total = 0;
  bool overflow = false;
  rc = J.tot.read(ctx, s0, &total, &overflow);
  if (rc) return fail(rc);
  tr.point("raster + d2h done", (long long)total);
  J.tl.mark(s0, "all done", 0, (long long)total);
  J.tl.host("totals read");
  J.tl.print();
  if (overflow) {   // the store was too small for the leaves: now their number is known, run again
    if ((int64_t)total <= est_blocks) return irt_fail(ctx, IRT_ERR_CAPACITY, "set store overflow");
    return voxelize_edges_core(ctx, rb, space, a, b, vstates, nv, pairs, state_size, n, env, store, flags, t_last,
                               nsamples, (int64_t)total);
  }
  return setstore_finalize(ctx, store, n, (int64_t)total, s0);
}

extern "C" {

int irt_voxelize_edges(irt_ctx *ctx, const irt_robot *rb, const irt_space *space, const double *a,
                       const double *b, int state_size, int64_t n, irt_setstore *store,
                       uint32_t *flags, double *t_last, int32_t *nsamples) {
  return voxelize_edges_core(ctx, rb, space, a, b, nullptr, 0, nullptr, state_size, n, nullptr, store, flags,
                             t_last, nsamples);
}

int irt_voxelize_edges_until_invalid(irt_ctx *ctx, const irt_robot *rb, const irt_space *space,
                                     const double *a, const double *b, int state_size, int64_t n,
                                     const irt_env *env, irt_setstore *store, uint32_t *flags,
                                     double *t_last, int32_t *nsamples) {
  if (!env) return IRT_ERR_INVALID_ARGUMENT;
  return voxelize_edges_core(ctx, rb, space, a, b, nullptr, 0, nullptr, state_size, n, env, store, flags,
                             t_last, nsamples);
}

int irt_voxelize_edges_indexed(irt_ctx *ctx, const irt_robot *rb, const irt_space *space,
                               const double *vertex_states, int state_size, int64_t n_vertices,
                               const int64_t *pairs, int64_t n_edges, irt_setstore *store,
                               uint32_t *flags, double *t_last, int32_t *nsamples) {
  if (n_edges > 0 && !pairs) return IRT_ERR_INVALID_ARGUMENT;
  static const int64_t dummy[2] = {0, 0};
  return voxelize_edges_core(ctx, rb, space, nullptr, nullptr, vertex_states, n_vertices,
                             pairs ? pairs : dummy, state_size, n_edges, nullptr, store, flags, t_last, nsamples);
}

}  // extern "C"
