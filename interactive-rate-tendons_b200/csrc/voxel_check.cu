// voxel_check.cu -- environment grid, cached set store and K3 `voxel_and_popc`.
//
// Replaces VoxelOctree::collides(const VoxelOctree&) (collision/VoxelOctree.cpp:973-978 ->
// TreeNode<N>::collides, collision/detail/TreeNode.hxx:165-174, leaf test `_tree & other._tree`
// :268) for every cached vertex/edge voxel set against the environment.
//
// Data layout in HBM (B200-first, not the reference's pointer octree):
//   environment  dense uint64[Nb^3] leaf blocks indexed by Morton key (x-major octant order =
//                the reference's child order, TreeNode.h:66-68), so 8 consecutive entries are one
//                512-bit 2x2x2 super-block (one 64-byte line); plus a 1-bit-per-leaf occupancy
//                bitmap (4 KiB at 128^3) that the kernel stages in shared memory: the bitmap plays
//                the role of the octree's "null child" early-out.
//   set store    CSR, structure-of-arrays: keys uint32[nb], bits uint64[nb], offsets uint64[n+1];
//                12 bytes per occupied leaf block = the algorithmic traffic of SURVEY 8(d).
// K3: one CTA per tile of 256 consecutive sets = 8 uint32 verdict words.  The tile's leaves are
// one contiguous CSR range that the CTA streams with 128-bit loads; a leaf whose `bits & env[key]`
// (behind the occupancy bitmap) is non-zero sets one bit in a shared-memory hit bitmap, and each
// thread then tests the bits of the one set it owns; the word is one __ballot_sync per warp: no
// global atomics, no memset, no search, no per-set divergence (details at the kernel).
#include <cstring>
#include <vector>

#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace {

constexpr int K3_THREADS = 256;

__global__ void env_build_occ_kernel(const uint64_t *__restrict__ blocks, int64_t nblk,
                                     uint32_t *__restrict__ occ) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nwords = (nblk + 31) / 32;
  if (w >= nwords) return;
  uint32_t m = 0;
  for (int b = 0; b < 32; b++) {
    const int64_t i = w * 32 + b;
    if (i < nblk && blocks[i] != 0) m |= 1u << b;
  }
  occ[w] = m;
}

__global__ void env_scatter_sparse_kernel(const uint8_t *__restrict__ bxyz,
                                          const uint64_t *__restrict__ bits, int64_t n, int levels,
                                          uint64_t *__restrict__ blocks) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t bx = bxyz[3 * i], by = bxyz[3 * i + 1], bz = bxyz[3 * i + 2];
  uint32_t key = 0;
  for (int l = 0; l < levels; l++)
    key |= (((bx >> l) & 1u) << (3 * l + 2)) | (((by >> l) & 1u) << (3 * l + 1)) | (((bz >> l) & 1u) << (3 * l));
  blocks[key] = bits[i];
}

__global__ void count_nonzero_kernel(const uint64_t *__restrict__ blocks, int64_t n,
                                     unsigned long long *__restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool nz = (i < n) && blocks[i] != 0;
  const unsigned m = __ballot_sync(0xffffffffu, nz);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(out, (unsigned long long)__popc(m));
}

// K3 `voxel_and_popc`
//
// One CTA per tile of K3_THREADS consecutive sets (= 8 verdict words).  The tile's leaves are one
// contiguous CSR range that all 256 threads stream as 16-byte aligned quads (uint4 of keys +
// 2 x ulonglong2 of bits per thread and step, two steps in flight, ld.global.cs).  A leaf whose
// `bits & env[key]` is non-zero sets ONE BIT at its tile-relative position in a shared-memory hit
// bitmap (atomicOr, only on a hit); after the stream thread t -- which owns set s0+t and holds its
// leaf range [lo,hi) -- tests the bits of its range (1-2 words for a typical 20-60 leaf set), and a
// __ballot_sync per warp is the verdict word.  No shuffles, no search and no per-set divergence in the
// streaming loop; tiles with more leaves than the bitmap holds are streamed in chunks.  Three hit bitmaps
// rotate, so a chunk costs ONE __syncthreads (the buffer cleared during chunk k was last read two barriers ago).
constexpr int K3_CHUNK_LEAVES = 32768;                      // hit-bitmap capacity per buffer (4 KiB)
constexpr int K3_BM_WORDS = K3_CHUNK_LEAVES / 32 + 2;       // +1 straddle word, +1 pad
constexpr int K3_GATHER_TILES = 256;                         // staged verdict words per CTA: 8 KiB
// staged tiles per P2P flush: peer stores trickle out while the sweep runs, so the fence at the end of a CTA only
// waits for its last few
constexpr int K3_GATHER_FLUSH_TILES = 4;
static_assert(K3_GATHER_FLUSH_TILES <= K3_GATHER_TILES, "a flush cannot hold more tiles than are staged");
constexpr int K3_SMEM_FIXED_WORDS = 3 * K3_BM_WORDS + (3 * K3_BM_WORDS & 1) + 2 * 2 * (K3_THREADS + 2);

// predicated 8-byte read-only load: the four environment look-ups of a quad are issued back to back
// (no branch per look-up), so their latencies overlap; lanes whose leaf is in an empty environment
// block issue nothing
__device__ __forceinline__ uint64_t ld_env_if(const uint64_t *p, uint32_t pred) {
  uint64_t v;
  asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\tmov.u64 %0, 0;\n\t@p ld.global.nc.u64 %0, [%2];\n\t}"
      : "=l"(v) : "r"(pred), "l"(p));
  return v;
}

__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// streaming 16-byte loads (evict-first); volatile keeps the issue order of the software pipeline
__device__ __forceinline__ uint4 ld_stream(const uint4 *p) {
  uint4 v;
  asm volatile("ld.global.cs.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ ulonglong2 ld_stream(const ulonglong2 *p) {
  ulonglong2 v;
  asm volatile("ld.global.cs.v2.u64 {%0,%1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p));
  return v;
}

// Verdict exchange fused into K3 (multi-GPU): every rank holds the gathered verdict array of ALL ranks
// in a buffer its peers can write (CUDA IPC over NVLink).  A CTA stages the verdict words of its finished tiles
// and stores them as 32-byte runs straight into every peer's copy; the last CTA to finish raises this rank's
// epoch flag on every peer and waits for the peers' flags.  No NCCL call, no extra kernel between the sweep and
// its consumers.
constexpr int IRT_MAX_PEERS = 16;
struct XchgDev {
  uint32_t *peer[IRT_MAX_PEERS];  // base of every rank's buffer as mapped in THIS process (own: local)
  int world, rank, parity;
  int flush_tiles;                // staged tiles per P2P flush (the host sets K3_GATHER_FLUSH_TILES)
  int64_t slot_words;             // words every rank contributes
  uint32_t epoch;
  unsigned int *done;             // local: [0] CTAs done, [1] error word, [2] dynamic tile counter
  // buffer layout (uint32): words[2][world][slot_words], flags[2][world]
  __device__ __forceinline__ uint32_t *words(int r) const {
    return peer[r] + ((int64_t)parity * world + rank) * slot_words;
  }
  __device__ __forceinline__ uint32_t *flag(int r) const {
    return peer[r] + (int64_t)2 * world * slot_words + parity * world + rank;
  }
  // rank r's flag of this parity in THIS rank's buffer
  __device__ __forceinline__ const uint32_t *flag_here(int r) const {
    return peer[rank] + (int64_t)2 * world * slot_words + parity * world + r;
  }
};

// last-CTA epilogue of a gathering kernel.  Ordering (PTX memory model, causality order is transitive across
// scopes): a CTA's peer stores -> CTA barrier -> thread 0: fence.gpu + atomicAdd(done)  [release at gpu scope]
// -> last CTA: atomicAdd observes all + fence.sys  [acquire at gpu scope, and the fence is cumulative]
// -> st.relaxed.sys flags  [release at sys scope] -> a peer's ld.acquire.sys of the flag.  The same CTA then waits
// (bounded) until every peer's flag of this sweep has arrived in this rank's buffer, so that when the kernel ends
// the gathered array is complete: no separate wait kernel.  (Every rank's kernel runs on its own GPU; nothing here
// waits for another launch on the same device.)
__device__ __forceinline__ void xchg_signal(const XchgDev &x) {
  // the CTA barrier orders every thread's peer stores before thread 0's fence (fences are cumulative), so ONE
  // fence per CTA publishes them all
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    // a CTA publishes its peer stores towards the LAST CTA with a gpu-scope fence and only the last CTA pays a
    // system-scope fence before the flags (-6 us per sweep: MEMBAR.SYS twice in a row on the critical path was
    // ~10 us)
    __threadfence();
    const unsigned prev = atomicAdd(x.done, 1u);
    s_last = (prev == gridDim.x - 1);
    if (s_last) {
      x.done[0] = 0;   // CTA counter and tile counter are ready for the next sweep
      x.done[2] = 0;
      // release pattern with ONE fence: fence.sys, then relaxed system-scope flag stores.  (st.release.sys is a
      // fence per store: with 8 peers the last CTA would sit through 7 more NVLink round trips.)
      __threadfence_system();
      for (int r = 0; r < x.world; r++)
        asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(x.flag(r)), "r"(x.epoch) : "memory");
    }
  }
  __syncthreads();
  if (s_last && threadIdx.x < x.world) {   // thread r waits for rank r's flag
    const uint32_t *f = x.flag_here(threadIdx.x);
    bool ok = false;
    for (long it = 0; it < (1L << 22); it++) {
      uint32_t v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
      if (v == x.epoch) { ok = true; break; }
      __nanosleep(100);
    }
    if (!ok) atomicExch(x.done + 1, 1u + (unsigned)threadIdx.x);   // a peer that never arrives: reported, no hang
  }
}

template <bool OCC_SMEM, bool STATS, bool GATHER = false>
__global__ void __launch_bounds__(K3_THREADS, 4)
voxel_and_popc_kernel(const uint32_t *__restrict__ keys, const uint64_t *__restrict__ bits,
                      const uint64_t *__restrict__ offsets, const uint64_t *__restrict__ env,
                      const uint32_t *__restrict__ occ, int occ_words,
                      int64_t set_begin, int64_t set_end, uint32_t *__restrict__ verdict,
                      unsigned long long *__restrict__ stats, const XchgDev xd) {
  // [0, 3*K3_BM_WORDS): three hit bitmaps (rotating, so a chunk costs ONE __syncthreads: the buffer
  // cleared during chunk k was last read two barriers ago); then two tiles of set offsets
  // (cp.async prefetch of the next tile's CSR offsets while this tile streams); then the
  // occupancy bitmap (OCC_SMEM)
  extern __shared__ __align__(16) uint32_t s_mem[];
  constexpr int OFF_OFF = 3 * K3_BM_WORDS + (3 * K3_BM_WORDS & 1);          // 8-byte aligned
  constexpr int OCC_OFF = OFF_OFF + 2 * 2 * (K3_THREADS + 2);
  uint64_t *s_off = reinterpret_cast<uint64_t *>(s_mem + OFF_OFF);          // [2][K3_THREADS + 2]
  const int tid = threadIdx.x;
  const int64_t n_sets = set_end - set_begin;
  const int64_t ntiles = (n_sets + K3_THREADS - 1) / K3_THREADS;
  const int64_t nwords_out = (n_sets + 31) >> 5;
  unsigned long long vox = 0, nhit = 0;

  // asynchronous copy of the offsets of tile t into s_off[buf]: entry i = offsets[s0 + min(i, n_valid)]
  auto prefetch_offsets = [&](int64_t t, int buf) {
    const int64_t s0 = set_begin + t * K3_THREADS;
    const int64_t n_valid = min((int64_t)K3_THREADS, set_end - s0);
    uint64_t *dst = s_off + buf * (K3_THREADS + 2);
    cp_async8(dst + tid, offsets + s0 + min((int64_t)tid, n_valid));
    if (tid == 0) cp_async8(dst + K3_THREADS, offsets + s0 + n_valid);
  };

  // tile schedule.  Plain sweeps: static stride over a grid of up to 8 CTAs per SM.  GATHER: one resident wave
  // whose CTAs take tile ids from a global counter (fetched two tiles ahead, so the id of the next tile is
  // known when its offsets are prefetched): no tail of unevenly loaded CTAs, however many tiles a shard has.
  __shared__ long long s_tile_id[2];
  int64_t tile = blockIdx.x, tile_next = (int64_t)blockIdx.x + gridDim.x;
  if (GATHER) {
    if (tid == 0) {
      s_tile_id[0] = (long long)atomicAdd(xd.done + 2, 1u);
      s_tile_id[1] = (long long)atomicAdd(xd.done + 2, 1u);
    }
    __syncthreads();
    tile = s_tile_id[0];
    tile_next = s_tile_id[1];
    __syncthreads();
  }
  if (tile < ntiles) prefetch_offsets(tile, 0);
  if (OCC_SMEM) {
    for (int i = tid; i < occ_words; i += K3_THREADS) s_mem[OCC_OFF + i] = occ[i];
  }
  for (int i = tid; i < K3_BM_WORDS; i += K3_THREADS) s_mem[i] = 0;
  cp_async_wait_all();
  __syncthreads();
  int hb = 0, mb = 0;   // current hit bitmap / offsets buffer
  // GATHER: verdict words of the tiles this CTA has finished, [K3_GATHER_TILES][8], and their tile ids
  uint32_t *s_gw = s_mem + OCC_OFF + (OCC_SMEM ? occ_words : 0);
  int32_t *s_gtile = reinterpret_cast<int32_t *>(s_gw + K3_GATHER_TILES * (K3_THREADS / 32));
  int kt = 0;
  auto flush_gathered = [&](int ntl) {   // block-uniform argument
    __syncthreads();
    for (int idx = tid; idx < ntl * (K3_THREADS / 32); idx += K3_THREADS) {
      const int64_t t = (int64_t)s_gtile[idx / (K3_THREADS / 32)];
      const int64_t wi = t * (K3_THREADS / 32) + idx % (K3_THREADS / 32);
      if (wi < nwords_out) {
        const uint32_t v = s_gw[idx];
        for (int r = 0; r < xd.world; r++) xd.words(r)[wi] = v;   // P2P stores over NVLink
      }
    }
    __syncthreads();
  };

  for (int it = 0; tile < ntiles; it++) {
    const uint64_t *my_off = s_off + mb * (K3_THREADS + 2);
    const uint64_t t_lo = my_off[0], t_hi = my_off[K3_THREADS];
    const uint64_t lo = my_off[tid], hi = my_off[tid + 1];
    if (tile_next < ntiles) prefetch_offsets(tile_next, mb ^ 1);
    mb ^= 1;
    if (GATHER && tid == 0)   // id of the tile after next; the barrier(s) of this tile publish it
      s_tile_id[it & 1] = (long long)atomicAdd(xd.done + 2, 1u);
    bool own = false;
    if (t_lo == t_hi) {   // a tile of empty sets: no chunk below, but the prefetch still needs its barrier
      cp_async_wait_all();
      __syncthreads();
    }

    for (uint64_t c_lo = t_lo; c_lo < t_hi; c_lo += K3_CHUNK_LEAVES) {   // block-uniform
      const uint64_t c_hi = min(c_lo + (uint64_t)K3_CHUNK_LEAVES, t_hi);
      const uint32_t c_n = (uint32_t)(c_hi - c_lo);
      const int hit_off = hb * K3_BM_WORDS;
      hb = (hb == 2) ? 0 : hb + 1;
      const int next_hit_off = hb * K3_BM_WORDS;

      const int64_t q_begin = (int64_t)(c_lo >> 2);
      const int nq = (int)((int64_t)((c_hi + 3) >> 2) - q_begin);          // <= 8193 quads
      const int32_t head = (int32_t)((q_begin << 2) - (int64_t)c_lo);      // in (-4, 0]

      auto process = [&](int32_t r0, const uint4 &kk, const ulonglong2 &b01, const ulonglong2 &b23) {
        const uint32_t k[4] = {kk.x, kk.y, kk.z, kk.w};
        const uint64_t b[4] = {b01.x, b01.y, b23.x, b23.y};
        uint32_t o[4];
        uint64_t ev[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {   // occupied environment leaf?
          const uint32_t w = OCC_SMEM ? s_mem[OCC_OFF + (k[e] >> 5)] : __ldg(occ + (k[e] >> 5));
          o[e] = (w >> (k[e] & 31)) & 1u;
        }
#pragma unroll
        for (int e = 0; e < 4; e++) ev[e] = ld_env_if(env + k[e], o[e]);
        uint32_t hitmask = 0;
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const uint64_t x = b[e] & ev[e];
          if (x != 0ull) hitmask |= 1u << e;
          if (STATS) {
            if (x != 0ull && (uint32_t)(r0 + e) < c_n) { vox += (unsigned long long)__popcll(x); nhit++; }
          }
        }
        if (hitmask) {
          // clip leaves of the neighbouring chunks / tiles (only the first and last quad can have any)
          if (r0 < 0) { hitmask >>= -r0; r0 = 0; }
          if ((uint32_t)r0 + 4u > c_n) hitmask &= (c_n > (uint32_t)r0) ? (0xFu >> ((uint32_t)r0 + 4u - c_n)) : 0u;
          const uint64_t m = (uint64_t)hitmask << (r0 & 31);
          if ((uint32_t)m) atomicOr(&s_mem[hit_off + (r0 >> 5)], (uint32_t)m);
          if ((uint32_t)(m >> 32)) atomicOr(&s_mem[hit_off + (r0 >> 5) + 1], (uint32_t)(m >> 32));
        }
      };

      // flat walk over the chunk's leaves: software-pipelined ping-pong, the loads of a thread's next
      // quad are issued before its current quad is processed (two quads per thread in flight)
      const uint4 *kp = reinterpret_cast<const uint4 *>(keys) + q_begin + tid;
      const ulonglong2 *bp = reinterpret_cast<const ulonglong2 *>(bits) + 2 * (q_begin + tid);
      int32_t ra = head + 4 * tid;
      uint4 ka = make_uint4(0, 0, 0, 0), kb = ka;
      ulonglong2 a01 = make_ulonglong2(0, 0), a23 = a01, b01 = a01, b23 = a01;
      if (tid < nq) { ka = ld_stream(kp); a01 = ld_stream(bp); a23 = ld_stream(bp + 1); }
      for (int i = tid; i < nq; i += 2 * K3_THREADS) {
        const bool vb = i + K3_THREADS < nq, vc = i + 2 * K3_THREADS < nq;
        if (vb) {
          kb = ld_stream(kp + K3_THREADS);
          b01 = ld_stream(bp + 2 * K3_THREADS);
          b23 = ld_stream(bp + 2 * K3_THREADS + 1);
        }
        process(ra, ka, a01, a23);
        if (vc) {
          ka = ld_stream(kp + 2 * K3_THREADS);
          a01 = ld_stream(bp + 4 * K3_THREADS);
          a23 = ld_stream(bp + 4 * K3_THREADS + 1);
        }
        if (vb) process(ra + 4 * K3_THREADS, kb, b01, b23);
        kp += 2 * K3_THREADS;
        bp += 4 * K3_THREADS;
        ra += 8 * K3_THREADS;
      }
      for (int i = tid; i < K3_BM_WORDS; i += K3_THREADS) s_mem[next_hit_off + i] = 0;
      cp_async_wait_all();
      __syncthreads();

      // does any hit bit fall into this thread's set range, clipped to the chunk?
      const uint64_t a64 = max(lo, c_lo), b64 = min(hi, c_hi);
      if (a64 < b64 && !own) {
        const uint32_t a = (uint32_t)(a64 - c_lo), b = (uint32_t)(b64 - c_lo);   // [a, b), b > a
        const uint32_t w0 = a >> 5, w1 = (b - 1) >> 5;
        for (uint32_t w = w0; w <= w1; w++) {
          uint32_t m = s_mem[hit_off + w];
          if (w == w0) m &= 0xffffffffu << (a & 31);
          if (w == w1) m &= 0xffffffffu >> (31 - ((b - 1) & 31));
          if (m) { own = true; break; }
        }
      }
    }
    const unsigned word = __ballot_sync(0xffffffffu, own);
    const int64_t wi = tile * (K3_THREADS / 32) + (tid >> 5);
    if (GATHER) {
      // stage this CTA's words in shared memory; they go to the peers as 32-byte runs (one tile = 8
      // consecutive words) instead of one 4-byte NVLink write per warp
      if ((tid & 31) == 0) s_gw[kt * (K3_THREADS / 32) + (tid >> 5)] = word;
      if (tid == 0) s_gtile[kt] = (int32_t)tile;
      if (++kt == xd.flush_tiles) { flush_gathered(kt); kt = 0; }
    } else if ((tid & 31) == 0 && wi < nwords_out) {
      verdict[wi] = word;
    }
    const int64_t tile_after = GATHER ? (int64_t)s_tile_id[it & 1] : tile_next + gridDim.x;
    tile = tile_next;
    tile_next = tile_after;
  }
  if (GATHER) {
    flush_gathered(kt);
    // padding words of this rank's slot (sets beyond the shard) read as "no collision" everywhere
    for (int64_t wi = nwords_out + (int64_t)blockIdx.x * K3_THREADS + tid; wi < xd.slot_words;
         wi += (int64_t)gridDim.x * K3_THREADS)
      for (int r = 0; r < xd.world; r++) xd.words(r)[wi] = 0u;
    xchg_signal(xd);
  }
  if (STATS) {
    for (int o = 16; o > 0; o >>= 1) {
      vox += __shfl_down_sync(0xffffffffu, vox, o);
      nhit += __shfl_down_sync(0xffffffffu, nhit, o);
    }
    if ((tid & 31) == 0 && (vox | nhit)) {
      atomicAdd(&stats[0], vox);
      atomicAdd(&stats[1], nhit);
    }
  }
}

// a rank whose shard is empty still has to clear its slot and raise its flag
__global__ void xchg_empty_shard_kernel(const XchgDev xd) {
  for (int64_t wi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; wi < xd.slot_words;
       wi += (int64_t)gridDim.x * blockDim.x)
    for (int r = 0; r < xd.world; r++) xd.words(r)[wi] = 0u;
  xchg_signal(xd);
}

int ensure_store_capacity(irt_ctx *ctx, irt_setstore *s, int64_t n_sets, int64_t n_blocks) {
  if ((size_t)(n_sets + 1) > s->cap_sets) {
    if (s->d_offsets) cudaFree(s->d_offsets);
    s->d_offsets = nullptr;
    s->cap_sets = 0;
    IRT_CUDA(ctx, cudaMalloc(&s->d_offsets, (size_t)(n_sets + 1) * 8));
    s->cap_sets = (size_t)(n_sets + 1);
  }
  if ((size_t)n_blocks + 4 > s->cap_blocks) {
    if (s->d_keys) cudaFree(s->d_keys);
    if (s->d_bits) cudaFree(s->d_bits);
    s->d_keys = nullptr; s->d_bits = nullptr; s->cap_blocks = 0;
    IRT_CUDA(ctx, cudaMalloc(&s->d_keys, ((size_t)n_blocks + 4) * 4));
    IRT_CUDA(ctx, cudaMalloc(&s->d_bits, ((size_t)n_blocks + 4) * 8));
    s->cap_blocks = (size_t)n_blocks + 4;
  }
  return IRT_OK;
}

// ---- append: stream compaction of a CSR range onto the end of another store ----------------------
// (kept leaves before set i, kept sets before set i): the exclusive scan of these gives every kept set its leaf
// position and its slot in the destination at once
struct __align__(16) AppendPos {
  unsigned long long leaves, sets;
};
struct AppendPosSum {
  __device__ __forceinline__ AppendPos operator()(const AppendPos &a, const AppendPos &b) const {
    return {a.leaves + b.leaves, a.sets + b.sets};
  }
};

// pos[i] = (leaf count, 1) of set begin + i if it is kept, else (0, 0); pos[n] = (0, 0), so that the exclusive scan
// of n + 1 entries ends with the totals
__global__ void append_count_kernel(const uint64_t *__restrict__ src_off, int64_t begin, int64_t n,
                                    const uint32_t *__restrict__ keep, AppendPos *__restrict__ pos) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  const bool kept = i < n && (!keep || ((keep[i >> 5] >> (i & 31)) & 1u));
  pos[i] = kept ? AppendPos{src_off[begin + i + 1] - src_off[begin + i], 1ull} : AppendPos{0ull, 0ull};
}

// one warp per source set: a kept set's keys and bits go to their scanned position (lanes over its leaves, so every
// load and store of a warp is one contiguous run) and its end offset to its slot
constexpr int APPEND_THREADS = 256;
__global__ void __launch_bounds__(APPEND_THREADS)
append_gather_kernel(const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_keys,
                     const uint64_t *__restrict__ src_bits, int64_t begin, int64_t n,
                     const AppendPos *__restrict__ pos, uint64_t dst_blocks, int64_t dst_sets,
                     uint64_t *__restrict__ dst_off, uint32_t *__restrict__ dst_keys,
                     uint64_t *__restrict__ dst_bits) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (APPEND_THREADS / 32);
  for (int64_t i = (int64_t)blockIdx.x * (APPEND_THREADS / 32) + (threadIdx.x >> 5); i < n; i += warps) {
    const AppendPos p = pos[i], q = pos[i + 1];
    if (q.sets == p.sets) continue;   // masked out
    const uint64_t len = q.leaves - p.leaves;
    const uint64_t from = src_off[begin + i], to = dst_blocks + p.leaves;
    for (uint64_t j = lane; j < len; j += 32) {
      dst_keys[to + j] = src_keys[from + j];
      dst_bits[to + j] = src_bits[from + j];
    }
    if (lane == 0) dst_off[dst_sets + 1 + (int64_t)p.sets] = dst_blocks + q.leaves;
  }
}

}  // namespace

// the start of every replacement of a store's content (import, and voxel_raster.cu before it fills the store)
int setstore_reserve(irt_ctx *ctx, irt_setstore *s, int64_t n_sets, int64_t n_blocks) {
  s->generation++;
  return ensure_store_capacity(ctx, s, n_sets, n_blocks);
}

// content-preserving growth of the keys/bits arrays (amortised x1.5)
int setstore_grow_blocks(irt_ctx *ctx, irt_setstore *s, int64_t need_blocks, int64_t keep_blocks,
                         cudaStream_t st) {
  if ((size_t)need_blocks + 4 <= s->cap_blocks) return IRT_OK;
  size_t cap = s->cap_blocks + s->cap_blocks / 2;
  if (cap < (size_t)need_blocks + 4) cap = (size_t)need_blocks + 4;
  uint32_t *nk = nullptr;
  uint64_t *nb = nullptr;
  IRT_CUDA(ctx, cudaMalloc(&nk, cap * 4));
  IRT_CUDA(ctx, cudaMalloc(&nb, cap * 8));
  if (keep_blocks > 0) {
    IRT_CUDA(ctx, cudaMemcpyAsync(nk, s->d_keys, (size_t)keep_blocks * 4, cudaMemcpyDeviceToDevice, st));
    IRT_CUDA(ctx, cudaMemcpyAsync(nb, s->d_bits, (size_t)keep_blocks * 8, cudaMemcpyDeviceToDevice, st));
    IRT_CUDA(ctx, cudaStreamSynchronize(st));
  }
  if (s->d_keys) cudaFree(s->d_keys);
  if (s->d_bits) cudaFree(s->d_bits);
  s->d_keys = nk;
  s->d_bits = nb;
  s->cap_blocks = cap;
  return IRT_OK;
}

// the same for the offsets array: room for need_sets sets (need_sets + 1 offsets), the first keep_sets + 1 offsets
// kept; a store that never held an offsets array gets offsets[0] = 0
static int setstore_grow_sets(irt_ctx *ctx, irt_setstore *s, int64_t need_sets, int64_t keep_sets,
                              cudaStream_t st) {
  if ((size_t)need_sets + 1 <= s->cap_sets) return IRT_OK;
  size_t cap = s->cap_sets + s->cap_sets / 2;
  if (cap < (size_t)need_sets + 1) cap = (size_t)need_sets + 1;
  uint64_t *no = nullptr;
  IRT_CUDA(ctx, cudaMalloc(&no, cap * 8));
  if (s->d_offsets) {
    IRT_CUDA(ctx, cudaMemcpyAsync(no, s->d_offsets, (size_t)(keep_sets + 1) * 8, cudaMemcpyDeviceToDevice, st));
    IRT_CUDA(ctx, cudaStreamSynchronize(st));
    cudaFree(s->d_offsets);
  } else {
    IRT_CUDA(ctx, cudaMemsetAsync(no, 0, 8, st));
  }
  s->d_offsets = no;
  s->cap_sets = cap;
  return IRT_OK;
}

int setstore_finalize(irt_ctx *ctx, irt_setstore *s, int64_t n_sets, int64_t n_blocks,
                      cudaStream_t st) {
  // K3 reads whole 16-byte quads: the (clipped) leaves past the end of the store must hold valid keys
  if (s->d_keys) IRT_CUDA(ctx, cudaMemsetAsync(s->d_keys + n_blocks, 0, 4 * sizeof(uint32_t), st));
  s->n_sets = n_sets;
  s->n_blocks = n_blocks;
  return IRT_OK;
}

extern "C" {

// ---- environment -------------------------------------------------------------------------
int irt_env_create(irt_ctx *ctx, const irt_grid *grid, irt_env **out) {
  if (!ctx || !out) return IRT_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  int rc = grid_check(ctx, grid);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  irt_env *e = new irt_env();
  e->ctx = ctx;
  e->grid = *grid;
  e->gd = make_grid_dev(*grid);
  const int64_t nblk = (int64_t)e->gd.Nb * e->gd.Nb * e->gd.Nb;
  e->n_blocks_total = nblk;
  const int64_t nwords = (nblk + 31) / 32;
  if (cudaMalloc(&e->d_blocks, (size_t)nblk * 8) != cudaSuccess ||
      cudaMalloc(&e->d_occ, (size_t)nwords * 4) != cudaSuccess) {
    irt_env_destroy(e);
    return irt_fail(ctx, IRT_ERR_CUDA, "environment allocation failed");
  }
  cudaMemsetAsync(e->d_blocks, 0, (size_t)nblk * 8, ctx->stream);
  cudaMemsetAsync(e->d_occ, 0, (size_t)nwords * 4, ctx->stream);
  IRT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *out = e;
  return IRT_OK;
}

void irt_env_destroy(irt_env *env) {
  if (!env) return;
  cudaSetDevice(env->ctx->device);
  if (env->d_blocks) cudaFree(env->d_blocks);
  if (env->d_occ) cudaFree(env->d_occ);
  delete env;
}

}  // extern "C"
int env_rebuild_occ(irt_ctx *ctx, irt_env *env, cudaStream_t st) {
  const int64_t nwords = (env->n_blocks_total + 31) / 32;
  const int T = 256;
  env_build_occ_kernel<<<(unsigned)((nwords + T - 1) / T), T, 0, st>>>(env->d_blocks,
                                                                      env->n_blocks_total, env->d_occ);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  return IRT_OK;
}
extern "C" {

int irt_env_update_dev(irt_ctx *ctx, irt_env *env, const uint64_t *d_blocks, void *stream) {
  if (!ctx || !env || !d_blocks) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  IRT_CUDA(ctx, cudaMemcpyAsync(env->d_blocks, d_blocks, (size_t)env->n_blocks_total * 8,
                                cudaMemcpyDeviceToDevice, st));
  return env_rebuild_occ(ctx, env, st);
}

int irt_env_update(irt_ctx *ctx, irt_env *env, const uint64_t *blocks) {
  if (!ctx || !env || !blocks) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  IRT_CUDA(ctx, cudaMemcpyAsync(env->d_blocks, blocks, (size_t)env->n_blocks_total * 8,
                                cudaMemcpyHostToDevice, ctx->stream));
  int rc = env_rebuild_occ(ctx, env, ctx->stream);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return IRT_OK;
}

int irt_env_update_sparse(irt_ctx *ctx, irt_env *env, const uint8_t *bxyz, const uint64_t *bits,
                          int64_t nblocks) {
  if (!ctx || !env || nblocks < 0 || (nblocks > 0 && (!bxyz || !bits)))
    return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  for (int64_t i = 0; i < nblocks; i++)
    if (bxyz[3 * i] >= env->gd.Nb || bxyz[3 * i + 1] >= env->gd.Nb || bxyz[3 * i + 2] >= env->gd.Nb)
      return irt_fail(ctx, IRT_ERR_OUT_OF_RANGE, "block index outside the grid");
  IRT_CUDA(ctx, cudaMemsetAsync(env->d_blocks, 0, (size_t)env->n_blocks_total * 8, st));
  if (nblocks > 0) {
    char *scr = (char *)ctx_scratch(ctx, (size_t)nblocks * 11 + 64);
    if (!scr) return irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc failed");
    uint64_t *d_bits = (uint64_t *)scr;
    uint8_t *d_xyz = (uint8_t *)(scr + (size_t)nblocks * 8);
    IRT_CUDA(ctx, cudaMemcpyAsync(d_bits, bits, (size_t)nblocks * 8, cudaMemcpyHostToDevice, st));
    IRT_CUDA(ctx, cudaMemcpyAsync(d_xyz, bxyz, (size_t)nblocks * 3, cudaMemcpyHostToDevice, st));
    const int T = 256;
    env_scatter_sparse_kernel<<<(unsigned)((nblocks + T - 1) / T), T, 0, st>>>(
        d_xyz, d_bits, nblocks, env->gd.levels, env->d_blocks);
    IRT_LAUNCHED(ctx);
  }
  int rc = env_rebuild_occ(ctx, env, st);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaStreamSynchronize(st));
  return IRT_OK;
}

int64_t irt_env_nblocks(irt_ctx *ctx, const irt_env *env) {
  if (!ctx || !env) return -1;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return -1;
  unsigned long long *d = (unsigned long long *)ctx_scratch(ctx, 64);
  if (!d) return -1;
  cudaMemsetAsync(d, 0, 8, ctx->stream);
  const int T = 256;
  count_nonzero_kernel<<<(unsigned)((env->n_blocks_total + T - 1) / T), T, 0, ctx->stream>>>(
      env->d_blocks, env->n_blocks_total, d);
  IRT_LAUNCHED(ctx);
  unsigned long long h = 0;
  if (cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) return -1;
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -1;
  return (int64_t)h;
}

// ---- set store ---------------------------------------------------------------------------
int irt_setstore_create(irt_ctx *ctx, const irt_grid *grid, irt_setstore **out) {
  if (!ctx || !out) return IRT_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  int rc = grid_check(ctx, grid);
  if (rc) return rc;
  irt_setstore *s = new irt_setstore();
  s->ctx = ctx;
  s->grid = *grid;
  s->gd = make_grid_dev(*grid);
  *out = s;
  return IRT_OK;
}

void irt_setstore_destroy(irt_setstore *s) {
  if (!s) return;
  cudaSetDevice(s->ctx->device);
  if (s->d_offsets) cudaFree(s->d_offsets);
  if (s->d_keys) cudaFree(s->d_keys);
  if (s->d_bits) cudaFree(s->d_bits);
  delete s;
}

int64_t irt_setstore_num_sets(const irt_setstore *s) { return s ? s->n_sets : -1; }
int64_t irt_setstore_num_blocks(const irt_setstore *s) { return s ? s->n_blocks : -1; }

int irt_setstore_import(irt_ctx *ctx, irt_setstore *s, int64_t n_sets, const uint64_t *offsets,
                        const uint32_t *keys, const uint64_t *bits) {
  if (!ctx || !s || n_sets < 0 || !offsets) return IRT_ERR_INVALID_ARGUMENT;
  if (offsets[0] != 0) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "offsets[0] must be 0");
  const int64_t nb = (int64_t)offsets[n_sets];
  if (nb > 0 && (!keys || !bits)) return IRT_ERR_INVALID_ARGUMENT;
  const uint32_t nkeys = (uint32_t)((int64_t)s->gd.Nb * s->gd.Nb * s->gd.Nb);
  for (int64_t i = 0; i < n_sets; i++)
    if (offsets[i + 1] < offsets[i]) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "offsets not monotone");
  for (int64_t i = 0; i < nb; i++)
    if (keys[i] >= nkeys) return irt_fail(ctx, IRT_ERR_OUT_OF_RANGE, "block key outside the grid");
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  int rc = setstore_reserve(ctx, s, n_sets, nb);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  IRT_CUDA(ctx, cudaMemcpyAsync(s->d_offsets, offsets, (size_t)(n_sets + 1) * 8, cudaMemcpyHostToDevice, st));
  if (nb > 0) {
    IRT_CUDA(ctx, cudaMemcpyAsync(s->d_keys, keys, (size_t)nb * 4, cudaMemcpyHostToDevice, st));
    IRT_CUDA(ctx, cudaMemcpyAsync(s->d_bits, bits, (size_t)nb * 8, cudaMemcpyHostToDevice, st));
  }
  rc = setstore_finalize(ctx, s, n_sets, nb, st);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaStreamSynchronize(st));
  return IRT_OK;
}

int irt_setstore_export(irt_ctx *ctx, const irt_setstore *s, uint64_t *offsets, uint32_t *keys,
                        uint64_t *bits) {
  if (!ctx || !s) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  if (offsets) {
    if (s->d_offsets)
      IRT_CUDA(ctx, cudaMemcpyAsync(offsets, s->d_offsets, (size_t)(s->n_sets + 1) * 8, cudaMemcpyDeviceToHost, st));
    else
      offsets[0] = 0;
  }
  if (keys && s->n_blocks > 0)
    IRT_CUDA(ctx, cudaMemcpyAsync(keys, s->d_keys, (size_t)s->n_blocks * 4, cudaMemcpyDeviceToHost, st));
  if (bits && s->n_blocks > 0)
    IRT_CUDA(ctx, cudaMemcpyAsync(bits, s->d_bits, (size_t)s->n_blocks * 8, cudaMemcpyDeviceToHost, st));
  IRT_CUDA(ctx, cudaStreamSynchronize(st));
  return IRT_OK;
}

int irt_setstore_device_ptrs(const irt_setstore *s, const uint64_t **d_offsets,
                             const uint32_t **d_keys, const uint64_t **d_bits) {
  if (!s) return IRT_ERR_INVALID_ARGUMENT;
  if (d_offsets) *d_offsets = s->d_offsets;
  if (d_keys) *d_keys = s->d_keys;
  if (d_bits) *d_bits = s->d_bits;
  return IRT_OK;
}

// count + scan (one CUB scan of (leaves, sets) pairs), one read-back of the totals to size the growth, then the
// gather; dst is only written once every argument has been checked and the scratch is in place
int irt_setstore_append(irt_ctx *ctx, irt_setstore *dst, const irt_setstore *src, int64_t begin, int64_t end,
                        const uint32_t *keep_words) {
  if (!ctx || !dst || !src) return IRT_ERR_INVALID_ARGUMENT;
  if (dst == src) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "a store cannot be appended to itself");
  if (dst->ctx->device != ctx->device || src->ctx->device != ctx->device)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "stores of another device");
  if (!same_grid(dst->grid, src->grid)) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "the stores' grids differ");
  if (begin < 0 || begin > end || end > src->n_sets)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "set range [%lld,%lld) outside [0,%lld]", (long long)begin,
                    (long long)end, (long long)src->n_sets);
  const int64_t n = end - begin;
  const int64_t nwords = (n + 31) / 32;
  if (keep_words) {
    int64_t kept = 0;
    for (int64_t w = 0; w < nwords; w++) {
      uint32_t m = keep_words[w];
      if (w == nwords - 1 && (n & 31)) m &= (1u << (n & 31)) - 1u;
      kept += __builtin_popcount(m);
    }
    if (kept == 0) return IRT_OK;
  }
  if (n == 0) return IRT_OK;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;

  AppendPos *d_pos = nullptr;
  size_t cub_bytes = 0;
  IRT_CUDA(ctx, cub::DeviceScan::ExclusiveScan(nullptr, cub_bytes, d_pos, d_pos, AppendPosSum(),
                                               AppendPos{0ull, 0ull}, n + 1, st));
  const size_t pos_bytes = ((size_t)(n + 1) * sizeof(AppendPos) + 255) & ~(size_t)255;
  const size_t cub_off = pos_bytes, keep_off = cub_off + ((cub_bytes + 255) & ~(size_t)255);
  char *scr = (char *)ctx_scratch(ctx, keep_off + (size_t)nwords * 4 + 64);
  if (!scr) return irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc failed");
  d_pos = (AppendPos *)scr;
  uint32_t *d_keep = nullptr;
  if (keep_words) {
    d_keep = (uint32_t *)(scr + keep_off);
    IRT_CUDA(ctx, cudaMemcpyAsync(d_keep, keep_words, (size_t)nwords * 4, cudaMemcpyHostToDevice, st));
  }
  const int T = 256;
  append_count_kernel<<<(unsigned)((n + T) / T), T, 0, st>>>(src->d_offsets, begin, n, d_keep, d_pos);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  IRT_CUDA(ctx, cub::DeviceScan::ExclusiveScan(scr + cub_off, cub_bytes, d_pos, d_pos, AppendPosSum(),
                                               AppendPos{0ull, 0ull}, n + 1, st));
  IRT_LAUNCHED(ctx);
  AppendPos total;
  IRT_CUDA(ctx, cudaMemcpyAsync(&total, d_pos + n, sizeof(total), cudaMemcpyDeviceToHost, st));
  IRT_CUDA(ctx, cudaStreamSynchronize(st));

  const int64_t new_sets = dst->n_sets + (int64_t)total.sets, new_blocks = dst->n_blocks + (int64_t)total.leaves;
  int rc = setstore_grow_sets(ctx, dst, new_sets, dst->n_sets, st);
  if (rc) return rc;
  rc = setstore_grow_blocks(ctx, dst, new_blocks, dst->n_blocks, st);
  if (rc) return rc;
  int64_t blocks = (n + APPEND_THREADS / 32 - 1) / (APPEND_THREADS / 32);
  if (blocks > (int64_t)ctx->sm_count * 16) blocks = (int64_t)ctx->sm_count * 16;
  append_gather_kernel<<<(unsigned)blocks, APPEND_THREADS, 0, st>>>(
      src->d_offsets, src->d_keys, src->d_bits, begin, n, d_pos, (uint64_t)dst->n_blocks, dst->n_sets,
      dst->d_offsets, dst->d_keys, dst->d_bits);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  rc = setstore_finalize(ctx, dst, new_sets, new_blocks, st);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaStreamSynchronize(st));
  return IRT_OK;
}

// ---- K3 ----------------------------------------------------------------------------------
static int check_sets_impl(irt_ctx *ctx, const irt_setstore *store, const irt_env *env,
                           int64_t begin, int64_t end, uint32_t *d_verdict,
                           unsigned long long *d_stats, cudaStream_t st, const XchgDev *xd = nullptr) {
  if (!ctx || !store || !env || (!d_verdict && !xd)) return IRT_ERR_INVALID_ARGUMENT;
  if (store->grid.Ng != env->grid.Ng)  // check_dims -- collision/VoxelOctree.cpp:46-53
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "voxel dimension mismatch (%d != %d)",
                    store->grid.Ng, env->grid.Ng);
  if (begin < 0 || end < begin || end > store->n_sets)
    return irt_fail(ctx, IRT_ERR_OUT_OF_RANGE, "set range [%lld,%lld) outside [0,%lld)",
                    (long long)begin, (long long)end, (long long)store->n_sets);
  const int64_t n = end - begin;
  if (xd && (n == 0 || store->n_blocks == 0)) {   // nothing to test: clear the slot, raise the flag
    xchg_empty_shard_kernel<<<8, 256, 0, st>>>(*xd);
    IRT_LAUNCHED(ctx);
    IRT_CUDA(ctx, cudaGetLastError());
    return IRT_OK;
  }
  if (n == 0) return IRT_OK;
  if (store->n_blocks == 0) {
    IRT_CUDA(ctx, cudaMemsetAsync(d_verdict, 0, (size_t)((n + 31) / 32) * 4, st));
    return IRT_OK;
  }
  const int occ_words = (int)((env->n_blocks_total + 31) / 32);
  const bool occ_smem = (size_t)occ_words * 4 <= 64 * 1024;
  int64_t blocks = (n + K3_THREADS - 1) / K3_THREADS;     // one CTA per tile of 256 sets ...
  // ... a grid of up to 8 CTAs per SM striding over the tiles: __launch_bounds__(256, 4) keeps 4 resident per
  // SM, i.e. two waves (the second wave's early CTAs start while the first wave's late ones drain)
  const int64_t max_blocks = (int64_t)ctx->sm_count * 8;
  if (blocks > max_blocks) blocks = max_blocks;
  const size_t smem = (size_t)K3_SMEM_FIXED_WORDS * 4 + (occ_smem ? (size_t)occ_words * 4 : 0);
#define K3_LAUNCH(OS, ST)                                                                          \
  do {                                                                                             \
    auto kfn = voxel_and_popc_kernel<OS, ST>;                                                      \
    if (smem > 48 * 1024)                                                                          \
      IRT_CUDA(ctx, cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kfn<<<(unsigned)blocks, K3_THREADS, smem, st>>>(store->d_keys, store->d_bits, store->d_offsets, \
                                                    env->d_blocks, env->d_occ, occ_words, begin,   \
                                                    end, d_verdict, d_stats, XchgDev());           \
  } while (0)
#define K3_LAUNCH_GATHER(OS)                                                                       \
  do {                                                                                             \
    auto kfn = voxel_and_popc_kernel<OS, false, true>;                                             \
    const size_t gsmem = smem + (size_t)K3_GATHER_TILES * (K3_THREADS / 32 + 1) * 4;               \
    if (gsmem > 48 * 1024)                                                                         \
      IRT_CUDA(ctx, cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsmem)); \
    kfn<<<(unsigned)blocks, K3_THREADS, gsmem, st>>>(store->d_keys, store->d_bits, store->d_offsets, \
                                                    env->d_blocks, env->d_occ, occ_words, begin,   \
                                                    end, nullptr, nullptr, *xd);                   \
  } while (0)
  if (xd) {
    // one resident wave with dynamic tile scheduling (the CTAs take tile ids from a counter): every CTA ends
    // with ONE system-scope fence, and no CTA is left with an extra tile at the end of the sweep
    if (blocks > (int64_t)ctx->sm_count * 4) blocks = (int64_t)ctx->sm_count * 4;
    if ((n + 31) / 32 > xd->slot_words)
      return irt_fail(ctx, IRT_ERR_CAPACITY, "shard of %lld sets exceeds the exchange slot (%lld words)",
                      (long long)n, (long long)xd->slot_words);
    if (occ_smem) K3_LAUNCH_GATHER(true); else K3_LAUNCH_GATHER(false);
  } else if (occ_smem) {
    if (d_stats) K3_LAUNCH(true, true); else K3_LAUNCH(true, false);
  } else {
    if (d_stats) K3_LAUNCH(false, true); else K3_LAUNCH(false, false);
  }
#undef K3_LAUNCH_GATHER
#undef K3_LAUNCH
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  return IRT_OK;
}

}  // extern "C"
int check_sets_launch(irt_ctx *ctx, const irt_setstore *store, const irt_env *env, int64_t begin, int64_t end,
                      uint32_t *d_verdict, cudaStream_t st) {
  return check_sets_impl(ctx, store, env, begin, end, d_verdict, nullptr, st);
}
extern "C" {

// ---- verdict exchange over peer memory (multi-GPU) ----------------------------------------------
struct irt_xchg {
  irt_ctx *ctx = nullptr;
  int rank = 0, world = 1;
  int64_t slot_words = 0;
  uint32_t *local = nullptr;          // words[2][world][slot_words], flags[2][world]
  uint32_t *peer[IRT_MAX_PEERS] = {};  // peers' buffers mapped here (peer[rank] == local)
  bool opened[IRT_MAX_PEERS] = {};
  unsigned int *d_done = nullptr;     // [0] CTA counter, [1] error word, [2] dynamic tile counter
  uint32_t epoch = 0;
  bool connected = false;
};

int irt_xchg_create(irt_ctx *ctx, int rank, int world, int64_t slot_words, irt_xchg **out) {
  if (!ctx || !out || world < 1 || world > IRT_MAX_PEERS || rank < 0 || rank >= world || slot_words < 1)
    return IRT_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  irt_xchg *x = new irt_xchg();
  x->ctx = ctx; x->rank = rank; x->world = world; x->slot_words = slot_words;
  const size_t bytes = ((size_t)2 * world * slot_words + (size_t)2 * world) * 4;
  if (cudaMalloc(&x->local, bytes) != cudaSuccess || cudaMalloc(&x->d_done, 64) != cudaSuccess) {
    irt_xchg_destroy(x);
    return irt_fail(ctx, IRT_ERR_CUDA, "exchange buffer allocation failed");
  }
  cudaMemset(x->local, 0, bytes);
  cudaMemset(x->d_done, 0, 64);
  x->peer[rank] = x->local;
  x->connected = (world == 1);
  *out = x;
  return IRT_OK;
}

void irt_xchg_destroy(irt_xchg *x) {
  if (!x) return;
  cudaSetDevice(x->ctx->device);
  cudaDeviceSynchronize();
  for (int r = 0; r < x->world; r++)
    if (x->opened[r]) cudaIpcCloseMemHandle(x->peer[r]);
  if (x->local) cudaFree(x->local);
  if (x->d_done) cudaFree(x->d_done);
  delete x;
}

int irt_xchg_handle_size(void) { return (int)sizeof(cudaIpcMemHandle_t); }

// the handle every rank publishes (host-side all-gather of irt_xchg_handle_size() bytes per rank)
int irt_xchg_export(irt_xchg *x, void *handle) {
  if (!x || !handle) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(x->ctx, cudaSetDevice(x->ctx->device));
  cudaIpcMemHandle_t h;
  IRT_CUDA(x->ctx, cudaIpcGetMemHandle(&h, x->local));
  std::memcpy(handle, &h, sizeof(h));
  return IRT_OK;
}

// handles: [world][irt_xchg_handle_size()] in rank order.  Collective in the sense that every rank must
// have created its buffer before any rank connects.
int irt_xchg_connect(irt_xchg *x, const void *handles) {
  if (!x || !handles) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(x->ctx, cudaSetDevice(x->ctx->device));
  for (int r = 0; r < x->world; r++) {
    if (r == x->rank || x->opened[r]) continue;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, (const char *)handles + (size_t)r * sizeof(h), sizeof(h));
    void *p = nullptr;
    IRT_CUDA(x->ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    x->peer[r] = (uint32_t *)p;
    x->opened[r] = true;
  }
  x->connected = true;
  return IRT_OK;
}

// K3 over sets [begin, end) of this rank's store with the verdict all-gather fused in: on return of
// the stream work, *d_gathered (device, [world][slot_words] words, rank-major) holds every rank's
// verdict words of this sweep.  Consumers must read it in stream order before the sweep after next
// (two buffers alternate).  Every rank must call this the same number of times.
int irt_check_sets_allgather_dev(irt_ctx *ctx, const irt_setstore *store, const irt_env *env,
                                 int64_t begin, int64_t end, irt_xchg *x, void *stream,
                                 const uint32_t **d_gathered) {
  if (!ctx || !x || !store || !env) return IRT_ERR_INVALID_ARGUMENT;
  if (!x->connected) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "exchange not connected");
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  x->epoch++;
  XchgDev xd;
  std::memset(&xd, 0, sizeof(xd));
  for (int r = 0; r < x->world; r++) xd.peer[r] = x->peer[r];
  xd.world = x->world; xd.rank = x->rank; xd.parity = (int)(x->epoch & 1u);
  xd.slot_words = x->slot_words; xd.epoch = x->epoch; xd.done = x->d_done;
  xd.flush_tiles = K3_GATHER_FLUSH_TILES;
  int rc = check_sets_impl(ctx, store, env, begin, end, nullptr, nullptr, st, &xd);
  if (rc) return rc;
  // (the kernel's last CTA has waited for every peer's flag: the gathered array is complete when it ends)
  if (d_gathered) *d_gathered = x->local + (size_t)xd.parity * x->world * x->slot_words;
  return IRT_OK;
}

// 0 when every wait so far saw all peers arrive; 1 + rank of a peer that timed out otherwise
int irt_xchg_status(irt_xchg *x) {
  if (!x) return -1;
  unsigned int e = 0;
  cudaSetDevice(x->ctx->device);
  cudaMemcpy(&e, x->d_done + 1, 4, cudaMemcpyDeviceToHost);
  return (int)e;
}

int irt_check_sets_dev(irt_ctx *ctx, const irt_setstore *store, const irt_env *env,
                       int64_t begin, int64_t end, uint32_t *d_verdict_words, void *stream) {
  if (!ctx) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  return check_sets_impl(ctx, store, env, begin, end, d_verdict_words, nullptr, st);
}

int irt_check_sets(irt_ctx *ctx, const irt_setstore *store, const irt_env *env, int64_t begin,
                   int64_t end, uint32_t *verdict_words) {
  if (!ctx || !verdict_words) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t n = end - begin;
  if (n <= 0) return (n == 0) ? IRT_OK : IRT_ERR_OUT_OF_RANGE;
  const size_t words = (size_t)((n + 31) / 32);
  uint32_t *d_v = (uint32_t *)ctx_scratch(ctx, words * 4 + 64);
  if (!d_v) return irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc failed");
  int rc = check_sets_impl(ctx, store, env, begin, end, d_v, nullptr, ctx->stream);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaMemcpyAsync(verdict_words, d_v, words * 4, cudaMemcpyDeviceToHost, ctx->stream));
  IRT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return IRT_OK;
}

// colliding-voxel popcount over the range: stats[0] = sum popc(bits & env), stats[1] = #leaves hit
int irt_check_sets_popcount(irt_ctx *ctx, const irt_setstore *store, const irt_env *env,
                            int64_t begin, int64_t end, uint64_t *stats) {
  if (!ctx || !stats) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t n = end - begin;
  stats[0] = stats[1] = 0;
  if (n <= 0) return (n == 0) ? IRT_OK : IRT_ERR_OUT_OF_RANGE;
  const size_t words = (size_t)((n + 31) / 32);
  char *scr = (char *)ctx_scratch(ctx, words * 4 + 128);
  if (!scr) return irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc failed");
  unsigned long long *d_stats = (unsigned long long *)scr;
  uint32_t *d_v = (uint32_t *)(scr + 64);
  IRT_CUDA(ctx, cudaMemsetAsync(d_stats, 0, 16, ctx->stream));
  int rc = check_sets_impl(ctx, store, env, begin, end, d_v, d_stats, ctx->stream);
  if (rc) return rc;
  IRT_CUDA(ctx, cudaMemcpyAsync(stats, d_stats, 16, cudaMemcpyDeviceToHost, ctx->stream));
  IRT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return IRT_OK;
}

int64_t irt_check_sets_algorithmic_bytes(const irt_setstore *store, int64_t begin, int64_t end) {
  if (!store || begin < 0 || end < begin || end > store->n_sets) return -1;
  if (end == begin) return 0;
  uint64_t lr[2] = {0, 0};
  if (cudaSetDevice(store->ctx->device) != cudaSuccess) return -1;
  if (cudaMemcpy(&lr[0], store->d_offsets + begin, 8, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  if (cudaMemcpy(&lr[1], store->d_offsets + end, 8, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  const int64_t nb = (int64_t)(lr[1] - lr[0]), n = end - begin;
  const int64_t Nb = store->gd.Nb;
  return 12 * nb + 8 * n + 8 * Nb * Nb * Nb + (n + 7) / 8;
}

}  // extern "C"
