// ctx.cu -- context, robot constants / routing tables, grid helpers, FP64 peak probe.
#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <limits>

#include <atomic>

#include "common.cuh"

int irt_fail(irt_ctx *ctx, int status, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->last_error = buf;
  }
  return status;
}

void irt_launched(irt_ctx *ctx, const char *file, int line) {
  ctx->launches.fetch_add(1, std::memory_order_relaxed);
  if (ctx->debug_sync) {
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
      std::fprintf(stderr, "[irt debug] kernel launched at %s:%d failed: %s\n", file, line, cudaGetErrorString(e));
      std::fflush(stderr);
      ctx->debug_sync = false;
    }
  }
}

void *ctx_scratch(irt_ctx *ctx, size_t bytes) {
  if (bytes <= ctx->scratch_bytes) return ctx->scratch;
  if (ctx->scratch) cudaFree(ctx->scratch);
  ctx->scratch = nullptr;
  ctx->scratch_bytes = 0;
  size_t want = bytes + bytes / 4;
  if (cudaMalloc(&ctx->scratch, want) != cudaSuccess) {
    if (cudaMalloc(&ctx->scratch, bytes) != cudaSuccess) return nullptr;
    want = bytes;
  }
  ctx->scratch_bytes = want;
  return ctx->scratch;
}

void *ctx_arena(irt_ctx *ctx, size_t bytes) {
  if (bytes <= ctx->arena_bytes) return ctx->arena;
  if (ctx->arena) cudaFree(ctx->arena);
  ctx->arena = nullptr;
  ctx->arena_bytes = 0;
  if (cudaMalloc(&ctx->arena, bytes) != cudaSuccess) return nullptr;
  ctx->arena_bytes = bytes;
  return ctx->arena;
}

void *ctx_io(irt_ctx *ctx, size_t bytes) {
  if (bytes <= ctx->io_bytes) return ctx->io;
  if (ctx->io) cudaFree(ctx->io);   // (the pinned host buffer is independent of this one: ctx_pinned owns it)
  ctx->io = nullptr;
  ctx->io_bytes = 0;
  if (cudaMalloc(&ctx->io, bytes) != cudaSuccess) return nullptr;
  ctx->io_bytes = bytes;
  return ctx->io;
}

void *ctx_pinned(irt_ctx *ctx, size_t bytes) {
  if (bytes <= ctx->pinned_bytes) return ctx->pinned;
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  ctx->pinned = nullptr;
  ctx->pinned_bytes = 0;
  if (cudaMallocHost(&ctx->pinned, bytes) != cudaSuccess) return nullptr;
  ctx->pinned_bytes = bytes;
  return ctx->pinned;
}

extern "C" {

int irt_abi_version(void) { return IRT_ABI_VERSION; }

const char *irt_status_string(int s) {
  switch (s) {
    case IRT_OK: return "ok";
    case IRT_ERR_NO_DEVICE: return "no CUDA device (there is no CPU fallback)";
    case IRT_ERR_INVALID_ARGUMENT: return "invalid argument";
    case IRT_ERR_OUT_OF_RANGE: return "out of range";
    case IRT_ERR_CUDA: return "CUDA error";
    case IRT_ERR_UNSUPPORTED: return "unsupported";
    case IRT_ERR_CAPACITY: return "capacity exceeded";
    case IRT_ERR_DOMAIN: return "point outside the voxel domain";
    default: return "unknown status";
  }
}

int irt_ctx_create(int device, irt_ctx **out) {
  if (!out) return IRT_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) return IRT_ERR_NO_DEVICE;
  if (device < 0 || device >= count) return IRT_ERR_INVALID_ARGUMENT;
  if (cudaSetDevice(device) != cudaSuccess) return IRT_ERR_CUDA;
  irt_ctx *ctx = new irt_ctx();
  ctx->device = device;
  {
    const char *dbg = getenv("IRT_B200_DEBUG_SYNC");
    ctx->debug_sync = dbg && dbg[0] == '1';
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return IRT_ERR_CUDA;
  }
  for (int b = 0; b < 2; b++) {
    cudaEventCreateWithFlags(&ctx->ev_computed[b], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ctx->ev_offsets[b], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ctx->ev_copied[b], cudaEventDisableTiming);
  }
  *out = ctx;
  return IRT_OK;
}

void irt_ctx_destroy(irt_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->scratch) cudaFree(ctx->scratch);
  if (ctx->arena) cudaFree(ctx->arena);
  if (ctx->io) cudaFree(ctx->io);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  for (int b = 0; b < 2; b++) {
    if (ctx->ev_computed[b]) cudaEventDestroy(ctx->ev_computed[b]);
    if (ctx->ev_offsets[b]) cudaEventDestroy(ctx->ev_offsets[b]);
    if (ctx->ev_copied[b]) cudaEventDestroy(ctx->ev_copied[b]);
  }
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
}

const char *irt_last_error(const irt_ctx *ctx) { return ctx ? ctx->last_error.c_str() : ""; }
int irt_ctx_device(const irt_ctx *ctx) { return ctx ? ctx->device : -1; }
int64_t irt_ctx_launch_count(const irt_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }

int irt_ctx_synchronize(irt_ctx *ctx) {
  if (!ctx) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  IRT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return IRT_OK;
}

uint32_t irt_morton_key(int bx, int by, int bz, int Nb) {
  uint32_t key = 0;
  for (int l = 0; (1 << l) < Nb; l++)
    key |= (uint32_t((bx >> l) & 1) << (3 * l + 2)) | (uint32_t((by >> l) & 1) << (3 * l + 1)) |
           (uint32_t((bz >> l) & 1) << (3 * l));
  return key;
}

void irt_morton_decode(uint32_t key, int Nb, int *bx, int *by, int *bz) {
  int x = 0, y = 0, z = 0;
  for (int l = 0; (1 << l) < Nb; l++) {
    x |= int((key >> (3 * l + 2)) & 1) << l;
    y |= int((key >> (3 * l + 1)) & 1) << l;
    z |= int((key >> (3 * l)) & 1) << l;
  }
  *bx = x; *by = y; *bz = z;
}

}  // extern "C"

int grid_check(irt_ctx *ctx, const irt_grid *g) {
  if (!g) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "null grid");
  int Ng = g->Ng;
  // collision/VoxelOctree.cpp:83-116: supported sizes 4..512, powers of two
  if (Ng < 4 || Ng > 512 || (Ng & (Ng - 1)) != 0)
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "unsupported voxel dimension: %d", Ng);
  for (int a = 0; a < 3; a++)  // set_xlim throws std::length_error when min >= max
    if (!(g->lim[2 * a] < g->lim[2 * a + 1]))
      return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "grid limits must be positive in size");
  return IRT_OK;
}

GridDev make_grid_dev(const irt_grid &g) {
  GridDev d;
  d.Ng = g.Ng;
  d.Nb = g.Ng / 4;
  d.levels = 0;
  while ((1 << d.levels) < d.Nb) d.levels++;
  for (int a = 0; a < 3; a++) {
    d.lo[a] = g.lim[2 * a];
    d.hi[a] = g.lim[2 * a + 1];
    d.d[a] = (g.lim[2 * a + 1] - g.lim[2 * a]) / g.Ng;  // VoxelOctree.cpp:152-177
    d.inv_d[a] = 1 / d.d[a];                            // VoxelOctree.cpp:338
  }
  bool ident = true;
  for (int i = 0; i < 9; i++) {
    d.inv_rot[i] = g.inv_rot[i];
    if (g.inv_rot[i] != ((i % 4 == 0) ? 1.0 : 0.0)) ident = false;
  }
  d.identity_rot = ident ? 1 : 0;
  return d;
}

// ---------------------------------------------------------------------------------------
// robot
// ---------------------------------------------------------------------------------------
namespace {

// tendon/get_r_info.cpp:17-40,105-144 -- evaluated once per table entry on the host
void routing_host(const irt_robot_desc &rb, double t, double *out /*[N][6]*/) {
  const int Nt = rb.n_tendons, Na = rb.n_c, Nm = rb.n_d;
  const int Ns = Na > Nm ? Na : Nm;
  double S[IRT_MAX_COEF], Sd[IRT_MAX_COEF], Sdd[IRT_MAX_COEF];
  S[0] = 1; Sd[0] = 0; Sdd[0] = 0;
  if (Ns >= 2) { S[1] = t; Sd[1] = 1; Sdd[1] = 0; }
  for (int i = 2; i < Ns; i++) {
    S[i] = t * S[i - 1];
    Sd[i] = i * S[i - 1];
    Sdd[i] = i * (i - 1) * S[i - 2];
  }
  for (int j = 0; j < Nt; j++) {
    const double *C = rb.C + j * IRT_MAX_COEF, *D = rb.D + j * IRT_MAX_COEF;
    double th = 0, th1 = 0, th2 = 0, rho = 0, rho1 = 0, rho2 = 0;
    for (int i = 0; i < Na; i++) { th += C[i] * S[i]; th1 += C[i] * Sd[i]; th2 += C[i] * Sdd[i]; }
    for (int i = 0; i < Nm; i++) { rho += D[i] * S[i]; rho1 += D[i] * Sd[i]; rho2 += D[i] * Sdd[i]; }
    double s = std::sin(th), c = std::cos(th);
    double *o = out + 6 * j;
    o[0] = rho * s;
    o[1] = rho * c;
    o[2] = rho1 * s + rho * (c * th1);
    o[3] = rho1 * c + rho * (-s * th1);
    o[4] = ((rho2 * s + (2 * rho1) * (c * th1)) - rho * (s * th1 * th1)) + rho * (c * th2);
    o[5] = ((rho2 * c + (2 * rho1) * (-s * th1)) - rho * (c * th1 * th1)) + rho * (-s * th2);
  }
}

int poly_degree(const double *coef, int n) {  // tendon/TendonSpecs.cpp:17-25
  if (n == 0) return 0;
  for (int i = n - 1; i > 0; i--)
    if (std::fabs(coef[i]) > 0.0) return i;
  return 0;
}

}  // namespace

extern "C" {

int irt_robot_create(irt_ctx *ctx, const irt_robot_desc *desc, irt_robot **out) {
  if (!ctx || !desc || !out) return IRT_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  const int N = desc->n_tendons;
  if (N < 1 || N > IRT_MAX_TENDONS)
    return irt_fail(ctx, IRT_ERR_OUT_OF_RANGE, "n_tendons=%d outside [1,%d]", N, IRT_MAX_TENDONS);
  if (desc->n_c < 1 || desc->n_c > IRT_MAX_COEF || desc->n_d < 1 || desc->n_d > IRT_MAX_COEF)
    return irt_fail(ctx, IRT_ERR_OUT_OF_RANGE, "coefficient counts outside [1,%d]", IRT_MAX_COEF);
  if (!(desc->L > 0) || !(desc->dL > 0) || !(desc->ro > desc->ri))
    return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "bad backbone specs");
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));

  irt_robot *rb = new irt_robot();
  {
    static std::atomic<unsigned long long> next_uid{1};
    rb->uid = next_uid.fetch_add(1);
  }
  rb->ctx = ctx;
  rb->desc = *desc;
  rb->state_size = N + (desc->enable_rotation ? 1 : 0) + (desc->enable_retraction ? 1 : 0);
  RobotDev &d = rb->dev;
  std::memset(&d, 0, sizeof(d));
  {  // stiffness -- tendon/TendonRobot.cpp:105-148
    double ro2 = desc->ro * desc->ro, ri2 = desc->ri * desc->ri;
    double I = (1.0 / 4.0) * M_PI * (ro2 * ro2 - ri2 * ri2);
    double Ar = M_PI * (ro2 - ri2);
    double J = 2 * I;
    double Gmod = desc->E / (2 * (1 + desc->nu));
    d.Kbt[0] = d.Kbt[1] = desc->E * I; d.Kbt[2] = J * Gmod;
    d.Kse[0] = d.Kse[1] = Gmod * Ar; d.Kse[2] = desc->E * Ar;
    d.KbtInv[0] = d.KbtInv[1] = 1 / (desc->E * I); d.KbtInv[2] = 1 / (J * Gmod);
    d.KseInv[0] = d.KseInv[1] = 1 / (Gmod * Ar); d.KseInv[2] = 1 / (desc->E * Ar);
  }
  d.L = desc->L; d.dL = desc->dL; d.r = desc->r; d.residual_threshold = desc->residual_threshold;
  std::memcpy(d.C, desc->C, sizeof(d.C));
  std::memcpy(d.D, desc->D, sizeof(d.D));
  d.n_tendons = N; d.n_c = desc->n_c; d.n_d = desc->n_d;
  d.enable_rotation = desc->enable_rotation ? 1 : 0;
  d.enable_retraction = desc->enable_retraction ? 1 : 0;
  {
    double tsum = 0.0;
    for (int j = 0; j < N; j++) tsum += desc->max_tension[j];
    d.tau_bin_scale = (tsum > 0.0) ? 8.0 / tsum : 0.0;   // FK_TAU_BINS bins over [0, sum(max_tension)]
    d.simple_routing = (desc->n_c <= 2 && desc->n_d == 1) ? 1 : 0;
    d.c1_uniform = d.simple_routing;
    d.c1_abs = 0.0;
    for (int j = 0; j < N && d.simple_routing; j++) {
      const double c0 = desc->C[j * IRT_MAX_COEF];
      const double c1 = (desc->n_c > 1) ? desc->C[j * IRT_MAX_COEF + 1] : 0.0;
      d.sin_c0[j] = std::sin(c0);
      d.cos_c0[j] = std::cos(c0);
      d.c1_sign[j] = (c1 > 0.0) ? 1.0 : ((c1 < 0.0) ? -1.0 : 0.0);
      if (c1 != 0.0) {
        if (d.c1_abs == 0.0) d.c1_abs = std::fabs(c1);
        else if (std::fabs(c1) != d.c1_abs) d.c1_uniform = 0;
      }
    }
  }
  for (int j = 0; j < N; j++) {  // home_shape closed forms -- tendon/TendonRobot.cpp:281-310
    const double *C = desc->C + j * IRT_MAX_COEF, *D = desc->D + j * IRT_MAX_COEF;
    int rdeg = poly_degree(D, desc->n_d), tdeg = poly_degree(C, desc->n_c);
    if (rdeg == 0 && tdeg == 0) d.home_factor[j] = 1.0;
    else if (rdeg == 0 && tdeg == 1) d.home_factor[j] = std::sqrt(1 + D[0] * D[0] * C[1] * C[1]);
    else d.home_factor[j] = std::numeric_limits<double>::quiet_NaN();  // reference UB (simpsons)
    d.min_length[j] = desc->min_length[j];
    d.max_length[j] = desc->max_length[j];
  }
  // canonical grid for s = 0: util::range + t_range (vector_ops.h:67-75, TendonRobot.cpp:69-84)
  std::vector<double> vals;
  for (double p = 0.0; p <= desc->L - (desc->dL / 2); p += desc->dL) vals.push_back(p);
  const int K = (int)vals.size();
  if (K + 1 > IRT_CAP_PTS_MAX) {
    delete rb;
    return irt_fail(ctx, IRT_ERR_CAPACITY, "L/dL too large: %d points > %d", K + 1, IRT_CAP_PTS_MAX);
  }
  rb->max_points = K + 1;
  rb->node_t.resize(K);
  for (int i = 0; i < K; i++) rb->node_t[i] = desc->L - (vals[i] - 0.0);  // node i ~ L - i*dL
  d.Kfull = K;
  d.n_table = 2 * K - 1;
  std::vector<double> table((size_t)d.n_table * N * 6);
  for (int i = 0; i < K; i++) routing_host(*desc, rb->node_t[i], &table[(size_t)(2 * i) * N * 6]);
  for (int q = 1; q < K; q++)  // RK4 mid stage of the step node q -> node q-1
    routing_host(*desc, rb->node_t[q] + 0.5 * desc->dL, &table[(size_t)(2 * q - 1) * N * 6]);
  // the wide rows of the constant-memory copy: each tendon's 6 values and the products of r (rounded on their own)
  std::vector<double> ctab((size_t)d.n_table * N * IRT_CT_WIDTH);
  for (size_t k = 0; k < (size_t)d.n_table * N; k++) {
    const double *src = &table[6 * k];
    double *dst = &ctab[IRT_CT_WIDTH * k];
    for (int i = 0; i < 6; i++) dst[i] = src[i];
    const double rxx = src[0] * src[0], ryy = src[1] * src[1];
    dst[6] = rxx;
    dst[7] = ryy;
    dst[8] = src[0] * src[1];
    dst[9] = rxx + ryy;
  }
  // head (first gap) stages for s = 0: times 0, h0/2 [, h0, h0 + h1/2]
  std::vector<double> head((size_t)4 * N * 6, 0.0);
  {
    const double eps = std::numeric_limits<double>::epsilon();
    double t0 = desc->L - (desc->L - 0.0);  // t_range's own first point
    double t1 = rb->node_t[K - 1];
    double h0 = std::fmin(desc->dL, t1 - t0);
    d.head_h[0] = h0;
    d.head_h[1] = 0.0;
    d.n_head = 2;
    routing_host(*desc, t0, &head[0]);
    routing_host(*desc, t0 + 0.5 * h0, &head[(size_t)1 * N * 6]);
    double tc = t0 + h0;
    if (t1 - tc > eps) {
      double h1 = std::fmin(desc->dL, t1 - tc);
      d.head_h[1] = h1;
      d.n_head = 4;
      routing_host(*desc, tc, &head[(size_t)2 * N * 6]);
      routing_host(*desc, tc + 0.5 * h1, &head[(size_t)3 * N * 6]);
    }
  }
  auto upload = [&](const std::vector<double> &v, double **dp) {
    if (cudaMalloc(dp, v.size() * sizeof(double)) != cudaSuccess) return false;
    return cudaMemcpy(*dp, v.data(), v.size() * sizeof(double), cudaMemcpyHostToDevice) == cudaSuccess;
  };
  if (!upload(table, &rb->d_table) || !upload(ctab, &rb->d_ctab) || !upload(head, &rb->d_head) ||
      !upload(rb->node_t, &rb->d_node_t)) {
    irt_robot_destroy(rb);
    return irt_fail(ctx, IRT_ERR_CUDA, "robot table upload failed: %s",
                    cudaGetErrorString(cudaGetLastError()));
  }
  d.table = rb->d_table;
  d.head = rb->d_head;
  d.node_t = rb->d_node_t;
  *out = rb;
  return IRT_OK;
}

void irt_robot_destroy(irt_robot *rb) {
  if (!rb) return;
  cudaSetDevice(rb->ctx->device);
  if (rb->d_table) cudaFree(rb->d_table);
  if (rb->d_ctab) cudaFree(rb->d_ctab);
  if (rb->d_head) cudaFree(rb->d_head);
  if (rb->d_node_t) cudaFree(rb->d_node_t);
  delete rb;
}

int irt_robot_state_size(const irt_robot *rb) { return rb ? rb->state_size : -1; }
int irt_robot_max_points(const irt_robot *rb) { return rb ? rb->max_points : -1; }

}  // extern "C"

// ---------------------------------------------------------------------------------------
// FP64 peak probe: 8 independent DFMA chains per thread, 2 FLOP per DFMA
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double *out, int iters, double seed) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5,
         a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
#pragma unroll 1
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int k = 0; k < 8; k++) {
      a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
      a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
  }
  double s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  if (s == 123.456) out[0] = s;  // keep the chains alive
}

// The same probe with other operand patterns (irt_measure_fp64_rate): what a DFMA costs when its sources are not
// served by the operand reuse cache.  MODE 1: a_k = fma(a_k, m, c_k) -- two new register pairs per instruction
// (m stays in the reuse cache); MODE 2: a_k = fma(a_k, b_k, c_k) -- three distinct register pairs, none shared with
// the previous instruction.  K1's stage loop has 245 of 445 DFMAs of the second kind.
template <int MODE>
__global__ void __launch_bounds__(256) dfma_operand_kernel(double *out, int iters, double seed) {
  double a[8], b[8], c[8];
#pragma unroll
  for (int k = 0; k < 8; k++) {
    a[k] = seed + threadIdx.x + k;
    b[k] = 1.0000001 + 1e-12 * seed * (threadIdx.x + k + 1);   // per thread: not a uniform-register operand
    c[k] = 1e-9 * seed * (threadIdx.x + k + 1);
  }
#pragma unroll 1
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int r = 0; r < 8; r++) {
#pragma unroll
      for (int k = 0; k < 8; k++) a[k] = (MODE == 1) ? fma(a[k], b[0], c[k]) : fma(a[k], b[k], c[k]);
    }
  }
  double s = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) s += a[k];
  if (s == 123.456) out[0] = s;
}

extern "C" int irt_measure_fp64_rate(irt_ctx *ctx, int mode, double *flops_per_s) {
  if (!ctx || !flops_per_s || mode < 0 || mode > 2) return IRT_ERR_INVALID_ARGUMENT;
  IRT_CUDA(ctx, cudaSetDevice(ctx->device));
  double *d_out = (double *)ctx_scratch(ctx, 256);
  if (!d_out) return irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc failed");
  const int iters = 4096, blocks = ctx->sm_count * 8, threads = 256;
  cudaEvent_t e0, e1;
  IRT_CUDA(ctx, cudaEventCreate(&e0));
  IRT_CUDA(ctx, cudaEventCreate(&e1));
  double best = 0;
  for (int rep = 0; rep < 5; rep++) {
    IRT_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
    if (mode == 0) dfma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 1.0);
    else if (mode == 1) dfma_operand_kernel<1><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 1.0);
    else dfma_operand_kernel<2><<<blocks, threads, 0, ctx->stream>>>(d_out, iters, 1.0);
    IRT_LAUNCHED(ctx);
    IRT_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    IRT_CUDA(ctx, cudaEventSynchronize(e1));
    float ms = 0;
    IRT_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
    double flops = 2.0 * 64.0 * iters * (double)blocks * threads;
    double rate = flops / (ms * 1e-3);
    if (rep > 0 && rate > best) best = rate;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *flops_per_s = best;
  return IRT_OK;
}

extern "C" int irt_measure_fp64_peak(irt_ctx *ctx, double *flops_per_s) {
  return irt_measure_fp64_rate(ctx, 0, flops_per_s);
}
