/*
 * irt_b200.h -- C ABI of the B200-native hot path of interactive-rate-tendons.
 *
 * The reference (Kuntz-Lab/interactive-rate-tendons) has no C ABI or plugin loader; its
 * "operator API" for this path is a pair of C++ virtual interfaces plus the value types they
 * exchange (SURVEY.md section 8b).  Every entry point below names the reference interface it
 * replaces (file:line relative to /root/reference/cpp/src/).  INTEGRATION.md shows the
 * reference-side C++ glue a maintainer would add.
 *
 * Conventions
 *   - plain C: opaque handles, POD structs, pointers + sizes; no exceptions cross the boundary.
 *   - every call returns an irt_status (0 = OK).  irt_last_error(ctx) has the detail string.
 *   - "host" entry points take HOST pointers and copy H2D/D2H internally;
 *     "_dev" entry points take DEVICE pointers (cudaMalloc'ed or torch tensors' data_ptr())
 *     and a cudaStream_t passed as void* (NULL = the context's own stream); they are
 *     asynchronous with respect to the host.
 *   - threading: a context owns one stream and grow-only device scratch; calls on the SAME context
 *     must be serialised by the caller (the reference calls its validators from many OpenMP
 *     threads, one item each -- here one call carries the whole batch).  Different contexts,
 *     robots, stores and environments can be used from different host threads concurrently.
 *     The "_dev" calls keep their per-call temporaries (bucket keys and order of K1, perturbed states
 *     of the Jacobian batch, candidate lists of the self-collision test) in that per-context scratch:
 *     all "_dev" calls on one context must therefore be STREAM-ORDERED with each other (same stream,
 *     or an event between them); two of them running concurrently on different streams would share
 *     the temporaries.  Use one context per concurrent stream.
 *   - robots: K1 keeps the routing table of the robot it last ran in the device's constant memory (one copy per
 *     device and process, shared by all contexts); a call for another robot on the same device drains the device
 *     and re-uploads (correct, but slow when two robots alternate).
 *   - there is NO CPU fallback: without a CUDA device irt_ctx_create fails with
 *     IRT_ERR_NO_DEVICE and nothing else can be called.
 *   - per-item problems (non-convergence, limits, ...) are NOT errors: they are reported in a
 *     per-item uint32 flag word (IRT_FLAG_*), mirroring TendonResult::converged
 *     (tendon/TendonRobot.cpp:470-474) and AbstractValidityChecker::is_valid_shape
 *     (motion-planning/AbstractValidityChecker.cpp:99-114).
 *
 * Data layouts
 *   state    double[S], S = N + [rotation] + [retraction]   (tendon/TendonRobot.h:60-64)
 *   points   double[n][cap_pts][3], first npts[i] rows valid (TendonResult::p)
 *   R        double[n][cap_pts][9] column-major               (TendonResult::R, Eigen storage)
 *   voxel block  uint64, bit = x*16 + y*4 + z                 (collision/VoxelOctree.cpp:1501-1503)
 *   block key    uint32 Morton code with x as the most significant bit of every 3-bit group:
 *                exactly the reference's octant order (collision/detail/TreeNode.h:66-68), so a
 *                key-sorted list is VoxelOctree::visit_leaves order and 8 consecutive keys are
 *                one 2x2x2 group of leaf blocks = one 512-bit super-block.
 *   set store    CSR: offsets uint64[n+1], keys uint32[nb], bits uint64[nb], key-sorted per set
 *   verdicts     uint32 words, bit (i % 32) of word (i / 32) = set i collides with the environment
 */
#ifndef IRT_B200_H
#define IRT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IRT_MAX_TENDONS 12
#define IRT_MAX_COEF 8
#define IRT_ABI_VERSION 1

typedef enum irt_status {
  IRT_OK = 0,
  IRT_ERR_NO_DEVICE = 1,        /* no CUDA device / driver: there is no CPU fallback */
  IRT_ERR_INVALID_ARGUMENT = 2, /* std::invalid_argument in the reference (wrong state size,
                                   grid size mismatch, dL too coarse for the grid) */
  IRT_ERR_OUT_OF_RANGE = 3,     /* std::out_of_range (tau / tendon count mismatch) */
  IRT_ERR_CUDA = 4,             /* a CUDA runtime call or kernel failed */
  IRT_ERR_UNSUPPORTED = 5,      /* routing the reference itself cannot handle (SURVEY App. B #2) */
  IRT_ERR_CAPACITY = 6,         /* an output buffer / per-set capacity is too small */
  IRT_ERR_DOMAIN = 7            /* std::domain_error: point outside the voxel grid */
} irt_status;

/* per-item flag word */
#define IRT_FLAG_NONCONVERGED 1u   /* TendonResult::converged == false */
#define IRT_FLAG_LENGTH_LIMIT 2u   /* !is_within_length_limits (tendon/TendonRobot.h:262-278) */
#define IRT_FLAG_SELF_COLLISION 4u /* collides_self (collision/collision.cpp:6-46) */
#define IRT_FLAG_OUT_OF_DOMAIN 8u  /* find_cell would throw std::domain_error */
#define IRT_FLAG_PARTIAL 16u       /* edge: PartialVoxelization::is_fully_valid == false */
#define IRT_FLAG_BAD_STATE 32u     /* retraction NaN, or so far below 0 that the grid exceeds max_points: outside the reference's state space */
#define IRT_FLAG_CAPACITY 64u      /* per-item scratch capacity exceeded (result incomplete) */
#define IRT_FLAG_ENV_COLLISION 128u /* until-invalid mode: the sample's own voxels hit the environment */

typedef struct irt_ctx irt_ctx;
typedef struct irt_robot irt_robot;
typedef struct irt_env irt_env;
typedef struct irt_setstore irt_setstore;

/* POD mirror of tendon::TendonRobot (tendon/TendonRobot.h:52-58), BackboneSpecs
 * (tendon/BackboneSpecs.h:15-21) and TendonSpecs (tendon/TendonSpecs.h:24-30). */
typedef struct irt_robot_desc {
  double r;
  double L, dL, ro, ri, E, nu;
  double residual_threshold;
  int32_t n_tendons;
  int32_t n_c;  /* theta-polynomial length (all tendons share tendon 0's, get_r_info.h:34-39) */
  int32_t n_d;  /* rho-polynomial length */
  int32_t enable_rotation;
  int32_t enable_retraction;
  int32_t _pad;
  double C[IRT_MAX_TENDONS * IRT_MAX_COEF]; /* row-major [tendon][coef] */
  double D[IRT_MAX_TENDONS * IRT_MAX_COEF];
  double max_tension[IRT_MAX_TENDONS];
  double min_length[IRT_MAX_TENDONS];
  double max_length[IRT_MAX_TENDONS];
} irt_robot_desc;

/* Voxel grid geometry: VoxelOctree limits (collision/VoxelOctree.h:310-329) and
 * VoxelEnvironment::inv_rotation (motion-planning/VoxelEnvironment.cpp:129-131). */
typedef struct irt_grid {
  int32_t Ng; /* voxels per axis, power of two in [4, 512] (VoxelOctree.cpp:83-116) */
  int32_t _pad;
  double lim[6];     /* xmin,xmax,ymin,ymax,zmin,zmax */
  double inv_rot[9]; /* row-major */
} irt_grid;

/* OMPL space constants fixed by Problem::create_space_information
 * (motion-planning/Problem.cpp:101-163, Problem.h:59-63). */
typedef struct irt_space {
  double min_tension_change;    /* default 0.02 */
  double min_rotation_change;   /* default 0.01 */
  double min_retraction_change; /* default 1e-4 */
} irt_space;

/* optional FK outputs; NULL members are skipped.  Host or device pointers depending on the
 * entry point.  Mirrors tendon::TendonResult (tendon/TendonResult.h:17-28). */
typedef struct irt_fk_outputs {
  double *p;       /* [n][cap_pts][3] */
  double *R;       /* [n][cap_pts][9] column-major */
  double *t;       /* [n][cap_pts] */
  int32_t *npts;   /* [n] */
  double *L;       /* [n] */
  double *L_i;     /* [n][N] */
  double *tip;     /* [n][3]  == p[npts-1] */
  double *uv;      /* [n][12]: u_i, u_f, v_i, v_f */
  uint32_t *flags; /* [n] IRT_FLAG_NONCONVERGED | LENGTH_LIMIT | SELF_COLLISION | BAD_STATE */
  int32_t *iters;  /* [n] fixed-point iterations (solve_initial_bending.cpp:41-70) */
  int32_t *nsteps; /* [n] RK4 steps taken */
} irt_fk_outputs;

/* ---- context ------------------------------------------------------------------------- */
int irt_abi_version(void);
const char *irt_status_string(int status);
int irt_ctx_create(int device, irt_ctx **out);
void irt_ctx_destroy(irt_ctx *ctx);
const char *irt_last_error(const irt_ctx *ctx);
int irt_ctx_device(const irt_ctx *ctx);
int irt_ctx_synchronize(irt_ctx *ctx);
/* kernels launched by this context since creation (bench.py "gpu_launches") */
int64_t irt_ctx_launch_count(const irt_ctx *ctx);
/* measured FP64 DFMA-chain peak of this device in FLOP/s (roofline denominator for K1) */
int irt_measure_fp64_peak(irt_ctx *ctx, double *flops_per_s);
/* the same probe with other operand patterns: mode 0 = the peak probe (a = fma(a, m, c): m and c stay in the
 * operand reuse cache), 1 = two new register pairs per DFMA, 2 = three distinct register pairs per DFMA (the
 * register file serves two per issue slot: what bounds K1's stage loop, DESIGN.md section 7) */
int irt_measure_fp64_rate(irt_ctx *ctx, int mode, double *flops_per_s);

/* ---- robot: replaces tendon::TendonRobot (tendon/TendonRobot.h:52-355) ------------------ */
int irt_robot_create(irt_ctx *ctx, const irt_robot_desc *desc, irt_robot **out);
void irt_robot_destroy(irt_robot *rb);
int irt_robot_state_size(const irt_robot *rb); /* TendonRobot::state_size, TendonRobot.h:60-64 */
int irt_robot_max_points(const irt_robot *rb); /* len(t_range(0, L, dL)), TendonRobot.cpp:69-84 */

/* K1: TendonRobot::shape(state) for n states (tendon/TendonRobot.h:105-131 ->
 * tension_shape TendonRobot.cpp:325-500), plus the validity epilogue
 * AbstractValidityChecker::is_valid_shape (AbstractValidityChecker.cpp:99-114) when
 * out->flags != NULL.  Replaces the OpenMP loops apps/estimate_length_discretization.cpp:62-71
 * and apps/roadmap2samples.cpp:64-78.
 * IRT_ERR_INVALID_ARGUMENT if state_size != irt_robot_state_size (TendonRobot.h:107-109),
 * IRT_ERR_CAPACITY if cap_pts < irt_robot_max_points. */
int irt_fk_batch(irt_ctx *ctx, const irt_robot *rb, const double *states, int state_size,
                 int64_t n, int cap_pts, const irt_fk_outputs *out);
int irt_fk_batch_dev(irt_ctx *ctx, const irt_robot *rb, const double *d_states, int state_size,
                     int64_t n, int cap_pts, const irt_fk_outputs *d_out, void *stream);
/* Packed form of irt_fk_batch (host pointers): out->p / R / t hold only the rows that exist, shape i
 * in rows [row_offsets[i], row_offsets[i+1]) -- the reference's per-shape std::vector<Point> /
 * vector<Matrix3d> / vector<double> (tendon/TendonResult.h:17-28) laid end to end; all other members
 * of `out` are per shape as in irt_fk_batch.  row_offsets has n+1 entries; cap_rows is the capacity
 * of the caller's p/R/t buffers in rows (n * irt_robot_max_points always suffices), IRT_ERR_CAPACITY
 * if it is too small.  With retraction this moves ~3/4 of the bytes of the dense form over PCIe. */
int irt_fk_batch_packed(irt_ctx *ctx, const irt_robot *rb, const double *states, int state_size,
                        int64_t n, const irt_fk_outputs *out, int64_t cap_rows, int64_t *row_offsets);
/* Batched finite-difference tip Jacobians (SURVEY 8(f) row 3): what the reference's IK and tip
 * controllers compute with one FK per perturbed parameter.  J is [n][3][S] (row i of seed k at
 * J[(k*3+i)*S + j], levmar's jac[i*m+j] layout), tips is [n][3] (may be NULL): the value the
 * differences are taken from.  One K1 launch over n*(S+1) or n*(2S+1) states.
 *   IRT_JAC_FORWARD_FIXED   tip_control::Jacobian (tip-control/tip_control.cpp:243-265):
 *                           (fk(state + delta e_j).back() - tip) / delta; the reference's `dist` is a C float
 *                           promoted to double, so pass delta = (double)(float)dist for the same step
 *   IRT_JAC_LEVMAR_FORWARD  levmar-2.6 dlevmar_fdif_forw_jac_approx (3rdparty/levmar-2.6/misc_core.c:137-172)
 *   IRT_JAC_LEVMAR_CENTRAL  dlevmar_fdif_cent_jac_approx (misc_core.c:175-211), the form
 *                           tip_control::inverse_kinematics_impl asks for (tip_control.cpp:85)
 * The two levmar modes differentiate the reference's wrapper fk_wrap (tip_control.cpp:92-122):
 * a retraction beyond L evaluates to (0, 0, L - s).  d = max(|1e-4 p_j|, delta). */
#define IRT_JAC_FORWARD_FIXED 0
#define IRT_JAC_LEVMAR_FORWARD 1
#define IRT_JAC_LEVMAR_CENTRAL 2
int irt_fk_tip_jacobian_batch(irt_ctx *ctx, const irt_robot *rb, const double *states, int state_size,
                              int64_t n, int mode, double delta, double *tips, double *J);
int irt_fk_tip_jacobian_batch_dev(irt_ctx *ctx, const irt_robot *rb, const double *d_states,
                                  int state_size, int64_t n, int mode, double delta, double *d_tips,
                                  double *d_J, void *stream);
/* collision::collides_self(CapsuleSequence{points, r}) (collision/collision.cpp:6-46) = TendonRobot::collides_self
 * (tendon/TendonRobot.cpp:955-974) for n given backbones: p[n][cap_pts][3], npts[n] (host); collides[i] = 0 / 1.
 * The validity epilogue of irt_fk_batch runs the same kernels on the shapes it has just computed. */
int irt_self_collision_shapes(irt_ctx *ctx, const double *p, const int32_t *npts, int cap_pts, int64_t n,
                              double r, uint8_t *collides);
/* TendonRobot::home_shape(state).L_i (tendon/TendonRobot.cpp:249-314), host arrays */
int irt_home_lengths_batch(irt_ctx *ctx, const irt_robot *rb, const double *states,
                           int state_size, int64_t n, double *L_i);

/* ---- environment: replaces the obstacle collision::VoxelOctree each validator copies at
 * construction (AbstractVoxelValidityChecker.h:22-25,64; AbstractVoxelMotionValidator.h:191) */
int irt_env_create(irt_ctx *ctx, const irt_grid *grid, irt_env **out);
void irt_env_destroy(irt_env *env);
/* dense upload: blocks[Nb^3] indexed by Morton key */
int irt_env_update(irt_ctx *ctx, irt_env *env, const uint64_t *blocks);
int irt_env_update_dev(irt_ctx *ctx, irt_env *env, const uint64_t *d_blocks, void *stream);
/* sparse upload from VoxelOctree::visit_leaves output: (bx,by,bz) uint8 triples + bits */
int irt_env_update_sparse(irt_ctx *ctx, irt_env *env, const uint8_t *bxyz,
                          const uint64_t *bits, int64_t nblocks);
int64_t irt_env_nblocks(irt_ctx *ctx, const irt_env *env); /* VoxelOctree::nblocks */
/* environment preparation on the device, in place (the steps apps apply to the obstacle tree
 * before planning).  Synchronous; bit-exact with the reference's trees.
 *   irt_env_dilate          VoxelOctree::dilate_6neighbor(num) (collision/VoxelOctree.cpp:757-787)
 *                           or, use_diagonal != 0, dilate_27neighbor(num) (:789-825, including
 *                           its neighbour list as written: (x+1,y+1,z+1) twice, no (x-1,y+1,z+1))
 *   irt_env_dilate_sphere   VoxelOctree::dilate_sphere(r) (:949-951) =
 *                           dilate_6neighbor(round(r / min(dx,dy,dz)))
 *   irt_env_remove_interior VoxelOctree::remove_interior_6neighbor (:533-600) or, keep_diagonal
 *                           != 0, remove_interior_27neighbor (:602-689, the default of
 *                           VoxelOctree::remove_interior, VoxelOctree.h:165); cells outside the
 *                           grid count as occupied
 *   irt_env_download        dense host copy blocks[Nb^3] indexed by Morton key */
/* Environment::voxelize(reference) (motion-planning/Environment.cpp:62-74): voxels->add(p) / add(s) / add(c) for
 * the environment's points [n][3], spheres [n][4] = (c, r) and capsules [n][7] = (a, b, r), OR-ed into the
 * grid (clear_first != 0: into an empty one, like the reference's empty_copy()).  A voxel is set when its
 * CENTRE is inside the object (VoxelOctree::add_sphere / add_capsule, collision/VoxelOctree.cpp:434-515;
 * collides(Sphere, Point) / collides(Capsule, Point), collision/collision.hxx:62-84), plus the cells of the
 * points, sphere centres and capsule end points themselves (add_point, :319-323).  Bit-exact with the
 * reference's trees.  Environment::voxelize(reference, dilate) (:76-101) is the same call with `dilate` added
 * to every radius and the points turned into spheres of that radius (host side, see the mirrors).
 * Meshes are not supported (the reference throws std::logic_error for them as well). */
int irt_env_add_primitives(irt_ctx *ctx, irt_env *env, const double *points, int64_t n_points,
                           const double *spheres, int64_t n_spheres, const double *capsules,
                           int64_t n_capsules, int clear_first);
int irt_env_dilate(irt_ctx *ctx, irt_env *env, int num, int use_diagonal);
int irt_env_dilate_sphere(irt_ctx *ctx, irt_env *env, double r);
int irt_env_remove_interior(irt_ctx *ctx, irt_env *env, int keep_diagonal);
int irt_env_download(irt_ctx *ctx, const irt_env *env, uint64_t *blocks);

/* ---- set store: replaces vertexVoxelsProperty_/edgeVoxelsProperty_
 * (std::shared_ptr<VoxelOctree> per vertex/edge, VoxelCachedLazyPRM.h:141,165-179) ------- */
int irt_setstore_create(irt_ctx *ctx, const irt_grid *grid, irt_setstore **out);
void irt_setstore_destroy(irt_setstore *s);
int64_t irt_setstore_num_sets(const irt_setstore *s);
int64_t irt_setstore_num_blocks(const irt_setstore *s);
/* import/export the CSR (host arrays); the .rmp record list {u8 bx,u8 by,u8 bz,u64 bits}
 * (VoxelCachedLazyPRM.cpp:1091-1095) converts 1:1 with irt_morton_key / irt_morton_decode */
int irt_setstore_import(irt_ctx *ctx, irt_setstore *s, int64_t n_sets, const uint64_t *offsets,
                        const uint32_t *keys, const uint64_t *bits);
int irt_setstore_export(irt_ctx *ctx, const irt_setstore *s, uint64_t *offsets, uint32_t *keys,
                        uint64_t *bits);
/* Append sets [begin, end) of src to the end of dst, in index order.  keep_words (host, may be NULL = keep all):
 * set begin+i is appended iff bit i % 32 of word i / 32 is set.  dst's existing sets, offsets, keys and bits are
 * unchanged; afterwards dst equals irt_setstore_import of the concatenated CSR, bit for bit.  Synchronous.
 * IRT_ERR_INVALID_ARGUMENT: dst == src, NULL handles, grids that differ (Ng, lim, inv_rot), begin/end outside
 * [0, num_sets(src)] or begin > end, stores of another context's device.  An empty range or an all-clear mask is a
 * no-op.  On any error dst is unchanged.  Device views of dst (irt_setstore_device_ptrs) are invalidated.
 * The batch form of the reference's compute-if-absent voxelizeVertex / voxelizeEdge (VoxelCachedLazyPRM.cpp:
 * 2803-2837, 2879-2902) and of the per-increment caches of createRoadmap(N) (.cpp:1380-1561): voxelise the new
 * items into a scratch store, then append the kept ones (INTEGRATION.md section B). */
int irt_setstore_append(irt_ctx *ctx, irt_setstore *dst, const irt_setstore *src, int64_t begin, int64_t end,
                        const uint32_t *keep_words);
/* device views (valid until the store is next modified) */
int irt_setstore_device_ptrs(const irt_setstore *s, const uint64_t **d_offsets,
                             const uint32_t **d_keys, const uint64_t **d_bits);
uint32_t irt_morton_key(int bx, int by, int bz, int Nb);
void irt_morton_decode(uint32_t key, int Nb, int *bx, int *by, int *bz);

/* K1+K2 (vertex mode): VoxelCachedLazyPRM::precomputeVertexVoxelCache /
 * voxelizeVertex (VoxelCachedLazyPRM.cpp:1687-1712,2803-2837): FK + is_valid_shape +
 * VoxelBackboneValidityChecker::voxelize_impl (VoxelBackboneValidityChecker.h:49-57).
 * Replaces the store content with n sets (an invalid shape gets an empty set and its flags).
 * tips (optional, [n][3]) = fk_shape.p.back(). */
int irt_voxelize_vertices(irt_ctx *ctx, const irt_robot *rb, const double *states,
                          int state_size, int64_t n, irt_setstore *store, uint32_t *flags,
                          double *tips);
/* K2 on given shapes: AbstractVoxelValidityChecker::voxelize(const TendonResult&)
 * (AbstractVoxelValidityChecker.h:33-41 -> VoxelBackboneValidityChecker::voxelize_impl,
 * VoxelBackboneValidityChecker.h:49-57): rotate_points + add_piecewise_line of n already computed
 * backbones p[n][cap_pts][3] (host), npts[n].  Replaces the store content with n sets. */
int irt_voxelize_shapes(irt_ctx *ctx, const double *p, const int32_t *npts, int cap_pts, int64_t n,
                        irt_setstore *store);
/* K1+K2 (edge mode): VoxelCachedLazyPRM::precomputeEdgeVoxelCache / voxelizeEdge
 * (VoxelCachedLazyPRM.cpp:1736-1782,2879-2902) -> AbstractVoxelMotionValidator::voxelize
 * (AbstractVoxelMotionValidator.h:98-107) -> VoxelBackboneMotionValidator::generic_voxelize
 * (VoxelBackboneMotionValidator.cpp:41-74) -> VoxelEnvironment::voxelize_valid_backbone_motion
 * (VoxelEnvironment.cpp:207-444).  a,b: [n][S] endpoint states.  Outputs (optional):
 * flags (IRT_FLAG_PARTIAL = !is_fully_valid), t_last = PartialVoxelization::t,
 * nsamples = FK evaluations spent on the edge. */
int irt_voxelize_edges(irt_ctx *ctx, const irt_robot *rb, const irt_space *space,
                       const double *a, const double *b, int state_size, int64_t n,
                       irt_setstore *store, uint32_t *flags, double *t_last, int32_t *nsamples);
/* AbstractVoxelMotionValidator::voxelize_until_invalid (AbstractVoxelMotionValidator.h:109-127 ->
 * VoxelBackboneMotionValidator::voxelize_until_invalid_impl, .cpp:83-91): like irt_voxelize_edges,
 * but a sample is also invalid when its backbone voxels collide with `env`
 * (is_valid_shape && !_vc->collides(shape)); the stored set is the swept volume up to the last
 * valid t, which is what checkMotion(s1, s2, last_valid) reports. */
int irt_voxelize_edges_until_invalid(irt_ctx *ctx, const irt_robot *rb, const irt_space *space,
                                     const double *a, const double *b, int state_size, int64_t n,
                                     const irt_env *env, irt_setstore *store, uint32_t *flags,
                                     double *t_last, int32_t *nsamples);
/* Same, for edges given as index pairs into one list of roadmap vertices (the planner's own
 * representation: boost::source(e) / boost::target(e), VoxelCachedLazyPRM.cpp:2888-2891).  The FK of
 * every vertex is computed once and shared by all incident edges.  pairs: int64[n_edges][2].
 * IRT_ERR_OUT_OF_RANGE if an index is outside [0, n_vertices). */
int irt_voxelize_edges_indexed(irt_ctx *ctx, const irt_robot *rb, const irt_space *space,
                               const double *vertex_states, int state_size, int64_t n_vertices,
                               const int64_t *pairs, int64_t n_edges, irt_setstore *store,
                               uint32_t *flags, double *t_last, int32_t *nsamples);
/* OMPL StateSpace::validSegmentCount for the compound space of Problem.cpp:101-163 (host) */
uint32_t irt_valid_segment_count(const irt_robot_desc *desc, const irt_space *space,
                                 const double *a, const double *b);

/* K3: VoxelOctree::collides(other) (collision/VoxelOctree.cpp:973-978) of every cached set in
 * [begin,end) against the environment; the batch form of computeVertexValidity /
 * computeEdgeValidity with warm caches (VoxelCachedLazyPRM.cpp:2607-2631) as driven by
 * precomputeVertexValidity / precomputeEdgeValidity (:1563-1647).
 * verdict_words: uint32[(end-begin+31)/32], bit i-begin set <=> set i collides.
 * IRT_ERR_INVALID_ARGUMENT if the grids' Ng differ (VoxelOctree.cpp:46-53). */
int irt_check_sets(irt_ctx *ctx, const irt_setstore *store, const irt_env *env, int64_t begin,
                   int64_t end, uint32_t *verdict_words);
int irt_check_sets_dev(irt_ctx *ctx, const irt_setstore *store, const irt_env *env,
                       int64_t begin, int64_t end, uint32_t *d_verdict_words, void *stream);
/* the popcount side of K3 over the same range: stats[0] = sum over leaves of
 * popcount(set_bits & env_bits) (colliding voxels), stats[1] = number of leaves that hit.
 * Not part of the reference API (its collides() stops at the first hit); used as a
 * size-independent checksum and for reporting. */
int irt_check_sets_popcount(irt_ctx *ctx, const irt_setstore *store, const irt_env *env,
                            int64_t begin, int64_t end, uint64_t *stats);

/* ---- incremental revalidation after an environment change (the replanning loop; the reference has no live-update
 * API and re-checks every item) ----------------------------------------------------------------------------------
 * A set's verdict can only change where one of its leaves overlaps a changed voxel: for a leaf with
 * bits & (old ^ new) == 0, bits & new == bits & old.  The index lists, per leaf-block key, the sets with a leaf there
 * and that leaf's bits, so a change re-checks only the sets whose leaves overlap it.
 *
 * Inverted index of a set store: for every leaf-block key, the (set index, leaf bits) of every set that has a leaf
 * there.  Covers sets [0, irt_setindex_num_sets(ix)) of the store as it was when built; ~12 B per leaf + 8 B per key.
 * IRT_ERR_CAPACITY when the store holds 2^32 sets or more.  The index belongs to its store and is built on the
 * device (synchronous); it holds no pointer into the store's arrays, which appends may move. */
typedef struct irt_setindex irt_setindex;
int irt_setindex_create(irt_ctx *ctx, const irt_setstore *store, irt_setindex **out);
void irt_setindex_destroy(irt_setindex *ix);
int64_t irt_setindex_num_sets(const irt_setindex *ix);

/* verdict_words (host, (end-begin+31)/32 words): on entry the words irt_check_sets(store, env_old, begin, end) gave,
 * on return the words irt_check_sets(store, env_new, begin, end) gives, bit for bit.  flipped (host, may be NULL):
 * the absolute indices of the sets whose bit changed, ascending; *n_flipped (may be NULL) their number.  stats (may
 * be NULL): [0] changed leaf blocks, [1] sets re-checked, [2] 1 if the call swept the whole range instead.
 * Synchronous.
 *   Tail sets: sets in [irt_setindex_num_sets(ix), end) were appended after the build (irt_setstore_append, which
 *     never changes existing sets); they are re-checked in full whenever a block changed.
 *   The path is chosen from the input: when the index lists of the changed blocks hold more entries than a fixed
 *     fraction of the range's leaves, the call sweeps the range with K3 instead (same words, same flips).
 *   IRT_ERR_INVALID_ARGUMENT: NULL handles; env_old / env_new grids that differ (Ng, lim, inv_rot); a store whose Ng
 *     differs from the environments'; begin < 0, end < begin or end > irt_setstore_num_sets(store); an index of
 *     another store, or a stale one (the store's content was replaced by irt_setstore_import or irt_voxelize_*
 *     after the build: rebuild the index); cap_flipped < 0; verdict_words NULL for a non-empty range.
 *   IRT_ERR_CAPACITY: flipped != NULL and more than cap_flipped sets flipped; *n_flipped is set to the number needed.
 *   Every argument is checked before anything runs; on any error verdict_words is unchanged.
 *   env_old == env_new, or two equal grids, is a no-op with no flips. */
int irt_check_sets_changed(irt_ctx *ctx, const irt_setstore *store, const irt_setindex *ix,
                           const irt_env *env_old, const irt_env *env_new, int64_t begin, int64_t end,
                           uint32_t *verdict_words, int64_t *flipped, int64_t cap_flipped, int64_t *n_flipped,
                           int64_t *stats);
/* ---- multi-GPU: verdict all-gather fused into K3 over peer memory (NVLink / NVSwitch) -----------
 * One process per GPU.  Every rank creates an exchange buffer, publishes its handle (host-side
 * all-gather of irt_xchg_handle_size() bytes, e.g. with torch.distributed / MPI) and connects.  A
 * sweep then stores every verdict word straight into all peers' copies of the gathered array; its
 * last CTA raises this rank's epoch flag on every peer and waits (bounded) for the peers' flags, so
 * the gathered array is complete when the sweep kernel ends -- ONE launch per sweep.  Replaces
 * K3 + ncclAllGather of the verdict words (VoxelCachedLazyPRM.cpp:1584-1591 sharded over GPUs).
 * slot_words = words every rank contributes (the same on all ranks, >= ceil(shard sets / 32)). */
typedef struct irt_xchg irt_xchg;
int irt_xchg_create(irt_ctx *ctx, int rank, int world, int64_t slot_words, irt_xchg **out);
void irt_xchg_destroy(irt_xchg *x);
int irt_xchg_handle_size(void);
int irt_xchg_export(irt_xchg *x, void *handle);
int irt_xchg_connect(irt_xchg *x, const void *handles /* [world][handle_size], rank order */);
int irt_check_sets_allgather_dev(irt_ctx *ctx, const irt_setstore *store, const irt_env *env,
                                 int64_t begin, int64_t end, irt_xchg *x, void *stream,
                                 const uint32_t **d_gathered /* [world][slot_words] device words */);
int irt_xchg_status(irt_xchg *x); /* 0, or 1 + rank of a peer whose flag never arrived */
/* algorithmic bytes one irt_check_sets call over [begin,end) moves (SURVEY 8d):
 * sum(12*nb + 8) + 8*Nb^3 + ceil(n/8) */
int64_t irt_check_sets_algorithmic_bytes(const irt_setstore *store, int64_t begin, int64_t end);

/* ---- exact k-nearest neighbours: replaces the host scans behind nn_->nearestK / nnTip_->nearestK
 * (KBoundedStrategy, VoxelCachedLazyPRM.cpp:1329-1345; roadmapIk .cpp:3095-3137; addMilestone .cpp:1854-1885) --
 * A device-resident, append-only point set with one metric.  The metric is the distance of OMPL's compound space
 * of Problem.cpp:118-141 as both host mirrors compute it, or plain R^n:
 *
 *   d(a,b) = ((e + w_so2*s) + w_lin*l)        a term whose column is -1 is left out (not added as zero)
 *   e = sqrt(((0 + t_0) + t_1) + ... + t_{n_euclid-1}),  t_j = (a_j - b_j)*(a_j - b_j)
 *   s = |a_c - b_c|, then 2*M_PI - s if s > M_PI          (c = so2_col, pi and 2 pi as doubles)
 *   l = |a_l - b_l|                                       (l = lin_col)
 *
 * in IEEE double, every operation rounded on its own (no FMA contraction), sums left to right, sqrt correctly
 * rounded: bit for bit what VoxelCachedLazyPRM::distance of host/irt_host.hpp computes.  The Euclidean columns are
 * the leading n_euclid columns; so2_col / lin_col must lie after them and differ.  Weights are finite and >= 0.
 * Other columns are stored but never read.
 *
 * irt_nnset_knn: for each of m query rows, the k nearest items in (distance, index) order -- exactly what a stable
 * sort by distance gives, also on exact ties -- skipping items whose exclude bit is set and returning only finite
 * distances <= bound (NaN distances never).  Entries past the last hit are idx -1 / dist +inf.  Host pointers,
 * synchronous.  IRT_ERR_INVALID_ARGUMENT for k outside [1, IRT_KNN_MAX_K], dim outside [1, 16] or a bad metric;
 * IRT_ERR_CAPACITY past 2^31 - 2 items.  n = 0 and m = 0 are valid. */
typedef struct irt_metric {
  int32_t n_euclid; /* leading columns under the L2 norm (tensions; 3 for tip positions) */
  int32_t so2_col;  /* column of an SO(2) angle, -1 = none */
  int32_t lin_col;  /* column under a weighted |difference| (retraction), -1 = none */
  int32_t _pad;
  double w_so2, w_lin;
} irt_metric;
#define IRT_KNN_MAX_K 64
typedef struct irt_nnset irt_nnset;
int irt_nnset_create(irt_ctx *ctx, int dim, const irt_metric *m, irt_nnset **out);
void irt_nnset_destroy(irt_nnset *s);
int64_t irt_nnset_size(const irt_nnset *s);
int irt_nnset_append(irt_ctx *ctx, irt_nnset *s, const double *rows /* [n][dim] host */, int64_t n);
int irt_nnset_clear(irt_ctx *ctx, irt_nnset *s);
int irt_nnset_knn(irt_ctx *ctx, const irt_nnset *s, const double *queries /* [m][dim] */, int64_t m, int k,
                  double bound, const uint32_t *exclude_words /* NULL, or bit i % 32 of word i / 32 */,
                  int64_t *idx /* [m][k] */, double *dist /* [m][k] or NULL */);

/* ---- .rmp roadmap files (SURVEY 8f "next" #1) ----------------------------------------------
 * The reference's binary roadmap format: LazyRmpParser / RmpStreamer
 * (motion-planning/VoxelCachedLazyPRM.cpp:862-1114, serialize_inner :636-657):
 *   u32 nV, u32 nE, bool has_voxels, [u8 Nb, f64 lims[6]],
 *   per vertex: u32 index, vector<f64> state (u32 count + data), optional<Vector3d> tip,
 *               [bool has, u32 nblocks, nblocks x {u8 bx, u8 by, u8 bz, u64 bits}]
 *   per edge:   u32 source, u32 target, f64 weight, [bool has, u32 nblocks, blocks...]
 * irt_rmp_read parses such a file into host arrays whose voxel part is already the CSR
 * (offsets / Morton keys / bits) that irt_setstore_import takes; irt_rmp_write is the inverse
 * (blocks are written in key order == the reference's visit_leaves order).  Host-side IO only. */
typedef struct irt_rmp {
  uint32_t n_verts, n_edges;
  int32_t has_voxels; /* reference voxel header present */
  int32_t Nb;         /* blocks per axis (Ng / 4) */
  double lims[6];
  int32_t state_size; /* all vertex states must have this many reals */
  int32_t _pad;
  uint32_t *v_index;  /* [nV] */
  double *v_state;    /* [nV][state_size] */
  uint8_t *v_has_tip; /* [nV] */
  double *v_tip;      /* [nV][3] */
  uint8_t *v_has_vox; /* [nV] */
  uint64_t *v_off;    /* [nV + 1] */
  uint32_t *v_keys;   /* [v_off[nV]] Morton keys */
  uint64_t *v_bits;
  uint32_t *e_src, *e_dst; /* [nE] */
  double *e_weight;        /* [nE] */
  uint8_t *e_has_vox;      /* [nE] */
  uint64_t *e_off;         /* [nE + 1] */
  uint32_t *e_keys;
  uint64_t *e_bits;
} irt_rmp;
int irt_rmp_read(const char *path, irt_rmp **out);
int irt_rmp_write(const char *path, const irt_rmp *r);
void irt_rmp_free(irt_rmp *r);

#ifdef __cplusplus
}
#endif
#endif /* IRT_B200_H */
