"""irt_b200 -- B200-native hot path of interactive-rate-tendons (FK / voxelise / voxel check).

Python host layer over the C ABI in include/irt_b200.h (libirt_b200.so, hand-written CUDA for
sm_100a).  It mirrors the reference's operator interface for this path:

  Robot            <-> tendon::TendonRobot            (tendon/TendonRobot.h:52-355)
  Env              <-> the obstacle collision::VoxelOctree held by the validators
                       (motion-planning/AbstractVoxelValidityChecker.h:22-25,64)
  SetStore         <-> vertexVoxelsProperty_/edgeVoxelsProperty_ caches
                       (motion-planning/VoxelCachedLazyPRM.h:141,165-179)
  Roadmap          <-> the batch entry points of VoxelCachedLazyPRM
                       (VoxelCachedLazyPRM.h:495-520; .cpp:1563-1782)
  NearestSet       <-> the exact scans behind nn_ / nnTip_ (ompl::NearestNeighbors) of the planner

There is no CPU fallback: if the CUDA library or a CUDA device is missing, construction fails
loudly.  Nothing in this package imports the oracle/ directory.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IRT_B200_LIB", os.path.join(_HERE, "libirt_b200.so"))

MAX_TENDONS = 12
MAX_COEF = 8

FLAG_NONCONVERGED = 1
FLAG_LENGTH_LIMIT = 2
FLAG_SELF_COLLISION = 4
FLAG_OUT_OF_DOMAIN = 8
FLAG_PARTIAL = 16
FLAG_BAD_STATE = 32
JAC_FORWARD_FIXED, JAC_LEVMAR_FORWARD, JAC_LEVMAR_CENTRAL = 0, 1, 2
FLAG_CAPACITY = 64
FLAG_ENV_COLLISION = 128
INVALID_MASK = FLAG_NONCONVERGED | FLAG_LENGTH_LIMIT | FLAG_SELF_COLLISION | FLAG_BAD_STATE

IRT_OK, IRT_ERR_NO_DEVICE, IRT_ERR_INVALID_ARGUMENT, IRT_ERR_OUT_OF_RANGE = 0, 1, 2, 3
IRT_ERR_CUDA, IRT_ERR_UNSUPPORTED, IRT_ERR_CAPACITY, IRT_ERR_DOMAIN = 4, 5, 6, 7


class IrtError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("irt_b200 status %d: %s" % (status, msg))
        self.status = status


class RobotDesc(C.Structure):
    _fields_ = [
        ("r", C.c_double),
        ("L", C.c_double), ("dL", C.c_double), ("ro", C.c_double), ("ri", C.c_double),
        ("E", C.c_double), ("nu", C.c_double),
        ("residual_threshold", C.c_double),
        ("n_tendons", C.c_int32), ("n_c", C.c_int32), ("n_d", C.c_int32),
        ("enable_rotation", C.c_int32), ("enable_retraction", C.c_int32), ("_pad", C.c_int32),
        ("C", C.c_double * (MAX_TENDONS * MAX_COEF)),
        ("D", C.c_double * (MAX_TENDONS * MAX_COEF)),
        ("max_tension", C.c_double * MAX_TENDONS),
        ("min_length", C.c_double * MAX_TENDONS),
        ("max_length", C.c_double * MAX_TENDONS),
    ]


class Grid(C.Structure):
    _fields_ = [("Ng", C.c_int32), ("_pad", C.c_int32), ("lim", C.c_double * 6),
                ("inv_rot", C.c_double * 9)]


class Space(C.Structure):
    _fields_ = [("min_tension_change", C.c_double), ("min_rotation_change", C.c_double),
                ("min_retraction_change", C.c_double)]


class Rmp(C.Structure):
    """irt_rmp: a roadmap file parsed into host arrays (voxels as CSR with Morton keys)"""
    _fields_ = [("n_verts", C.c_uint32), ("n_edges", C.c_uint32), ("has_voxels", C.c_int32),
                ("Nb", C.c_int32), ("lims", C.c_double * 6), ("state_size", C.c_int32), ("_pad", C.c_int32),
                ("v_index", C.c_void_p), ("v_state", C.c_void_p), ("v_has_tip", C.c_void_p),
                ("v_tip", C.c_void_p), ("v_has_vox", C.c_void_p), ("v_off", C.c_void_p),
                ("v_keys", C.c_void_p), ("v_bits", C.c_void_p), ("e_src", C.c_void_p),
                ("e_dst", C.c_void_p), ("e_weight", C.c_void_p), ("e_has_vox", C.c_void_p),
                ("e_off", C.c_void_p), ("e_keys", C.c_void_p), ("e_bits", C.c_void_p)]


class Metric(C.Structure):
    """irt_metric: d = ((e + w_so2 s) + w_lin l), e = the L2 norm of the leading n_euclid columns (include/irt_b200.h)"""
    _fields_ = [("n_euclid", C.c_int32), ("so2_col", C.c_int32), ("lin_col", C.c_int32), ("_pad", C.c_int32),
                ("w_so2", C.c_double), ("w_lin", C.c_double)]


KNN_MAX_K = 64


class FkOutputs(C.Structure):
    _fields_ = [("p", C.c_void_p), ("R", C.c_void_p), ("t", C.c_void_p), ("npts", C.c_void_p),
                ("L", C.c_void_p), ("L_i", C.c_void_p), ("tip", C.c_void_p), ("uv", C.c_void_p),
                ("flags", C.c_void_p), ("iters", C.c_void_p), ("nsteps", C.c_void_p)]


# every symbol include/irt_b200.h declares (tests check the library exports each one)
ABI_SYMBOLS = [
    "irt_abi_version", "irt_status_string", "irt_ctx_create", "irt_ctx_destroy", "irt_last_error",
    "irt_ctx_device", "irt_ctx_synchronize", "irt_ctx_launch_count", "irt_measure_fp64_peak", "irt_measure_fp64_rate",
    "irt_robot_create", "irt_robot_destroy", "irt_robot_state_size", "irt_robot_max_points",
    "irt_fk_batch", "irt_fk_batch_dev", "irt_fk_batch_packed", "irt_home_lengths_batch", "irt_self_collision_shapes",
    "irt_fk_tip_jacobian_batch", "irt_fk_tip_jacobian_batch_dev",
    "irt_env_create", "irt_env_destroy", "irt_env_update", "irt_env_update_dev",
    "irt_env_update_sparse", "irt_env_nblocks",
    "irt_env_add_primitives",
    "irt_env_dilate", "irt_env_dilate_sphere", "irt_env_remove_interior", "irt_env_download",
    "irt_setstore_create", "irt_setstore_destroy", "irt_setstore_num_sets",
    "irt_setstore_num_blocks", "irt_setstore_import", "irt_setstore_export", "irt_setstore_append",
    "irt_setstore_device_ptrs", "irt_morton_key", "irt_morton_decode",
    "irt_voxelize_vertices", "irt_voxelize_shapes", "irt_voxelize_edges", "irt_voxelize_edges_until_invalid", "irt_voxelize_edges_indexed",
    "irt_valid_segment_count",
    "irt_check_sets", "irt_check_sets_dev", "irt_check_sets_popcount",
    "irt_check_sets_algorithmic_bytes",
    "irt_setindex_create", "irt_setindex_destroy", "irt_setindex_num_sets", "irt_check_sets_changed",
    "irt_xchg_create", "irt_xchg_destroy", "irt_xchg_handle_size", "irt_xchg_export", "irt_xchg_connect",
    "irt_check_sets_allgather_dev", "irt_xchg_status",
    "irt_rmp_read", "irt_rmp_write", "irt_rmp_free",
    "irt_nnset_create", "irt_nnset_destroy", "irt_nnset_size", "irt_nnset_append", "irt_nnset_clear",
    "irt_nnset_knn",
]

_lib = None


def lib():
    """Load libirt_b200.so (fails loudly when it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "irt_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a).  There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint32
    sig = {
        "irt_abi_version": (i32, []),
        "irt_status_string": (C.c_char_p, [i32]),
        "irt_ctx_create": (i32, [i32, C.POINTER(vp)]),
        "irt_ctx_destroy": (None, [vp]),
        "irt_last_error": (C.c_char_p, [vp]),
        "irt_ctx_device": (i32, [vp]),
        "irt_ctx_synchronize": (i32, [vp]),
        "irt_ctx_launch_count": (i64, [vp]),
        "irt_measure_fp64_peak": (i32, [vp, C.POINTER(C.c_double)]),
        "irt_measure_fp64_rate": (i32, [vp, i32, C.POINTER(C.c_double)]),
        "irt_robot_create": (i32, [vp, C.POINTER(RobotDesc), C.POINTER(vp)]),
        "irt_robot_destroy": (None, [vp]),
        "irt_robot_state_size": (i32, [vp]),
        "irt_robot_max_points": (i32, [vp]),
        "irt_fk_batch": (i32, [vp, vp, vp, i32, i64, i32, C.POINTER(FkOutputs)]),
        "irt_fk_batch_dev": (i32, [vp, vp, vp, i32, i64, i32, C.POINTER(FkOutputs), vp]),
        "irt_fk_batch_packed": (i32, [vp, vp, vp, i32, i64, C.POINTER(FkOutputs), i64, vp]),
        "irt_home_lengths_batch": (i32, [vp, vp, vp, i32, i64, vp]),
        "irt_self_collision_shapes": (i32, [vp, vp, vp, i32, i64, C.c_double, vp]),
        "irt_fk_tip_jacobian_batch": (i32, [vp, vp, vp, i32, i64, i32, C.c_double, vp, vp]),
        "irt_fk_tip_jacobian_batch_dev": (i32, [vp, vp, vp, i32, i64, i32, C.c_double, vp, vp, vp]),
        "irt_env_create": (i32, [vp, C.POINTER(Grid), C.POINTER(vp)]),
        "irt_env_destroy": (None, [vp]),
        "irt_env_update": (i32, [vp, vp, vp]),
        "irt_env_update_dev": (i32, [vp, vp, vp, vp]),
        "irt_env_update_sparse": (i32, [vp, vp, vp, vp, i64]),
        "irt_env_nblocks": (i64, [vp, vp]),
        "irt_env_add_primitives": (i32, [vp, vp, vp, i64, vp, i64, vp, i64, i32]),
        "irt_env_dilate": (i32, [vp, vp, i32, i32]),
        "irt_env_dilate_sphere": (i32, [vp, vp, C.c_double]),
        "irt_env_remove_interior": (i32, [vp, vp, i32]),
        "irt_env_download": (i32, [vp, vp, vp]),
        "irt_setstore_create": (i32, [vp, C.POINTER(Grid), C.POINTER(vp)]),
        "irt_setstore_destroy": (None, [vp]),
        "irt_setstore_num_sets": (i64, [vp]),
        "irt_setstore_num_blocks": (i64, [vp]),
        "irt_setstore_import": (i32, [vp, vp, i64, vp, vp, vp]),
        "irt_setstore_export": (i32, [vp, vp, vp, vp, vp]),
        "irt_setstore_append": (i32, [vp, vp, vp, i64, i64, vp]),
        "irt_setstore_device_ptrs": (i32, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
        "irt_morton_key": (u32, [i32, i32, i32, i32]),
        "irt_morton_decode": (None, [u32, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
        "irt_voxelize_vertices": (i32, [vp, vp, vp, i32, i64, vp, vp, vp]),
        "irt_voxelize_shapes": (i32, [vp, vp, vp, i32, i64, vp]),
        "irt_voxelize_edges": (i32, [vp, vp, C.POINTER(Space), vp, vp, i32, i64, vp, vp, vp, vp]),
        "irt_voxelize_edges_until_invalid": (i32, [vp, vp, C.POINTER(Space), vp, vp, i32, i64, vp, vp, vp, vp, vp]),
        "irt_voxelize_edges_indexed": (i32, [vp, vp, C.POINTER(Space), vp, i32, i64, vp, i64, vp, vp, vp, vp]),
        "irt_valid_segment_count": (u32, [C.POINTER(RobotDesc), C.POINTER(Space), vp, vp]),
        "irt_check_sets": (i32, [vp, vp, vp, i64, i64, vp]),
        "irt_check_sets_dev": (i32, [vp, vp, vp, i64, i64, vp, vp]),
        "irt_check_sets_popcount": (i32, [vp, vp, vp, i64, i64, vp]),
        "irt_check_sets_algorithmic_bytes": (i64, [vp, i64, i64]),
        "irt_setindex_create": (i32, [vp, vp, C.POINTER(vp)]),
        "irt_setindex_destroy": (None, [vp]),
        "irt_setindex_num_sets": (i64, [vp]),
        "irt_check_sets_changed": (i32, [vp, vp, vp, vp, vp, i64, i64, vp, vp, i64, vp, vp]),
        "irt_xchg_create": (i32, [vp, i32, i32, i64, C.POINTER(vp)]),
        "irt_xchg_destroy": (None, [vp]),
        "irt_xchg_handle_size": (i32, []),
        "irt_xchg_export": (i32, [vp, vp]),
        "irt_xchg_connect": (i32, [vp, vp]),
        "irt_check_sets_allgather_dev": (i32, [vp, vp, vp, i64, i64, vp, vp, C.POINTER(vp)]),
        "irt_xchg_status": (i32, [vp]),
        "irt_rmp_read": (i32, [C.c_char_p, C.POINTER(C.POINTER(Rmp))]),
        "irt_rmp_write": (i32, [C.c_char_p, C.POINTER(Rmp)]),
        "irt_rmp_free": (None, [C.POINTER(Rmp)]),
        "irt_nnset_create": (i32, [vp, i32, C.POINTER(Metric), C.POINTER(vp)]),
        "irt_nnset_destroy": (None, [vp]),
        "irt_nnset_size": (i64, [vp]),
        "irt_nnset_append": (i32, [vp, vp, vp, i64]),
        "irt_nnset_clear": (i32, [vp, vp]),
        "irt_nnset_knn": (i32, [vp, vp, vp, i64, i32, C.c_double, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args
    _lib = L
    return L


def robot_desc(spec):
    """dict (see workloads.robot_a) -> RobotDesc"""
    rb = RobotDesc()
    for k in ("r", "L", "dL", "ro", "ri", "E", "nu", "residual_threshold"):
        setattr(rb, k, float(spec[k]))
    Cc, Dd = spec["C"], spec["D"]
    n = len(Cc)
    if n > MAX_TENDONS:
        raise IrtError(IRT_ERR_OUT_OF_RANGE, "too many tendons")
    rb.n_tendons = n
    rb.n_c = len(Cc[0]) if n else 0
    rb.n_d = len(Dd[0]) if n else 0
    for j in range(n):
        if len(Cc[j]) != rb.n_c or len(Dd[j]) != rb.n_d:
            # get_r_info.h:34-39: all tendons use tendon 0's coefficient counts
            raise IrtError(IRT_ERR_INVALID_ARGUMENT, "tendons must share coefficient counts (pad with 0)")
        for i, c in enumerate(Cc[j]):
            rb.C[j * MAX_COEF + i] = float(c)
        for i, d in enumerate(Dd[j]):
            rb.D[j * MAX_COEF + i] = float(d)
        rb.max_tension[j] = float(spec["max_tension"][j])
        rb.min_length[j] = float(spec["min_length"][j])
        rb.max_length[j] = float(spec["max_length"][j])
    rb.enable_rotation = int(bool(spec.get("enable_rotation", False)))
    rb.enable_retraction = int(bool(spec.get("enable_retraction", False)))
    return rb


def make_grid(Ng, lim, inv_rot=None):
    g = Grid()
    g.Ng = int(Ng)
    for i, v in enumerate(lim):
        g.lim[i] = float(v)
    R = np.eye(3) if inv_rot is None else np.asarray(inv_rot, dtype=np.float64).reshape(3, 3)
    for i, v in enumerate(R.reshape(-1)):
        g.inv_rot[i] = float(v)
    return g


def make_space(min_tension_change=0.02, min_rotation_change=0.01, min_retraction_change=0.0001):
    return Space(min_tension_change, min_rotation_change, min_retraction_change)


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(int(a.data_ptr()))  # torch tensor


class Context:
    """irt_ctx: one CUDA device + stream.  Raises IrtError(IRT_ERR_NO_DEVICE) without a GPU."""

    def __init__(self, device=0):
        self.L = lib()
        h = C.c_void_p()
        rc = self.L.irt_ctx_create(int(device), C.byref(h))
        if rc != IRT_OK:
            raise IrtError(rc, self.L.irt_status_string(rc).decode())
        self.h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            self.L.irt_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != IRT_OK:
            raise IrtError(rc, "%s: %s" % (self.L.irt_status_string(rc).decode(),
                                           self.L.irt_last_error(self.h).decode()))

    def synchronize(self):
        self.check(self.L.irt_ctx_synchronize(self.h))

    def launch_count(self):
        return int(self.L.irt_ctx_launch_count(self.h))

    def fp64_peak(self):
        v = C.c_double()
        self.check(self.L.irt_measure_fp64_peak(self.h, C.byref(v)))
        return v.value

    def fp64_rate(self, mode):
        """DFMA rate (FLOP/s) of the probe with 0 / 2 / 3 register pairs per instruction that the operand reuse
        cache does not serve (mode 0 / 1 / 2)"""
        v = C.c_double()
        self.check(self.L.irt_measure_fp64_rate(self.h, int(mode), C.byref(v)))
        return v.value


def self_collision_shapes(ctx, p, npts, r):
    """collides_self(CapsuleSequence{points, r}) (collision/collision.cpp:6-46) for backbones p[n][cap][3], npts[n]"""
    p, npts = _np(p, np.float64), _np(npts, np.int32)
    n, cap = p.shape[0], p.shape[1]
    out = np.zeros(n, dtype=np.uint8)
    ctx.check(ctx.L.irt_self_collision_shapes(ctx.h, _ptr(p), _ptr(npts), cap, n, float(r), _ptr(out)))
    return out.astype(bool)


class Robot:
    """Mirror of tendon::TendonRobot for the batched FK path."""

    def __init__(self, ctx, spec):
        self.ctx, self.spec = ctx, spec
        self.desc = robot_desc(spec)
        h = C.c_void_p()
        ctx.check(ctx.L.irt_robot_create(ctx.h, C.byref(self.desc), C.byref(h)))
        self.h = h
        self.n_tendons = self.desc.n_tendons
        self.state_size = int(ctx.L.irt_robot_state_size(h))
        self.max_points = int(ctx.L.irt_robot_max_points(h))

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.L.irt_robot_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def shape_batch(self, states, want=("p", "npts", "L", "L_i", "tip", "flags"), cap_pts=None):
        """TendonRobot::shape for every row of `states` (host numpy in, host numpy out).
        `want` selects TendonResult members: p R t npts L L_i tip uv flags iters nsteps."""
        states = _np(states, np.float64)
        if states.ndim != 2:
            raise IrtError(IRT_ERR_INVALID_ARGUMENT, "states must be [n][S]")
        n, S = states.shape
        cap = cap_pts or self.max_points
        N = self.n_tendons
        shapes = dict(p=((n, cap, 3), np.float64), R=((n, cap, 9), np.float64),
                      t=((n, cap), np.float64), npts=((n,), np.int32), L=((n,), np.float64),
                      L_i=((n, N), np.float64), tip=((n, 3), np.float64), uv=((n, 12), np.float64),
                      flags=((n,), np.uint32), iters=((n,), np.int32), nsteps=((n,), np.int32))
        want = set(want)  # (flags alone is fine: the library keeps the points on the device)
        out = {k: np.zeros(*shapes[k]) for k in want}
        o = FkOutputs()
        for k, a in out.items():
            setattr(o, k, a.ctypes.data)
        self.ctx.check(self.ctx.L.irt_fk_batch(self.ctx.h, self.h, _ptr(states), S, n, cap, C.byref(o)))
        if "R" in out:  # column-major 3x3 -> [n][cap][row][col]
            out["R"] = out["R"].reshape(n, cap, 3, 3).transpose(0, 1, 3, 2)
        return out

    def shape_batch_packed(self, states, want=("p", "npts", "L", "L_i", "tip", "flags"), out=None,
                           cap_rows=None):
        """Like shape_batch, but p / R / t are packed: shape i owns rows
        [row_offsets[i], row_offsets[i+1]) (the reference's per-shape vectors laid end to end).
        `out` may carry preallocated (e.g. pinned) arrays; returns the dict with "row_offsets" and
        "rows" (total) added."""
        states = _np(states, np.float64)
        if states.ndim != 2:
            raise IrtError(IRT_ERR_INVALID_ARGUMENT, "states must be [n][S]")
        n, S = states.shape
        N = self.n_tendons
        cap_rows = int(cap_rows if cap_rows is not None else n * self.max_points)
        shapes = dict(p=((cap_rows, 3), np.float64), R=((cap_rows, 9), np.float64),
                      t=((cap_rows,), np.float64), npts=((n,), np.int32), L=((n,), np.float64),
                      L_i=((n, N), np.float64), tip=((n, 3), np.float64), uv=((n, 12), np.float64),
                      flags=((n,), np.uint32), iters=((n,), np.int32), nsteps=((n,), np.int32))
        res = dict(out) if out is not None else {}
        for k in want:
            if k not in res:
                res[k] = np.empty(*shapes[k])
        if "row_offsets" not in res:
            res["row_offsets"] = np.zeros(n + 1, dtype=np.int64)
        o = FkOutputs()
        for k in shapes:
            if k in res:
                setattr(o, k, _ptr(res[k]).value if hasattr(res[k], "data_ptr") else res[k].ctypes.data)
        self.ctx.check(self.ctx.L.irt_fk_batch_packed(self.ctx.h, self.h, _ptr(states), S, n, C.byref(o),
                                                      cap_rows, _ptr(res["row_offsets"])))
        res["rows"] = int(np.asarray(res["row_offsets"])[-1]) if not hasattr(res["row_offsets"], "data_ptr") \
            else int(res["row_offsets"][-1])
        return res

    def shape_batch_dev(self, d_states, n, outputs, cap_pts=None, stream=None):
        """Device-resident form: d_states and every value of `outputs` are torch CUDA tensors
        (or objects with data_ptr()).  Asynchronous."""
        o = FkOutputs()
        for k, a in outputs.items():
            setattr(o, k, int(a.data_ptr()))
        cap = cap_pts or self.max_points
        self.ctx.check(self.ctx.L.irt_fk_batch_dev(
            self.ctx.h, self.h, _ptr(d_states), self.state_size, int(n), cap, C.byref(o),
            C.c_void_p(stream) if stream else None))

    def tip_jacobian_batch(self, states, mode=JAC_LEVMAR_CENTRAL, delta=1e-4):
        """Finite-difference tip Jacobians of every row of `states` in one FK batch: returns
        (tips [n][3], J [n][3][S]).  mode: JAC_FORWARD_FIXED = tip_control::Jacobian
        (tip-control/tip_control.cpp:243-265); JAC_LEVMAR_FORWARD / JAC_LEVMAR_CENTRAL = the rule of
        levmar-2.6 behind tip_control::inverse_kinematics (misc_core.c:137-211).
        tip_control::Jacobian takes its step as a C `float`: pass delta=float(np.float32(dist)) to take exactly
        the step the reference takes (oracle == the reference's own text bit for bit with that step)."""
        states = _np(states, np.float64)
        if states.ndim != 2:
            raise IrtError(IRT_ERR_INVALID_ARGUMENT, "states must be [n][S]")
        n, S = states.shape
        tips, J = np.zeros((n, 3)), np.zeros((n, 3, S))
        self.ctx.check(self.ctx.L.irt_fk_tip_jacobian_batch(
            self.ctx.h, self.h, _ptr(states), S, n, int(mode), float(delta), _ptr(tips), _ptr(J)))
        return tips, J

    def home_lengths(self, states):
        states = _np(states, np.float64)
        n, S = states.shape
        out = np.zeros((n, self.n_tendons))
        self.ctx.check(self.ctx.L.irt_home_lengths_batch(self.ctx.h, self.h, _ptr(states), S, n, _ptr(out)))
        return out

    def valid_segment_count(self, space, a, b):
        a, b = _np(a, np.float64), _np(b, np.float64)
        return int(self.ctx.L.irt_valid_segment_count(C.byref(self.desc), C.byref(space), _ptr(a), _ptr(b)))


class Env:
    """Device-resident obstacle voxel grid (dense, Morton-ordered leaf blocks)."""

    def __init__(self, ctx, grid):
        self.ctx, self.grid = ctx, grid
        h = C.c_void_p()
        ctx.check(ctx.L.irt_env_create(ctx.h, C.byref(grid), C.byref(h)))
        self.h = h
        self.Nb = grid.Ng // 4

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.L.irt_env_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def update(self, blocks):
        """blocks: uint64[Nb^3] indexed by Morton key (host numpy)."""
        blocks = _np(blocks, np.uint64)
        if blocks.size != self.Nb ** 3:
            raise IrtError(IRT_ERR_INVALID_ARGUMENT, "env needs Nb^3 blocks")
        self.ctx.check(self.ctx.L.irt_env_update(self.ctx.h, self.h, _ptr(blocks)))

    def update_dev(self, d_blocks, stream=None):
        self.ctx.check(self.ctx.L.irt_env_update_dev(self.ctx.h, self.h, _ptr(d_blocks),
                                                     C.c_void_p(stream) if stream else None))

    def update_sparse(self, bxyz, bits):
        """VoxelOctree::visit_leaves style input: uint8[n,3] block coords + uint64[n] bits."""
        bxyz, bits = _np(bxyz, np.uint8), _np(bits, np.uint64)
        self.ctx.check(self.ctx.L.irt_env_update_sparse(self.ctx.h, self.h, _ptr(bxyz), _ptr(bits), len(bits)))

    def nblocks(self):
        return int(self.ctx.L.irt_env_nblocks(self.ctx.h, self.h))

    def add_primitives(self, points=None, spheres=None, capsules=None, clear=False, dilate=0.0):
        """Environment::voxelize (motion-planning/Environment.cpp:62-101) on the device: points [n][3], spheres
        [n][4] = (c, r), capsules [n][7] = (a, b, r) OR-ed into the grid (clear=True: into an empty one).
        dilate > 0 is the reference's second overload: every radius grows by `dilate` and the points become
        spheres of that radius; dilate == 0 there voxelises NOTHING (its `dummy` environment stays empty,
        Environment.cpp:86-99) -- use dilate=0.0 here for the plain overload."""
        def arr(a, w):
            a = np.zeros((0, w)) if a is None else np.ascontiguousarray(a, dtype=np.float64).reshape(-1, w)
            return a
        pts, sph, cap = arr(points, 3), arr(spheres, 4), arr(capsules, 7)
        if dilate < 0.0:
            raise IrtError(IRT_ERR_INVALID_ARGUMENT, "Negative dilation value given")   # Environment.cpp:83-85
        if dilate > 0.0:
            sph = np.concatenate([np.concatenate([pts, np.full((len(pts), 1), dilate)], axis=1),
                                  sph + np.array([0, 0, 0, dilate])], axis=0)
            cap = cap + np.array([0, 0, 0, 0, 0, 0, dilate])
            pts = np.zeros((0, 3))
        sph, cap, pts = (np.ascontiguousarray(x) for x in (sph, cap, pts))
        self.ctx.check(self.ctx.L.irt_env_add_primitives(
            self.ctx.h, self.h, _ptr(pts) if len(pts) else None, len(pts), _ptr(sph) if len(sph) else None, len(sph),
            _ptr(cap) if len(cap) else None, len(cap), int(bool(clear))))

    def dilate(self, num=1, use_diagonal=False):
        """VoxelOctree::dilate_6neighbor / dilate_27neighbor, in place on the device."""
        self.ctx.check(self.ctx.L.irt_env_dilate(self.ctx.h, self.h, int(num), int(bool(use_diagonal))))

    def dilate_sphere(self, r):
        """VoxelOctree::dilate_sphere(r)."""
        self.ctx.check(self.ctx.L.irt_env_dilate_sphere(self.ctx.h, self.h, float(r)))

    def remove_interior(self, keep_diagonal=True):
        """VoxelOctree::remove_interior(keep_diagonal)."""
        self.ctx.check(self.ctx.L.irt_env_remove_interior(self.ctx.h, self.h, int(bool(keep_diagonal))))

    def download(self):
        """Dense host copy: uint64[Nb^3] indexed by Morton key."""
        out = np.zeros(self.Nb ** 3, np.uint64)
        self.ctx.check(self.ctx.L.irt_env_download(self.ctx.h, self.h, _ptr(out)))
        return out


class SetStore:
    """CSR store of cached vertex / edge voxel sets on the device."""

    def __init__(self, ctx, grid):
        self.ctx, self.grid = ctx, grid
        h = C.c_void_p()
        ctx.check(ctx.L.irt_setstore_create(ctx.h, C.byref(grid), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.L.irt_setstore_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def num_sets(self):
        return int(self.ctx.L.irt_setstore_num_sets(self.h))

    @property
    def num_blocks(self):
        return int(self.ctx.L.irt_setstore_num_blocks(self.h))

    def import_csr(self, offsets, keys, bits):
        offsets, keys, bits = _np(offsets, np.uint64), _np(keys, np.uint32), _np(bits, np.uint64)
        self.ctx.check(self.ctx.L.irt_setstore_import(self.ctx.h, self.h, len(offsets) - 1,
                                                      _ptr(offsets), _ptr(keys), _ptr(bits)))

    def export_csr(self):
        n, nb = self.num_sets, self.num_blocks
        offsets = np.zeros(n + 1, dtype=np.uint64)
        keys = np.zeros(max(nb, 1), dtype=np.uint32)
        bits = np.zeros(max(nb, 1), dtype=np.uint64)
        self.ctx.check(self.ctx.L.irt_setstore_export(self.ctx.h, self.h, _ptr(offsets), _ptr(keys), _ptr(bits)))
        return offsets, keys[:nb], bits[:nb]

    def append(self, src, keep=None, begin=0, end=None):
        """Append sets [begin, end) of the store `src` after this store's last set, in index order; keep (bool[end -
        begin], optional) selects the sets that are appended.  The sets already here stay as they are."""
        end = src.num_sets if end is None else end
        words = None
        if keep is not None:
            keep = np.asarray(keep, dtype=bool)
            if keep.shape != (max(end - begin, 0),):
                raise IrtError(IRT_ERR_INVALID_ARGUMENT, "keep must hold one flag per set of the range")
            words = pack_mask(keep)
        self.ctx.check(self.ctx.L.irt_setstore_append(self.ctx.h, self.h, src.h, begin, end,
                                                      _ptr(words) if words is not None else None))

    def voxelize_vertices(self, robot, states):
        """precomputeVertexVoxelCache: FK + is_valid_shape + voxelize for every state.
        Returns (flags uint32[n], tips float64[n,3])."""
        states = _np(states, np.float64)
        n, S = states.shape
        flags = np.zeros(n, dtype=np.uint32)
        tips = np.zeros((n, 3))
        self.ctx.check(self.ctx.L.irt_voxelize_vertices(self.ctx.h, robot.h, _ptr(states), S, n, self.h,
                                                        _ptr(flags), _ptr(tips)))
        return flags, tips

    def voxelize_shapes(self, p, npts):
        """AbstractVoxelValidityChecker::voxelize for already computed backbones p[n][cap][3]."""
        p, npts = _np(p, np.float64), _np(npts, np.int32)
        n, cap = p.shape[0], p.shape[1]
        self.ctx.check(self.ctx.L.irt_voxelize_shapes(self.ctx.h, _ptr(p), _ptr(npts), cap, n, self.h))

    def voxelize_edges(self, robot, space, a, b):
        """precomputeEdgeVoxelCache: swept volume of every edge a[i] -> b[i].
        Returns dict(flags, t_last, nsamples)."""
        a, b = _np(a, np.float64), _np(b, np.float64)
        n, S = a.shape
        flags = np.zeros(n, dtype=np.uint32)
        t_last = np.zeros(n)
        nsamples = np.zeros(n, dtype=np.int32)
        self.ctx.check(self.ctx.L.irt_voxelize_edges(self.ctx.h, robot.h, C.byref(space), _ptr(a), _ptr(b),
                                                     S, n, self.h, _ptr(flags), _ptr(t_last), _ptr(nsamples)))
        return dict(flags=flags, t_last=t_last, nsamples=nsamples)

    def voxelize_edges_until_invalid(self, robot, space, a, b, env):
        """voxelize_until_invalid: swept volume up to the first configuration that is invalid or
        whose backbone hits `env`.  Returns dict(flags, t_last, nsamples)."""
        a, b = _np(a, np.float64), _np(b, np.float64)
        n, S = a.shape
        flags = np.zeros(n, dtype=np.uint32)
        t_last = np.zeros(n)
        nsamples = np.zeros(n, dtype=np.int32)
        self.ctx.check(self.ctx.L.irt_voxelize_edges_until_invalid(
            self.ctx.h, robot.h, C.byref(space), _ptr(a), _ptr(b), S, n, env.h, self.h,
            _ptr(flags), _ptr(t_last), _ptr(nsamples)))
        return dict(flags=flags, t_last=t_last, nsamples=nsamples)

    def voxelize_edges_indexed(self, robot, space, vertex_states, pairs):
        """precomputeEdgeVoxelCache with edges given as (source, target) vertex indices; every
        vertex's FK is computed once and shared by its incident edges."""
        vs = _np(vertex_states, np.float64)
        pr = _np(pairs, np.int64).reshape(-1, 2)
        nv, S = vs.shape
        n = pr.shape[0]
        flags = np.zeros(n, dtype=np.uint32)
        t_last = np.zeros(n)
        nsamples = np.zeros(n, dtype=np.int32)
        self.ctx.check(self.ctx.L.irt_voxelize_edges_indexed(
            self.ctx.h, robot.h, C.byref(space), _ptr(vs), S, nv, _ptr(pr), n, self.h,
            _ptr(flags), _ptr(t_last), _ptr(nsamples)))
        return dict(flags=flags, t_last=t_last, nsamples=nsamples)

    def check(self, env, begin=0, end=None):
        """precomputeVertexValidity / precomputeEdgeValidity with warm caches: returns a bool
        array, True where the cached set collides with the environment."""
        end = self.num_sets if end is None else end
        n = end - begin
        words = np.zeros(max((n + 31) // 32, 1), dtype=np.uint32)
        self.ctx.check(self.ctx.L.irt_check_sets(self.ctx.h, self.h, env.h, begin, end, _ptr(words)))
        return unpack_verdicts(words, n)

    def check_dev(self, env, d_words, begin=0, end=None, stream=None):
        end = self.num_sets if end is None else end
        self.ctx.check(self.ctx.L.irt_check_sets_dev(self.ctx.h, self.h, env.h, begin, end, _ptr(d_words),
                                                     C.c_void_p(stream) if stream else None))

    def popcount(self, env, begin=0, end=None):
        end = self.num_sets if end is None else end
        stats = np.zeros(2, dtype=np.uint64)
        self.ctx.check(self.ctx.L.irt_check_sets_popcount(self.ctx.h, self.h, env.h, begin, end, _ptr(stats)))
        return int(stats[0]), int(stats[1])

    def algorithmic_bytes(self, begin=0, end=None):
        end = self.num_sets if end is None else end
        return int(self.ctx.L.irt_check_sets_algorithmic_bytes(self.h, begin, end))

    def check_changed(self, index, env_old, env_new, words, begin=0, end=None):
        """Revalidation after an environment change (irt_check_sets_changed): `words` (uint32, the packed verdicts
        check(env_old, begin, end) gave) become the words of check(env_new, begin, end), in place when they are a
        contiguous uint32 array.  Only the sets whose leaves overlap the changed voxels, and the sets appended after
        `index` was built, are re-checked.  Returns (words, flipped: int64 indices of the sets whose verdict changed,
        ascending; stats: [changed leaf blocks, sets re-checked, 1 if the whole range was swept instead])."""
        end = self.num_sets if end is None else end
        words = _np(words, np.uint32)
        if len(words) < (max(end - begin, 0) + 31) // 32:
            raise IrtError(IRT_ERR_INVALID_ARGUMENT, "words must hold (end - begin + 31) // 32 entries")
        stats = np.zeros(3, dtype=np.int64)
        n_flipped = C.c_int64(0)
        flipped = np.zeros(1024, dtype=np.int64)
        for attempt in range(2):      # a change that flips more sets than the buffer holds: grow it, try once more
            rc = self.ctx.L.irt_check_sets_changed(self.ctx.h, self.h, index.h, env_old.h, env_new.h, begin, end,
                                                   _ptr(words), _ptr(flipped), len(flipped), C.byref(n_flipped),
                                                   _ptr(stats))
            if rc != IRT_ERR_CAPACITY or attempt == 1 or n_flipped.value <= len(flipped):
                break
            flipped = np.zeros(n_flipped.value, dtype=np.int64)
        self.ctx.check(rc)
        return words, flipped[:n_flipped.value].copy(), stats


class SetIndex:
    """Inverted index of a SetStore (irt_setindex): per leaf-block key, the sets with a leaf there and that leaf's
    bits.  It covers the store's sets as they are when it is built; sets appended later are its tail, and replacing
    the store's content makes it stale (SetStore.check_changed then raises)."""

    def __init__(self, ctx, store):
        self.ctx, self.store = ctx, store
        h = C.c_void_p()
        ctx.check(ctx.L.irt_setindex_create(ctx.h, store.h, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.L.irt_setindex_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def num_sets(self):
        return int(self.ctx.L.irt_setindex_num_sets(self.h))


def state_metric(spec):
    """irt_metric of the compound state space (Problem.cpp:118-141) with the weights computed exactly as
    roadmap.VoxelCachedLazyPRM.distance computes them: tensions under L2, rotation weighted ext / (4 pi), retraction
    weighted 2 ext / L, ext = |max_tension|.  Returns (state size, Metric)."""
    N = len(spec["C"])
    ext = float(np.linalg.norm(np.asarray(spec["max_tension"], dtype=np.float64)[:N]))
    m = Metric(N, -1, -1, 0, 0.0, 0.0)
    k = N
    if spec.get("enable_rotation"):
        m.so2_col, m.w_so2 = k, ext / (4 * np.pi)
        k += 1
    if spec.get("enable_retraction"):
        m.lin_col, m.w_lin = k, 2 * ext / spec["L"]
        k += 1
    return k, m


def tip_metric():
    """plain R^3, as np.linalg.norm(tips - request, axis=1)"""
    return Metric(3, -1, -1, 0, 0.0, 0.0)


def pack_mask(flags):
    """bool[n] -> the uint32 exclude words of NearestSet.knn (bit i % 32 of word i / 32)"""
    b = np.packbits(np.asarray(flags, dtype=bool), bitorder="little")
    w = np.zeros(-(-len(b) // 4) * 4, dtype=np.uint8)
    w[:len(b)] = b
    return w.view(np.uint32)


class NearestSet:
    """Device-resident, append-only point set with exact k-nearest-neighbour queries (irt_nnset_*): the answers are
    the same indices in the same order as a stable sort of the distances of the contract in include/irt_b200.h."""

    def __init__(self, ctx, dim, metric):
        self.ctx, self.dim, self.metric = ctx, int(dim), metric
        h = C.c_void_p()
        ctx.check(ctx.L.irt_nnset_create(ctx.h, self.dim, C.byref(metric), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.L.irt_nnset_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def size(self):
        return int(self.ctx.L.irt_nnset_size(self.h))

    def append(self, rows):
        rows = _np(rows, np.float64).reshape(-1, self.dim)
        if len(rows):
            self.ctx.check(self.ctx.L.irt_nnset_append(self.ctx.h, self.h, _ptr(rows), len(rows)))

    def clear(self):
        self.ctx.check(self.ctx.L.irt_nnset_clear(self.ctx.h, self.h))

    def knn(self, queries, k, bound=np.inf, exclude=None):
        """queries [m][dim] -> (idx int64[m][k], dist float64[m][k]); missing entries are -1 / inf.  exclude: None,
        bool[size()] or uint32 words (pack_mask)."""
        q = _np(queries, np.float64).reshape(-1, self.dim)
        m, k = len(q), int(k)
        idx = np.empty((m, max(k, 0)), dtype=np.int64)
        dist = np.empty((m, max(k, 0)))
        words = None
        if exclude is not None:
            exclude = np.asarray(exclude)
            words = pack_mask(exclude) if exclude.dtype == bool else _np(exclude, np.uint32)
            if len(words) * 32 < self.size():
                raise IrtError(IRT_ERR_INVALID_ARGUMENT, "exclude mask shorter than the set")
        self.ctx.check(self.ctx.L.irt_nnset_knn(self.ctx.h, self.h, _ptr(q), m, k, float(bound), _ptr(words),
                                                _ptr(idx), _ptr(dist)))
        return idx, dist


class _DeviceWords:
    """zero-copy view of device words for torch.as_tensor(..., device="cuda")"""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": "<i4", "data": (int(ptr), False),
                                         "version": 2}


class VerdictExchange:
    """Verdict all-gather fused into K3 over peer memory (include/irt_b200.h, irt_xchg_*).
    `dist` is an initialised torch.distributed (NCCL) used once, to publish the IPC handles."""

    def __init__(self, ctx, rank, world, slot_words, dist=None):
        self.ctx, self.rank, self.world, self.slot_words = ctx, rank, world, int(slot_words)
        h = C.c_void_p()
        ctx.check(ctx.L.irt_xchg_create(ctx.h, rank, world, self.slot_words, C.byref(h)))
        self.h = h
        if world > 1:
            import torch
            hs = ctx.L.irt_xchg_handle_size()
            mine = np.zeros(hs, dtype=np.uint8)
            ctx.check(ctx.L.irt_xchg_export(self.h, _ptr(mine)))
            dev = torch.device("cuda", ctx.device)
            t = torch.from_numpy(mine).to(dev)
            allh = torch.empty(world * hs, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(allh, t)
            handles = np.ascontiguousarray(allh.cpu().numpy())
            ctx.check(ctx.L.irt_xchg_connect(self.h, _ptr(handles)))
            dist.barrier()   # every rank has mapped every buffer before the first sweep

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.L.irt_xchg_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, store, env, begin=0, end=None, stream=None):
        """K3 + fused all-gather (asynchronous on `stream`).  Returns a zero-copy torch int32 view
        [world * slot_words] of this sweep's gathered verdict words (valid until the sweep after next)."""
        import torch
        end = store.num_sets if end is None else end
        out = C.c_void_p()
        self.ctx.check(self.ctx.L.irt_check_sets_allgather_dev(
            self.ctx.h, store.h, env.h, int(begin), int(end), self.h,
            C.c_void_p(stream) if stream else None, C.byref(out)))
        return torch.as_tensor(_DeviceWords(out.value, self.world * self.slot_words),
                               device=torch.device("cuda", self.ctx.device))

    def status(self):
        return int(self.ctx.L.irt_xchg_status(self.h))


def _arr(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype).copy()


def read_rmp(path):
    """Parse a reference `.rmp` roadmap (VoxelCachedLazyPRM.cpp:862-1114) into numpy arrays; the
    vertex / edge voxel caches come back as CSR triples ready for SetStore.import_csr."""
    L = lib()
    p = C.POINTER(Rmp)()
    rc = L.irt_rmp_read(os.fsencode(path), C.byref(p))
    if rc != IRT_OK:
        raise IrtError(rc, "cannot parse %s" % path)
    r = p.contents
    nv, ne, S = r.n_verts, r.n_edges, r.state_size
    voff = _arr(r.v_off, nv + 1, np.uint64)
    eoff = _arr(r.e_off, ne + 1, np.uint64)
    out = dict(
        n_verts=nv, n_edges=ne, has_voxels=bool(r.has_voxels), Ng=r.Nb * 4, lims=list(r.lims),
        v_index=_arr(r.v_index, nv, np.uint32), v_state=_arr(r.v_state, nv * S, np.float64).reshape(nv, S),
        v_has_tip=_arr(r.v_has_tip, nv, np.uint8).astype(bool), v_tip=_arr(r.v_tip, nv * 3, np.float64).reshape(nv, 3),
        v_has_vox=_arr(r.v_has_vox, nv, np.uint8).astype(bool), v_off=voff,
        v_keys=_arr(r.v_keys, int(voff[-1]), np.uint32), v_bits=_arr(r.v_bits, int(voff[-1]), np.uint64),
        e_src=_arr(r.e_src, ne, np.uint32), e_dst=_arr(r.e_dst, ne, np.uint32),
        e_weight=_arr(r.e_weight, ne, np.float64), e_has_vox=_arr(r.e_has_vox, ne, np.uint8).astype(bool),
        e_off=eoff, e_keys=_arr(r.e_keys, int(eoff[-1]), np.uint32), e_bits=_arr(r.e_bits, int(eoff[-1]), np.uint64))
    L.irt_rmp_free(p)
    return out


def write_rmp(path, d):
    """Inverse of read_rmp: `d` has the same keys (numpy arrays)."""
    L = lib()
    keep = []

    def ptr(a, dt):
        a = np.ascontiguousarray(a, dtype=dt)
        if a.size == 0:
            a = np.zeros(1, dtype=dt)
        keep.append(a)
        return a.ctypes.data

    r = Rmp()
    r.n_verts, r.n_edges = int(d["n_verts"]), int(d["n_edges"])
    r.has_voxels = int(bool(d["has_voxels"]))
    r.Nb = int(d["Ng"]) // 4
    for i, v in enumerate(d["lims"]):
        r.lims[i] = float(v)
    r.state_size = int(np.asarray(d["v_state"]).shape[1]) if r.n_verts else 0
    r.v_index = ptr(d["v_index"], np.uint32); r.v_state = ptr(d["v_state"], np.float64)
    r.v_has_tip = ptr(d["v_has_tip"], np.uint8); r.v_tip = ptr(d["v_tip"], np.float64)
    r.v_has_vox = ptr(d["v_has_vox"], np.uint8); r.v_off = ptr(d["v_off"], np.uint64)
    r.v_keys = ptr(d["v_keys"], np.uint32); r.v_bits = ptr(d["v_bits"], np.uint64)
    r.e_src = ptr(d["e_src"], np.uint32); r.e_dst = ptr(d["e_dst"], np.uint32)
    r.e_weight = ptr(d["e_weight"], np.float64); r.e_has_vox = ptr(d["e_has_vox"], np.uint8)
    r.e_off = ptr(d["e_off"], np.uint64); r.e_keys = ptr(d["e_keys"], np.uint32); r.e_bits = ptr(d["e_bits"], np.uint64)
    rc = L.irt_rmp_write(os.fsencode(path), C.byref(r))
    if rc != IRT_OK:
        raise IrtError(rc, "cannot write %s" % path)


def unpack_verdicts(words, n):
    w8 = np.ascontiguousarray(words, dtype=np.uint32).view(np.uint8)
    return np.unpackbits(w8, count=n, bitorder="little").view(bool)   # bytes 0 / 1: a bool view, no copy


def shard_range(n, rank, world, align=64):
    """Contiguous index range of `rank` among `world` shards, boundaries aligned to `align`
    so verdict words never straddle shards (SURVEY 8e)."""
    per = -(-n // world)
    per = -(-per // align) * align
    lo = min(n, rank * per)
    hi = min(n, lo + per)
    return lo, hi
