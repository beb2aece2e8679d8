"""irt_setstore_append (csrc/voxel_check.cu) on the B200: every appended store equals, bit for bit, the export of a store
imported from the numpy-concatenated CSR -- synthetic stores of every shape, every kind of keep mask, many small
appends against one large one, K3 over the result, real vertex / edge sets -- every argument error leaves dst as it
was, and extendVoxelCache of both planner mirrors gives a fresh planner's caches and validity tables."""
import ctypes as C
import os
import subprocess
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NG = 128
NKEYS = (NG // 4) ** 3


@pytest.fixture(scope="module")
def irt():
    import irt_b200
    return irt_b200


@pytest.fixture(scope="module")
def ctx(irt):
    return irt.Context(0)


@pytest.fixture(scope="module")
def grid(irt):
    return irt.make_grid(NG, [-0.2, 0.2, -0.2, 0.2, -0.2, 0.2])


def _random_csr(rng, sizes):
    """CSR with sets of the given leaf counts (at most 2000): strictly increasing Morton keys, random non-zero bits"""
    sizes = np.asarray(sizes, dtype=np.int64)
    off = np.zeros(len(sizes) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(sizes)
    inc = rng.integers(1, 16, size=int(off[-1]))
    cs = np.concatenate([[0], np.cumsum(inc)])
    set_id = np.repeat(np.arange(len(sizes)), sizes)
    start = rng.integers(0, NKEYS - 15 * sizes)
    keys = (start[set_id] + cs[1:] - cs[off[:-1].astype(np.int64)][set_id] - 1).astype(np.uint32)
    bits = rng.integers(1, 2 ** 63, size=len(keys), dtype=np.int64).astype(np.uint64)
    return off, keys, bits


def _concat(dst, src, begin, end, keep):
    """numpy restatement of the contract: dst's sets, then the kept sets of src[begin:end]"""
    off, keys, bits = (np.asarray(a) for a in dst)
    so, sk, sb = src
    out_off, out_k, out_b = [off], [keys], [bits]
    last = int(off[-1])
    for i in range(end - begin):
        if keep is not None and not keep[i]:
            continue
        lo, hi = int(so[begin + i]), int(so[begin + i + 1])
        out_k.append(sk[lo:hi])
        out_b.append(sb[lo:hi])
        last += hi - lo
        out_off.append(np.array([last], dtype=np.uint64))
    return (np.concatenate(out_off).astype(np.uint64), np.concatenate(out_k).astype(np.uint32),
            np.concatenate(out_b).astype(np.uint64))


def _store(irt, ctx, grid, csr=None):
    s = irt.SetStore(ctx, grid)
    if csr is not None:
        s.import_csr(*csr)
    return s


def _assert_same(irt, ctx, grid, store, want):
    got = store.export_csr()
    ref = _store(irt, ctx, grid, want).export_csr()
    for g, r, w in zip(got, ref, want):
        assert g.dtype == r.dtype and np.array_equal(g, r) and np.array_equal(g, w)


def _sizes(rng, kind, n):
    if kind == "typical":
        return rng.poisson(23, size=n)
    if kind == "wide":
        return rng.integers(1, 2001, size=n)
    if kind == "empty_sets":
        return np.where(rng.random(n) < 0.5, 0, rng.integers(1, 40, size=n))
    if kind == "zero_leaves":
        return np.zeros(n, dtype=np.int64)
    raise ValueError(kind)


@pytest.mark.parametrize("kind,n_dst,n_src,begin,end", [
    ("typical", 0, 1, 0, 1),                 # one set onto a store that never held anything
    ("typical", 37, 1, 0, 1),
    ("empty_sets", 33, 517, 3, 514),          # range and leaf counts not divisible by 4
    ("zero_leaves", 0, 70, 0, 70),            # a store without leaves
    ("zero_leaves", 19, 70, 5, 69),
    ("wide", 11, 300, 1, 299),                # sets of 1 to 2000 leaves
    ("typical", 200_000, 200_000, 0, 200_000),
    ("typical", 1001, 200_001, 7, 199_990),
])
@pytest.mark.parametrize("mask", ["none", "all_clear", "all_set", "random"])
def test_append_equals_import_of_concatenation(irt, ctx, grid, kind, n_dst, n_src, begin, end, mask):
    rng = np.random.default_rng(zlib.crc32(repr((kind, n_dst, n_src, begin, end, mask)).encode()))
    dst_csr = _random_csr(rng, _sizes(rng, kind, n_dst))
    src_csr = _random_csr(rng, _sizes(rng, kind, n_src))
    n = end - begin
    keep = {"none": None, "all_clear": np.zeros(n, dtype=bool), "all_set": np.ones(n, dtype=bool),
            "random": rng.random(n) < 0.9}[mask]
    dst = _store(irt, ctx, grid, dst_csr if n_dst else None)
    src = _store(irt, ctx, grid, src_csr)
    dst.append(src, keep=keep, begin=begin, end=end)
    _assert_same(irt, ctx, grid, dst, _concat(dst_csr, src_csr, begin, end, keep))
    assert src.export_csr()[0].tobytes() == src_csr[0].tobytes()


def test_partial_last_mask_word_ignores_bits_past_the_range(irt, ctx, grid):
    """bits of the last keep word past the range are not sets of the range: they neither add nor count"""
    rng = np.random.default_rng(5)
    src_csr = _random_csr(rng, rng.poisson(23, size=100))
    for begin, end in ((0, 45), (10, 43), (60, 61)):
        n = end - begin
        keep = rng.random(n) < 0.5
        words = irt.pack_mask(keep)
        words[-1] |= np.uint32(0xffffffff) << np.uint32(n % 32) if n % 32 else np.uint32(0)
        dst = _store(irt, ctx, grid)
        src = _store(irt, ctx, grid, src_csr)
        ctx.check(ctx.L.irt_setstore_append(ctx.h, dst.h, src.h, begin, end, words.ctypes.data_as(C.c_void_p)))
        _assert_same(irt, ctx, grid, dst, _concat((np.zeros(1, np.uint64), np.zeros(0, np.uint32),
                                                   np.zeros(0, np.uint64)), src_csr, begin, end, keep))


def test_many_small_appends_equal_one_large(irt, ctx, grid):
    """100 appends grow the store's arrays many times over; every growth keeps what was there"""
    rng = np.random.default_rng(9)
    src_csr = _random_csr(rng, rng.poisson(23, size=30_000))
    src = _store(irt, ctx, grid, src_csr)
    keep = rng.random(30_000) < 0.8
    one = _store(irt, ctx, grid)
    one.append(src, keep=keep)
    many = _store(irt, ctx, grid)
    cuts = np.sort(rng.choice(np.arange(1, 30_000), size=99, replace=False))
    for lo, hi in zip(np.r_[0, cuts], np.r_[cuts, 30_000]):
        many.append(src, keep=keep[lo:hi], begin=int(lo), end=int(hi))
    for a, b in zip(one.export_csr(), many.export_csr()):
        assert np.array_equal(a, b)
    _assert_same(irt, ctx, grid, many, _concat((np.zeros(1, np.uint64), np.zeros(0, np.uint32),
                                                np.zeros(0, np.uint64)), src_csr, 0, 30_000, keep))


def test_check_sets_over_appended_store(irt, ctx, grid):
    """K3 reads the appended store like the imported one: the same verdicts and the same popcount checksums"""
    rng = np.random.default_rng(13)
    dst_csr = _random_csr(rng, rng.poisson(23, size=5001))
    src_csr = _random_csr(rng, rng.poisson(23, size=7003))
    keep = rng.random(7000) < 0.9
    env = irt.Env(ctx, grid)
    blocks = np.where(rng.random(NKEYS) < 0.05, rng.integers(1, 2 ** 63, size=NKEYS, dtype=np.int64), 0).astype(np.uint64)
    env.update(blocks)
    dst = _store(irt, ctx, grid, dst_csr)
    dst.append(_store(irt, ctx, grid, src_csr), keep=keep, begin=2, end=7002)
    ref = _store(irt, ctx, grid, _concat(dst_csr, src_csr, 2, 7002, keep))
    assert dst.num_sets == ref.num_sets
    hits = dst.check(env)
    assert hits.any() and not hits.all()
    assert np.array_equal(hits, ref.check(env))
    for b, e in ((0, dst.num_sets), (5001, dst.num_sets), (4999, 5003), (17, 12_000)):
        e = min(e, dst.num_sets)
        assert np.array_equal(dst.check(env, b, e), ref.check(env, b, e))
        assert dst.popcount(env, b, e) == ref.popcount(env, b, e)


def test_real_sets_in_two_batches_equal_one_call(irt, ctx, wl):
    """vertex sets and indexed edge sets voxelised in two batches and appended equal one call over all of them"""
    spec = wl.robot_b(0.003, rotation=True)
    g = wl.workspace_grid(spec)
    grid = irt.make_grid(g["Ng"], g["lim"])
    rb = irt.Robot(ctx, spec)
    states = wl.sample_states(spec, 3001, stream=77)
    pairs = wl.knn_edges(spec, states, k=5)
    space = irt.make_space()
    whole = irt.SetStore(ctx, grid)
    f_all, tips_all = whole.voxelize_vertices(rb, states)
    parts = irt.SetStore(ctx, grid)
    f0, _ = parts.voxelize_vertices(rb, states[:1234])
    scratch = irt.SetStore(ctx, grid)
    f1, _ = scratch.voxelize_vertices(rb, states[1234:])
    parts.append(scratch)
    assert np.array_equal(np.r_[f0, f1], f_all)
    for a, b in zip(parts.export_csr(), whole.export_csr()):
        assert np.array_equal(a, b)
    ewhole = irt.SetStore(ctx, grid)
    i_all = ewhole.voxelize_edges_indexed(rb, space, states, pairs)
    eparts = irt.SetStore(ctx, grid)
    cut = len(pairs) // 3 + 1
    i0 = eparts.voxelize_edges_indexed(rb, space, states, pairs[:cut])
    i1 = scratch.voxelize_edges_indexed(rb, space, states, pairs[cut:])
    eparts.append(scratch)
    assert np.array_equal(np.r_[i0["flags"], i1["flags"]], i_all["flags"])
    assert np.array_equal(np.r_[i0["t_last"], i1["t_last"]], i_all["t_last"])
    for a, b in zip(eparts.export_csr(), ewhole.export_csr()):
        assert np.array_equal(a, b)


def test_argument_errors_leave_dst_unchanged(irt, ctx, grid):
    rng = np.random.default_rng(17)
    dst_csr = _random_csr(rng, rng.poisson(23, size=300))
    src_csr = _random_csr(rng, rng.poisson(23, size=200))
    dst = _store(irt, ctx, grid, dst_csr)
    src = _store(irt, ctx, grid, src_csr)
    L = ctx.L

    def unchanged():
        for a, b in zip(dst.export_csr(), dst_csr):
            assert np.array_equal(a, b)

    bad = [(ctx.h, dst.h, dst.h, 0, 10), (ctx.h, None, src.h, 0, 10), (ctx.h, dst.h, None, 0, 10),
           (None, dst.h, src.h, 0, 10), (ctx.h, dst.h, src.h, -1, 10), (ctx.h, dst.h, src.h, 0, 201),
           (ctx.h, dst.h, src.h, 11, 10), (ctx.h, dst.h, src.h, 201, 201)]
    lim = [-0.2, 0.2, -0.2, 0.2, -0.2, 0.2]
    rot = np.eye(3)
    rot[0, 0], rot[0, 1], rot[1, 0], rot[1, 1] = 0.0, -1.0, 1.0, 0.0
    for other in (irt.make_grid(64, lim), irt.make_grid(NG, lim[:5] + [0.3]), irt.make_grid(NG, lim, rot)):
        o = irt.SetStore(ctx, other)
        o.import_csr(np.zeros(201, dtype=np.uint64), np.zeros(0, dtype=np.uint32), np.zeros(0, dtype=np.uint64))
        bad.append((ctx.h, dst.h, o.h, 0, 10))
        bad.append((ctx.h, o.h, src.h, 0, 10))
    for args in bad:
        assert L.irt_setstore_append(*args, None) == irt.IRT_ERR_INVALID_ARGUMENT, args
        unchanged()
    # empty ranges and all-clear masks are no-ops
    for b in (0, 57, 200):
        dst.append(src, begin=b, end=b)
        unchanged()
    dst.append(src, keep=np.zeros(200, dtype=bool))
    unchanged()
    with pytest.raises(irt.IrtError):
        dst.append(src, keep=np.ones(199, dtype=bool))
    unchanged()
    import torch
    if torch.cuda.device_count() > 1:
        ctx1 = irt.Context(1)
        far = irt.SetStore(ctx1, grid)
        far.import_csr(*src_csr)
        assert L.irt_setstore_append(ctx.h, dst.h, far.h, 0, 10, None) == irt.IRT_ERR_INVALID_ARGUMENT
        unchanged()


def _roadmap_with_newcomers(irt, ctx, wl, R):
    spec = wl.robot_b(0.003, rotation=True)
    g = wl.workspace_grid(spec)
    grid = irt.make_grid(g["Ng"], g["lim"])
    rb = irt.Robot(ctx, spec)
    env_blocks = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    prm = R.VoxelCachedLazyPRM(ctx, rb, grid)
    prm.setEnvironment(env_blocks)
    prm.createRoadmap(400, opt=R.VoxelizeVertices)
    prm.precomputeVoxelCache()
    prm.precomputeValidity()
    rng = np.random.default_rng(23)
    nv0 = len(prm.states)
    for m in range(25):
        x = prm.states[(7 * m) % nv0].copy()
        x[:6] = np.maximum(0.0, x[:6] + rng.normal(size=6) * 0.5)
        prm.addMilestone(x)
    return prm, rb, grid, env_blocks


def test_extend_voxel_cache_python_mirror(irt, ctx, wl):
    from irt_b200 import roadmap as R
    prm, rb, grid, env_blocks = _roadmap_with_newcomers(irt, ctx, wl, R)
    nv, ne = len(prm.states), len(prm.edges)
    assert len(prm.vertex_flags) < nv and len(prm.edge_flags) < ne
    prm.nearest_tips(prm.tips[0], 5)                     # the device copy of the tips exists before the extension
    vstore, estore = prm.vertex_store, prm.edge_store
    prm.extendVoxelCache()
    assert prm.vertex_store is vstore and prm.edge_store is estore
    assert vstore.num_sets == nv and estore.num_sets == ne

    fresh = R.VoxelCachedLazyPRM(ctx, rb, grid)
    fresh.setEnvironment(env_blocks)
    fresh.set_roadmap(prm.states.copy(), prm.edges.copy())
    fresh.precomputeVoxelCache()
    for a, b in ((vstore, fresh.vertex_store), (estore, fresh.edge_store)):
        for x, y in zip(a.export_csr(), b.export_csr()):
            assert np.array_equal(x, y)
    assert np.array_equal(prm.vertex_flags, fresh.vertex_flags)
    assert np.array_equal(prm.edge_flags, fresh.edge_flags)
    assert np.array_equal(prm.tips, fresh.tips)
    assert np.array_equal(prm.edge_info["t_last"], fresh.edge_info["t_last"])
    full = (fresh.edge_flags & R.FLAG_PARTIAL) == 0
    assert np.array_equal(prm.edge_info["nsamples"][full], fresh.edge_info["nsamples"][full])
    # the k-NN copy of the tips follows
    rng = np.random.default_rng(1)
    for v in rng.integers(nv, size=20):
        req = prm.tips[v] + rng.normal(size=3) * 0.003
        d = np.linalg.norm(prm.tips - req[None], axis=1)
        assert list(prm.nearest_tips(req, 5)) == list(np.lexsort((np.arange(nv), d))[:5])

    def no_scratch(ids):
        raise AssertionError("a scratch batch ran for %d items" % len(ids))

    prm._check_vertices_now = prm._check_edges_now = no_scratch
    prm.clearValidity()
    prm.precomputeValidity()
    fresh.precomputeValidity()
    assert prm.vertex_store is vstore and prm.edge_store is estore
    assert np.array_equal(prm.vertex_validity, fresh.vertex_validity)
    assert np.array_equal(prm.edge_validity, fresh.edge_validity)


def test_extend_voxel_cache_cpp_mirror(tmp_path):
    exe = str(tmp_path / "test_extend_voxel_cache")
    pkg = os.path.join(ROOT, "interactive-rate-tendons_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", os.path.join(ROOT, "tests", "cpp", "test_extend_voxel_cache.cpp"),
                           "-o", exe, "-L" + pkg, "-lirt_b200", "-Wl,-rpath," + pkg, "-fopenmp"])
    out = subprocess.run([exe, "400"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "extend voxel cache ok" in out.stdout
