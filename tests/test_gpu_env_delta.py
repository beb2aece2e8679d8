"""irt_check_sets_changed and irt_setindex (csrc/env_delta.cu) on the B200: after every call the words equal, bit for
bit, irt_check_sets against the new grid, and the flip list is exactly the XOR of the old and new words -- synthetic
stores and the real vertex / edge sets of a K2-voxelised roadmap; single bits, blobs mid-workspace and at the robot
base, adds only, removes only, keys 0 and Nb^3 - 1, empty sets, unaligned ranges, identical grids, a whole-grid
replacement (the full-sweep path) and a one-block change (the delta path), an index with appended tail sets, and every
argument and capacity error with the words unchanged.  Then updateEnvironment of both planner mirrors over 20 blob
ticks against a twin planner that calls setEnvironment + precomputeValidity."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NG = 128
NB = NG // 4
NKEYS = NB ** 3
LIM = [-0.2, 0.2, -0.2, 0.2, -0.2, 0.2]


@pytest.fixture(scope="module")
def irt():
    import irt_b200
    return irt_b200


@pytest.fixture(scope="module")
def ctx(irt):
    return irt.Context(0)


@pytest.fixture(scope="module")
def grid(irt):
    return irt.make_grid(NG, LIM)


def _random_csr(rng, sizes):
    """CSR with sets of the given leaf counts: strictly increasing Morton keys, random non-zero bits"""
    sizes = np.asarray(sizes, dtype=np.int64)
    off = np.zeros(len(sizes) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(sizes)
    keys, bits = [], []
    for s in sizes:
        keys.append(np.sort(rng.choice(NKEYS, size=int(s), replace=False)).astype(np.uint32))
        bits.append(rng.integers(1, 2 ** 63, size=int(s), dtype=np.int64).astype(np.uint64)
                    & rng.integers(0, 2 ** 63, size=int(s), dtype=np.int64).astype(np.uint64) | np.uint64(1))
    return off, np.concatenate(keys + [np.zeros(0, np.uint32)]), np.concatenate(bits + [np.zeros(0, np.uint64)])


def _store(irt, ctx, grid, csr):
    s = irt.SetStore(ctx, grid)
    s.import_csr(*csr)
    return s


def _env(irt, ctx, grid, blocks):
    e = irt.Env(ctx, grid)
    e.update(blocks)
    return e


def _words(ctx, store, env, begin, end):
    w = np.zeros(max((end - begin + 31) // 32, 1), dtype=np.uint32)
    ctx.check(ctx.L.irt_check_sets(ctx.h, store.h, env.h, begin, end, w.ctypes.data))
    return w


def _call(irt, ctx, store, ix, eo, en, words, begin, end, cap=1 << 20, flipped=True):
    w = words.copy()
    fl = np.zeros(max(cap, 1), dtype=np.int64)
    nf = C.c_int64(-1)
    stats = np.full(3, -1, dtype=np.int64)
    rc = ctx.L.irt_check_sets_changed(ctx.h, store.h, ix.h if ix is not None else None, eo.h if eo else None,
                                      en.h if en else None, begin, end, w.ctypes.data,
                                      fl.ctypes.data if flipped else None, cap, C.byref(nf), stats.ctypes.data)
    return rc, w, fl[:max(nf.value, 0)], stats


def _assert_exact(irt, ctx, store, ix, eo, en, begin=0, end=None, path=None):
    """the contract: words of env_new bit for bit, flips = XOR of old and new, ascending"""
    end = store.num_sets if end is None else end
    n = end - begin
    old = _words(ctx, store, eo, begin, end)
    new = _words(ctx, store, en, begin, end)
    rc, w, fl, stats = _call(irt, ctx, store, ix, eo, en, old, begin, end)
    assert rc == 0, ctx.L.irt_last_error(ctx.h)
    assert np.array_equal(w[:(n + 31) // 32], new[:(n + 31) // 32])
    x = irt.unpack_verdicts(old, n) != irt.unpack_verdicts(new, n)
    assert np.array_equal(fl, begin + np.nonzero(x)[0])
    if path is not None:
        assert stats[2] == path, stats
    return fl, stats


def _sparse_env(rng, density=0.05):
    b = np.zeros(NKEYS, dtype=np.uint64)
    k = rng.choice(NKEYS, size=int(NKEYS * density), replace=False)
    b[k] = rng.integers(1, 2 ** 63, size=len(k), dtype=np.int64).astype(np.uint64)
    return b


def _blob(blocks, center, radius):
    import irt_b200.workloads as wl
    return wl.toggle_blob(blocks, {"Ng": NG, "lim": LIM}, np.asarray(center, dtype=np.float64), radius)


def test_synthetic_changes(irt, ctx, grid):
    rng = np.random.default_rng(1)
    sizes = rng.integers(0, 60, size=5003)
    sizes[[0, 17, 5002]] = 0                        # empty sets, also at the ends
    csr = _random_csr(rng, sizes)
    store = _store(irt, ctx, grid, csr)
    ix = irt.SetIndex(ctx, store)
    assert ix.num_sets == 5003
    base = _sparse_env(rng, 0.3)
    eo = _env(irt, ctx, grid, base)
    hot = int(np.bincount(csr[1], minlength=NKEYS).argmax())

    def with_blocks(b):
        return _env(irt, ctx, grid, b)

    cases = []
    b = base.copy(); b[hot] ^= np.uint64(1) << np.uint64(int(rng.integers(64))); cases.append(("one bit", b, 0))
    cases.append(("blob mid", _blob(base, [0.03, -0.02, 0.05], 0.012), None))
    cases.append(("blob corner", _blob(base, [-0.19, -0.19, -0.19], 0.015), None))
    b = base.copy(); nz = np.nonzero(b)[0][:200]; b[nz] = np.uint64(0); cases.append(("removes only", b, None))
    b = base.copy(); z = np.nonzero(b == 0)[0][:200]; b[z] = np.uint64(0xFFFFFFFFFFFFFFFF); cases.append(("adds only", b, None))
    b = base.copy(); b[0] ^= np.uint64(0xF0F0); b[NKEYS - 1] ^= np.uint64(0x8000000000000001); cases.append(("ends", b, None))
    b = base.copy(); b[hot] = ~b[hot]; cases.append(("one block", b, 0))
    cases.append(("whole grid", _sparse_env(rng, 0.5), 1))
    for name, blocks, path in cases:
        en = with_blocks(blocks)
        for begin, end in ((0, 5003), (13, 4001), (0, 1), (4970, 5003)):
            _assert_exact(irt, ctx, store, ix, eo, en, begin, end, path if (begin, end) == (0, 5003) else None)
        # and back: the other direction of the same change
        _assert_exact(irt, ctx, store, ix, en, eo)
    # identical grids: no-op, no flips, nothing re-checked
    same = with_blocks(base)
    for a, b_ in ((eo, eo), (eo, same)):
        fl, stats = _assert_exact(irt, ctx, store, ix, a, b_)
        assert len(fl) == 0 and stats[0] == 0 and stats[1] == 0 and stats[2] == 0
    # the candidate bitmap is left clear: a second identical call gives the same answer
    en = with_blocks(_blob(base, [0.0, 0.0, 0.0], 0.015))
    f1, s1 = _assert_exact(irt, ctx, store, ix, eo, en)
    f2, s2 = _assert_exact(irt, ctx, store, ix, eo, en)
    assert np.array_equal(f1, f2) and np.array_equal(s1, s2)


def test_tail_sets_appended_after_the_index(irt, ctx, grid):
    rng = np.random.default_rng(2)
    store = _store(irt, ctx, grid, _random_csr(rng, rng.integers(1, 40, size=3000)))
    ix = irt.SetIndex(ctx, store)
    more = _store(irt, ctx, grid, _random_csr(rng, rng.integers(0, 40, size=201)))
    store.append(more)
    assert store.num_sets == 3201 and ix.num_sets == 3000
    base = _sparse_env(rng, 0.3)
    eo = _env(irt, ctx, grid, base)
    for c in ([0.0, 0.0, 0.0], [0.1, 0.05, -0.1]):
        en = _env(irt, ctx, grid, _blob(base, c, 0.014))
        fl, stats = _assert_exact(irt, ctx, store, ix, eo, en, path=0)
        assert stats[1] >= 201                       # every tail set is re-checked
        _assert_exact(irt, ctx, store, ix, eo, en, 2990, 3100)
        _assert_exact(irt, ctx, store, ix, eo, en, 3100, 3201)


def test_real_roadmap_sets(irt, ctx, wl):
    from irt_b200 import roadmap as R
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    grid = irt.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    prm = R.VoxelCachedLazyPRM(ctx, irt.Robot(ctx, spec), grid)
    prm.createRoadmap(3000, opt=R.LazyRoadmap)
    prm.precomputeVoxelCache()
    base = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    eo = _env(irt, ctx, grid, base)
    rng = np.random.default_rng(3)
    flips = 0
    for store in (prm.vertex_store, prm.edge_store):
        ix = irt.SetIndex(ctx, store)
        for i in range(12):
            at_base = i % 3 == 0
            c = (np.r_[rng.uniform(-0.004, 0.004, 2), 0.0] if at_base else
                 rng.uniform(-0.1, 0.1, 3) + np.array([0.0, 0.0, 0.1]))
            en = _env(irt, ctx, grid, wl.toggle_blob(base, g, c, rng.uniform(0.005, 0.015)))
            fl, _ = _assert_exact(irt, ctx, store, ix, eo, en)
            flips += len(fl)
        full = rng.integers(1, 2 ** 63, size=base.size, dtype=np.int64).astype(np.uint64)   # every block changes
        _assert_exact(irt, ctx, store, ix, eo, _env(irt, ctx, grid, full), path=1)
    assert flips > 0


def test_argument_and_capacity_errors_leave_words_unchanged(irt, ctx, grid):
    rng = np.random.default_rng(4)
    store = _store(irt, ctx, grid, _random_csr(rng, rng.integers(1, 40, size=1000)))
    other = _store(irt, ctx, grid, _random_csr(rng, rng.integers(1, 40, size=1000)))
    ix, ix_other = irt.SetIndex(ctx, store), irt.SetIndex(ctx, other)
    base = _sparse_env(rng, 0.3)
    eo = _env(irt, ctx, grid, base)
    en = _env(irt, ctx, grid, _sparse_env(rng, 0.3))
    g2 = irt.make_grid(NG, [-0.3, 0.3, -0.2, 0.2, -0.2, 0.2])
    e_other_grid = _env(irt, ctx, g2, base)
    g64 = irt.make_grid(64, LIM)
    s64 = _store(irt, ctx, g64, (np.zeros(3, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint64)))
    ix64 = irt.SetIndex(ctx, s64)
    old = _words(ctx, store, eo, 0, 1000)
    INV, CAP = irt.IRT_ERR_INVALID_ARGUMENT, irt.IRT_ERR_CAPACITY
    bad = [
        (store, None, eo, en, 0, 1000), (store, ix, None, en, 0, 1000), (store, ix, eo, None, 0, 1000),
        (store, ix, eo, e_other_grid, 0, 1000), (store, ix, e_other_grid, en, 0, 1000),
        (store, ix, eo, en, -1, 1000), (store, ix, eo, en, 0, 1001), (store, ix, eo, en, 500, 499),
        (store, ix_other, eo, en, 0, 1000), (s64, ix64, eo, en, 0, 2),
    ]
    for st, x, a, b, lo, hi in bad:
        rc, w, _, _ = _call(irt, ctx, st, x, a, b, old, lo, hi)
        assert rc == INV, (lo, hi)
        assert np.array_equal(w, old)
    rc = ctx.L.irt_check_sets_changed(None, store.h, ix.h, eo.h, en.h, 0, 1000, old.ctypes.data, None, 0, None, None)
    assert rc == INV
    rc, w, _, _ = _call(irt, ctx, store, ix, eo, en, old, 0, 1000, cap=-1)
    assert rc == INV and np.array_equal(w, old)
    # capacity: the number needed comes back, the words stay; with room the same call succeeds
    n_need = int(np.count_nonzero(irt.unpack_verdicts(old, 1000) != irt.unpack_verdicts(_words(ctx, store, en, 0, 1000), 1000)))
    assert n_need > 2
    w = old.copy()
    nf = C.c_int64(0)
    fl = np.zeros(2, dtype=np.int64)
    rc = ctx.L.irt_check_sets_changed(ctx.h, store.h, ix.h, eo.h, en.h, 0, 1000, w.ctypes.data, fl.ctypes.data, 2,
                                      C.byref(nf), None)
    assert rc == CAP and nf.value == n_need and np.array_equal(w, old)
    words, flipped, stats = store.check_changed(ix, eo, en, old.copy())      # the binding grows its buffer
    assert len(flipped) == n_need and np.array_equal(words, _words(ctx, store, en, 0, 1000))
    # without a flip list there is no capacity limit
    rc, w, _, _ = _call(irt, ctx, store, ix, eo, en, old, 0, 1000, cap=0, flipped=False)
    assert rc == 0 and np.array_equal(w, _words(ctx, store, en, 0, 1000))
    # a stale index: the store's content was replaced after the build (append keeps it valid)
    store.append(other, end=10)
    _assert_exact(irt, ctx, store, ix, eo, en)
    store.import_csr(*_random_csr(rng, rng.integers(1, 40, size=1000)))
    old = _words(ctx, store, eo, 0, 1000)
    rc, w, _, _ = _call(irt, ctx, store, ix, eo, en, old, 0, 1000)
    assert rc == INV and np.array_equal(w, old)
    _assert_exact(irt, ctx, store, irt.SetIndex(ctx, store), eo, en)


def _roadmap(irt, ctx, wl, R, n):
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    grid = irt.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    rb = irt.Robot(ctx, spec)
    prm = R.VoxelCachedLazyPRM(ctx, rb, grid)
    prm.createRoadmap(n, opt=R.VoxelizeVertices)
    return prm, rb, grid, g, spec


def test_update_environment_python_mirror(irt, ctx, wl):
    from irt_b200 import roadmap as R
    prm, rb, grid, g, spec = _roadmap(irt, ctx, wl, R, 2000)
    env = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    prm.setEnvironment(env)
    prm.precomputeVoxelCache()
    prm.precomputeValidity()
    rng = np.random.default_rng(6)
    flips = 0
    for t in range(20):
        nv0, ne0 = len(prm.states), len(prm.edges)
        if t % 5 == 2:                               # a milestone joins (unchecked tail)
            x = prm.states[t].copy()
            x[0] += 0.3
            prm.addMilestone(x)
        c = (np.r_[rng.uniform(-0.004, 0.004, 2), 0.0] if t % 4 == 1 else
             rng.uniform(-0.1, 0.1, 3) + np.array([0.0, 0.0, 0.1]))
        env = wl.toggle_blob(env, g, c, rng.uniform(0.005, 0.015))
        vold, eold = prm.vertex_validity.copy(), prm.edge_validity.copy()
        sweeps = prm.lookups["sweeps"]
        ch = prm.updateEnvironment(env)
        assert prm.lookups["sweeps"] == sweeps
        twin = R.VoxelCachedLazyPRM(ctx, rb, grid)
        twin.set_roadmap(prm.states.copy(), prm.edges.copy())
        twin.precomputeVoxelCache()
        twin.setEnvironment(env)
        twin.precomputeValidity()
        vk, ek = np.arange(len(prm.states)) < nv0, np.arange(len(prm.edges)) < ne0
        assert np.array_equal(prm.vertex_validity[vk], twin.vertex_validity[vk])
        assert np.array_equal(prm.edge_validity[ek], twin.edge_validity[ek])
        assert np.array_equal(ch["vertices"], np.nonzero(vold != prm.vertex_validity)[0])
        assert np.array_equal(ch["edges"], np.nonzero(eold != prm.edge_validity)[0])
        flips += len(ch["vertices"]) + len(ch["edges"])
        for v in range(len(prm.states)):
            assert prm.computeVertexValidity(v) == twin.computeVertexValidity(v)
        for e in range(len(prm.edges)):
            assert prm.computeEdgeValidity(e) == twin.computeEdgeValidity(e)
    assert flips > 0


def test_update_environment_cpp_mirror(tmp_path):
    exe = str(tmp_path / "test_env_delta_mirror")
    pkg = os.path.join(ROOT, "interactive-rate-tendons_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", os.path.join(ROOT, "tests", "cpp", "test_env_delta_mirror.cpp"),
                           "-o", exe, "-L" + pkg, "-lirt_b200", "-Wl,-rpath," + pkg, "-fopenmp"])
    out = subprocess.run([exe, "400", "20"], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "env delta mirror ok" in out.stdout
