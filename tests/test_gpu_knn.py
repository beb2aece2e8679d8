"""irt_nnset_* (csrc/knn.cu) on the B200 against the numpy restatement of its contract (tests/knn_reference.py): equal
indices and bit-equal distances, both kernels (small / large query batches) bit for bit, and the two host mirrors
giving the same roadmaps and query answers as their host scans."""
import os
import subprocess
import zlib

import numpy as np
import pytest

from tests import knn_reference as ref

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL_M = 64          # KNN_SMALL_M of csrc/knn.cu: batches of at least this many queries take the large-m kernel


@pytest.fixture(scope="module")
def irt():
    import irt_b200
    return irt_b200


@pytest.fixture(scope="module")
def ctx(irt):
    return irt.Context(0)


def _metrics(irt, wl):
    out = {"tips": (3, irt.tip_metric())}
    out["robot_a"] = irt.state_metric(wl.robot_a())
    out["robot_b"] = irt.state_metric(wl.robot_b())
    out["rot_ret"] = irt.state_metric(wl.robot_b(rotation=True))
    out["12_tendons"] = (12, irt.Metric(12, -1, -1, 0, 0.0, 0.0))
    return out


def _rows(rng, dim, metric, n):
    x = rng.uniform(0.0, 20.0, size=(n, dim))
    if metric.so2_col >= 0:
        x[:, metric.so2_col] = rng.uniform(-np.pi, np.pi, n)
    if metric.lin_col >= 0:
        x[:, metric.lin_col] = rng.uniform(0.0, 0.25, n)
    return x


def _check(ns, rows, q, metric, k, bound=np.inf, exclude=None):
    gi, gd = ns.knn(q, k, bound, exclude)
    wi, wd = ref.knn(rows, q, metric, k, bound, exclude)
    assert np.array_equal(gi, wi)
    assert np.array_equal(gd.view(np.uint64), wd.view(np.uint64))
    return gi


@pytest.mark.parametrize("name", ["tips", "robot_a", "robot_b", "rot_ret", "12_tendons"])
def test_knn_equals_the_contract(irt, ctx, wl, name):
    dim, metric = _metrics(irt, wl)[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    for n in (0, 1, 31, 32, 33, 1000, 200003):
        rows = _rows(rng, dim, metric, n)
        ns = irt.NearestSet(ctx, dim, metric)
        ns.append(rows)
        assert ns.size() == n
        q = _rows(rng, dim, metric, 3)
        if n:
            q[0] = rows[n // 2]                              # distance 0 to one item
        for k in (1, 5, 17, 64):
            _check(ns, rows, q, metric, k)
        mask = rng.random(n) < 0.3
        r = float(np.median(ref.distances(rows, q[1], metric))) if n else 1.0
        for bound in (np.inf, r, 0.0, -1.0):
            _check(ns, rows, q, metric, 17, bound, mask)
        _check(ns, rows, q, metric, 5, exclude=np.ones(n, dtype=bool))
        if n > 100:                                          # the large-m kernel on the same set
            _check(ns, rows, _rows(rng, dim, metric, SMALL_M + 5), metric, 17, r, mask)


def test_large_batch_equals_small_chunks(irt, ctx, wl):
    for name in ("robot_b", "rot_ret", "tips"):
        dim, metric = _metrics(irt, wl)[name]
        rng = np.random.default_rng(7)
        rows = _rows(rng, dim, metric, 50000)
        rows[1000:1100] = rows[5]                            # exact ties across tiles and slices
        ns = irt.NearestSet(ctx, dim, metric)
        ns.append(rows)
        q = np.concatenate([rows[:2000], _rows(rng, dim, metric, 1000)])
        mask = rng.random(len(rows)) < 0.05
        for k, bound in ((5, 2.0), (17, np.inf), (64, np.inf)):
            big_i, big_d = ns.knn(q, k, bound, mask)
            parts = [ns.knn(q[s:s + SMALL_M - 1], k, bound, mask) for s in range(0, len(q), SMALL_M - 1)]
            assert np.array_equal(big_i, np.concatenate([p[0] for p in parts]))
            assert np.array_equal(big_d.view(np.uint64), np.concatenate([p[1] for p in parts]).view(np.uint64))
            sample = rng.choice(len(q), 40, replace=False)
            wi, wd = ref.knn(rows, q[sample], metric, k, bound, mask)
            assert np.array_equal(big_i[sample], wi) and np.array_equal(big_d[sample], wd)


def test_exact_ties_come_out_in_index_order(irt, ctx):
    n = 300000
    rng = np.random.default_rng(3)
    metric = irt.tip_metric()
    rows = rng.uniform(-1, 1, size=(n, 3))
    p = np.array([0.25, -0.5, 0.125])
    spots = [0, 31, 32, 255, 256, 4095, 4096, 70001, 150000, 200000, n - 1]
    rows[spots] = p
    # integer lattice points at equal distance sqrt(1) / sqrt(2) from the query
    lat = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [-1, 0, 0], [0, -1, 0], [0, 0, -1], [1, 1, 0], [0, 1, 1]], float)
    lat_at = rng.choice(np.setdiff1d(np.arange(n), spots), len(lat), replace=False)
    rows[lat_at] = lat + 10.0
    ns = irt.NearestSet(ctx, 3, metric)
    ns.append(rows)
    idx = _check(ns, rows, np.stack([p, np.full(3, 10.0)]), metric, 64)
    assert list(idx[0, :len(spots)]) == spots
    for m in (1, SMALL_M + 1):                               # both kernels
        i, _ = ns.knn(np.repeat(p[None], m, axis=0), 11)
        assert np.all(i == np.array(spots))


def test_so2_wrap_and_nan_rows(irt, ctx, wl):
    dim, metric = irt.state_metric(wl.robot_b(rotation=True))
    c = metric.so2_col
    rng = np.random.default_rng(9)
    rows = _rows(rng, dim, metric, 4000)
    rows[:, :c] = 1.0
    rows[:, metric.lin_col] = 0.1
    angles = [np.pi, -np.pi, 0.0, np.nextafter(np.pi, 0), np.nextafter(0.0, 1), 1e-300]
    rows[:len(angles), c] = angles
    rows[10:20, 0] = np.nan
    rows[20:25, c] = np.nan
    rows[25, metric.lin_col] = np.inf
    ns = irt.NearestSet(ctx, dim, metric)
    ns.append(rows)
    q = rows[:8].copy()
    q[6] = rows[10]                                          # a NaN query: nothing comes back
    q[7, c] = np.nextafter(np.pi, 4)                         # dr just above pi against -pi
    for k in (5, 64):
        idx = _check(ns, rows, q, metric, k)
        assert not np.isin(idx, np.arange(10, 26)).any()
        assert np.all(idx[6] == -1)
    for m in (1, SMALL_M):
        i, d = ns.knn(np.repeat(q[:1], m, axis=0), 64)
        assert not np.isin(i, np.arange(10, 26)).any() and np.isfinite(d[i >= 0]).all()


def test_small_appends_equal_one_append(irt, ctx, wl):
    dim, metric = irt.state_metric(wl.robot_b())
    rng = np.random.default_rng(4)
    rows = _rows(rng, dim, metric, 5000)
    a = irt.NearestSet(ctx, dim, metric)
    s = 0
    while s < len(rows):
        step = int(rng.integers(1, 700))
        a.append(rows[s:s + step])
        s += step
    b = irt.NearestSet(ctx, dim, metric)
    b.append(rows[:100])
    b.clear()
    assert b.size() == 0
    b.append(rows)
    q = _rows(rng, dim, metric, 100)
    mask = rng.random(len(rows)) < 0.2
    for k in (1, 17):
        for ex in (None, mask):
            ia, da = a.knn(q, k, exclude=ex)
            ib, db = b.knn(q, k, exclude=ex)
            assert np.array_equal(ia, ib) and np.array_equal(da, db)
        _check(a, rows, q, metric, k)


def test_argument_errors(irt, ctx):
    bad = irt.IRT_ERR_INVALID_ARGUMENT
    M = irt.Metric
    for dim, m in ((0, M(1, -1, -1, 0, 0, 0)), (17, M(3, -1, -1, 0, 0, 0)), (3, M(0, -1, -1, 0, 0, 0)),
                   (3, M(4, -1, -1, 0, 0, 0)), (4, M(3, 3, 3, 0, 1, 1)), (4, M(3, 2, -1, 0, 1, 0)),
                   (4, M(3, -1, 4, 0, 0, 1)), (4, M(3, -1, -2, 0, 0, 1)), (4, M(3, 3, -1, 0, -1.0, 0)),
                   (4, M(3, -1, 3, 0, 0, np.nan)), (4, M(3, -1, 3, 0, 0, np.inf))):
        with pytest.raises(irt.IrtError) as e:
            irt.NearestSet(ctx, dim, m)
        assert e.value.status == bad
    ns = irt.NearestSet(ctx, 3, irt.tip_metric())
    ns.append(np.zeros((4, 3)))
    for k in (0, -1, irt.KNN_MAX_K + 1):
        with pytest.raises(irt.IrtError) as e:
            ns.knn(np.zeros((1, 3)), k)
        assert e.value.status == bad
    i, d = ns.knn(np.zeros((0, 3)), 5)                       # m = 0
    assert i.shape == (0, 5)
    empty = irt.NearestSet(ctx, 3, irt.tip_metric())        # n = 0: every entry is padding
    i, d = empty.knn(np.zeros((2, 3)), 3)
    assert np.all(i == -1) and np.all(np.isinf(d))


# ---- the mirrors ------------------------------------------------------------------------------------------------
def _host_twin(prm):
    """the same planner object answering every nearest-neighbour question with the host scans"""
    prm._nn = None
    return prm


def test_python_mirror_create_roadmap_equals_host_loop(irt, ctx, wl):
    from irt_b200 import roadmap as R
    spec = wl.robot_b(dL=0.003)
    rb = irt.Robot(ctx, spec)
    g = wl.workspace_grid(spec)
    grid = irt.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    dev = R.VoxelCachedLazyPRM(ctx, rb, grid)
    dev.createRoadmap(5000, opt=R.LazyRoadmap)
    host = _host_twin(R.VoxelCachedLazyPRM(ctx, rb, grid))
    host.createRoadmap(5000, sampler=lambda cnt, rnd: dev.states, opt=R.LazyRoadmap)
    assert np.array_equal(dev.states, host.states)
    assert np.array_equal(dev.edges, host.edges) and len(dev.edges) > 5000
    # widths up to 7: the device's lists are the Python mirror's own host function's
    for v in range(0, 5000, 97):
        idx, _ = dev._nn["states"][0].knn(dev.states[v], 5, dev.maximum_extent() * 0.2)
        assert np.array_equal(idx[0][idx[0] >= 0], host.k_bounded_neighbors(v))


def test_python_mirror_queries_equal_host_scans(irt, ctx, wl):
    from irt_b200 import roadmap as R
    from tests.test_roadmap_host_logic import _dls_solver
    spec = wl.robot_b(dL=0.003)
    rb = irt.Robot(ctx, spec)
    g = wl.workspace_grid(spec)
    grid = irt.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    env = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    prms = []
    for _ in range(2):
        p = R.VoxelCachedLazyPRM(ctx, rb, grid)
        p.setEnvironment(env)
        p.createRoadmap(3000, opt=R.VoxelizeVertices)
        p.precomputeVoxelCache()
        prms.append(p)
    dev, host = prms[0], _host_twin(prms[1])
    assert np.array_equal(dev.edges, host.edges)
    rng = np.random.default_rng(17)
    lb, ub = np.zeros(7), np.array([float(t) for t in spec["max_tension"][:6]] + [spec["L"]])
    solver = _dls_solver(lb, ub)
    for trial in range(4):
        goal = np.clip(dev.states[rng.integers(len(dev.states))] + rng.normal(size=7) * [1, 1, 1, 1, 1, 1, 0.004],
                       lb, ub)
        request = rb.shape_batch(goal[None], want=("tip",))["tip"][0]
        for k in (1, 5, 17):
            assert np.array_equal(dev.nearest_tips(request, k), host.nearest_tips(request, k))
        for kw in (dict(), dict(auto_add=True), dict(auto_add=True, accurate=True)):
            a = dev.roadmapIk(request, 1e-4, 4, solver, **kw)
            b = host.roadmapIk(request, 1e-4, 4, solver, **kw)
            assert (a is None) == (b is None)
            if a is not None:
                assert np.array_equal(a["controls"], b["controls"]) and a["vertex"] == b["vertex"]
        x = np.clip(goal + rng.normal(size=7) * 0.3, lb, ub)
        assert dev.addMilestone(x) == host.addMilestone(x)
        assert np.array_equal(dev.edges, host.edges) and np.array_equal(dev.states, host.states)
        for p in (dev, host):                                # removals of a search, then the reload
            p.solveWithRoadmap(0, len(p.states) - 1, max_iterations=20)
        assert np.array_equal(dev.vertex_removed, host.vertex_removed)
        assert np.array_equal(dev.edge_removed, host.edge_removed)
        if trial == 2:
            for p in (dev, host):
                p.restoreRemoved()


def test_cpp_mirror_knn(tmp_path, orc):
    exe = str(tmp_path / "test_knn_mirror")
    pkg = os.path.join(ROOT, "interactive-rate-tendons_b200")
    cmd = ["g++", "-std=c++17", "-O1", os.path.join(ROOT, "tests", "cpp", "test_knn_mirror.cpp"), "-o", exe,
           "-L" + pkg, "-lirt_b200", "-Wl,-rpath," + pkg, "-fopenmp"]
    subprocess.check_call(cmd, env=dict(os.environ, CXX="g++"))
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    print(out.stdout[-3000:], out.stderr[-2000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "knn mirror ok" in out.stdout
