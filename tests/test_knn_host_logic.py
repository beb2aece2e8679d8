"""Host logic of the Python mirror's device k-NN path (roadmap.py: NearestSet behind createRoadmap's connection,
nearest_tips, addMilestone, roadmapIk and _ik_nearest) WITHOUT a GPU: NearestSet is replaced, in this file only, by
the numpy restatement of its contract (tests/knn_reference.py), and every result is compared with the same planner
running the host scans (ctx=None).  Checks the batched connection and its vectorised edge dedup, and that the device
copies follow the host arrays: appends, replacements, in-place tip writes and removal masks."""
import numpy as np
import pytest

from tests.knn_reference import NumpyNearestSet
from tests.test_roadmap_host_logic import _Ctx, _Env, _Robot, _Store, _dls_solver


def _pair(R, orc, wl, spec, g, oenv, monkeypatch):
    """(host planner, planner on the stand-in "device") over the same oracle-backed robot / store / environment"""
    ogrid = orc.grid(g["Ng"], g["lim"])
    monkeypatch.setattr(R, "SetStore", lambda ctx, grid: _Store(orc, ogrid))
    monkeypatch.setattr(R, "Env", lambda ctx, grid: _Env(oenv))
    monkeypatch.setattr(R, "NearestSet", NumpyNearestSet)
    monkeypatch.setattr(R, "Context", _Ctx)

    class PRM(R.VoxelCachedLazyPRM):
        def _sweep(self, store, n_total, flags):
            return store.check(self.env)

    robot = _Robot(orc, spec, wl)
    host, dev = PRM(None, robot, None), PRM(_Ctx(), robot, None)
    assert host._nn is None and dev._nn is not None
    return host, dev


def test_connection_edges_equal_the_loop():
    from irt_b200 import roadmap as R
    rng = np.random.default_rng(5)
    for trial in range(200):
        n = int(rng.integers(1, 60))
        nv0 = int(rng.integers(0, n))
        k = int(rng.integers(1, 8))
        nbr = rng.integers(-1, n, size=(n - nv0, k))
        nbr[rng.random(nbr.shape) < 0.2] = -1
        for i in range(len(nbr)):                       # self pairs, as nn_->nearestK returns them
            if rng.random() < 0.5:
                nbr[i, 0] = nv0 + i
        old = rng.integers(0, max(nv0, 1), size=(int(rng.integers(0, 20)), 2)) if nv0 else np.zeros((0, 2), np.int64)
        have = set(map(tuple, np.sort(old, axis=1).tolist()))
        want = []
        for v in range(nv0, n):
            for u in nbr[v - nv0].tolist():
                key = (min(v, u), max(v, u))
                if u >= 0 and u != v and key not in have:
                    have.add(key)
                    want.append((v, u))
        got = R.connection_edges(nbr, nv0, old, n)
        assert np.array_equal(got, np.array(want, dtype=np.int64).reshape(-1, 2)), trial


@pytest.mark.parametrize("rotation", [False, True])
def test_create_roadmap_connection_batch_equals_host_loop(orc, wl, monkeypatch, rotation):
    from irt_b200 import roadmap as R
    spec = wl.robot_b(0.003, rotation=rotation)
    g = wl.workspace_grid(spec)
    oenv = orc.octree(orc.grid(g["Ng"], g["lim"]))
    host, dev = _pair(R, orc, wl, spec, g, oenv, monkeypatch)
    prev = 0
    for n in (150, 260, 400):                           # growing keeps the prefix: the device set only appends
        sampler = lambda cnt, rnd, n=n: wl.sample_states(spec, cnt, stream=40 + n + rnd)
        host.createRoadmap(n, sampler, opt=R.LazyRoadmap)
        q0 = dev._nn["states"][0].queries
        dev.createRoadmap(n, sampler, opt=R.LazyRoadmap)
        assert np.array_equal(host.states, dev.states)
        assert np.array_equal(host.edges, dev.edges) and len(dev.edges) > n
        nn = dev._nn["states"][0]
        assert nn.queries - q0 == n - prev               # one batched query per new vertex
        assert nn.clears == 0 and nn.appended == n and nn.size() == n
        prev = n
    # a replaced roadmap is uploaded again
    dev.set_roadmap(host.states[:200], host.edges[:10])
    host.set_roadmap(host.states[:200], host.edges[:10])
    host.createRoadmap(230, lambda cnt, rnd: wl.sample_states(spec, cnt, stream=7 + rnd), opt=R.LazyRoadmap)
    dev.createRoadmap(230, lambda cnt, rnd: wl.sample_states(spec, cnt, stream=7 + rnd), opt=R.LazyRoadmap)
    assert np.array_equal(host.edges, dev.edges)
    assert dev._nn["states"][0].clears == 1 and dev._nn["states"][0].size() == 230
    # k above the device limit: the host loop answers
    dev.max_nearest_neighbors = host.max_nearest_neighbors = R.KNN_MAX_K + 1
    q0 = dev._nn["states"][0].queries
    host.createRoadmap(240, lambda cnt, rnd: wl.sample_states(spec, cnt, stream=9 + rnd), opt=R.LazyRoadmap)
    dev.createRoadmap(240, lambda cnt, rnd: wl.sample_states(spec, cnt, stream=9 + rnd), opt=R.LazyRoadmap)
    assert np.array_equal(host.edges, dev.edges) and dev._nn["states"][0].queries == q0


def test_queries_and_device_copies_follow_the_host_arrays(orc, wl, monkeypatch):
    from irt_b200 import roadmap as R
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    ogrid = orc.grid(g["Ng"], g["lim"])
    oenv = orc.octree(ogrid)
    oenv.add_sphere([0.05, 0.0, 0.12], 0.03)
    host, dev = _pair(R, orc, wl, spec, g, oenv, monkeypatch)
    for p in (host, dev):
        p.world = 1
        p.createRoadmap(120, lambda cnt, rnd: wl.sample_states(spec, cnt, stream=300 + rnd),
                        lambda st: wl.knn_edges(spec, st, k=4), opt=R.VoxelizeVertices)
        p.precomputeVoxelCache()
    tips = dev._nn["tips"][0]
    rng = np.random.default_rng(11)
    lb, ub = np.zeros(7), np.array([20.0] * 6 + [spec["L"]])
    # nearest_tips / addMilestone / _ik_nearest under removals; _ik_nearest of a roadmap state ties the temporary
    # vertex (distance 0, highest index) with that state
    for step in range(8):
        req = dev.tips[rng.integers(len(dev.tips))] + rng.normal(size=3) * 0.003
        for k in (1, 5, 17):
            assert np.array_equal(host.nearest_tips(req, k), dev.nearest_tips(req, k))
        x = np.clip(dev.states[rng.integers(len(dev.states))] + rng.normal(size=7) * 0.5, lb, ub)
        removed = rng.random(len(dev.states)) < 0.1
        for own in (-1, 3):
            for accurate in (False, True):
                assert host._ik_nearest(x, own, 7, accurate, removed) == dev._ik_nearest(x, own, 7, accurate, removed)
        assert host._ik_nearest(dev.states[4], -1, 7, True, removed) == dev._ik_nearest(dev.states[4], -1, 7, True, removed)
        host.vertex_removed[rng.integers(len(host.states))] = True
        dev.vertex_removed[:] = host.vertex_removed
        hv, hadd = host.addMilestone(x)
        dv, dadd = dev.addMilestone(x)
        assert (hv, hadd) == (dv, dadd) and np.array_equal(host.edges, dev.edges)
        assert np.array_equal(host.tips, dev.tips)
    dev.nearest_tips(req, 1)
    assert tips.clears == 1 and tips.size() == len(dev.tips)   # appends by _append_vertex reach the device as appends
    host.restoreRemoved()
    dev.restoreRemoved()
    # an in-place tip write is uploaded again before the next query
    v = 10
    for p in (host, dev):
        p.tips[v] = p.tips[20] + 1e-6
        p._replaced("tips")
    c0 = tips.clears
    req = dev.tips[20]
    assert np.array_equal(host.nearest_tips(req, 3), dev.nearest_tips(req, 3)) and tips.clears == c0 + 1
    # roadmapIk, plain / auto_add / accurate, on both
    solver = _dls_solver(lb, ub)
    for trial in range(3):
        goal = np.clip(dev.states[rng.integers(120)] + rng.normal(size=7) * [1, 1, 1, 1, 1, 1, 0.004], lb, ub)
        request = orc.fk_batch(dev.robot.orb, goal[None], 128, want_p=False)["tip"][0]
        for kw in (dict(), dict(auto_add=True), dict(auto_add=True, accurate=True)):
            a = host.roadmapIk(request, 1e-4, 4, solver, **kw)
            b = dev.roadmapIk(request, 1e-4, 4, solver, **kw)
            assert (a is None) == (b is None)
            if a is not None:
                assert np.array_equal(a["controls"], b["controls"]) and a["vertex"] == b["vertex"]
                assert np.array_equal(a["neighbors"], b["neighbors"])
            assert np.array_equal(host.states, dev.states) and np.array_equal(host.edges, dev.edges)
            assert np.array_equal(host.tips, dev.tips)
            assert np.array_equal(host.vertex_removed, dev.vertex_removed)
    # clearVertexVoxelCache drops the tips; the next query rebuilds the device copy from the new ones
    for p in (host, dev):
        p.clearVertexVoxelCache()
    assert np.array_equal(host.nearest_tips(req, 4), dev.nearest_tips(req, 4))
    assert tips.size() == len(dev.tips)
