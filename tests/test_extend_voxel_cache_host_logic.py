"""extendVoxelCache of both planner mirrors WITHOUT a GPU.  The Python mirror (interactive-rate-tendons_b200/roadmap.py)
runs over oracle-backed stand-ins of Robot / SetStore / Env whose store can append (concatenating the oracle's sets);
the C++ mirror (host/irt_host.hpp) is linked against the test-only stand-in of the C ABI plus
tests/cpp/setstore_append_standin.hpp.  After addMilestone has added vertices and lazy edges, extending the caches must
give the sets, flags, edge info and tips of a fresh planner's precompute*VoxelCache, voxelise only the newcomers, and
leave the next sweep one pass over the caches with no scratch batch and no rebuild.  The same checks run on the real
library in tests/test_gpu_setstore_append.py."""
import os
import subprocess

import numpy as np
import pytest

from tests.test_roadmap_host_logic import _Env, _Robot, _Store

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _AppendStore(_Store):
    """the oracle-backed store stand-in, plus append: a new oracle store holding this store's sets, then the kept
    sets of the source range"""

    def append(self, src, keep=None, begin=0, end=None):
        end = src.num_sets if end is None else end
        picked = [begin + i for i in range(end - begin) if keep is None or keep[i]]
        out = self.orc.setstore(self.ogrid, self.num_sets + len(picked))
        for i in range(self.num_sets):
            out.get(i).add_voxels(self.store.get(i))
        for j, s in enumerate(picked):
            out.get(self.num_sets + j).add_voxels(src.store.get(s))
        self.store = out


def _csr(store):
    return store.store.export() if store.store is not None else (np.zeros(1, np.uint64), [], [])


def _planner(R, orc, wl, spec, g, oenv, monkeypatch):
    ogrid = orc.grid(g["Ng"], g["lim"])
    made = []

    def make_store(ctx, grid):
        made.append(_AppendStore(orc, ogrid))
        return made[-1]

    monkeypatch.setattr(R, "SetStore", make_store)
    monkeypatch.setattr(R, "Env", lambda ctx, grid: _Env(oenv))

    class PRM(R.VoxelCachedLazyPRM):
        def _sweep(self, store, n_total, flags):
            assert store.num_sets == n_total
            return store.check(self.env)

    prm = PRM(None, _Robot(orc, spec, wl), None)
    prm.world = 1
    return prm, made


def test_extend_voxel_cache_python_mirror(orc, wl, monkeypatch):
    from irt_b200 import roadmap as R
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    oenv = orc.octree(orc.grid(g["Ng"], g["lim"]))
    oenv.add_sphere([0.05, 0.0, 0.12], 0.03)
    prm, made = _planner(R, orc, wl, spec, g, oenv, monkeypatch)
    prm.createRoadmap(120, lambda cnt, rnd: wl.sample_states(spec, cnt, stream=1700 + rnd),
                      lambda st: wl.knn_edges(spec, st, k=5), opt=R.VoxelizeVertices)
    prm.precomputeVoxelCache()
    prm.precomputeValidity()
    nv0, ne0 = len(prm.states), len(prm.edges)
    rng = np.random.default_rng(3)
    for m in range(10):
        x = prm.states[(3 * m) % nv0].copy()
        x[:6] = np.maximum(0.0, x[:6] + rng.normal(size=6) * 0.5)
        prm.addMilestone(x)
    nv, ne = len(prm.states), len(prm.edges)
    assert nv > nv0 and ne > ne0
    assert prm._tail(prm.vertex_flags, nv) == nv - nv0 and prm._tail(prm.edge_flags, ne) == ne - ne0
    vstore, estore = prm.vertex_store, prm.edge_store
    calls = (vstore.calls, estore.calls)
    validity = (prm.vertex_validity.copy(), prm.edge_validity.copy())
    unchecked = (set(prm._vertex_unchecked), set(prm._edge_unchecked))
    n_made = len(made)

    prm.extendVoxelCache()
    assert prm.vertex_store is vstore and prm.edge_store is estore
    assert (vstore.calls, estore.calls) == calls, "the cached stores were appended to, not rebuilt"
    scratch = made[n_made:]
    assert len(scratch) == 2 and scratch[0].num_sets == nv - nv0 and scratch[1].num_sets == ne - ne0
    assert prm._tail(prm.vertex_flags, nv) == 0 and prm._tail(prm.edge_flags, ne) == 0
    assert np.array_equal(prm.vertex_validity, validity[0]) and np.array_equal(prm.edge_validity, validity[1])
    assert (prm._vertex_unchecked, prm._edge_unchecked) == unchecked

    fresh, _ = _planner(R, orc, wl, spec, g, oenv, monkeypatch)
    fresh.set_roadmap(prm.states.copy(), prm.edges.copy())
    fresh.precomputeVoxelCache()
    for a, b in ((prm.vertex_store, fresh.vertex_store), (prm.edge_store, fresh.edge_store)):
        for x, y in zip(_csr(a), _csr(b)):
            assert np.array_equal(x, y)
    assert np.array_equal(prm.vertex_flags, fresh.vertex_flags)
    assert np.array_equal(prm.edge_flags, fresh.edge_flags)
    assert prm.edge_info["flags"] is prm.edge_flags
    assert np.array_equal(prm.edge_info["t_last"], fresh.edge_info["t_last"])
    full = (fresh.edge_flags & R.FLAG_PARTIAL) == 0
    assert np.array_equal(prm.edge_info["nsamples"][full], fresh.edge_info["nsamples"][full])
    assert np.array_equal(prm.tips, fresh.tips)

    # the next sweep: every item from the caches, no scratch batch, no rebuild, the fresh planner's tables
    def no_scratch(ids):
        raise AssertionError("a scratch batch ran for %d items" % len(ids))

    prm._check_vertices_now = prm._check_edges_now = no_scratch
    prm.clearValidity()
    prm.precomputeValidity()
    fresh.precomputeValidity()
    assert (vstore.calls, estore.calls) == calls
    assert np.array_equal(prm.vertex_validity, fresh.vertex_validity)
    assert np.array_equal(prm.edge_validity, fresh.edge_validity)

    # nothing left to extend: nothing is voxelised; a cleared cache is built whole
    n_made = len(made)
    prm.extendVoxelCache()
    assert len(made) == n_made and (vstore.calls, estore.calls) == calls
    prm.clearEdgeVoxelCache()
    prm.extendVoxelCache()
    assert prm.edge_store.calls == 1 and np.array_equal(prm.edge_flags, fresh.edge_flags)

    prm.world = 2
    with pytest.raises(NotImplementedError):
        prm.extendVoxelCache()


def test_extend_voxel_cache_cpp_mirror(tmp_path, orc):
    exe = str(tmp_path / "test_extend_voxel_cache")
    cpp = os.path.join(ROOT, "tests", "cpp")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-DIRT_TEST_OVER_STANDIN",
                           os.path.join(cpp, "test_extend_voxel_cache.cpp"),
                           os.path.join(cpp, "abi_standin_over_oracle.cpp"), "-o", exe,
                           "-L" + os.path.join(ROOT, "oracle"), "-loracle",
                           "-Wl,-rpath," + os.path.join(ROOT, "oracle"), "-fopenmp"])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "extend voxel cache ok" in out.stdout
