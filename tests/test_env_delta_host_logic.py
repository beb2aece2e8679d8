"""updateEnvironment of both planner mirrors WITHOUT a GPU.  The Python mirror (interactive-rate-tendons_b200/roadmap.py)
runs over the oracle-backed stand-ins of test_extend_voxel_cache_host_logic.py, extended with an environment that can
be re-uploaded, an index stand-in and SetStore.check_changed answered by re-checking the range with the oracle; the C++
mirror (host/irt_host.hpp) is linked against the test-only stand-in of the C ABI plus tests/cpp/env_delta_standin.hpp.
Over blob ticks the tables must equal a twin planner's after setEnvironment + precomputeValidity, the look-ups must
answer alike, the flips must be the items whose validity bit changed, and no sweep may be counted; tables that are not
current are reset.  The same checks run on the real library in tests/test_gpu_env_delta.py."""
import os
import subprocess

import numpy as np
import pytest

from tests.test_extend_voxel_cache_host_logic import _AppendStore, _csr
from tests.test_roadmap_host_logic import _Robot

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _DeltaEnv:
    """the oracle octree behind Env, re-uploadable from Morton-ordered dense blocks"""

    def __init__(self, orc, ogrid, wl, oenv=None):
        self.orc, self.ogrid, self.wl = orc, ogrid, wl
        self.oenv = oenv if oenv is not None else orc.octree(ogrid)

    def update(self, blocks):
        blocks = np.asarray(blocks, dtype=np.uint64)
        Nb = round(len(blocks) ** (1 / 3))
        t = self.orc.octree(self.ogrid)
        for k in np.nonzero(blocks)[0]:
            bx, by, bz = self.wl.morton_decode(int(k), Nb)
            t.set_block(int(bx), int(by), int(bz), int(blocks[k]))
        self.oenv = t


class _Index:
    """the index stand-in: a copy of the sets it covers (a store whose first sets differ from it is stale)"""

    def __init__(self, ctx, store):
        self.store = store
        self.csr = [np.array(a) for a in _csr(store)]
        self.num_sets = len(self.csr[0]) - 1
        store.indexes = getattr(store, "indexes", 0) + 1

    def close(self):
        pass


class _DeltaStore(_AppendStore):
    def check_changed(self, index, env_old, env_new, words, begin=0, end=None):
        end = self.num_sets if end is None else end
        assert index.store is self
        off, keys, bits = _csr(self)
        n_ix = index.num_sets
        assert np.array_equal(off[:n_ix + 1], index.csr[0]), "stale index"
        assert np.array_equal(keys[:int(off[n_ix])], index.csr[1]) and np.array_equal(bits[:int(off[n_ix])], index.csr[2])
        old = np.unpackbits(np.asarray(words, dtype=np.uint32).view(np.uint8), count=end - begin, bitorder="little")
        new = self.check(env_new, begin, end).astype(np.uint8)
        b = np.zeros(len(words) * 32, dtype=np.uint8)
        b[:end - begin] = new
        words[:] = np.packbits(b, bitorder="little").view(np.uint32)
        return words, begin + np.nonzero(old != new)[0].astype(np.int64), np.array([0, end - begin, 1])


def _planner(R, orc, wl, spec, g, env_now, monkeypatch):
    from irt_b200 import pack_mask
    ogrid = orc.grid(g["Ng"], g["lim"])
    monkeypatch.setattr(R, "SetStore", lambda ctx, grid: _DeltaStore(orc, ogrid))
    monkeypatch.setattr(R, "SetIndex", _Index)
    monkeypatch.setattr(R, "Env", lambda ctx, grid: _DeltaEnv(orc, ogrid, wl))

    class PRM(R.VoxelCachedLazyPRM):
        def _sweep(self, store, n_total, flags):
            collides = store.check(self.env)
            self._swept_words = pack_mask(collides) if len(collides) else np.zeros(0, np.uint32)
            return collides

    prm = PRM(None, _Robot(orc, spec, wl), None)
    prm.world = 1
    prm.env.update(env_now)
    return prm


def test_update_environment_python_mirror(orc, wl, monkeypatch):
    from irt_b200 import roadmap as R
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    base = orc.octree(orc.grid(g["Ng"], g["lim"]))
    base.add_sphere([0.05, 0.0, 0.12], 0.03)
    env = base.dense_morton()
    prm = _planner(R, orc, wl, spec, g, env, monkeypatch)
    prm.createRoadmap(80, lambda cnt, rnd: wl.sample_states(spec, cnt, stream=2100 + rnd),
                      lambda st: wl.knn_edges(spec, st, k=5), opt=R.VoxelizeVertices)
    prm.precomputeVoxelCache()
    prm.precomputeValidity()
    rng = np.random.default_rng(7)
    flips_seen = 0
    for t in range(8):
        kind = t % 6     # as in tests/cpp/test_env_delta_mirror.cpp
        nv0, ne0 = len(prm.states), len(prm.edges)
        if kind == 2:
            x = prm.states[t % nv0].copy()
            x[0] += 0.3
            prm.addMilestone(x)
        elif kind == 3:
            x = prm.states[(3 * t) % nv0].copy()
            x[1] += 0.4
            prm.addMilestone(x)
            prm.extendVoxelCache()
        elif kind == 4:
            prm.clearValidity()
        elif kind == 5:
            builds = prm.vertex_store.calls
            prm.precomputeVoxelCache()
            assert prm.vertex_store.calls == builds + 1
        c = (np.r_[rng.uniform(-0.005, 0.005, 2), 0.0] if kind == 1 else
             rng.uniform(-0.1, 0.1, 3) + np.array([0.0, 0.0, 0.1]))
        env = wl.toggle_blob(env, g, c, rng.uniform(0.005, 0.015))
        vold, eold = prm.vertex_validity.copy(), prm.edge_validity.copy()
        sweeps = prm.lookups["sweeps"]
        indexes = (getattr(prm.vertex_store, "indexes", 0), getattr(prm.edge_store, "indexes", 0))
        ch = prm.updateEnvironment(env)
        assert prm.lookups["sweeps"] == sweeps
        if kind == 5:    # the caches were rebuilt: so are their indexes
            assert (prm.vertex_store.indexes, prm.edge_store.indexes) == (indexes[0] + 1, indexes[1] + 1)
        elif t > 0 and kind != 4:
            assert (prm.vertex_store.indexes, prm.edge_store.indexes) == indexes, "the indexes were reused"
        twin = _planner(R, orc, wl, spec, g, env, monkeypatch)
        twin.set_roadmap(prm.states.copy(), prm.edges.copy())
        twin.precomputeVoxelCache()
        twin.setEnvironment(env)
        if kind == 4:    # not current: reset like setEnvironment
            assert not len(ch["vertices"]) and not len(ch["edges"])
            assert np.array_equal(prm.vertex_validity, twin.vertex_validity)
            assert np.array_equal(prm.edge_validity, twin.edge_validity)
        twin.precomputeValidity()
        if kind != 4:
            vskip = np.arange(len(prm.states)) >= nv0       # this tick's milestones: still unchecked
            eskip = np.arange(len(prm.edges)) >= ne0
            assert set(prm._vertex_unchecked) == set(np.nonzero(vskip)[0].tolist())
            assert np.array_equal(prm.vertex_validity[~vskip], twin.vertex_validity[~vskip])
            assert np.array_equal(prm.edge_validity[~eskip], twin.edge_validity[~eskip])
            assert np.array_equal(ch["vertices"], np.nonzero(vold != prm.vertex_validity)[0])
            assert np.array_equal(ch["edges"], np.nonzero(eold != prm.edge_validity)[0])
            flips_seen += len(ch["vertices"]) + len(ch["edges"])
        for v in range(len(prm.states)):
            assert prm.computeVertexValidity(v) == twin.computeVertexValidity(v)
        for e in range(len(prm.edges)):
            assert prm.computeEdgeValidity(e) == twin.computeEdgeValidity(e)
        if kind == 4:
            prm.precomputeValidity()
    assert flips_seen > 0
    # the index follows the cache: a cleared cache drops it, the next update builds it again
    prm.clearEdgeVoxelCache()
    assert prm._index["edge"] is None
    prm.updateEnvironment(env)
    assert prm._index["edge"] is not None and prm._index["edge"][1] is prm.edge_store
    # a tail past max_uncached makes the index be rebuilt
    prm.max_uncached = 0
    for m in range(2):
        x = prm.states[m].copy()
        x[2] += 0.2
        prm.addMilestone(x)
    prm.extendVoxelCache()
    prm.precomputeValidity()
    old_ix = prm._index["vertex"][0]
    prm.updateEnvironment(env)
    assert prm._index["vertex"][0] is not old_ix and prm._index["vertex"][0].num_sets == len(prm.states)
    prm.world = 2
    with pytest.raises(NotImplementedError):
        prm.updateEnvironment(env)


def test_update_environment_cpp_mirror(tmp_path, orc):
    exe = str(tmp_path / "test_env_delta_mirror")
    cpp = os.path.join(ROOT, "tests", "cpp")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-DIRT_TEST_OVER_STANDIN",
                           os.path.join(cpp, "test_env_delta_mirror.cpp"),
                           os.path.join(cpp, "abi_standin_over_oracle.cpp"), "-o", exe,
                           "-L" + os.path.join(ROOT, "oracle"), "-loracle",
                           "-Wl,-rpath," + os.path.join(ROOT, "oracle"), "-fopenmp"])
    out = subprocess.run([exe, "60", "12"], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "env delta mirror ok" in out.stdout
