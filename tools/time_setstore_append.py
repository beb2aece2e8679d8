"""Times irt_setstore_append (csrc/voxel_check.cu behind irt_b200.SetStore.append) and extendVoxelCache in one run:

  * a C4-sized roadmap (Robot B, 1M vertices) is built by the planner's createRoadmap at k = 17 (9.5M edges; the
    edge generator of bench.py gives ~10.09M) and its edge cache voxelised (K1 + K2, also timed: the rebuild an append
    avoids);
  * the 2.56M edge sets of a createRoadmap(1M) k = 5 increment (real edge sets: the first 2.56M of the C4 store) are
    appended onto the C4 store, repeatedly onto the same growing store, with no mask and with a random 90 % keep mask;
    appends that had to grow the store's arrays (amortised x1.5, content copied) are reported apart from those that
    did not;
  * a 4096-set tail appended the same way;
  * extendVoxelCache for a tail of 4096 edges that joined the C4 roadmap after its cache was built, against the
    precomputeEdgeVoxelCache rebuild it replaces.

GB/s is over the bytes an append must move: 2 x 12 B per kept leaf (key + bits, read and written) + 8 B per set
(its offset).  Timings are host clocks around synchronous calls (every append ends in a stream synchronise).  The
stores are far larger than the 126 MB L2, so nothing is served from a warm cache except the 4096-set tail.
Usage: python tools/time_setstore_append.py --out profiles/setstore_append_b200.json"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn):
    t = time.perf_counter()
    fn()
    return time.perf_counter() - t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--k", type=int, default=17)
    ap.add_argument("--increment", type=int, default=2_560_000)
    ap.add_argument("--tail", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import irt_b200
    import irt_b200.workloads as wl
    from irt_b200 import roadmap as R

    res = dict(gpu=gpu_info(), n_vertices=a.n, k=a.k)
    print("GPU:", res["gpu"], flush=True)
    ctx = irt_b200.Context(0)
    spec = wl.robot_b(dL=0.003)
    rb = irt_b200.Robot(ctx, spec)
    g = wl.workspace_grid(spec)
    grid = irt_b200.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    prm = R.VoxelCachedLazyPRM(ctx, rb, grid)
    prm.max_nearest_neighbors = a.k
    prm.createRoadmap(a.n, opt=R.LazyRoadmap)
    prm.precomputeEdgeVoxelCache()                     # warm-up of K1 + K2 at this size
    res["rebuild_s"] = [timed(prm.precomputeEdgeVoxelCache) for _ in range(2)]
    c4 = prm.edge_store
    res["c4_sets"], res["c4_leaves"] = c4.num_sets, c4.num_blocks
    print("C4 store: %d sets, %d leaves (%.2f per set); rebuild %s s" % (
        c4.num_sets, c4.num_blocks, c4.num_blocks / c4.num_sets, res["rebuild_s"]), flush=True)

    c4_off = c4.export_csr()[0].astype(np.int64)
    inc = irt_b200.SetStore(ctx, grid)
    inc.append(c4, end=min(a.increment, c4.num_sets))
    tail = irt_b200.SetStore(ctx, grid)
    tail.append(c4, end=a.tail)

    def grow(cap, need):                               # the store's amortised growth (setstore_grow_*)
        return cap if need <= cap else max(cap + cap // 2, need)

    rng = np.random.default_rng(7)
    for name, src, mask in (("increment", inc, False), ("increment_keep90", inc, True), ("tail", tail, False)):
        n = src.num_sets
        keep = (rng.random(n) < 0.9) if mask else None
        per = np.diff(c4_off[:n + 1])                  # src holds the first n sets of the C4 store
        kept_sets, kept_leaves = (n, int(per.sum())) if keep is None else (int(keep.sum()), int(per[keep].sum()))
        nbytes = 24 * kept_leaves + 8 * kept_sets
        dst = irt_b200.SetStore(ctx, grid)
        dst.append(c4)                                 # arrays of exactly the C4 store's size
        cap_s, cap_b = c4.num_sets + 1, c4.num_blocks + 4
        grew, steady = [], []
        for r in range(a.reps + 1):
            ns, nb = dst.num_sets + kept_sets + 1, dst.num_blocks + kept_leaves + 4
            t = timed(lambda: dst.append(src, keep=keep))
            grows = grow(cap_s, ns) != cap_s or grow(cap_b, nb) != cap_b
            cap_s, cap_b = grow(cap_s, ns), grow(cap_b, nb)
            if r > 0:                                  # the first call is the warm-up
                (grew if grows else steady).append(t)
        del dst
        row = dict(sets=n, kept_sets=kept_sets, kept_leaves=kept_leaves, bytes=nbytes, steady_s=steady, grew_s=grew)
        if steady:
            row["steady_gbps"] = nbytes / float(np.median(steady)) / 1e9
        res[name] = row
        print(name, json.dumps(row), flush=True)

    # extendVoxelCache: a tail of edges between existing vertices that the cache lacks
    prm.precomputeVertexVoxelCache()
    ext = []
    for rep in range(3):
        nn = prm._nearest_set("states", 8)
        v = rng.integers(len(prm.states), size=a.tail)
        idx, _ = nn.knn(prm.states[v], 8, np.inf)
        pairs = np.stack([v, idx[:, 7]], axis=1)
        prm._append_edges(pairs, R.VALIDITY_UNKNOWN)
        ext.append(timed(prm.extendVoxelCache))
        assert prm.edge_store.num_sets == len(prm.edges)
    res["extend_tail_s"] = ext
    print("extendVoxelCache(%d edges): %s s; rebuild %s s" % (a.tail, ext, res["rebuild_s"]), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
