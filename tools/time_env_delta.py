"""Times incremental revalidation after an environment change (irt_check_sets_changed, csrc/env_delta.cu, behind
irt_b200.SetStore.check_changed and the planners' updateEnvironment) in one run:

  * a C4-sized roadmap (Robot B, 1M vertices, k = 17: 9.5M edges) is built the way tools/time_setstore_append.py
    builds it, its vertex and edge caches voxelised, and the lung-like environment of bench.py uploaded;
  * the inverted index of each cache: build time and bytes;
  * ticks on the edge cache: blobs of 5-15 mm away from the base (bench.py's C5 tick, workloads.toggle_blob), blobs
    at the base, and changes of growing size (k random blocks replaced, up to a whole-grid replacement).  Per tick:
    changed blocks, index entries scanned (the summed list lengths of the changed keys, counted on the host from the
    exported store), sets re-checked, flips, the path taken, and the time of irt_check_sets_changed against a plain
    K3 sweep of the same range into host words plus the host diff (XOR + nonzero) that finds the flips;
  * updateEnvironment against setEnvironment + precomputeValidity (bench.py's replanning_tick_with_path
    ms_words_on_host), alternating on one planner, host clock.

Every timing is a host clock around synchronous calls (median of --reps).  The edge store (145M leaves, 1.7 GB) is far
larger than the 126 MB L2; a sweep streams it from HBM.  The delta path touches a few MB.
Usage: python tools/time_env_delta.py --out profiles/env_delta_b200.json"""
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


def median_time(fn, reps):
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--k", type=int, default=17)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ticks", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import irt_b200
    import irt_b200.workloads as wl
    from irt_b200 import roadmap as R

    res = dict(gpu=gpu_info(), n_vertices=a.n, k=a.k, reps=a.reps)
    print("GPU:", res["gpu"], flush=True)
    ctx = irt_b200.Context(0)
    spec = wl.robot_b(dL=0.003)
    rb = irt_b200.Robot(ctx, spec)
    g = wl.workspace_grid(spec)
    grid = irt_b200.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    prm = R.VoxelCachedLazyPRM(ctx, rb, grid)
    prm.max_nearest_neighbors = a.k
    prm.createRoadmap(a.n, opt=R.LazyRoadmap)
    prm.precomputeVoxelCache()
    env_blocks = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    prm.setEnvironment(env_blocks)
    Nb = g["Ng"] // 4
    res["vertex_sets"], res["edge_sets"] = prm.vertex_store.num_sets, prm.edge_store.num_sets
    res["edge_leaves"] = prm.edge_store.num_blocks
    print("roadmap: %d vertices, %d edges, %d edge leaves" % (res["vertex_sets"], res["edge_sets"], res["edge_leaves"]),
          flush=True)

    # ---- index build
    res["index"] = {}
    for name, store in (("vertex", prm.vertex_store), ("edge", prm.edge_store)):
        irt_b200.SetIndex(ctx, store).close()          # warm-up (module load, scratch growth)
        t = median_time(lambda: irt_b200.SetIndex(ctx, store).close(), 3)
        res["index"][name] = {"build_ms": t * 1e3, "sets": store.num_sets, "leaves": store.num_blocks,
                              "bytes": 12 * store.num_blocks + 8 * (Nb ** 3 + 1) + 4 * ((store.num_sets + 31) // 32)}
        print("index %s: %.2f ms, %.2f GB" % (name, t * 1e3, res["index"][name]["bytes"] / 1e9), flush=True)

    store = prm.edge_store
    ix = irt_b200.SetIndex(ctx, store)
    n = store.num_sets
    per_key = np.bincount(store.export_csr()[1], minlength=Nb ** 3).astype(np.int64)
    e_old = irt_b200.Env(ctx, grid)
    e_old.update(env_blocks)
    e_new = irt_b200.Env(ctx, grid)
    words_old = np.zeros((n + 31) // 32, dtype=np.uint32)
    ctx.check(ctx.L.irt_check_sets(ctx.h, store.h, e_old.h, 0, n, words_old.ctypes.data))

    def sweep_and_diff():
        w = np.zeros_like(words_old)
        ctx.check(ctx.L.irt_check_sets(ctx.h, store.h, e_new.h, 0, n, w.ctypes.data))
        x = np.bitwise_xor(w, words_old)
        return np.nonzero(irt_b200.unpack_verdicts(x, n))[0]

    def tick(kind, blocks):
        e_new.update(blocks)
        changed = np.nonzero(blocks != env_blocks)[0]
        out = {}
        words, flipped, stats = store.check_changed(ix, e_old, e_new, words_old.copy())   # warm-up + result
        ref = sweep_and_diff()
        assert np.array_equal(flipped, ref), "flips differ from the sweep"
        out.update(kind=kind, changed_blocks=int(stats[0]), entries_scanned=int(per_key[changed].sum()),
                   entries_over_range_leaves=float(per_key[changed].sum() / max(store.num_blocks, 1)),
                   sets_rechecked=int(stats[1]), flips=int(len(flipped)), full_sweep=bool(stats[2]))
        out["check_changed_ms"] = median_time(lambda: store.check_changed(ix, e_old, e_new, words_old.copy()),
                                              a.reps) * 1e3
        out["sweep_plus_host_diff_ms"] = median_time(sweep_and_diff, a.reps) * 1e3
        print(kind, {k: (round(v, 3) if isinstance(v, float) else v) for k, v in out.items() if k != "kind"},
              flush=True)
        return out

    rng = np.random.default_rng(wl.SEED + 5)
    ticks = []
    for _ in range(a.ticks):          # bench.py's C5 tick: a 5-15 mm blob in the workspace
        c = rng.uniform(-0.1, 0.1, 3) + np.array([0.0, 0.0, 0.1])
        ticks.append(tick("blob", wl.toggle_blob(env_blocks, g, c, rng.uniform(0.005, 0.015))))
    for _ in range(a.ticks):          # at the robot base: the block every backbone starts in
        c = np.r_[rng.uniform(-0.004, 0.004, 2), 0.0]
        ticks.append(tick("blob_at_base", wl.toggle_blob(env_blocks, g, c, rng.uniform(0.005, 0.015))))
    for k in (1, 4, 16, 64, 256, 1024, 2048, 4096, 8192, 16384, Nb ** 3):   # growing changes
        b = env_blocks.copy()
        keys = rng.choice(Nb ** 3, size=k, replace=False)
        b[keys] = rng.integers(1, 2 ** 63, size=k, dtype=np.int64).astype(np.uint64)
        ticks.append(tick("random_blocks_%d" % k, b))
    res["edge_ticks"] = ticks

    # ---- the planner: updateEnvironment against setEnvironment + precomputeValidity (host clock, alternating)
    prm.setEnvironment(env_blocks)
    prm.precomputeValidity()
    envs = []
    for _ in range(2 * a.ticks + 2):
        c = rng.uniform(-0.1, 0.1, 3) + np.array([0.0, 0.0, 0.1])
        envs.append(wl.toggle_blob(env_blocks, g, c, rng.uniform(0.005, 0.015)))
    prm.updateEnvironment(envs[0])                    # builds both indexes
    prm.setEnvironment(envs[1])
    prm.precomputeValidity()
    upd, full, nflip = [], [], []
    for i in range(a.ticks):
        t = time.perf_counter()
        ch = prm.updateEnvironment(envs[2 + 2 * i])
        upd.append(time.perf_counter() - t)
        nflip.append(len(ch["vertices"]) + len(ch["edges"]))
        t = time.perf_counter()
        prm.setEnvironment(envs[3 + 2 * i])
        prm.precomputeValidity()
        full.append(time.perf_counter() - t)
    res["planner_tick"] = {
        "update_environment_ms": float(np.median(upd)) * 1e3, "update_environment_ms_all": [x * 1e3 for x in upd],
        "set_environment_plus_precompute_validity_ms": float(np.median(full)) * 1e3,
        "set_environment_plus_precompute_validity_ms_all": [x * 1e3 for x in full],
        "flips_per_tick": nflip,
        "what": "Python mirror, 1M vertices + %d edges, blob ticks of 5-15 mm: updateEnvironment (upload, patch of "
                "both current tables) against setEnvironment + precomputeValidity (upload, both sweeps, D2H of the "
                "words, validity tables); host clock" % res["edge_sets"]}
    print(res["planner_tick"], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
