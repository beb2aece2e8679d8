"""Times the exact k-NN path (csrc/knn.cu behind irt_b200.NearestSet) where the planner uses it, in one run:

  * createRoadmap(1_000_000) of Robot B on the 128^3 grid, phase by phase (sampling with the FK validity filter,
    connection, edge voxel cache), at k = 5 (the mirrors' default) and k = 17 (bench.py's); the connection through
    each kernel: one call over all new vertices (large-batch kernel) and calls of 63 queries (small-batch kernel,
    timed on a prefix and scaled);
  * the single-query latency of nearest_tips and addMilestone's neighbour search through the Python mirror over 1M
    vertices (median / p99 of 1000 queries, mask packing and copies included), and of the whole addMilestone call;
  * the host scans they replace on a sample of the same queries, and bench.py's torch topk generator (FP32, not
    exact) as a comparison;
  * mismatches of sampled device answers against tests/knn_reference.py (the numpy restatement of the contract).

Timings are host clocks around synchronous calls (every NearestSet call ends in a stream synchronise).  L2 is not
flushed: the 1M-row sets (24 / 56 MB) stay resident in the 126 MB L2 between queries as they do in the planner.
Usage: python tools/time_knn.py --out profiles/knn_b200.json"""
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


def stats(ts):
    ts = np.asarray(ts) * 1e3
    return dict(median_ms=float(np.median(ts)), p99_ms=float(np.percentile(ts, 99)), mean_ms=float(ts.mean()),
                n=len(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--queries", type=int, default=1000)
    ap.add_argument("--check", type=int, default=2000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import irt_b200
    import irt_b200.workloads as wl
    from irt_b200 import roadmap as R
    from tests import knn_reference as ref

    res = dict(gpu=gpu_info(), n=a.n)
    print("GPU:", res["gpu"], flush=True)
    ctx = irt_b200.Context(0)
    spec = wl.robot_b(dL=0.003)          # the dL the 128^3 grid's validity checker accepts
    rb = irt_b200.Robot(ctx, spec)
    g = wl.workspace_grid(spec)
    grid = irt_b200.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    dim, metric = irt_b200.state_metric(spec)

    # ---- createRoadmap(n) phase by phase ----
    prm = R.VoxelCachedLazyPRM(ctx, rb, grid)
    warm = R.VoxelCachedLazyPRM(ctx, rb, grid)
    warm.createRoadmap(20000, opt=R.VoxelizeVertices | R.VoxelizeEdges)          # modules, scratch, algorithms
    t0 = time.perf_counter()
    cand = prm.random_states(int(a.n * 1.25) + 64, 0)
    ok = (rb.shape_batch(cand, want=("flags",))["flags"] & irt_b200.INVALID_MASK) == 0
    states = np.ascontiguousarray(cand[ok][:a.n])
    t_sample = time.perf_counter() - t0
    assert len(states) == a.n
    bound = 0.2 * prm.maximum_extent()
    phases = {}
    for k in (5, 17):
        ns = irt_b200.NearestSet(ctx, dim, metric)
        t0 = time.perf_counter()
        ns.append(states)
        t_up = time.perf_counter() - t0
        ns.knn(states[:4096], k, bound)                                          # warm-up of this k
        t0 = time.perf_counter()
        nbr, _ = ns.knn(states, k, bound)
        t_knn = time.perf_counter() - t0
        t0 = time.perf_counter()
        edges = R.connection_edges(nbr, 0, np.zeros((0, 2), np.int64), a.n)
        t_edges = time.perf_counter() - t0
        pre = 64 * 63 * 16                                                       # 64k queries in calls of 63
        t0 = time.perf_counter()
        small = [ns.knn(states[s:s + 63], k, bound)[0] for s in range(0, pre, 63)]
        t_small = time.perf_counter() - t0
        small_eq = bool(np.array_equal(np.concatenate(small)[:pre], nbr[:pre]))
        ph = dict(upload_s=t_up, knn_large_kernel_one_call_s=t_knn, edge_list_s=t_edges,
                  connection_s=t_up + t_knn + t_edges, n_edges=int(len(edges)),
                  knn_small_kernel_calls_of_63_s_for_prefix=t_small, small_kernel_prefix_queries=pre,
                  knn_small_kernel_scaled_to_all_s=t_small * a.n / pre, small_equals_large_on_prefix=small_eq)
        if k == 5:
            store = irt_b200.SetStore(ctx, grid)
            t0 = time.perf_counter()
            store.voxelize_edges_indexed(rb, prm.space, states, edges)
            ph["edge_voxel_cache_s"] = time.perf_counter() - t0
            del store
        phases["k%d" % k] = ph
        print("k=%d" % k, json.dumps(ph), flush=True)
        if k == 5:
            nbr5, edges5 = nbr, edges
    res["create_roadmap"] = dict(sampling_s=t_sample, phases=phases)

    # ---- torch topk generator of bench.py (FP32, not exact) on the same states ----
    import torch
    import bench
    torch.cuda.synchronize()
    bench.knn_edges_gpu(torch, states[:50000], spec, 17, "cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    te = bench.knn_edges_gpu(torch, states, spec, 17, "cuda")
    torch.cuda.synchronize()
    res["torch_topk_fp32_not_exact_k17_s"] = time.perf_counter() - t0
    res["torch_topk_edges"] = int(len(te))
    del te
    torch.cuda.empty_cache()

    # ---- single queries through the Python mirror over n vertices ----
    prm.set_roadmap(states, edges5)
    prm.precomputeVertexVoxelCache()
    rng = np.random.default_rng(1)
    reqs = prm.tips[rng.integers(a.n, size=a.queries)] + rng.normal(size=(a.queries, 3)) * 0.002
    xs = np.clip(states[rng.integers(a.n, size=a.queries)] + rng.normal(size=(a.queries, dim)) * 0.2, 0, None)
    prm.vertex_removed[rng.integers(a.n, size=100)] = True
    for r in reqs[:20]:
        prm.nearest_tips(r, 5)
        prm._connection_neighbors(xs[0], prm.vertex_removed)
    tt, tm = [], []
    for r, x in zip(reqs, xs):
        t0 = time.perf_counter()
        prm.nearest_tips(r, 5)
        tt.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        prm._connection_neighbors(x, prm.vertex_removed)
        tm.append(time.perf_counter() - t0)
    res["nearest_tips_k5"] = stats(tt)
    res["addMilestone_neighbour_search_k5"] = stats(tm)
    host = R.VoxelCachedLazyPRM(ctx, rb, grid)
    host._nn = None
    host.set_roadmap(states, edges5)
    host.tips, host.vertex_removed = prm.tips, prm.vertex_removed
    host._have_vcache = True
    ht, hm = [], []
    for r, x in zip(reqs[:5], xs[:5]):
        t0 = time.perf_counter()
        host.nearest_tips(r, 5)
        ht.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        d = np.where(host.vertex_removed, np.inf, host.distance(x, host.states))
        order = np.lexsort((np.arange(len(d)), d))[:5]
        hm.append(time.perf_counter() - t0)
    res["host_nearest_tips_k5"] = stats(ht)
    res["host_addMilestone_scan_k5"] = stats(hm)
    full = []
    for x in xs[:200]:
        t0 = time.perf_counter()
        prm.addMilestone(x)
        full.append(time.perf_counter() - t0)
    res["addMilestone_whole_call"] = stats(full)
    print(json.dumps({k: res[k] for k in res if k.startswith(("nearest", "addM", "host", "torch"))}), flush=True)

    # ---- sampled check against the numpy restatement ----
    half = a.check // 2
    mism = 0
    qi = rng.choice(a.n, half, replace=False)
    for i in qi:      # the connection lists of k = 5
        wi, _ = ref.knn(states, states[i], metric, 5, bound)
        mism += int(not np.array_equal(wi[0], nbr5[i]))
    tns = irt_b200.NearestSet(ctx, 3, irt_b200.tip_metric())
    tns.append(prm.tips[:a.n])
    gi, gd = tns.knn(reqs[:half], 17)
    for j in range(min(half, len(reqs))):
        wi, wd = ref.knn(prm.tips[:a.n], reqs[j], irt_b200.tip_metric(), 17)
        mism += int(not (np.array_equal(wi[0], gi[j]) and np.array_equal(wd[0], gd[j])))
    res["sampled_check"] = dict(queries=int(half + min(half, len(reqs))), mismatches=mism)
    print("sampled check:", res["sampled_check"], flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
