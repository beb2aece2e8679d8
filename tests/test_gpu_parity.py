"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on identical
seeded inputs.  Bars (BASELINE.json north_star): backbone points within 1e-9 relative;
flags, voxel sets and collision verdicts bit-exact (flips counted and required to be zero here).
"""
import numpy as np
import pytest

from tests.test_fk_precision_vectors import TOL_P_REL

pytestmark = pytest.mark.gpu

FK_REL_TOL = 1e-9  # relative to the backbone length L (north_star tolerance)


@pytest.fixture(scope="module")
def irt():
    import irt_b200
    return irt_b200


@pytest.fixture(scope="module")
def ctx(irt):
    return irt.Context(0)


def _fk_compare(irt, ctx, orc, spec, states, want_all=False):
    rb = irt.Robot(ctx, spec)
    want = ("p", "R", "t", "npts", "L", "L_i", "tip", "uv", "flags", "iters", "nsteps") if want_all \
        else ("p", "npts", "L_i", "tip", "flags")
    out = rb.shape_batch(states, want=want)
    ref = orc.fk_batch(orc.robot(spec), states, rb.max_points)
    assert np.array_equal(out["npts"], ref["npts"])
    L = spec["L"]
    err = np.abs(out["p"] - ref["p"]).max() / L
    assert err < FK_REL_TOL, "backbone points differ by %g L" % err
    assert np.abs(out["L_i"] - ref["L_i"]).max() / L < FK_REL_TOL
    assert np.abs(out["tip"] - ref["tip"]).max() / L < FK_REL_TOL
    assert np.array_equal(out["flags"], ref["flags"])
    if want_all:
        assert np.array_equal(out["iters"], ref["iters"])
        assert np.array_equal(out["nsteps"], ref["nsteps"])
    return rb, out, ref


@pytest.mark.parametrize("robot,dL,rot", [("a", 0.005, False), ("a", 0.003, False),
                                          ("b", 0.005, False), ("b", 0.003, False),
                                          ("b", 0.005, True)])
def test_fk_parity(irt, ctx, orc, wl, robot, dL, rot):
    spec = wl.robot_a(dL) if robot == "a" else wl.robot_b(dL, rotation=rot)
    states = wl.sample_states(spec, 3000, stream=31)
    _fk_compare(irt, ctx, orc, spec, states, want_all=True)


def test_fk_full_tendon_result(irt, ctx, orc, wl):
    """every TendonResult member (t, p, R, L, L_i, u_i, u_f, v_i, v_f, converged)"""
    spec = wl.robot_b(0.005, rotation=True)
    states = wl.sample_states(spec, 64, stream=32)
    rb = irt.Robot(ctx, spec)
    out = rb.shape_batch(states, want=("p", "R", "t", "npts", "L", "L_i", "uv", "flags"))
    orb = orc.robot(spec)
    for i in range(64):
        s = orc.shape(orb, states[i])
        n = len(s["t"])
        assert out["npts"][i] == n
        assert np.allclose(out["t"][i, :n], s["t"], atol=1e-15)
        assert np.abs(out["p"][i, :n] - s["p"]).max() < FK_REL_TOL * spec["L"]
        assert np.abs(out["R"][i, :n] - s["R"]).max() < 1e-9
        assert abs(out["L"][i] - s["L"]) < FK_REL_TOL * spec["L"]
        uv = out["uv"][i]
        for got, want in ((uv[0:3], s["u_i"]), (uv[3:6], s["u_f"]), (uv[6:9], s["v_i"]), (uv[9:12], s["v_f"])):
            assert np.allclose(got, want, rtol=1e-9, atol=1e-10)
        assert bool(out["flags"][i] & irt.FLAG_NONCONVERGED) == (not s["converged"])
        assert np.all(out["p"][i, n:] == 0)  # padding rows are zero


def test_fk_other_tendon_counts(irt, ctx, orc, wl):
    """1, 2, 3, 5, 7, 8 and 12 tendons, mixed straight / helical / quadratic routing"""
    base = wl.robot_b(0.005)
    for n_t in (1, 2, 3, 5, 7, 8, 12):
        spec = dict(base)
        spec["C"] = [[0.4 * k, (-1) ** k * 9.0, 20.0 * (k % 2)] for k in range(n_t)]
        spec["D"] = [[0.008 + 0.0005 * k, 0.01 * (k % 3)] for k in range(n_t)]
        spec["max_tension"] = [20.0] * n_t
        spec["min_length"] = [-1.0] * n_t   # general routing: home lengths are unsupported
        spec["max_length"] = [1.0] * n_t    # (reference UB), keep the limits out of play
        states = wl.sample_states(spec, 300, stream=33 + n_t)
        rb = irt.Robot(ctx, spec)
        out = rb.shape_batch(states, want=("p", "npts", "L_i"))
        ref = orc.fk_batch(orc.robot(spec), states, rb.max_points)
        assert np.array_equal(out["npts"], ref["npts"])
        assert np.abs(out["p"] - ref["p"]).max() < FK_REL_TOL * spec["L"]
        assert np.abs(out["L_i"] - ref["L_i"]).max() < FK_REL_TOL * spec["L"]


def test_fk_edge_cases(irt, ctx, orc, wl):
    spec = wl.robot_b(0.005)
    rb = irt.Robot(ctx, spec)
    L = spec["L"]
    tau = [3.0, 7.5, 1.0, 0.0, 12.0, 4.0]
    # s == L, s > L, K == 0 (L - dL/2 < s < L), exact node, two-step and one-step first gaps, s = 0
    ss = [L, L + 0.05, 0.199, 0.1975, 0.195, 0.0131, 0.0169, 0.0, 1e-300]
    states = np.array([tau + [s] for s in ss])
    _fk_compare(irt, ctx, orc, spec, states, want_all=True)
    out = rb.shape_batch(states, want=("p", "npts", "flags"))
    assert out["npts"][0] == 1 and out["npts"][1] == 1 and out["npts"][2] == 1
    # a base slightly before 0 (what the reference's finite-difference Jacobians evaluate): same grid
    # size, longer first gap -- integrated like the reference does
    neg = np.array([tau + [s] for s in (-1e-7, -1e-4, -0.0005, -0.0014, -0.002, -0.00249)])
    _fk_compare(irt, ctx, orc, spec, neg, want_all=True)
    # NaN, or so far before 0 that the grid would not fit max_points: BAD_STATE, no points
    bad = rb.shape_batch(np.array([tau + [-0.0026], tau + [-0.01], tau + [-1e30], tau + [float("nan")]]),
                         want=("p", "npts", "flags"))
    assert np.all(bad["flags"] & irt.FLAG_BAD_STATE) and np.all(bad["npts"] == 0)
    # zero tension
    z = rb.shape_batch(np.array([[0.0] * 6 + [0.05]]), want=("p", "npts", "t"))
    n = z["npts"][0]
    assert np.all(z["p"][0, :n, :2] == 0) and np.allclose(z["p"][0, :n, 2], z["t"][0, :n] - 0.05, atol=1e-15)
    # empty batch
    e = rb.shape_batch(np.zeros((0, 7)))
    assert e["p"].shape[0] == 0
    # error convention (TendonRobot.h:107-109 -> std::invalid_argument)
    with pytest.raises(irt.IrtError) as ei:
        rb.shape_batch(np.zeros((4, 6)))
    assert ei.value.status == irt.IRT_ERR_INVALID_ARGUMENT
    with pytest.raises(irt.IrtError) as ei:
        rb.shape_batch(np.zeros((4, 7)), cap_pts=8)
    assert ei.value.status == irt.IRT_ERR_CAPACITY


def test_fk_self_collision_and_limits(irt, ctx, orc, wl):
    """a softer backbone curls enough to self-collide; flags must agree bit for bit"""
    spec = wl.robot_a(0.005)
    spec["E"] = 1.0e6
    states = wl.sample_states(spec, 4000, stream=35)
    rb, out, ref = _fk_compare(irt, ctx, orc, spec, states)
    assert (ref["flags"] & irt.FLAG_SELF_COLLISION).sum() > 20, "fixture must exercise self-collision"
    assert (ref["flags"] & irt.FLAG_LENGTH_LIMIT).sum() > 20
    spec = wl.robot_b(0.003)
    spec["E"] = 1.4e6  # also exercises non-convergence and the 1000-iteration cap
    states = wl.sample_states(spec, 4000, stream=36)
    _, _, ref = _fk_compare(irt, ctx, orc, spec, states, want_all=True)
    assert (ref["flags"] & irt.FLAG_NONCONVERGED).sum() > 50 and ref["iters"].max() == 1000


def test_fk_device_resident_matches_host_api(irt, ctx, wl):
    torch = pytest.importorskip("torch")
    spec = wl.robot_b(0.005)
    rb = irt.Robot(ctx, spec)
    n = 5000
    states = wl.sample_states(spec, n, stream=37)
    host = rb.shape_batch(states, want=("p", "npts", "flags"))
    d_states = torch.from_numpy(states).cuda()
    d = dict(p=torch.zeros(n, rb.max_points, 3, dtype=torch.float64, device="cuda"),
             npts=torch.zeros(n, dtype=torch.int32, device="cuda"),
             flags=torch.zeros(n, dtype=torch.int32, device="cuda"))
    rb.shape_batch_dev(d_states, n, d)
    ctx.synchronize()
    assert np.array_equal(d["p"].cpu().numpy(), host["p"])
    assert np.array_equal(d["npts"].cpu().numpy(), host["npts"])
    assert np.array_equal(d["flags"].cpu().numpy().view(np.uint32), host["flags"])


# ---------------------------------------------------------------------------------------------
# K2 vertex mode
# ---------------------------------------------------------------------------------------------
def _csr_flips(got, want):
    """number of differing voxels between two CSR stores (0 when bit-exact)"""
    go, gk, gb = got
    wo, wk, wb = want
    if np.array_equal(go, wo) and np.array_equal(gk, wk) and np.array_equal(gb, wb):
        return 0
    flips = 0
    for i in range(len(wo) - 1):
        a = dict(zip(gk[int(go[i]):int(go[i + 1])].tolist(), gb[int(go[i]):int(go[i + 1])].tolist()))
        b = dict(zip(wk[int(wo[i]):int(wo[i + 1])].tolist(), wb[int(wo[i]):int(wo[i + 1])].tolist()))
        for k in set(a) | set(b):
            flips += bin(a.get(k, 0) ^ b.get(k, 0)).count("1")
    return max(flips, 1)


@pytest.mark.parametrize("robot,rotated", [("a", False), ("b", False), ("b", True)])
def test_vertex_voxel_sets_bit_exact(irt, ctx, orc, wl, robot, rotated):
    spec = wl.robot_a(0.003) if robot == "a" else wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    inv_rot = np.eye(3)
    if rotated:
        c, s = np.cos(0.3), np.sin(0.3)
        inv_rot = np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]]) @ np.array([[1, 0, 0], [0, c, -s], [0, s, c]])
    states = wl.sample_states(spec, 3000, stream=41)
    rb = irt.Robot(ctx, spec)
    store = irt.SetStore(ctx, irt.make_grid(g["Ng"], g["lim"], inv_rot))
    flags, tips = store.voxelize_vertices(rb, states)
    ogrid = orc.grid(g["Ng"], g["lim"], inv_rot)
    ostore, oflags = orc.voxelize_vertices_batch(orc.robot(spec), ogrid, states)
    assert np.array_equal(flags, oflags)
    assert _csr_flips(store.export_csr(), ostore.export()) == 0
    ref = orc.fk_batch(orc.robot(spec), states, rb.max_points, want_p=False)
    assert np.abs(tips - ref["tip"]).max() < FK_REL_TOL * spec["L"]
    assert store.num_sets == 3000 and store.num_blocks == int(ostore.export()[0][-1])


def test_vertex_voxel_sets_invalid_and_empty(irt, ctx, orc, wl):
    spec = wl.robot_a(0.003)
    spec["E"] = 1.0e6  # many invalid shapes -> empty sets + flags
    g = wl.workspace_grid(spec)
    grid = irt.make_grid(g["Ng"], g["lim"])
    states = wl.sample_states(spec, 1500, stream=42)
    rb = irt.Robot(ctx, spec)
    store = irt.SetStore(ctx, grid)
    flags, _ = store.voxelize_vertices(rb, states)
    ostore, oflags = orc.voxelize_vertices_batch(orc.robot(spec), orc.grid(g["Ng"], g["lim"]), states)
    assert np.array_equal(flags, oflags) and (flags != 0).sum() > 50
    assert _csr_flips(store.export_csr(), ostore.export()) == 0
    off = store.export_csr()[0]
    assert np.all((off[1:] - off[:-1])[flags != 0] == 0)
    # empty batch
    store.voxelize_vertices(rb, np.zeros((0, 4)))
    assert store.num_sets == 0 and store.num_blocks == 0
    # dL coarser than the voxels: VoxelBackboneValidityChecker ctor throws std::invalid_argument
    coarse = irt.Robot(ctx, wl.robot_a(0.005))
    with pytest.raises(irt.IrtError) as ei:
        store.voxelize_vertices(coarse, wl.sample_states(wl.robot_a(0.005), 4))
    assert ei.value.status == irt.IRT_ERR_INVALID_ARGUMENT


# ---------------------------------------------------------------------------------------------
# K2 edge mode
# ---------------------------------------------------------------------------------------------
def _edges(wl, spec, n_vertices, k, stream, max_edges):
    states = wl.sample_states(spec, n_vertices, stream=stream)
    pairs = wl.knn_edges(spec, states, k=k)[:max_edges]
    return states[pairs[:, 0]].copy(), states[pairs[:, 1]].copy()


@pytest.mark.parametrize("robot", ["a", "b", "brot"])
def test_edge_swept_volumes_bit_exact(irt, ctx, orc, wl, robot):
    spec = {"a": wl.robot_a(0.003), "b": wl.robot_b(0.003), "brot": wl.robot_b(0.003, rotation=True)}[robot]
    g = wl.workspace_grid(spec)
    a, b = _edges(wl, spec, 400, 4, 51, 600)
    rb = irt.Robot(ctx, spec)
    store = irt.SetStore(ctx, irt.make_grid(g["Ng"], g["lim"]))
    info = store.voxelize_edges(rb, irt.make_space(), a, b)
    ostore, oinfo = orc.voxelize_edges_batch(orc.robot(spec), orc.grid(g["Ng"], g["lim"]), orc.space(), a, b)
    assert np.array_equal(info["flags"], oinfo["flags"])
    assert np.array_equal(info["t_last"], oinfo["t_last"])
    fully = (oinfo["flags"] & irt.FLAG_PARTIAL) == 0
    # below the first invalid t the sample set equals the reference's depth-first one, so for
    # fully valid edges even the FK-sample count must agree
    assert np.array_equal(info["nsamples"][fully], oinfo["nsamples"][fully])
    assert _csr_flips(store.export_csr(), ostore.export()) == 0
    assert info["nsamples"].mean() > 2.5, "fixture must exercise the bisection"


def test_edge_partial_validity(irt, ctx, orc, wl):
    """edges that run into invalid configurations: PARTIAL flag, t_last and the voxels of the
    valid prefix agree with the reference's LIFO order"""
    spec = wl.robot_a(0.003)
    spec["E"] = 1.4e6
    g = wl.workspace_grid(spec)
    a, b = _edges(wl, spec, 300, 4, 52, 500)
    rb = irt.Robot(ctx, spec)
    store = irt.SetStore(ctx, irt.make_grid(g["Ng"], g["lim"]))
    info = store.voxelize_edges(rb, irt.make_space(), a, b)
    ostore, oinfo = orc.voxelize_edges_batch(orc.robot(spec), orc.grid(g["Ng"], g["lim"]), orc.space(), a, b)
    assert (oinfo["flags"] & irt.FLAG_PARTIAL).sum() > 20, "fixture must contain partial edges"
    assert np.array_equal(info["flags"], oinfo["flags"])
    assert np.array_equal(info["t_last"], oinfo["t_last"])
    assert _csr_flips(store.export_csr(), ostore.export()) == 0
    assert np.all(info["nsamples"] >= oinfo["nsamples"])  # level-synchronous order may add samples past t*


def test_edge_degenerate_inputs(irt, ctx, orc, wl):
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    rb = irt.Robot(ctx, spec)
    store = irt.SetStore(ctx, irt.make_grid(g["Ng"], g["lim"]))
    x = wl.sample_states(spec, 3, stream=53)
    a = np.stack([x[0], x[1], x[2]])
    b = np.stack([x[0], x[1] + 1e-9, x[2]])  # identical endpoints: nseg = 0 -> threshold = inf
    info = store.voxelize_edges(rb, irt.make_space(), a, b)
    ostore, oinfo = orc.voxelize_edges_batch(orc.robot(spec), orc.grid(g["Ng"], g["lim"]), orc.space(), a, b)
    assert np.array_equal(info["nsamples"], oinfo["nsamples"]) and np.all(info["nsamples"] == 2)
    assert _csr_flips(store.export_csr(), ostore.export()) == 0
    store.voxelize_edges(rb, irt.make_space(), np.zeros((0, 7)), np.zeros((0, 7)))
    assert store.num_sets == 0
    assert rb.valid_segment_count(irt.make_space(), x[0], x[1]) == orc.valid_segment_count(
        orc.robot(spec), orc.space(), x[0], x[1])


# ---------------------------------------------------------------------------------------------
# K3
# ---------------------------------------------------------------------------------------------
def _oracle_env(orc, wl, ogrid, env_blocks, Nb):
    oenv = orc.octree(ogrid)
    nz = np.nonzero(env_blocks)[0]
    bx, by, bz = wl.morton_decode(nz.astype(np.uint32), Nb)
    for x, y, z, k in zip(bx.tolist(), by.tolist(), bz.tolist(), nz.tolist()):
        oenv.set_block(x, y, z, int(env_blocks[k]))
    return oenv


def test_check_sets_vs_tree_recursion(irt, ctx, orc, wl):
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    Nb = g["Ng"] // 4
    grid = irt.make_grid(g["Ng"], g["lim"])
    ogrid = orc.grid(g["Ng"], g["lim"])
    states = wl.sample_states(spec, 6000, stream=61)
    ostore, _ = orc.voxelize_vertices_batch(orc.robot(spec), ogrid, states)
    env_blocks = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    frac = np.count_nonzero(env_blocks) / env_blocks.size
    assert 0.005 < frac < 0.2
    oenv = _oracle_env(orc, wl, ogrid, env_blocks, Nb)
    want = orc.check_sets_batch(ostore, oenv).astype(bool)
    assert 0.02 < want.mean() < 0.98, "fixture must mix colliding and free sets"
    # device store imported from the oracle's CSR (the .rmp-style import path)
    store = irt.SetStore(ctx, grid)
    off, keys, bits = ostore.export()
    store.import_csr(off, keys, bits)
    env = irt.Env(ctx, grid)
    env.update(env_blocks)
    assert env.nblocks() == np.count_nonzero(env_blocks) == oenv.nblocks()
    got = store.check(env)
    assert np.array_equal(got, want)
    # ragged sub-ranges (heads/tails not multiple of 4 leaves or 32 sets)
    for lo, hi in ((0, 1), (1, 2), (5, 37), (33, 4097), (5999, 6000), (100, 100)):
        assert np.array_equal(store.check(env, lo, hi), want[lo:hi])
    # popcount checksum against numpy
    vox, hits = store.popcount(env)
    x = bits & env_blocks[keys]
    assert hits == int(np.count_nonzero(x))
    assert vox == int(sum(bin(int(v)).count("1") for v in x[x != 0]))
    # round trip
    o2, k2, b2 = store.export_csr()
    assert np.array_equal(o2, off) and np.array_equal(k2, keys) and np.array_equal(b2, bits)
    # sparse environment upload (visit_leaves style) gives the same verdicts
    bxyz, ebits = oenv.export()
    env2 = irt.Env(ctx, grid)
    env2.update_sparse(bxyz, ebits)
    assert np.array_equal(store.check(env2), want)
    # algorithmic bytes formula of SURVEY 8(d)
    assert store.algorithmic_bytes() == 12 * len(keys) + 8 * 6000 + 8 * Nb ** 3 + (6000 + 7) // 8


def test_check_sets_edge_cases(irt, ctx, wl):
    g = dict(Ng=16, lim=[0, 1, 0, 1, 0, 1])
    grid = irt.make_grid(g["Ng"], g["lim"])
    store = irt.SetStore(ctx, grid)
    env = irt.Env(ctx, grid)
    Nb = 4
    blocks = np.zeros(Nb ** 3, dtype=np.uint64)
    blocks[5] = 1 << 63
    blocks[63] = 1
    env.update(blocks)
    # sets: empty, hit on high bit, miss on same block, hit in last block, empty, zero-bits leaf
    off = np.array([0, 0, 1, 2, 4, 4, 5], dtype=np.uint64)
    keys = np.array([5, 5, 10, 63, 63], dtype=np.uint32)
    bits = np.array([1 << 63, 1 << 62, 7, 3, 0], dtype=np.uint64)
    store.import_csr(off, keys, bits)
    assert store.check(env).tolist() == [False, True, False, True, False, False]
    env.update(np.zeros(Nb ** 3, dtype=np.uint64))
    assert not store.check(env).any()
    env.update(np.full(Nb ** 3, 2 ** 64 - 1, dtype=np.uint64))
    assert store.check(env).tolist() == [False, True, True, True, False, False]
    # empty store
    store.import_csr(np.zeros(1, dtype=np.uint64), np.zeros(0, dtype=np.uint32), np.zeros(0, dtype=np.uint64))
    assert store.check(env).size == 0
    # grid-size mismatch -> std::invalid_argument (VoxelOctree.cpp:46-53)
    env32 = irt.Env(ctx, irt.make_grid(32, g["lim"]))
    store.import_csr(off, keys, bits)
    with pytest.raises(irt.IrtError) as ei:
        store.check(env32)
    assert ei.value.status == irt.IRT_ERR_INVALID_ARGUMENT
    # key outside the grid is rejected at import
    with pytest.raises(irt.IrtError):
        store.import_csr(np.array([0, 1], dtype=np.uint64), np.array([64], dtype=np.uint32),
                         np.array([1], dtype=np.uint64))


def test_check_sets_other_grid_sizes(irt, ctx, wl):
    """Ng = 4 (single leaf) up to 512 (occupancy bitmap too large for shared memory)"""
    rng = np.random.default_rng(7)
    for Ng in (4, 8, 64, 256, 512):
        Nb = Ng // 4
        grid = irt.make_grid(Ng, [0, 1, 0, 1, 0, 1])
        nkeys = Nb ** 3
        env_blocks = np.zeros(nkeys, dtype=np.uint64)
        occ = rng.choice(nkeys, size=max(1, nkeys // 20), replace=False)
        env_blocks[occ] = rng.integers(1, 2 ** 63, size=len(occ), dtype=np.uint64)
        n_sets = 500
        sizes = rng.integers(0, min(30, nkeys) + 1, size=n_sets)
        off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
        keys = np.concatenate([np.sort(rng.choice(nkeys, size=s, replace=False)) for s in sizes] + [np.zeros(0, dtype=np.int64)]).astype(np.uint32)
        bits = rng.integers(1, 2 ** 63, size=len(keys), dtype=np.uint64)
        want = np.array([np.any(bits[int(off[i]):int(off[i + 1])] & env_blocks[keys[int(off[i]):int(off[i + 1])]])
                         for i in range(n_sets)])
        store = irt.SetStore(ctx, grid)
        store.import_csr(off, keys, bits)
        env = irt.Env(ctx, grid)
        env.update(env_blocks)
        assert np.array_equal(store.check(env), want), Ng


# ---------------------------------------------------------------------------------------------
# size-independent properties at BASELINE.json's full sizes
# ---------------------------------------------------------------------------------------------
def test_full_size_fk_properties(irt, ctx, wl):
    """1M configurations (config C2): rotation equivariance and zero-tension home shape"""
    spec = wl.robot_b(0.005, rotation=True)
    rb = irt.Robot(ctx, spec)
    n = 1 << 20
    st = wl.sample_states(spec, n, stream=71)
    st0 = st.copy()
    st0[:, 6] = 0.0
    a = rb.shape_batch(st, want=("tip", "npts", "L_i"))
    b = rb.shape_batch(st0, want=("tip", "npts", "L_i"))
    c, s = np.cos(st[:, 6]), np.sin(st[:, 6])
    rot = np.stack([c * b["tip"][:, 0] - s * b["tip"][:, 1], s * b["tip"][:, 0] + c * b["tip"][:, 1], b["tip"][:, 2]], axis=1)
    assert np.abs(a["tip"] - rot).max() < 1e-12
    assert np.array_equal(a["npts"], b["npts"]) and np.array_equal(a["L_i"], b["L_i"])
    # tip never farther than the unretracted length; node count follows the retraction
    assert np.all(np.linalg.norm(a["tip"], axis=1) <= spec["L"] - st[:, 7] + 1e-9)
    k = np.floor((spec["L"] - st[:, 7]) / spec["dL"] - 0.5).astype(int) + 2
    assert np.abs(a["npts"] - k).max() <= 1
    z = st.copy()
    z[:, :6] = 0.0
    h = rb.shape_batch(z, want=("tip", "L_i", "npts"))
    m = h["npts"] > 1  # L - dL/2 < s < L gives the reference's single-point grid {s}: nothing integrated
    assert np.abs(np.linalg.norm(h["tip"], axis=1) - (spec["L"] - st[:, 7]))[m].max() < 1e-12
    assert np.abs(h["L_i"] - rb.home_lengths(z))[m].max() < 1e-12
    assert np.all(h["tip"][~m] == 0)


def test_full_size_check_properties(irt, ctx, wl):
    """10M synthetic sets (config C4 scale): monotonicity in the environment, idempotence,
    all-ones / all-zeros environments, checksum of checksums"""
    rng = np.random.default_rng(8)
    Ng, Nb = 128, 32
    grid = irt.make_grid(Ng, [-0.21, 0.21] * 3)
    n_sets = 2_000_000
    sizes = rng.integers(5, 60, size=n_sets)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    nb = int(off[-1])
    keys = rng.integers(0, Nb ** 3, size=nb, dtype=np.uint32)
    bits = rng.integers(1, 2 ** 63, size=nb, dtype=np.uint64)
    store = irt.SetStore(ctx, grid)
    store.import_csr(off, keys, bits)
    env = irt.Env(ctx, grid)
    e1 = np.zeros(Nb ** 3, dtype=np.uint64)
    occ = rng.choice(Nb ** 3, size=Nb ** 3 // 25, replace=False)
    e1[occ] = rng.integers(1, 2 ** 62, size=len(occ), dtype=np.uint64)
    e2 = e1.copy()
    more = rng.choice(Nb ** 3, size=Nb ** 3 // 25, replace=False)
    e2[more] |= rng.integers(1, 2 ** 62, size=len(more), dtype=np.uint64)
    env.update(e1)
    v1 = store.check(env)
    assert np.array_equal(v1, store.check(env))            # idempotent
    vox, hits = store.popcount(env)
    x = bits & e1[keys]
    assert hits == int(np.count_nonzero(x))                 # checksum of checksums
    seg = np.add.reduceat((x != 0).astype(np.int64), off[:-1].astype(np.int64))
    assert np.array_equal(v1, seg > 0)
    env.update(e2)
    v2 = store.check(env)
    assert np.all(v2 | ~v1)                                 # env1 subset env2 -> v1 implies v2
    env.update(np.zeros(Nb ** 3, dtype=np.uint64))
    assert not store.check(env).any()
    env.update(np.full(Nb ** 3, 2 ** 64 - 1, dtype=np.uint64))
    assert store.check(env).all()


def test_edge_indexed_form_matches_per_edge_form(irt, ctx, orc, wl):
    """edges given as (source, target) vertex indices share the endpoints' FK; results must be
    identical to the per-edge (a, b) form and to the oracle"""
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    states = wl.sample_states(spec, 500, stream=54)
    pairs = wl.knn_edges(spec, states, k=4)[:900]
    rb = irt.Robot(ctx, spec)
    grid = irt.make_grid(g["Ng"], g["lim"])
    s1, s2 = irt.SetStore(ctx, grid), irt.SetStore(ctx, grid)
    i1 = s1.voxelize_edges(rb, irt.make_space(), states[pairs[:, 0]], states[pairs[:, 1]])
    i2 = s2.voxelize_edges_indexed(rb, irt.make_space(), states, pairs)
    for k in ("flags", "t_last", "nsamples"):
        assert np.array_equal(i1[k], i2[k]), k
    assert _csr_flips(s1.export_csr(), s2.export_csr()) == 0
    ostore, oinfo = orc.voxelize_edges_batch(orc.robot(spec), orc.grid(g["Ng"], g["lim"]), orc.space(),
                                             states[pairs[:, 0]], states[pairs[:, 1]])
    assert _csr_flips(s2.export_csr(), ostore.export()) == 0
    with pytest.raises(irt.IrtError) as ei:
        s2.voxelize_edges_indexed(rb, irt.make_space(), states, np.array([[0, 500]]))
    assert ei.value.status == irt.IRT_ERR_OUT_OF_RANGE
    s2.voxelize_edges_indexed(rb, irt.make_space(), states, np.zeros((0, 2), dtype=np.int64))
    assert s2.num_sets == 0


def test_edge_until_invalid_matches_oracle(irt, ctx, orc, wl):
    """voxelize_until_invalid: bisection stops at the first sample whose backbone hits the
    environment; PARTIAL flag, last valid t and the voxels of the valid prefix are bit-exact"""
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    Nb = g["Ng"] // 4
    a, b = _edges(wl, spec, 150, 3, 55, 220)
    env_blocks = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    grid = irt.make_grid(g["Ng"], g["lim"])
    ogrid = orc.grid(g["Ng"], g["lim"])
    oenv = _oracle_env(orc, wl, ogrid, env_blocks, Nb)
    env = irt.Env(ctx, grid)
    env.update(env_blocks)
    rb = irt.Robot(ctx, spec)
    store = irt.SetStore(ctx, grid)
    info = store.voxelize_edges_until_invalid(rb, irt.make_space(), a, b, env)
    got_off, got_keys, got_bits = store.export_csr()
    orb = orc.robot(spec)
    n_partial = 0
    for i in range(len(a)):
        tree, oi = orc.voxelize_edge(orb, ogrid, orc.space(), a[i], b[i], env=oenv)
        assert bool(info["flags"][i] & irt.FLAG_PARTIAL) == (not oi["is_fully_valid"]), i
        assert info["t_last"][i] == oi["t"], i
        bxyz, bits = tree.export()
        keys = [orc.morton_key(int(x), int(y), int(z), Nb) for x, y, z in bxyz]
        lo, hi = int(got_off[i]), int(got_off[i + 1])
        assert list(got_keys[lo:hi]) == keys and np.array_equal(got_bits[lo:hi], bits), i
        n_partial += not oi["is_fully_valid"]
    assert 20 < n_partial < len(a) - 20, "fixture must mix blocked and free motions (%d)" % n_partial
    # the valid prefix never touches the environment
    assert not store.check(env).any()


@pytest.mark.parametrize("Ng,dL,lim", [(64, 0.005, [-0.21, 0.21, -0.21, 0.21, -0.21, 0.21]),
                                       (256, 0.0015, [-0.21, 0.21, -0.21, 0.21, -0.21, 0.21]),
                                       (128, 0.003, [-0.25, 0.22, -0.21, 0.30, -0.05, 0.40])])
def test_voxelisation_other_grids(irt, ctx, orc, wl, Ng, dL, lim):
    """coarser / finer grids and non-cubic cells (dx != dy != dz), vertices and edges"""
    spec = wl.robot_b(dL)
    states = wl.sample_states(spec, 400, stream=56)
    # include degenerate shapes: fully retracted (one point) and the single-point grid {s}
    states[0, -1] = spec["L"]
    states[1, -1] = spec["L"] - 0.2 * dL
    rb = irt.Robot(ctx, spec)
    grid = irt.make_grid(Ng, lim)
    ogrid = orc.grid(Ng, lim)
    vs = irt.SetStore(ctx, grid)
    flags, _ = vs.voxelize_vertices(rb, states)
    ostore, oflags = orc.voxelize_vertices_batch(orc.robot(spec), ogrid, states)
    assert np.array_equal(flags, oflags)
    assert _csr_flips(vs.export_csr(), ostore.export()) == 0
    off = vs.export_csr()[0]
    assert off[1] == off[0] and off[2] == off[1]  # one-point shapes voxelise to the empty set
    pairs = wl.knn_edges(spec, states, k=3)[:300]
    es = irt.SetStore(ctx, grid)
    info = es.voxelize_edges_indexed(rb, irt.make_space(), states, pairs)
    oes, oinfo = orc.voxelize_edges_batch(orc.robot(spec), ogrid, orc.space(), states[pairs[:, 0]], states[pairs[:, 1]])
    assert np.array_equal(info["flags"], oinfo["flags"]) and np.array_equal(info["t_last"], oinfo["t_last"])
    assert _csr_flips(es.export_csr(), oes.export()) == 0


def test_edge_large_swept_volumes_use_big_table(irt, ctx, orc, wl):
    """long edges at a fine grid: hundreds of leaf blocks per set, more than the rasteriser's
    small per-warp hash holds -> the big-table fallback pass must give the same bit-exact sets"""
    spec = wl.robot_a(0.0015)
    g = wl.workspace_grid(spec, Ng=256)
    st = wl.sample_states(spec, 60, stream=57) * 0.6   # moderate tensions: mostly valid shapes
    a, b = st[:30], st[30:]
    rb = irt.Robot(ctx, spec)
    grid = irt.make_grid(g["Ng"], g["lim"])
    store = irt.SetStore(ctx, grid)
    info = store.voxelize_edges(rb, irt.make_space(), a, b)
    ostore, oinfo = orc.voxelize_edges_batch(orc.robot(spec), orc.grid(g["Ng"], g["lim"]), orc.space(), a, b)
    assert np.array_equal(info["flags"], oinfo["flags"])
    assert not (info["flags"] & irt.FLAG_CAPACITY).any()
    off = ostore.export()[0].astype(np.int64)
    assert np.diff(off).max() > 192, "fixture must exceed the small hash (max %d blocks)" % np.diff(off).max()
    assert _csr_flips(store.export_csr(), ostore.export()) == 0


def test_config_c1_full(irt, ctx, orc, wl):
    """BASELINE.json configs[0] in full: default 4-tendon straight-routed robot, FK of 10k random
    tension configurations + vertex voxelisation at 128^3, against the CPU path"""
    spec = wl.robot_a(0.003)
    states = wl.sample_states(spec, 10_000, stream=1)
    rb, out, ref = _fk_compare(irt, ctx, orc, spec, states, want_all=True)
    g = wl.workspace_grid(spec)
    store = irt.SetStore(ctx, irt.make_grid(g["Ng"], g["lim"]))
    flags, _ = store.voxelize_vertices(rb, states)
    ostore, oflags = orc.voxelize_vertices_batch(orc.robot(spec), orc.grid(g["Ng"], g["lim"]), states)
    assert np.array_equal(flags, oflags)
    assert _csr_flips(store.export_csr(), ostore.export()) == 0


# ---------------------------------------------------------------------------------------------
# environment preparation on the device (irt_env_dilate / dilate_sphere / remove_interior)
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_env_preparation_bit_exact(irt, ctx, orc, wl):
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    Nb = g["Ng"] // 4
    grid = irt.make_grid(g["Ng"], g["lim"])
    ogrid = orc.grid(g["Ng"], g["lim"])
    env_blocks = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    # scatter single cells on faces, edges and corners of the grid and of leaf blocks
    rng = np.random.default_rng(5)
    for bx, by, bz in [(0, 0, 0), (Nb - 1, Nb - 1, Nb - 1), (0, Nb - 1, 3), (Nb - 1, 0, 0), (7, 0, Nb - 1)]:
        env_blocks[wl.morton_key(np.array([bx]), np.array([by]), np.array([bz]), Nb)[0]] |= np.uint64(
            (1 << 0) | (1 << 63) | (1 << int(rng.integers(0, 64))))
    oenv0 = _oracle_env(orc, wl, ogrid, env_blocks, Nb)
    env = irt.Env(ctx, grid)
    cases = [("dilate", (1, False)), ("dilate", (2, False)), ("dilate", (5, False)), ("dilate", (0, False)),
             ("dilate", (1, True)), ("dilate", (3, True)), ("dilate_sphere", (2.6 * oenv0_d(g),)),
             ("remove_interior", (False,)), ("remove_interior", (True,))]
    for name, args in cases:
        env.update(env_blocks)
        getattr(env, name)(*args)
        o = oenv0.copy()
        getattr(o, name)(*args)
        got, want = env.download(), o.dense_morton()
        flips = int(np.count_nonzero(got != want))
        assert flips == 0, (name, args, flips)
        assert env.nblocks() == o.nblocks()
    # the pipeline apps run on an obstacle tree before planning, chained on the device
    env.update(env_blocks)
    env.dilate_sphere(spec["r"])
    env.remove_interior()
    o = oenv0.copy(); o.dilate_sphere(spec["r"]); o.remove_interior(True)
    assert np.array_equal(env.download(), o.dense_morton())
    # the prepared environment drives K3 like an uploaded one (occupancy bitmap was rebuilt)
    states = wl.sample_states(spec, 2000, stream=91)
    store = irt.SetStore(ctx, grid)
    store.voxelize_vertices(irt.Robot(ctx, spec), states)
    env2 = irt.Env(ctx, grid)
    env2.update(o.dense_morton())
    assert np.array_equal(store.check(env), store.check(env2))


def oenv0_d(g):
    lim, Ng = g["lim"], g["Ng"]
    return min(lim[1] - lim[0], lim[3] - lim[2], lim[5] - lim[4]) / Ng


@pytest.mark.gpu
@pytest.mark.parametrize("Ng", [4, 16, 64])
def test_env_preparation_small_grids(irt, ctx, orc, wl, Ng):
    lim = [0, 1, -1, 1, 0, 0.5]
    Nb = Ng // 4
    grid, ogrid = irt.make_grid(Ng, lim), orc.grid(Ng, lim)
    rng = np.random.default_rng(Ng)
    blocks = np.zeros(Nb ** 3, np.uint64)
    pick = rng.integers(0, Nb ** 3, max(1, Nb ** 3 // 6))
    blocks[pick] = rng.integers(1, 2 ** 63, len(pick), dtype=np.uint64) & rng.integers(1, 2 ** 63, len(pick), dtype=np.uint64)
    oenv0 = _oracle_env(orc, wl, ogrid, blocks, Nb)
    env = irt.Env(ctx, grid)
    for name, args in [("dilate", (1, False)), ("dilate", (4, False)), ("dilate", (2, True)),
                       ("remove_interior", (False,)), ("remove_interior", (True,))]:
        env.update(blocks)
        getattr(env, name)(*args)
        o = oenv0.copy()
        getattr(o, name)(*args)
        assert np.array_equal(env.download(), o.dense_morton()), (name, args)
    # all-full grid: everything is interior, outside counts as occupied
    env.update(np.full(Nb ** 3, np.uint64(2 ** 64 - 1)))
    env.remove_interior()
    assert env.nblocks() == 0 and not env.download().any()


@pytest.mark.parametrize("mode,delta", [(0, 1e-3), (0, 1e-4), (1, 1e-4), (2, 1e-4), (2, 1e-6)])
def test_tip_jacobian_batch(irt, ctx, orc, wl, mode, delta):
    """SURVEY 8(f) row 3: finite-difference tip Jacobians of a batch of IK seeds in one FK launch vs
    the sequential rules of tip_control::Jacobian (tip_control.cpp:243-265) and levmar-2.6
    (misc_core.c:137-211 on fk_wrap, tip_control.cpp:92-122)."""
    spec = wl.robot_b(0.005, rotation=True)
    rb = irt.Robot(ctx, spec)
    orb = orc.robot(spec)
    L = spec["L"]
    states = wl.sample_states(spec, 300, stream=91)
    states[0, -1] = 0.0            # s - d < 0: the base before the origin is integrated like the reference
    states[1, -1] = L - 0.3 * delta  # s + d > L: fk_wrap returns (0, 0, L - s)
    states[2, -1] = L              # degenerate one-point shape
    states[3, :6] = 0.0            # tau = 0: tau - d < 0
    tips, J = rb.tip_jacobian_batch(states, mode=mode, delta=delta)
    assert J.shape == (300, 3, rb.state_size)
    worst_t = worst_J = 0.0
    for i, s in enumerate(states):
        t_ref, J_ref = orc.tip_jacobian(orb, s, mode, delta)
        worst_t = max(worst_t, np.abs(tips[i] - t_ref).max() / L)
        worst_J = max(worst_J, np.abs(J[i] - J_ref).max())
    assert worst_t < FK_REL_TOL
    # a Jacobian entry is a difference of two tips over the step, and the GPU's and the oracle's tips are each within
    # TOL_P_REL * L of the exact one (tests/test_gpu_fk_precision.py, tests/test_fk_precision_vectors.py)
    assert worst_J < 4 * TOL_P_REL * L / min(delta, 1e-4), worst_J
    # the batched Jacobian predicts the tip displacement of a small step (sanity, all modes)
    if mode == 2 and delta == 1e-4:
        dq = np.zeros_like(states[10]); dq[:6] = 1e-3
        t1 = rb.shape_batch((states[10] + dq)[None], want=("tip",))["tip"][0]
        assert np.abs(tips[10] + J[10] @ dq - t1).max() < 1e-6
    # error convention
    with pytest.raises(irt.IrtError):
        rb.tip_jacobian_batch(states[:, :-1])
    with pytest.raises(irt.IrtError):
        rb.tip_jacobian_batch(states, mode=7)
    with pytest.raises(irt.IrtError):
        rb.tip_jacobian_batch(states, delta=0.0)
    assert rb.tip_jacobian_batch(states[:0])[1].shape == (0, 3, rb.state_size)


def test_full_size_roadmap_generation_properties(irt, ctx, orc, wl):
    """Config C3 at full size: 100k vertices / ~1M k-NN edges, 128^3 grid.  Size-independent properties
    of the swept-volume build (determinism, shard invariance, endpoint containment, verdict
    monotonicity) plus the oracle on a random sample of its edges."""
    import torch
    from bench import knn_edges_gpu
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    Nb = g["Ng"] // 4
    grid = irt.make_grid(g["Ng"], g["lim"])
    rb = irt.Robot(ctx, spec)
    nv = 100_000
    st = wl.sample_states(spec, nv, stream=200)
    pairs = knn_edges_gpu(torch, st, spec, 17, torch.device("cuda"))   # ~1M undirected edges after dedupe
    assert 900_000 <= len(pairs) <= 1_250_000
    sp = irt.make_space()
    full = irt.SetStore(ctx, grid)
    info = full.voxelize_edges_indexed(rb, sp, st, pairs)
    off, keys, bits = full.export_csr()
    ne = len(pairs)
    assert len(off) == ne + 1 and np.all(np.diff(off.astype(np.int64)) >= 0)
    # keys sorted strictly inside every set (visit_leaves order), no empty leaves
    inner = np.ones(len(keys), dtype=bool)
    inner[off[:-1][off[:-1] < len(keys)].astype(np.int64)] = False
    assert np.all(np.diff(keys.astype(np.int64))[inner[1:]] > 0) and np.all(bits != 0)
    # determinism: a second build is identical
    again = irt.SetStore(ctx, grid)
    info2 = again.voxelize_edges_indexed(rb, sp, st, pairs)
    o2, k2, b2 = again.export_csr()
    assert np.array_equal(off, o2) and np.array_equal(keys, k2) and np.array_equal(bits, b2)
    assert all(np.array_equal(info[k], info2[k]) for k in ("flags", "t_last", "nsamples"))
    # shard invariance: the edge list split at an arbitrary point gives the same sets (what N ranks hold)
    cut = 333_337
    lo_s, hi_s = irt.SetStore(ctx, grid), irt.SetStore(ctx, grid)
    lo_s.voxelize_edges_indexed(rb, sp, st, pairs[:cut])
    hi_s.voxelize_edges_indexed(rb, sp, st, pairs[cut:])
    ol, kl, bl = lo_s.export_csr()
    oh, kh, bh = hi_s.export_csr()
    assert np.array_equal(np.concatenate([kl, kh]), keys) and np.array_equal(np.concatenate([bl, bh]), bits)
    assert np.array_equal(np.concatenate([ol, oh[1:] + ol[-1]]), off)
    # endpoint containment: a fully valid edge's swept volume contains both endpoint vertex sets
    vs = irt.SetStore(ctx, grid)
    vflags, _ = vs.voxelize_vertices(rb, st)
    vo, vk, vb = vs.export_csr()
    rng = np.random.default_rng(3)
    full_valid = np.nonzero(info["flags"] == 0)[0]
    for e in rng.choice(full_valid, size=2000, replace=False):
        es = dict(zip(keys[int(off[e]):int(off[e + 1])].tolist(), bits[int(off[e]):int(off[e + 1])].tolist()))
        for v in pairs[e]:
            for k, b in zip(vk[int(vo[v]):int(vo[v + 1])].tolist(), vb[int(vo[v]):int(vo[v + 1])].tolist()):
                assert es.get(k, 0) & b == b
    # verdict monotonicity: an edge whose endpoint vertex collides collides itself
    env = irt.Env(ctx, grid)
    env.update(wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g)))
    ev, vv = full.check(env), vs.check(env)
    ok = info["flags"] == 0
    assert np.all(ev[ok] | ~(vv[pairs[ok, 0]] | vv[pairs[ok, 1]]))
    assert 0.05 < ev.mean() < 0.95
    # the oracle on a random sample of these edges: bit-exact sets, flags and sample counts
    sample = np.sort(rng.choice(ne, size=400, replace=False))
    ostore, oinfo = orc.voxelize_edges_batch(orc.robot(spec), orc.grid(g["Ng"], g["lim"]), orc.space(),
                                             st[pairs[sample, 0]], st[pairs[sample, 1]])
    oo, ok_, ob = ostore.export()
    for j, e in enumerate(sample):
        assert np.array_equal(keys[int(off[e]):int(off[e + 1])], ok_[int(oo[j]):int(oo[j + 1])])
        assert np.array_equal(bits[int(off[e]):int(off[e + 1])], ob[int(oo[j]):int(oo[j + 1])])
    assert np.array_equal(info["flags"][sample], oinfo["flags"])
    assert np.array_equal(info["t_last"][sample], oinfo["t_last"])


@pytest.mark.parametrize("robot,rot,n", [("b", True, 250_000), ("a", False, 5000), ("b", False, 1)])
def test_fk_packed_outputs_equal_dense(irt, ctx, wl, robot, rot, n):
    """irt_fk_batch_packed: shape i's rows [row_offsets[i], row_offsets[i+1]) are exactly the first
    npts[i] rows of the dense form (bit for bit, across chunk boundaries of the pipeline), every per-shape
    output identical, self-collision flags computed from the packed rows."""
    spec = wl.robot_a(0.005) if robot == "a" else wl.robot_b(0.005, rotation=rot)
    rb = irt.Robot(ctx, spec)
    st = wl.sample_states(spec, n, stream=77)
    if spec.get("enable_retraction") and n >= 8:
        L = spec["L"]
        st[0, -1], st[1, -1], st[2, -1], st[3, -1], st[4, -1] = L, L + 0.01, 0.1995, -0.001, -0.01
    want = ("p", "R", "t", "npts", "L", "L_i", "tip", "uv", "flags", "iters", "nsteps")
    if n > 100_000:
        want = ("p", "t", "npts", "L_i", "tip", "flags")
    d = rb.shape_batch(st, want=want)
    k = rb.shape_batch_packed(st, want=want)
    ro = k["row_offsets"]
    assert ro[0] == 0 and np.array_equal(np.diff(ro), d["npts"]) and k["rows"] == int(d["npts"].sum())
    for name in ("npts", "L", "L_i", "tip", "uv", "flags", "iters", "nsteps"):
        if name in want:
            assert np.array_equal(d[name], k[name]), name
    cap = rb.max_points
    mask = np.arange(cap)[None, :] < d["npts"][:, None]
    assert np.array_equal(d["p"][mask], k["p"][:k["rows"]])
    assert np.array_equal(d["t"][mask], k["t"][:k["rows"]])
    if "R" in want:   # dense R is returned as [n][cap][row][col]; packed stays column-major 9-vectors
        assert np.array_equal(d["R"].transpose(0, 1, 3, 2).reshape(n, cap, 9)[mask], k["R"][:k["rows"]])
    # capacity error: one row too few
    if k["rows"] > 0:
        with pytest.raises(irt.IrtError) as ei:
            rb.shape_batch_packed(st, want=("p", "npts"), cap_rows=k["rows"] - 1)
        assert ei.value.status == irt.IRT_ERR_CAPACITY
    assert rb.shape_batch_packed(st[:0], want=("p", "npts"))["rows"] == 0


def test_create_roadmap_options(irt, ctx, orc, wl):
    """createRoadmap(N, opt) of the batch mirror (VoxelCachedLazyPRM.cpp:1380-1561): with every option on, each
    kept vertex is a valid shape that misses the environment, and the kept edges are exactly those candidate
    edges (k nearest incl. the vertex itself, range-bounded, new vertices in index order) that the oracle finds
    fully valid and collision free; growing the roadmap only touches what is added."""
    from irt_b200 import roadmap as R
    spec = wl.robot_b(0.003, rotation=True)
    g = wl.workspace_grid(spec)
    Nb = g["Ng"] // 4
    grid = irt.make_grid(g["Ng"], g["lim"])
    rb = irt.Robot(ctx, spec)
    prm = R.VoxelCachedLazyPRM(ctx, rb, grid)
    env_blocks = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    prm.setEnvironment(env_blocks)
    prm.createRoadmap(150, opt=R.VoxelizeVertices | R.ValidateVertices | R.VoxelizeEdges | R.ValidateEdges)
    assert prm.states.shape == (150, 8)
    orb, ogrid, osp = orc.robot(spec), orc.grid(g["Ng"], g["lim"]), orc.space()
    oenv = _oracle_env(orc, wl, ogrid, env_blocks, Nb)
    ostore, oflags = orc.voxelize_vertices_batch(orb, ogrid, prm.states)
    assert np.all(oflags == 0) and not orc.check_sets_batch(ostore, oenv).any()
    assert np.all(prm.vertex_validity == R.VALIDITY_TRUE) and np.all(prm.vertex_flags == 0)
    assert _csr_flips(prm.vertex_store.export_csr(), ostore.export()) == 0
    # replay the connection loop and ask the oracle about every candidate
    have, cand = set(), []
    for v in range(150):
        d = prm.distance(prm.states[v], prm.states)
        order = np.lexsort((np.arange(150), d))[:5]
        assert order[0] == v
        for n in order[d[order] <= 0.2 * prm.maximum_extent()].tolist():
            key = (min(v, n), max(v, n))
            if n != v and key not in have:
                have.add(key)
                cand.append((v, n))
    cand = np.array(cand, dtype=np.int64)
    oes, oinfo = orc.voxelize_edges_batch(orb, ogrid, osp, prm.states[cand[:, 0]], prm.states[cand[:, 1]])
    ok = ((oinfo["flags"] & irt.FLAG_PARTIAL) == 0) & ~orc.check_sets_batch(oes, oenv).astype(bool)
    assert ok.sum() > 0
    assert np.array_equal(prm.edges, cand[ok])
    assert np.all(prm.edge_validity == R.VALIDITY_TRUE) and np.all(prm.edge_flags == 0)
    assert prm.edge_store.num_sets == len(prm.edges)
    # growing: N <= size is a no-op; lazy growth keeps what was there and validates nothing new
    states0, edges0 = prm.states.copy(), prm.edges.copy()
    prm.createRoadmap(100)
    assert len(prm.states) == 150 and np.array_equal(prm.edges, edges0)
    prm.createRoadmap(200, opt=R.LazyRoadmap)
    assert len(prm.states) == 200 and np.array_equal(prm.states[:150], states0)
    assert np.array_equal(prm.edges[:len(edges0)], edges0) and len(prm.edges) > len(edges0)
    assert np.all(prm.vertex_validity[:150] == R.VALIDITY_TRUE) and not prm.vertex_validity[150:].any()
    assert np.all(prm.edge_validity[:len(edges0)] == R.VALIDITY_TRUE) and not prm.edge_validity[len(edges0):].any()
    assert prm.vertex_store.num_sets == 200 and prm.edge_store.num_sets == len(prm.edges)   # caches follow
    # the default sampler is TendonRobot::random_state: inside the state bounds
    s = prm.random_states(1000, 3)
    assert s[:, :6].min() >= 0 and s[:, :6].max() <= 20 and np.abs(s[:, 6]).max() <= np.pi
    assert s[:, 7].min() >= 0 and s[:, 7].max() <= spec["L"]


@pytest.mark.parametrize("Ng,lim", [(16, [0, 1, 0, 1, 0, 1]), (64, [-0.3, 0.2, -0.1, 0.4, 0.0, 0.25]),
                                     (128, [-0.21, 0.21, -0.21, 0.21, -0.21, 0.21])])
def test_env_add_primitives_bit_exact(irt, ctx, orc, wl, Ng, lim):
    """Environment::voxelize on the device (irt_env_add_primitives) against the oracle's add_point / add_sphere /
    add_capsule (pinned by the reference's own text): objects inside, straddling a face, outside the grid,
    degenerate capsules, radii below a cell and beyond the grid; 0 flips."""
    rng = np.random.default_rng(4321 + Ng)
    lo, hi = np.array(lim[0::2]), np.array(lim[1::2])
    ext = hi - lo
    grid, og = irt.make_grid(Ng, lim), orc.grid(Ng, lim)
    want = orc.octree(og)
    pts, sph, cap = [], [], []
    for k in range(90):
        c = lo + ext * rng.uniform(-0.3, 1.3, 3)
        r = float(ext.min() * rng.choice([0.001, 0.01, 0.05, 0.12, 0.02, 0.2]))
        if k % 3 == 0:
            want.add_point(c); pts.append(c)
        elif k % 3 == 1:
            want.add_sphere(c, r); sph.append(np.append(c, r))
        else:
            b = c if k % 9 == 2 else c + ext * rng.uniform(-0.5, 0.5, 3)
            want.add_capsule(c, b, r); cap.append(np.concatenate([c, b, [r]]))
    for p in (lo, hi, lo + ext / Ng * 3, hi + np.array([1e-12, 0, 0])):
        want.add_point(p); pts.append(p)
    env = irt.Env(ctx, grid)
    env.update(np.full((Ng // 4) ** 3, 0xFFFF, dtype=np.uint64))         # stale content: clear=True must drop it
    env.add_primitives(pts, sph, cap, clear=True)
    got, ref = env.download(), want.dense_morton()
    flips = int(sum(bin(int(x)).count("1") for x in (got ^ ref)[got != ref]))
    assert flips == 0, "%d voxel flips" % flips
    assert 0 < np.count_nonzero(ref) and env.nblocks() == np.count_nonzero(ref)
    # OR-ing more objects into the existing grid (clear=False), one kind at a time
    big = np.append(lo + ext / 2, 3.0 * ext.max())
    want.add_sphere(big[:3], big[3])
    env.add_primitives(spheres=[big])
    assert np.array_equal(env.download(), want.dense_morton()) and np.all(env.download() == ~np.uint64(0))
    # nothing to add is a no-op; empty arrays are accepted
    env.add_primitives(clear=True)
    assert env.nblocks() == 0


def test_env_voxelize_lung_capsules_and_dilate(irt, ctx, orc, wl):
    """the benchmark environment's capsule tree through Environment::voxelize(reference[, dilate]) on the device,
    followed by the preparation steps the apps apply (dilate by the robot radius, shell only)"""
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    grid, og = irt.make_grid(g["Ng"], g["lim"]), orc.grid(g["Ng"], g["lim"])
    caps = np.array([np.concatenate([a, b, [r]]) for a, b, r in wl.lung_like_capsules(spec)])
    for dilate in (0.0, 0.004):
        want = orc.octree(og)
        for c in caps:
            want.add_capsule(c[:3], c[3:6], c[6] + dilate)
        env = irt.Env(ctx, grid)
        env.add_primitives(capsules=caps, clear=True, dilate=dilate)
        assert np.array_equal(env.download(), want.dense_morton()) and env.nblocks() > 100
        env.dilate_sphere(spec["r"]); want.dilate_sphere(spec["r"])
        env.remove_interior(); want.remove_interior()
        assert np.array_equal(env.download(), want.dense_morton())
    with pytest.raises(irt.IrtError):
        irt.Env(ctx, grid).add_primitives(capsules=caps, dilate=-1.0)


def test_fused_verdict_exchange_single_rank_and_empty_shard(irt, ctx, orc, wl):
    """The verdict all-gather fused into K3 (voxel_and_popc_kernel<..., GATHER> + its last-CTA flag wait, and
    xchg_empty_shard_kernel), exercised on ONE GPU as a self-exchange (world = 1: the rank's own buffer is the
    only peer): the gathered words equal irt_check_sets' on full ranges, sub-ranges, ranges that end inside a
    verdict word, an empty shard, and over several sweeps (the two alternating buffers and the epoch flags)."""
    import torch
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    grid = irt.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    rb = irt.Robot(ctx, spec)
    states = wl.sample_states(spec, 5000, stream=41)
    store = irt.SetStore(ctx, grid)
    store.voxelize_vertices(rb, states)
    env = irt.Env(ctx, grid)
    env_blocks = wl.dense_to_morton_blocks(wl.lung_like_env_dense(spec, g))
    env.update(env_blocks)
    n = store.num_sets
    want = store.check(env)
    assert 0.05 < want.mean() < 0.95
    slot = (n + 63) // 64 * 2
    x = irt.VerdictExchange(ctx, 0, 1, slot)
    for sweep, (b, e) in enumerate([(0, n), (0, n), (0, 1000), (64, 64 + 777), (0, 0), (128, 128), (0, n), (4992, n)]):
        words = x.check(store, env, b, e).cpu().numpy().view(np.uint32)
        ctx.synchronize()
        assert len(words) == slot and x.status() == 0
        got = irt.unpack_verdicts(words, e - b) if e > b else np.zeros(0, dtype=bool)
        assert np.array_equal(got, want[b:e]), "sweep %d [%d, %d)" % (sweep, b, e)
        assert not words[(e - b + 31) // 32:].any(), "padding words of the slot must read 'no collision'"
    # a changed environment between sweeps (the replanning tick): the next gathered table follows it
    env.update(np.zeros_like(env_blocks))
    assert not irt.unpack_verdicts(x.check(store, env, 0, n).cpu().numpy().view(np.uint32), n).any()
    # an empty STORE is an empty shard too
    empty = irt.SetStore(ctx, grid)
    x2 = irt.VerdictExchange(ctx, 0, 1, 4)
    assert not x2.check(empty, env, 0, 0).cpu().numpy().any() and x2.status() == 0


def test_raster_arbitrary_segments_vs_oracle(irt, ctx, orc, wl):
    """K2's rasteriser on polylines that are NOT backbones (irt_voxelize_shapes): the golden segments of every kind
    (short, long across / past the grid, axis-aligned, zero-length, on cell faces, near-degenerate directions:
    tests/golden/reference_vectors.npz, generated with the reference's own add_line) as two-point shapes, and random
    polylines of long steps that cross many blocks (division-free traversal over paths of any length, hand-over to
    the literal code on close calls, block accumulator across segments, hash overflow into the big-table pass).
    Leaves and bits equal to the oracle's add_piecewise_line, in visit_leaves order."""
    import os
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors.npz"))
    lim = gold["vo_lim"].tolist()
    Ng, Nb = 128, 32
    rng = np.random.default_rng(77)
    shapes = [np.array(sg) for sg in gold["vo_segs"]]
    dxv = (lim[1] - lim[0]) / Ng
    for i in range(400):
        crossing = i >= 380                      # the last 20: 20-30 long steps through the grid, > 192 blocks
        n = int(rng.integers(20, 31)) if crossing else int(rng.integers(2, 13))
        pts = [rng.uniform(-0.24, 0.24, 3)]
        for _ in range(n - 1):
            kind = 1 if crossing else int(rng.integers(0, 6))
            a = pts[-1]
            if kind == 0:
                b = a + rng.normal(size=3) * 0.004
            elif kind == 1:
                b = rng.uniform(-0.3, 0.3, 3)
            elif kind == 2:
                b = a.copy(); b[rng.integers(0, 3)] += rng.uniform(-0.2, 0.2)
            elif kind == 3:
                b = a.copy()
            elif kind == 4:
                b = np.round(a / dxv) * dxv + rng.integers(-6, 7, 3) * dxv
            else:
                b = a + rng.uniform(-1, 1, 3) * np.array([1e-12, 0.08, 1e-11])[rng.permutation(3)]
            pts.append(b)
        shapes.append(np.array(pts))
    cap = max(len(sh) for sh in shapes)
    p = np.zeros((len(shapes), cap, 3))
    npts = np.zeros(len(shapes), dtype=np.int32)
    for i, sh in enumerate(shapes):
        p[i, :len(sh)] = sh
        npts[i] = len(sh)
    store = irt.SetStore(ctx, irt.make_grid(Ng, lim))
    store.voxelize_shapes(p, npts)
    off, keys, bits = store.export_csr()
    og = orc.grid(Ng, lim)
    flips = 0
    for i, sh in enumerate(shapes):
        t = orc.octree(og)
        t.add_piecewise_line(sh)
        xyz, rbits = t.export()
        rkeys = wl.morton_key(xyz[:, 0].astype(np.int64), xyz[:, 1].astype(np.int64), xyz[:, 2].astype(np.int64), Nb) \
            if len(xyz) else np.zeros(0, dtype=np.uint32)
        gk, gb = keys[int(off[i]):int(off[i + 1])], bits[int(off[i]):int(off[i + 1])]
        if not (np.array_equal(gk, np.asarray(rkeys, dtype=np.uint32)) and np.array_equal(gb, rbits)):
            flips += 1
    assert flips == 0, "%d of %d polylines differ from the oracle's add_piecewise_line" % (flips, len(shapes))
    nblk = np.diff(off.astype(np.int64))
    assert nblk.max() > 192, "no shape reached the big-table pass (%d blocks at most)" % nblk.max()
    # the golden groups (three segments per tree, leaves written by the reference's add_line): union of the three
    # single-segment sets
    goff = gold["vo_leaf_off"]
    for k in range(0, 600, 3):
        acc = {}
        for i in range(k, k + 3):
            for kk, bb in zip(keys[int(off[i]):int(off[i + 1])], bits[int(off[i]):int(off[i + 1])]):
                acc[int(kk)] = acc.get(int(kk), 0) | int(bb)
        xyz = gold["vo_leaf_xyz"][goff[k // 3]:goff[k // 3 + 1]].astype(np.int64)
        want = dict(zip(wl.morton_key(xyz[:, 0], xyz[:, 1], xyz[:, 2], Nb).tolist() if len(xyz) else [],
                        gold["vo_leaf_bits"][goff[k // 3]:goff[k // 3 + 1]].tolist()))
        assert acc == want, "golden group %d" % (k // 3)


def test_pinned_staging_survives_io_growth(irt, ctx, wl):
    """ADVICE r1 (high): packed(small) -> dense(large) -> packed(small) on ONE context.  Growing the device
    staging buffer used to free the pinned row-offset buffer and leave the dangling pointer in the context."""
    spec = wl.robot_b(0.005)
    rb = irt.Robot(ctx, spec)
    small = wl.sample_states(spec, 300, stream=51)
    big = wl.sample_states(spec, 300_000, stream=52)
    a = rb.shape_batch_packed(small, want=("p", "npts", "flags"))
    dense = rb.shape_batch(big, want=("p", "npts", "L_i", "flags"))
    b = rb.shape_batch_packed(small, want=("p", "npts", "flags"))
    rows = int(a["row_offsets"][-1])
    assert np.array_equal(a["row_offsets"], b["row_offsets"]) and np.array_equal(a["p"][:rows], b["p"][:rows])
    assert np.array_equal(a["npts"], b["npts"]) and int(a["row_offsets"][-1]) == int(a["npts"].sum())
    assert dense["npts"].shape == (300_000,)


def test_lazy_path_consumers_on_device_tables(irt, ctx, orc, wl):
    """SURVEY 8(f) row 2 on the real library: constructSolution / solveWithRoadmap validate A* paths by look-ups
    into the verdict words of ONE vertex sweep and ONE edge sweep (D2H included); paths are valid by the oracle's
    per-item checks, removed items are invalid ones (collisions and IRT_FLAG_PARTIAL edges)."""
    from irt_b200 import roadmap as R
    spec = wl.robot_b(0.003)
    g = wl.workspace_grid(spec)
    grid = irt.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    rb = irt.Robot(ctx, spec)
    prm = R.VoxelCachedLazyPRM(ctx, rb, grid)
    n = 400
    prm.createRoadmap(n, lambda cnt, rnd: wl.sample_states(spec, cnt, stream=700 + rnd),
                      lambda st: wl.knn_edges(spec, st, k=6), opt=R.VoxelizeVertices)
    prm.precomputeEdgeVoxelCache()
    ogrid, osp = orc.grid(g["Ng"], g["lim"]), orc.space()
    oenv = orc.octree(ogrid)
    oenv.add_sphere([0.04, 0.0, 0.13], 0.035)
    oenv.add_sphere([-0.05, 0.03, 0.10], 0.03)
    env = irt.Env(ctx, grid)
    env.add_primitives(spheres=[[0.04, 0.0, 0.13, 0.035], [-0.05, 0.03, 0.10, 0.03]], clear=True)
    prm.setEnvironment(env.download())
    orb = orc.robot(spec)
    vs, vf = orc.voxelize_vertices_batch(orb, ogrid, prm.states)
    v_ok = (vf == 0) & ~orc.check_sets_batch(vs, oenv).astype(bool)
    es, einfo = orc.voxelize_edges_batch(orb, ogrid, osp, prm.states[prm.edges[:, 0]], prm.states[prm.edges[:, 1]])
    e_ok = ((einfo["flags"] & 16) == 0) & ~orc.check_sets_batch(es, oenv).astype(bool)
    rng = np.random.default_rng(5)
    solved = 0
    for _ in range(10):
        a, b = (int(x) for x in rng.choice(np.nonzero(v_ok)[0], 2, replace=False))
        path, _ = prm.solveWithRoadmap(a, b)
        if path is None:
            continue
        solved += 1
        assert path[0] == a and path[-1] == b and all(v_ok[v] for v in path[1:-1])
        assert all(e_ok[prm.edge_index(u, v)] for u, v in zip(path[:-1], path[1:]))
    assert solved >= 5 and prm.lookups["sweeps"] == 2
    assert np.array_equal(prm.vertex_validity.astype(bool), v_ok) and np.array_equal(prm.edge_validity.astype(bool), e_ok)
    assert not v_ok[prm.vertex_removed].any() and not e_ok[prm.edge_removed].any()


def _adversarial_backbones(rng, r, cap):
    """polylines that sit on the decision boundaries of collides_self (collision/collision.cpp:6-46)"""
    shapes = []

    def put(pts):
        pts = np.asarray(pts, dtype=np.float64)
        if 2 <= len(pts) <= cap:
            shapes.append(pts)

    def rigid(pts):
        q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        return np.asarray(pts) @ q.T + rng.uniform(-0.15, 0.15, 3)

    dl = 0.005
    # (1) hairpins: two parallel runs D apart, D = 2r +- a few ulp and +- small relative steps (parallel-segment
    #     branch of closest_st_segment; the FP32 filter must keep every D <= 2r)
    for j in list(range(-4, 5)) + [-1000, 1000, -10 ** 6, 10 ** 6]:
        D = np.nextafter(2 * r, np.inf) if j == 0 else 2 * r * (1 + j * 2.2e-16)
        for nleg in (10, 14, 20):
            out = [[i * dl, 0.0, 0.0] for i in range(nleg)]
            nb = 6
            bend = [[(nleg - 1) * dl + 0.5 * D * np.sin(np.pi * k / nb), 0.5 * D * (1 - np.cos(np.pi * k / nb)), 0.0]
                    for k in range(1, nb)]
            back = [[(nleg - 1 - i) * dl, D, 0.0] for i in range(nleg)]
            put(out + bend + back)
            put(rigid(out + bend + back))
    # (2) V shapes: legs of n segments, turning theta at the corner; arc gaps around the 3r rule, distances around 2r
    for theta in np.linspace(0.3, 3.1, 29):
        for n1 in (3, 5, 8, 9, 10, 12):
            for scale in (1.0, 1.0 - 1e-12, 1.0 + 1e-12, 0.9, 1.1):
                d2 = np.array([np.cos(np.pi - theta), np.sin(np.pi - theta), 0.0])
                a = [[-(n1 - i) * dl * scale, 0.0, 0.0] for i in range(n1)] + [[0.0, 0.0, 0.0]]
                b = [list(d2 * (i + 1) * dl * scale) for i in range(n1)]
                put(rigid(a + b))
    # (3) arcs and spirals: constant and growing curvature, turning from below the early-out to several turns
    for turn in np.concatenate([np.linspace(1.2, 2.2, 21), np.linspace(2.5, 14.0, 24)]):
        for n in (20, 40, cap - 1):
            s = np.arange(n + 1) * dl
            for grow in (0.0, 1.0):
                kappa = turn / s[-1] * (1 + grow * s / s[-1]) / (1 + grow / 2)
                ang = np.concatenate([[0], np.cumsum(kappa[:-1] * dl)])
                pts = np.concatenate([[[0, 0, 0]], np.cumsum(np.stack([np.cos(ang[:-1]), np.sin(ang[:-1]),
                                                                         0.02 * np.ones(n)], 1) * dl, 0)])
                put(rigid(pts))
    # (4) random walks with bounded turning per step (many true collisions, many near misses)
    for _ in range(3000):
        n = int(rng.integers(8, cap))
        d = rng.normal(size=3)
        d /= np.linalg.norm(d)
        pts = [np.zeros(3)]
        for _k in range(n - 1):
            d = d + rng.normal(size=3) * rng.uniform(0.05, 0.6)
            d /= np.linalg.norm(d)
            pts.append(pts[-1] + d * dl * rng.uniform(0.6, 1.2))
        put(rigid(pts))
    # (5) degenerate: repeated points, very short shapes
    put(np.zeros((10, 3)))
    put([[0, 0, 0], [dl, 0, 0]])
    put([[0, 0, 0], [dl, 0, 0], [0, 0, 0], [dl, 0, 0], [0, 0, 0], [dl, 0, 0]])
    return shapes


def test_self_collision_adversarial_boundaries(irt, ctx, orc, wl):
    """collides_self on backbones built to sit on its decision boundaries: capsule pairs at 2r +- ulps (parallel
    and skew), arc gaps at the 3r skip rule, sharp corners, arcs around the turning bound of the filter's early
    out, spirals, random walks.  The FP32 pair filter and the turning early-out must never drop a true hit, and
    the exact stage must reproduce the reference's arithmetic: verdicts identical to the oracle on every shape."""
    r, cap = 0.015, 68
    shapes = _adversarial_backbones(np.random.default_rng(11), r, cap)
    n = len(shapes)
    p = np.zeros((n, cap, 3))
    npts = np.zeros(n, dtype=np.int32)
    for i, s in enumerate(shapes):
        p[i, :len(s)] = s
        npts[i] = len(s)
    got = irt.self_collision_shapes(ctx, p, npts, r)
    want = np.array([orc.collides_self(np.ascontiguousarray(s), r) for s in shapes])
    assert n > 4000 and 0.1 < want.mean() < 0.9
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, "verdict differs on %d shapes, first: %s" % (len(bad), bad[:5])
    # the same shapes through a narrower layout (cap 41 -> half a warp per shape in the filter)
    short = np.nonzero(npts <= 41)[0]
    got41 = irt.self_collision_shapes(ctx, np.ascontiguousarray(p[short, :41]), npts[short], r)
    assert np.array_equal(got41, want[short]) and want[short].any() and not want[short].all()
