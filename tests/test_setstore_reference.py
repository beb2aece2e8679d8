"""The set-store reference (tests/setstore_reference.py) against the oracle's tree recursion, and every layout builder
against its claims, without a GPU: so the GPU cases of tests/test_gpu_setstore_boundaries.py test the K3 edges they
say they test.  The reference is checked on reduced layouts (chunks of 64 or 128 leaves, tiles of 8 or 32 sets) at
Ng = 16 and 64; the claims at the full chunk and tile sizes."""
import numpy as np
import pytest

from oracle.oracle import SetStore
from tests import setstore_reference as R

C, T = R.CHUNK_LEAVES, R.TILE_SETS


def _reduced(kind, Nb, rng):
    if kind == "L1":
        return R.chunk_edges(Nb, rng, chunk=64, tile=8)
    if kind == "L2":
        return R.giant_sets(Nb, rng, chunk=64, tile=8, giant=300)
    if kind == "L3":
        return R.quad_phases(Nb, rng, chunk=128, tile=32)
    if kind == "L4":
        return R.empty_tiles(Nb, rng, chunk=64, tile=8, p_hit=1 / 20)
    if kind == "L4 no leaves":
        return R.no_leaves(Nb, n=50)
    if kind == "L5":
        return R.stride(Nb, rng, n_sets=200, grid_tiles=6, chunk=64, tile=8, common_key=8)
    raise ValueError(kind)


def _oracle(orc, wl, Nb, csr, env):
    """the CSR and the environment as the oracle's octrees"""
    grid = orc.grid(4 * Nb, [0, 1, 0, 1, 0, 1])
    off, keys, bits = (np.asarray(a) for a in csr)
    store = SetStore(orc, grid, len(off) - 1)
    bx, by, bz = wl.morton_decode(keys, Nb)
    for i in range(len(off) - 1):
        t = store.get(i)
        for j in range(int(off[i]), int(off[i + 1])):
            if bits[j]:
                t.union_block(int(bx[j]), int(by[j]), int(bz[j]), int(bits[j]))   # a key twice in a set: OR
    oenv = orc.octree(grid)
    nz = np.nonzero(env)[0]
    ex, ey, ez = wl.morton_decode(nz.astype(np.uint32), Nb)
    for x, y, z, k in zip(ex.tolist(), ey.tolist(), ez.tolist(), nz.tolist()):
        oenv.set_block(x, y, z, int(env[k]))
    return store, oenv


def _popcount_loop(off, keys, bits, env, begin, end):
    vox = hits = 0
    for j in range(int(off[begin]), int(off[end])):
        x = int(bits[j]) & int(env[keys[j]])
        vox += x.bit_count()
        hits += x != 0
    return vox, hits


@pytest.mark.parametrize("Ng", [16, 64])
@pytest.mark.parametrize("kind", ["L1", "L2", "L3", "L4", "L4 no leaves", "L5"])
def test_reference_matches_oracle_tree_recursion(orc, wl, Ng, kind):
    Nb = Ng // 4
    lay = _reduced(kind, Nb, np.random.default_rng(Ng))
    store, oenv = _oracle(orc, wl, Nb, lay.csr, lay.env)
    n = lay.n
    want = orc.check_sets_batch(store, oenv).astype(bool)
    got = R.verdicts(*lay.csr, lay.env)
    assert np.array_equal(got, want)
    assert np.array_equal(R.leaf_and(lay.keys, lay.bits, lay.env) != 0, lay.hit)      # the builder's own claim
    if kind != "L4 no leaves":
        assert 0 < got.sum() < n
    for begin, end in ((0, n), (1, n - 1), (3, 31), (n // 3, n // 2), (n - 1, n), (5, 5)):
        v = R.verdicts(*lay.csr, lay.env, begin, end)
        assert np.array_equal(v, want[begin:end])
        assert np.array_equal(v, orc.check_sets_batch(store, oenv, begin, end).astype(bool))
        assert R.popcount(*lay.csr, lay.env, begin, end) == _popcount_loop(*lay.csr, lay.env, begin, end)


@pytest.mark.parametrize("Ng", [16, 64])
def test_edge_keys_and_bits(orc, wl, Ng):
    """keys 0 and Nb^3 - 1, bits 0 and 63, zero-bit leaves (which never hit, even on the all-ones block of key 0)"""
    Nb = Ng // 4
    last = Nb ** 3 - 1
    env = R.pattern_env(Nb)
    sets = [
        [(0, 1)],                               # bit 0 of key 0: hit
        [(0, 1 << 63)],                         # bit 63 of key 0: hit
        [(0, 0)],                               # zero bits on the all-ones block: no hit
        [(last, 1 << 63)],                      # the last key, its only bit
        [(last, (1 << 63) - 1)],                # the last key, every other bit: no hit
        [(5, 0xFFFFFFFFFFFFFFFF)],              # an empty block (class 5): no hit
        [(2, 1 << 63), (3, 1)],                 # class 2 = bits 0 and 63; class 3 = the low half
        [(2, 0x7FFFFFFFFFFFFFFE), (last, 0), (0, 0)],
        [],
    ]
    off = np.concatenate([[0], np.cumsum([len(s) for s in sets])]).astype(np.uint64)
    keys = np.array([k for s in sets for k, _ in s], dtype=np.uint32)
    bits = np.array([b for s in sets for _, b in s], dtype=np.uint64)
    want = np.array([1, 1, 0, 1, 0, 0, 1, 0, 0], dtype=bool)
    assert np.array_equal(R.verdicts(off, keys, bits, env), want)
    store, oenv = _oracle(orc, wl, Nb, (off, keys, bits), env)
    assert np.array_equal(orc.check_sets_batch(store, oenv).astype(bool), want)
    assert R.popcount(off, keys, bits, env) == (1 + 1 + 1 + 1 + 1, 5)
    assert R.popcount(off, keys, bits, env, 6, 7) == (2, 2)


def test_pack_and_flips():
    rng = np.random.default_rng(0)
    for n in (0, 1, 31, 32, 33, 1000):
        v = rng.random(n) < 0.5
        w = R.pack(v)
        assert w.dtype == np.uint32 and len(w) == (n + 31) // 32
        for i in np.nonzero(v)[0]:
            assert (int(w[i // 32]) >> (i % 32)) & 1
        assert int(sum(bin(int(x)).count("1") for x in w)) == int(v.sum())
        u = rng.random(n) < 0.5
        assert np.array_equal(R.flips(v, u, 7), 7 + np.array([i for i in range(n) if v[i] != u[i]], dtype=np.int64))


def test_k3_position_restates_the_kernel_geometry():
    off = np.array([0, 6, 6, 70000, 70003], dtype=np.uint64)        # tiles of 2 sets: [0, 6), [6, 70003)
    p = R.k3_position(off, 6, tile=2)
    assert (p["tile"], p["chunk"], p["r"], p["head"], p["straddle"]) == (1, 0, 0, -2, False)
    p = R.k3_position(off, 6 + C, tile=2)
    assert (p["chunk"], p["r"], p["head"]) == (1, 0, -2)
    p = R.k3_position(off, 6 + 32, tile=2)          # quad 36..39 is tile positions 30..33: position 32 straddles
    assert p["word"] == 1 and p["straddle"]
    assert not R.k3_position(off, 6 + 30, tile=2)["straddle"]
    assert R.k3_position(off, 5, tile=2)["word"] == 0


@pytest.fixture(scope="module")
def full():
    return {k: f(64, np.random.default_rng(11)) for k, f in
            (("L1", R.chunk_edges), ("L2", R.giant_sets), ("L3", R.quad_phases), ("L4", R.empty_tiles))}


def test_l1_tiles_span_the_chunks_they_claim(full):
    lay = full["L1"]
    t_lo, t_hi = R.tile_leaves(lay.off)
    counts = {t: int(t_hi[t] - t_lo[t]) for t in range(len(t_lo))}
    for t, leaves in lay.claims["tile_leaves"].items():
        assert counts[t] == leaves and -(-leaves // C) == lay.claims["chunks"][t]
    assert {C - 1, C, C + 1, 2 * C, 3 * C + 1} <= set(lay.claims["tile_leaves"].values())
    assert {1, 2, 3, 4} <= set(lay.claims["chunks"].values())
    run = [t for t in range(len(counts)) if all(counts.get(t + i, 0) > C for i in range(4))]
    assert run, "four consecutive multi-chunk tiles"
    assert {int(x) % 4 for x in t_lo} >= {0, 1, 3}                 # tiles starting mid-quad


def test_l2_giant_sets_hold_one_hit_where_claimed(full):
    lay = full["L2"]
    off = lay.off.astype(np.int64)
    kinds = set()
    for s, p in lay.claims["giants"]:
        lo, hi = off[s], off[s + 1]
        assert hi - lo >= 140_000 and s % T == 0 and lo % 4 == 2
        h = np.nonzero(lay.hit[lo:hi])[0]
        assert h.tolist() == ([] if p is None else [p])
        assert lay.hit[lo - 1] and lay.hit[hi]                      # the neighbours hit next to the giant
        if p is None:
            continue
        w = lay.claims["where"][p]
        assert w == R.k3_position(off, lo + p)
        kinds.add(("chunk start", w["chunk"] > 0 and w["r"] == 0))
        kinds.add(("word 0", w["word"] == 0))
        kinds.add(("word 1023", w["word"] == C // 32 - 1))
        kinds.add(("straddle", w["straddle"]))
        kinds.add(("last", p == hi - lo - 1))
    assert {k for k, v in kinds if v} == {"chunk start", "word 0", "word 1023", "straddle", "last"}
    s = lay.claims["giants"][0][0]
    assert lay.claims["giants"][0][1] is None
    assert np.nonzero(lay.keys == lay.claims["lone_key"])[0].tolist() == [off[s + 1] - 1]
    assert {p for _, p in lay.claims["giants"]} >= {None, 0, C - 1, C, C + 1}


def test_l3_boundaries_fall_at_every_quad_phase(full):
    lay = full["L3"]
    off = lay.off.astype(np.int64)
    sizes = np.diff(off)
    seen, inside = set(), 0
    for leaf, kind, ph, d in lay.claims["boundaries"]:
        assert leaf % 4 == ph
        pos = R.k3_position(off, leaf)
        if kind == "tile":
            assert off[pos["tile"] * T] == leaf and pos["chunk"] == 0 and pos["r"] == 0
        else:
            assert pos["chunk"] == 1 and pos["r"] == 0
            inside += R.set_of(off, leaf)[1] != 0
        assert pos["head"] == -(ph % 4) if ph else pos["head"] == 0
        w = np.arange(leaf - R.QUAD_WINDOW, leaf + R.QUAD_WINDOW)
        assert all(1 <= sizes[R.set_of(off, x)[0]] <= 3 for x in w)
        assert np.nonzero(lay.hit[w])[0].tolist() == [d + R.QUAD_WINDOW]
        seen.add((kind, ph, d))
    assert len(seen) == 2 * 4 * 2 * R.QUAD_WINDOW
    assert inside > 0                                               # a chunk boundary inside a set


def test_l4_empty_runs_and_empty_tiles(full):
    lay = full["L4"]
    sizes = np.diff(lay.off.astype(np.int64))
    assert [n for _, n in lay.claims["empty_runs"]] == [300, 512, 700]
    for s, n in lay.claims["empty_runs"]:
        assert not sizes[s:s + n].any()
    t_lo, t_hi = R.tile_leaves(lay.off)
    assert (t_lo == t_hi).any() and (t_hi - t_lo > C).sum() == 2
    assert R.no_leaves(64).off.sum() == 0


def test_l5_one_cta_strides_over_several_heavy_tiles():
    G = 1184
    lay = R.stride(64, np.random.default_rng(5), grid_tiles=G)
    off = lay.off.astype(np.int64)
    t_lo, t_hi = R.tile_leaves(off)
    assert len(t_lo) > 2 * G
    heavy = set(lay.claims["heavy"])
    assert all(t_hi[t] - t_lo[t] > C for t in heavy)
    assert any({t, t + G, t + 2 * G} <= heavy for t in heavy)
    assert all(off[s + 1] - off[s] >= C and not lay.hit[off[s]:off[s + 1]].any() for s in lay.claims["giants"])
    k = lay.claims["common_key"]
    set_id = np.repeat(np.arange(lay.n), np.diff(off))
    at = lay.keys == k
    assert np.array_equal(np.unique(set_id[at]), np.arange(lay.n))   # every set has the common key
    assert not lay.hit[at].any()
    # the common key's list is under a quarter of the store's leaves: a change there takes the delta path
    assert at.sum() < 0.25 * off[-1]
