"""K3 (irt_check_sets, irt_check_sets_popcount, irt_check_sets_dev, the fused single-rank exchange), irt_setstore_append
and irt_check_sets_changed on the B200 against the exact numpy reference of tests/setstore_reference.py, on stores whose
tiles span several hit-bitmap chunks: tiles of 1 to 4 chunks and runs of them (L1), 140k-leaf sets with one hit at
every chunk / word / straddle position (L2), tiles and chunks starting at every phase inside a quad with 1-3 leaf sets
around them (L3), runs of empty sets and a store without leaves (L4), more tiles than one grid holds (L5), stale bits
past a shrunk store's last leaf (L6) and real K2 edge sets of Robot A at Ng = 512 (L7).  Ng = 256 keeps K3's
occupancy bitmap in shared memory, Ng = 512 reads it from global memory.  Every verdict word, popcount and flip is
compared with the reference, never with another GPU path.  tests/test_setstore_reference.py checks, without a GPU,
that the layouts put their boundaries where they claim."""
import numpy as np
import pytest

from tests import setstore_reference as R

pytestmark = pytest.mark.gpu
LIM = [-0.2, 0.2, -0.2, 0.2, -0.2, 0.2]
CANARY = 0x5A5A5A5A
KINDS = ["L1", "L2", "L3", "L4", "L4 no leaves", "L5"]


@pytest.fixture(scope="module")
def irt():
    import irt_b200
    return irt_b200


@pytest.fixture(scope="module")
def ctx(irt):
    return irt.Context(0)


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


@pytest.fixture(scope="module")
def grid_tiles(torch):
    """tiles one plain K3 grid covers before its CTAs stride (8 CTAs per SM)"""
    return torch.cuda.get_device_properties(0).multi_processor_count * 8


_LAYOUTS = {}


@pytest.fixture(scope="module")
def layout(irt, ctx, grid_tiles):
    """(Layout, imported SetStore) of a kind at a grid size, built once"""
    def get(kind, Ng):
        if (kind, Ng) not in _LAYOUTS:
            Nb, rng = Ng // 4, np.random.default_rng([KINDS.index(kind), Ng])
            lay = {"L1": lambda: R.chunk_edges(Nb, rng), "L2": lambda: R.giant_sets(Nb, rng),
                   "L3": lambda: R.quad_phases(Nb, rng), "L4": lambda: R.empty_tiles(Nb, rng),
                   "L4 no leaves": lambda: R.no_leaves(Nb),
                   "L5": lambda: R.stride(Nb, rng, grid_tiles=grid_tiles)}[kind]()
            _LAYOUTS[(kind, Ng)] = (lay, _store(irt, ctx, Ng, lay.csr))
        return _LAYOUTS[(kind, Ng)]
    return get


def _grid(irt, Ng):
    return irt.make_grid(Ng, LIM)


def _store(irt, ctx, Ng, csr):
    s = irt.SetStore(ctx, _grid(irt, Ng))
    s.import_csr(*csr)
    return s


def _env(irt, ctx, Ng, blocks):
    e = irt.Env(ctx, _grid(irt, Ng))
    e.update(blocks)
    return e


class _Expected:
    """the reference over the whole store once; any range's verdicts and popcount are slices of it"""

    def __init__(self, csr, env):
        self.off = np.asarray(csr[0], dtype=np.int64)
        self.v = R.verdicts(*csr, env)
        x = R.leaf_and(csr[1], csr[2], env)
        self.vox = np.concatenate([[0], np.cumsum(np.bitwise_count(x), dtype=np.int64)])
        self.hits = np.concatenate([[0], np.cumsum(x != 0, dtype=np.int64)])
        assert (int(self.vox[-1]), int(self.hits[-1])) == R.popcount(*csr, env)

    def words(self, b, e):
        return R.pack(self.v[b:e])

    def popcount(self, b, e):
        lo, hi = self.off[b], self.off[e]
        return int(self.vox[hi] - self.vox[lo]), int(self.hits[hi] - self.hits[lo])


def _ranges(lay):
    """every begin < end from {0, 1, 3, 31, 32, 255, 256, 257, inside the heaviest tile, n - 1, n}"""
    n = lay.n
    t_lo, t_hi = R.tile_leaves(lay.off)
    heavy = int(np.argmax(t_hi - t_lo)) * R.TILE_SETS
    pts = sorted({p for p in (0, 1, 3, 31, 32, 255, 256, 257, heavy, heavy + 1, heavy + 37, n - 1, n) if 0 <= p <= n})
    return [(b, e) for i, b in enumerate(pts) for e in pts[i + 1:]]


def _check_all_paths(irt, ctx, torch, store, env, want, ranges):
    """check, popcount, check_dev on a side stream into a canary-filled buffer, and the fused exchange"""
    dev = torch.device("cuda", 0)
    side = torch.cuda.Stream(device=dev)
    n = store.num_sets
    xchg = irt.VerdictExchange(ctx, 0, 1, (n + 31) // 32 + 5)
    slot = xchg.slot_words
    for b, e in ranges:
        W = (e - b + 31) // 32
        w = want.words(b, e)
        got = irt.pack_mask(store.check(env, b, e))[:W]
        assert np.array_equal(got, w), ("check", b, e)
        assert store.popcount(env, b, e) == want.popcount(b, e), ("popcount", b, e)
        buf = torch.full((W + 48,), CANARY, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        store.check_dev(env, buf[16:], b, e, stream=side.cuda_stream)
        side.synchronize()
        h = buf.cpu().numpy().view(np.uint32)
        assert np.array_equal(h[16:16 + W], w), ("check_dev", b, e)
        assert (h[:16] == CANARY).all() and (h[16 + W:] == CANARY).all(), ("check_dev canary", b, e)
        out = xchg.check(store, env, b, e, stream=side.cuda_stream)
        side.synchronize()
        h = out.cpu().numpy().view(np.uint32)
        assert np.array_equal(h[:W], w) and not h[W:slot].any(), ("exchange", b, e)
        out.fill_(CANARY)              # the sweep after next writes over this buffer: its padding must be cleared
        torch.cuda.synchronize()
    assert xchg.status() == 0


@pytest.mark.parametrize("Ng", [256, 512])
@pytest.mark.parametrize("kind", KINDS)
def test_sweeps_match_reference(irt, ctx, torch, layout, kind, Ng):
    lay, store = layout(kind, Ng)
    env = _env(irt, ctx, Ng, lay.env)
    want = _Expected(lay.csr, lay.env)
    if kind != "L4 no leaves":
        assert 0 < want.v.sum() < lay.n
    _check_all_paths(irt, ctx, torch, store, env, want, _ranges(lay))


def _shrunk(rng, env, n_sets, mod):
    """a small CSR whose leaf count is = mod (mod 4) and whose last set does not hit"""
    sizes = rng.integers(1, 40, size=n_sets)
    sizes[-1] += (mod - sizes.sum()) % 4
    off = np.concatenate([[0], np.cumsum(sizes)])
    quiet = np.zeros(int(off[-1]), dtype=bool)
    quiet[off[-2]:] = True
    return R.fill(sizes, env, rng, p_hit=1 / 50, quiet=quiet)[:3]


@pytest.mark.parametrize("Ng", [256, 512])
def test_stale_bits_past_the_last_leaf(irt, ctx, torch, layout, Ng):
    """L6: K3 reads whole quads, so the 1-3 leaves after a store's last leaf are read: their keys are zeroed (key 0 is
    all ones here) but their bits are whatever a previous, larger content left.  Only the clip keeps them out of the
    verdicts and the popcount."""
    big, _ = layout("L1", Ng)
    rng = np.random.default_rng(Ng + 6)
    src = _store(irt, ctx, Ng, R.giant_sets(Ng // 4, rng).csr)
    env = _env(irt, ctx, Ng, big.env)

    def check(store, csr):
        nb = int(csr[0][-1])
        assert nb % 4 and store.num_blocks == nb
        want = _Expected(csr, big.env)
        n = len(csr[0]) - 1
        _check_all_paths(irt, ctx, torch, store, env, want, [(0, n), (n - 1, n), (n - 3, n), (1, n)])

    for mod in (1, 2, 3):
        small = _shrunk(rng, big.env, 5000 + mod, mod)
        nb = int(small[0][-1])
        assert big.bits[nb:(nb + 3) // 4 * 4].any()       # the stale leaves of the last quad would hit
        store = _store(irt, ctx, Ng, big.csr)
        store.import_csr(*small)
        check(store, small)
        # the same after an append has grown the store: import, append the giants, import a small content again
        store = _store(irt, ctx, Ng, small)
        store.append(src)
        store.import_csr(*small)
        check(store, small)
        # an append that ends mid-quad, over the stale leaves of the larger content before it
        store = _store(irt, ctx, Ng, big.csr)
        store.import_csr(*small)
        tail = _shrunk(rng, big.env, 7, 0)
        store.append(_store(irt, ctx, Ng, tail))
        both = (np.concatenate([small[0], small[0][-1] + tail[0][1:]]), np.concatenate([small[1], tail[1]]),
                np.concatenate([small[2], tail[2]]))
        assert big.bits[int(both[0][-1]):(int(both[0][-1]) + 3) // 4 * 4].any()
        check(store, both)


def _concat(dst, src, keep):
    off, keys, bits = (np.asarray(a) for a in dst)
    so, sk, sb = (np.asarray(a) for a in src)
    so = so.astype(np.int64)
    kept = np.nonzero(keep)[0]
    sizes = so[kept + 1] - so[kept]
    idx = np.concatenate([np.arange(so[i], so[i + 1]) for i in kept] + [np.zeros(0, np.int64)])
    return (np.concatenate([off, off[-1] + np.cumsum(sizes).astype(np.uint64)]).astype(np.uint64),
            np.concatenate([keys, sk[idx]]).astype(np.uint32), np.concatenate([bits, sb[idx]]).astype(np.uint64))


@pytest.mark.parametrize("Ng", [256, 512])
def test_append_heavy_sets(irt, ctx, torch, layout, Ng):
    """append the giants of L2 (with masks that drop the hitting sets next to them, or a giant itself) onto L3: the
    export is the reference concatenation, and every sweep of the result matches the reference"""
    dst_lay, _ = layout("L3", Ng)
    src_lay, src = layout("L2", Ng)
    rng = np.random.default_rng(Ng + 7)
    giants = [s for s, _ in src_lay.claims["giants"]]
    masks = []
    keep = rng.random(src_lay.n) < 0.9
    keep[giants] = True
    keep[[g - 1 for g in giants] + [g + 1 for g in giants]] = False          # heavy neighbours' hits dropped
    masks.append(keep)
    keep = np.ones(src_lay.n, dtype=bool)
    keep[giants[1::2]] = False                                               # every other giant dropped
    masks.append(keep)
    for keep in masks:
        store = _store(irt, ctx, Ng, dst_lay.csr)
        store.append(src, keep=keep)
        want_csr = _concat(dst_lay.csr, src_lay.csr, keep)
        for g, w in zip(store.export_csr(), want_csr):
            assert g.dtype == w.dtype and np.array_equal(g, w)
        env = _env(irt, ctx, Ng, dst_lay.env)
        want = _Expected(want_csr, dst_lay.env)
        n0, n = dst_lay.n, store.num_sets
        _check_all_paths(irt, ctx, torch, store, env, want,
                         [(0, n), (n0 - 1, n), (n0, n), (n0 + 1, n - 1), (n0 - 300, n0 + 300), (3, n0 + 1)])


def _revalidate(irt, ctx, store, ix, csr, blocks_old, blocks_new, eo, en, begin=0, end=None, path=None):
    end = store.num_sets if end is None else end
    old = R.verdicts(*csr, blocks_old, begin, end)
    new = R.verdicts(*csr, blocks_new, begin, end)
    words, fl, stats = store.check_changed(ix, eo, en, R.pack(old).copy(), begin, end)
    assert np.array_equal(words[:(end - begin + 31) // 32], R.pack(new)), (begin, end)
    assert np.array_equal(fl, R.flips(old, new, begin)), (begin, end)
    if path is not None:
        assert stats[2] == path, stats
    return fl, stats


def _revalidate_both_ways(irt, ctx, store, ix, csr, b_old, b_new, Ng, ranges, path=None):
    """old -> new, then new -> old with the same index (the candidate bitmap must have been left clear)"""
    eo, en = _env(irt, ctx, Ng, b_old), _env(irt, ctx, Ng, b_new)
    fl = None
    for b, e in ranges:
        f, _ = _revalidate(irt, ctx, store, ix, csr, b_old, b_new, eo, en, b, e, path if (b, e) == ranges[0] else None)
        fl = f if fl is None else fl
        _revalidate(irt, ctx, store, ix, csr, b_new, b_old, en, eo, b, e, path if (b, e) == ranges[0] else None)
        _revalidate(irt, ctx, store, ix, csr, b_old, b_new, eo, en, b, e)
    return fl


def _add_bit(blocks, key, bit):
    b = blocks.copy()
    b[key] |= np.uint64(bit)
    return b


NG_IX = 256


def test_revalidation_giant_last_leaf(irt, ctx, layout):
    """a change that overlaps only a giant set's last leaf; a whole-grid change (the sweep path)"""
    lay, store = layout("L2", NG_IX)
    ix = irt.SetIndex(ctx, store)
    off = lay.off.astype(np.int64)
    n = lay.n
    s, p = lay.claims["giants"][0]
    k = lay.claims["lone_key"]
    last = int(off[s + 1]) - 1
    assert p is None and lay.keys[last] == k and not (lay.bits[last] & lay.env[k])
    new = _add_bit(lay.env, k, 1 << 0)                # the last leaf's bits are the even ones
    fl = _revalidate_both_ways(irt, ctx, store, ix, lay.csr, lay.env, new, NG_IX,
                               [(0, n), (s, s + 1), (s - 1, s + 2), (s - 255, n - 1)], path=0)
    assert fl.tolist() == [s]
    _revalidate_both_ways(irt, ctx, store, ix, lay.csr, lay.env, R.pattern_env(NG_IX // 4, 0.5, np.random.default_rng(8)),
                          NG_IX, [(0, n), (1, n - 1)], path=1)


def test_revalidation_common_key_and_tail(irt, ctx, layout):
    """L5: a key in every set of a 700k-set store; a change that overlaps the bits of some of them takes the delta path
    and re-checks the giants; then heavy tail sets (a 140k-leaf set among them) appended after the index"""
    lay, store = layout("L5", NG_IX)
    ix = irt.SetIndex(ctx, store)
    n = lay.n
    k = lay.claims["common_key"]
    giants = lay.claims["giants"]
    for bit in (1 << 1, 1 << 63):
        new = _add_bit(lay.env, k, bit)
        fl = _revalidate_both_ways(irt, ctx, store, ix, lay.csr, lay.env, new, NG_IX,
                                   [(0, n), (giants[0], giants[0] + 300), (257, n - 1)], path=0)
        assert set(giants) <= set(fl.tolist()) and len(fl) < n // 2
    src_lay, src = layout("L2", NG_IX)
    g = src_lay.claims["giants"][0][0]
    store.append(src, begin=g - 3, end=g + 300)
    csr = _concat(lay.csr, src_lay.csr, np.r_[np.zeros(g - 3, bool), np.ones(303, bool),
                                              np.zeros(src_lay.n - g - 300, bool)])
    m = store.num_sets
    assert m == n + 303 and ix.num_sets == n
    # the giant's own keys change: it is a tail set, re-checked whatever the index says
    gk = src_lay.keys[int(src_lay.off[g]) + 5]
    new = _add_bit(lay.env, k, 1 << 3)
    new[gk] = ~new[gk]
    _revalidate_both_ways(irt, ctx, store, ix, csr, lay.env, new, NG_IX, [(0, m), (n - 2, m), (n + 3, n + 4)], path=0)
    _revalidate_both_ways(irt, ctx, store, ix, csr, lay.env, R.pattern_env(NG_IX // 4, 0.5, np.random.default_rng(9)),
                          NG_IX, [(0, m)], path=1)


def test_revalidation_chunk_edges(irt, ctx, layout):
    """L1: removing the blocks of the hits placed at the chunk boundaries, and a whole-grid change"""
    lay, store = layout("L1", NG_IX)
    ix = irt.SetIndex(ctx, store)
    off = lay.off.astype(np.int64)
    t_lo = off[0::R.TILE_SETS]
    bounds = [t_lo[t] + c * R.CHUNK_LEAVES for t, nc in lay.claims["chunks"].items() for c in range(1, nc)]
    near = [j for b in bounds for j in range(b - 1, b + 2) if lay.hit[j]]
    assert len(near) >= len(bounds)
    new = lay.env.copy()
    new[lay.keys[near]] = 0
    new[0] = lay.env[0]
    fl = _revalidate_both_ways(irt, ctx, store, ix, lay.csr, lay.env, new, NG_IX, [(0, lay.n), (255, lay.n - 1)])
    assert len(fl) > 0
    _revalidate_both_ways(irt, ctx, store, ix, lay.csr, lay.env, R.pattern_env(NG_IX // 4, 0.3, np.random.default_rng(10)),
                          NG_IX, [(0, lay.n)], path=1)


def test_real_robot_a_edge_sets_at_ng_512(irt, ctx, torch, wl):
    """L7: K2 edge sets of short Robot A edges at Ng = 512, where a 256-edge tile spans more than one chunk (dL under
    the voxel size that Ng = 512 accepts)"""
    spec = wl.robot_a(0.0008)
    g = wl.workspace_grid(spec, Ng=512)
    grid = irt.make_grid(g["Ng"], g["lim"], g["inv_rot"])
    st = wl.sample_states(spec, 2048, stream=5)
    a, b = st[:1024], st[1024:]
    b = a + 0.05 * (b - a)
    store = irt.SetStore(ctx, grid)
    store.voxelize_edges(irt.Robot(ctx, spec), irt.make_space(), a, b)
    csr = store.export_csr()
    t_lo, t_hi = R.tile_leaves(csr[0])
    assert (t_hi - t_lo).max() > R.CHUNK_LEAVES, (t_hi - t_lo).max()
    blocks = R.pattern_env(128, 0.004, np.random.default_rng(12))
    env = irt.Env(ctx, grid)
    env.update(blocks)
    want = _Expected(csr, blocks)
    assert 0.05 < want.v.mean() < 0.95, want.v.mean()
    n = store.num_sets
    _check_all_paths(irt, ctx, torch, store, env, want,
                     [(0, n), (1, n), (3, 257), (255, n - 1), (256, 512), (n - 1, n), (31, 1000)])
