"""Exact numpy restatement of what K3 (irt_check_sets, irt_check_sets_popcount, the fused verdict exchange) and
irt_check_sets_changed compute over a CSR set store, and builders of stores whose tiles put K3's chunk and quad
boundaries at known leaves.  The reference of tests/test_gpu_setstore_boundaries.py; tests/test_setstore_reference.py
checks it against the oracle's tree recursion and checks every builder's claims.

K3 geometry restated here (csrc/voxel_check.cu): the sets [begin, end) are cut into tiles of TILE_SETS sets; a tile's
leaves [t_lo, t_hi) are streamed in chunks of CHUNK_LEAVES leaves starting at t_lo, each chunk as 16-byte quads of 4
leaves aligned to the store (not to the chunk), into a hit bitmap of 32-leaf words indexed by the leaf's position in
the chunk.  A chunk or tile whose first leaf is not a multiple of 4 starts mid-quad, and a quad whose 4 leaves span
two bitmap words writes the second one (the straddle).

Every builder returns a Layout: the CSR, `hit` (the leaves built to hit `pattern_env`) and `claims`, the positions it
says it puts on K3's edges; the CPU suite asserts each claim from the CSR alone."""
import numpy as np

TILE_SETS = 256          # K3_THREADS: sets per tile
CHUNK_LEAVES = 32768     # K3_CHUNK_LEAVES: leaves per hit-bitmap pass
WORD_LEAVES = 32

ALL_ONES = np.uint64(0xFFFFFFFFFFFFFFFF)
# environment block of a key by its class k % 8; class 5 is an empty block (skipped by K3's occupancy bitmap)
CLASS_MASKS = np.array([0x5555555555555555, 0xAAAAAAAAAAAAAAAA, 0x8000000000000001, 0x00000000FFFFFFFF,
                        0xFFFFFFFF00000000, 0, 0x0F0F0F0F0F0F0F0F, 0xF0F0F0F0F0F0F0F0], dtype=np.uint64)


# ---- the reference ---------------------------------------------------------------------------------------------
def _range(off, begin, end):
    off = np.asarray(off, dtype=np.int64)
    end = len(off) - 1 if end is None else int(end)
    return off, int(begin), end


def leaf_and(keys, bits, env):
    """bits & env[key] of every leaf"""
    return np.asarray(bits, dtype=np.uint64) & np.asarray(env, dtype=np.uint64)[np.asarray(keys, dtype=np.int64)]


def verdicts(off, keys, bits, env, begin=0, end=None):
    """bool[end - begin]: set i collides when any of its leaves has bits & env[key] != 0"""
    off, begin, end = _range(off, begin, end)
    lo, hi = off[begin], off[end]
    pos = lo + np.nonzero(leaf_and(keys[lo:hi], bits[lo:hi], env))[0]
    v = np.zeros(end - begin, dtype=bool)
    # the set of a hitting leaf: the last set that starts at or before it (empty sets share their start)
    v[np.searchsorted(off[begin:end + 1], pos, side="right") - 1] = True
    return v


def popcount(off, keys, bits, env, begin=0, end=None):
    """(sum of popcount(bits & env[key]), number of hitting leaves) over the leaves [off[begin], off[end])"""
    off, begin, end = _range(off, begin, end)
    x = leaf_and(keys[off[begin]:off[end]], bits[off[begin]:off[end]], env)
    return int(np.bitwise_count(x).sum(dtype=np.int64)), int(np.count_nonzero(x))


def pack(v):
    """bool[n] -> the (n + 31) // 32 verdict words of the ABI: set i is bit i % 32 of word i // 32"""
    v = np.asarray(v, dtype=bool)
    b = np.packbits(v, bitorder="little")
    w = np.zeros(-(-len(b) // 4) * 4, dtype=np.uint8)
    w[:len(b)] = b
    return w.view(np.uint32)[:(len(v) + 31) // 32]


def flips(old, new, begin=0):
    """ascending set indices whose verdict differs between the two bool arrays of the range starting at `begin`"""
    return begin + np.nonzero(np.asarray(old, dtype=bool) ^ np.asarray(new, dtype=bool))[0].astype(np.int64)


# ---- K3 geometry -----------------------------------------------------------------------------------------------
def tile_leaves(off, begin=0, end=None, tile=TILE_SETS):
    """(t_lo, t_hi) of every tile of the range"""
    off, begin, end = _range(off, begin, end)
    starts = np.arange(begin, end, tile)
    return off[starts], off[np.minimum(starts + tile, end)]


def k3_position(off, leaf, begin=0, end=None, chunk=CHUNK_LEAVES, tile=TILE_SETS):
    """where K3 puts leaf `leaf` of a sweep of [begin, end): dict(tile, chunk (in the tile), r (position in the chunk),
    word (r // 32), head (first quad's offset, in (-4, 0]), straddle (the leaf's bit reaches the bitmap through the
    quad's second word))"""
    off, begin, end = _range(off, begin, end)
    t = int(np.searchsorted(off[begin:end + 1:tile], leaf, side="right") - 1)
    # the last tile that starts at or before the leaf and is not empty
    t_lo = int(off[begin + t * tile])
    k = (leaf - t_lo) // chunk
    c_lo = t_lo + k * chunk
    r = leaf - c_lo
    head = (c_lo // 4) * 4 - c_lo
    r0 = r - ((r - head) % 4)               # the quad's first position
    return dict(tile=t, chunk=k, r=r, word=r // WORD_LEAVES, head=head,
                straddle=max(r0, 0) // WORD_LEAVES != r // WORD_LEAVES)


def set_of(off, leaf):
    """(set, leaf within it) of a store leaf"""
    off = np.asarray(off, dtype=np.int64)
    s = int(np.searchsorted(off, leaf, side="right") - 1)
    return s, int(leaf - off[s])


# ---- environment and leaf content --------------------------------------------------------------------------------
def pattern_env(Nb, density=1.0, rng=None):
    """uint64[Nb^3]: CLASS_MASKS by key class, key 0 all ones (K3 reads the zeroed keys past a store's last leaf as
    key 0, so stale bits there would hit), key Nb^3 - 1 only bit 63; density < 1 empties that share of the other
    blocks at random"""
    nk = Nb ** 3
    env = CLASS_MASKS[np.arange(nk) % 8].copy()
    if density < 1.0:
        env[rng.random(nk) >= density] = 0
    env[nk - 1] = np.uint64(1) << np.uint64(63)
    env[0] = ALL_ONES
    return env


def _one_bit(e, high):
    """lowest, or where `high`, highest set bit of every non-zero e"""
    lo = e & (~e + np.uint64(1))
    h = e.copy()
    for sh in (1, 2, 4, 8, 16, 32):
        h |= h >> np.uint64(sh)
    return np.where(high, h ^ (h >> np.uint64(1)), lo)


def fill(sizes, env, rng, hit_leaves=(), p_hit=0.0, quiet=None, zero_share=0.03):
    """CSR with sets of the given leaf counts whose leaves hit `env` exactly at `hit_leaves` (store positions) and,
    with probability p_hit, at the other leaves that `quiet` (bool per leaf) does not exclude.  Keys of a set are
    distinct (an affine map of the leaf's rank with an odd factor is a bijection of the 2^k keys), except where a
    hitting leaf lands on an empty block and moves to a random non-empty one.  A hitting leaf's bits hold the
    lowest or the highest bit of its block (bits 0 and 63 at key 0) plus random bits; a missing leaf's bits are
    random bits outside its block, or 0 for a `zero_share` of them.  Returns (off, keys, bits, hit)."""
    sizes = np.asarray(sizes, dtype=np.int64)
    nk = len(env)
    off = np.zeros(len(sizes) + 1, dtype=np.int64)
    off[1:] = np.cumsum(sizes)
    n = int(off[-1])
    set_id = np.repeat(np.arange(len(sizes)), sizes)
    j = np.arange(n, dtype=np.int64) - off[:-1][set_id]
    h = rng.integers(0, nk, size=len(sizes))
    m = 2 * rng.integers(0, nk // 2, size=len(sizes)) + 1
    keys = (h[set_id] + j * m[set_id]) % nk
    hit = rng.random(n) < p_hit
    if quiet is not None:
        hit &= ~np.asarray(quiet, dtype=bool)
    hit[np.asarray(hit_leaves, dtype=np.int64)] = True
    move = hit & (env[keys] == 0)
    if move.any():
        nonempty = np.nonzero(env)[0]
        keys[move] = nonempty[rng.integers(0, len(nonempty), size=int(move.sum()))]
    e = env[keys]
    r = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64)
    r2 = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64)
    bits = np.where(hit, _one_bit(e, rng.random(n) < 0.5) | (r & (r2 | ~e)), r & ~e)
    bits[~hit & (rng.random(n) < zero_share)] = 0
    return off.astype(np.uint64), keys.astype(np.uint32), bits.astype(np.uint64), hit


class Layout:
    def __init__(self, name, csr, env, claims):
        self.name = name
        self.off, self.keys, self.bits, self.hit = csr
        self.env = env
        self.claims = claims

    @property
    def n(self):
        return len(self.off) - 1

    @property
    def csr(self):
        return self.off, self.keys, self.bits


def _split(rng, total, parts):
    """`parts` non-negative sizes summing to `total`, at random"""
    cuts = np.sort(rng.integers(0, total + 1, size=parts - 1))
    return np.diff(np.concatenate([[0], cuts, [total]]))


def _light(rng, n, mean=6):
    return rng.poisson(mean, size=n) + 1


# ---- layouts -----------------------------------------------------------------------------------------------------
def chunk_edges(Nb, rng, chunk=CHUNK_LEAVES, tile=TILE_SETS):
    """L1: tiles of chunk - 1, chunk, chunk + 1, 2 chunk and 3 chunk + 1 leaves (1 to 4 chunks, three or more rotate
    all three hit bitmaps inside one tile), then a run of four consecutive multi-chunk tiles (the rotation carries
    over from tile to tile) between light tiles.  A hit at one of the three leaves around every chunk boundary, the
    rest at random.  claims: tile_leaves {tile: leaves}, chunks {tile: number of chunks}"""
    env = pattern_env(Nb)
    heavy = [chunk - 1, chunk, chunk + 1, 2 * chunk, 3 * chunk + 1, None, 2 * chunk + 3, chunk + 2, 3 * chunk + 2,
             2 * chunk + 1, None]
    sizes, claims = [], dict(tile_leaves={}, chunks={})
    for t, total in enumerate(heavy):
        if total is None:
            sizes.append(_light(rng, tile))
            continue
        sizes.append(_split(rng, total, tile))
        claims["tile_leaves"][t] = total
        claims["chunks"][t] = -(-total // chunk)
    sizes = np.concatenate(sizes)
    off = np.concatenate([[0], np.cumsum(sizes)])
    bounds = [off[t * tile] + k * chunk for t in claims["chunks"] for k in range(1, claims["chunks"][t])]
    hits = [b + int(rng.integers(-1, 2)) for b in bounds]
    return Layout("L1 chunk edges", fill(sizes, env, rng, hits, p_hit=1 / 400), env, claims)


GIANT_LEAVES = 140_003
LONE_KEY = 8 * 7 + 1


def giant_sets(Nb, rng, chunk=CHUNK_LEAVES, tile=TILE_SETS, giant=GIANT_LEAVES):
    """L2: giant sets of `giant` leaves, each the first set of its tile (whose first leaf is = 2 mod 4, so that quads
    straddle bitmap words), each with exactly one hitting leaf -- at its position 0, chunk - 1, chunk, chunk + 1 and
    last, in bitmap word 0 and word 1023 of a chunk, in the straddle word -- or none.  The set before a giant (the
    last of a light tile) hits at its last leaf, the set after it at its first.  claims: giants [(set, position of
    the hit in the set or None)], where {position: k3_position of the hit in a whole-store sweep}, lone_key (the key of
    the first giant's last leaf, which no other leaf has)"""
    env = pattern_env(Nb)
    words = chunk // WORD_LEAVES
    positions = [None, 0, chunk - 1, chunk, chunk + 1, giant - 1, chunk + 5, 2 * chunk + (words - 1) * WORD_LEAVES + 17,
                 3 * chunk + WORD_LEAVES * (words // 2)]
    sizes, hits, claims = [], [], dict(giants=[], where={})
    leaves = 0
    for p in positions:
        light = _light(rng, tile)
        light[-1] += (2 - (leaves + light.sum()) % 4) % 4       # the giant's tile starts at a leaf = 2 mod 4
        sizes.append(light)
        leaves += int(light.sum())
        hits.append(leaves - 1)                                 # the last leaf before the giant
        g0 = leaves
        tail = rng.integers(1, 4, size=tile - 1)
        sizes.append(np.concatenate([[giant], tail]))
        hits.append(g0 + giant)                                 # the first leaf after it
        if p is not None:
            hits.append(g0 + p)
        claims["giants"].append((len(np.concatenate(sizes)) - tile, p))
        leaves += giant + int(tail.sum())
    sizes.append(_light(rng, tile))
    sizes = np.concatenate(sizes)
    off = np.concatenate([[0], np.cumsum(sizes)])
    quiet = np.zeros(int(off[-1]), dtype=bool)
    for s, _ in claims["giants"]:
        quiet[off[s]:off[s + 1]] = True                         # no hit in a giant but the one placed
    o, keys, bits, hit = fill(sizes, env, rng, hits, p_hit=1 / 20, quiet=quiet)
    # the last leaf of the giant without a hit is the only leaf at LONE_KEY (class 1), with bits outside its block
    nk = len(env)
    keys[keys == LONE_KEY % nk] = (LONE_KEY + 8) % nk
    last = off[claims["giants"][0][0] + 1] - 1
    keys[last], bits[last] = LONE_KEY % nk, np.uint64(0x5555555555555555)
    claims["lone_key"] = LONE_KEY % nk
    lay = Layout("L2 giant sets", (o, keys, bits, hit), env, claims)
    for s, p in claims["giants"]:
        if p is not None:
            claims["where"][p] = k3_position(off, int(off[s]) + p, chunk=chunk, tile=tile)
    return lay


QUAD_WINDOW = 4     # leaves on each side of a boundary that L3 covers with tiny sets


def quad_phases(Nb, rng, chunk=CHUNK_LEAVES, tile=TILE_SETS):
    """L3: after a first tile of phase 0, one tile per (phase, d) with phase in 0..3 and d in -4..3: the tile's first
    leaf is = phase mod 4, so its chunk boundary (tile leaf `chunk`) is at the same phase inside a quad.  Sets of 1 to
    3 leaves cover the leaves within QUAD_WINDOW of the tile start and of the chunk boundary (which may fall inside one
    of them), and in each such window exactly one leaf hits: the one at boundary + d.  Other sets hit only in their
    middle.  claims: boundaries [(store leaf, kind ("tile" or "chunk"), phase, d)]"""
    env = pattern_env(Nb)
    cases = [(ph, d) for ph in range(4) for d in range(-QUAD_WINDOW, QUAD_WINDOW)]

    def tiny(k):                           # sets of 1 to 3 leaves, at least k leaves in all
        s = rng.integers(1, 4, size=k)
        while s.sum() < k:
            s = np.concatenate([s, rng.integers(1, 4, size=1)])
        return s

    sizes, claims, hits = [], dict(boundaries=[]), []
    leaves = 0
    for i, case in enumerate([None] + cases):
        t_lo = leaves
        head = tiny(QUAD_WINDOW) if case else np.zeros(0, np.int64)
        before, after, tail = tiny(QUAD_WINDOW), tiny(QUAD_WINDOW + 3), tiny(QUAD_WINDOW)
        n_fill = tile - len(head) - len(before) - len(after) - len(tail)
        # `before` starts 4 to 6 leaves ahead of the chunk boundary, and before + after reach 4 leaves past it
        f1 = _split(rng, chunk - QUAD_WINDOW - int(head.sum()) - int(rng.integers(0, 3)), n_fill // 2)
        next_phase = cases[i][0] if i < len(cases) else 0
        f2_total = chunk // 8 + int(rng.integers(0, chunk // 8))
        rest = int(head.sum() + f1.sum() + before.sum() + after.sum() + tail.sum())
        f2_total += (next_phase - (t_lo + rest + f2_total)) % 4
        f2 = _split(rng, f2_total, n_fill - n_fill // 2)
        tile_sizes = np.concatenate([head, f1, before, after, f2, tail])
        assert len(tile_sizes) == tile
        if case:
            ph, d = case
            claims["boundaries"] += [(t_lo, "tile", ph, d), (t_lo + chunk, "chunk", ph, d)]
            hits += [t_lo + d, t_lo + chunk + d]
        sizes.append(tile_sizes)
        leaves += int(tile_sizes.sum())
    sizes.append(tiny(QUAD_WINDOW))
    sizes = np.concatenate(sizes)
    off = np.concatenate([[0], np.cumsum(sizes)])
    mid = (off[:-1] + off[1:]) // 2
    hits += mid[(sizes >= 16) & (rng.random(len(sizes)) < 0.5)].tolist()
    quiet = np.ones(int(off[-1]), dtype=bool)          # hits only where placed
    return Layout("L3 quad phases", fill(sizes, env, rng, hits, quiet=quiet), env, claims)


def empty_tiles(Nb, rng, chunk=CHUNK_LEAVES, tile=TILE_SETS, p_hit=1 / 300):
    """L4: runs of 300, 512 and 700 empty sets before, between and after tiles of 2.5 and 1.5 chunks and a light
    tile.  claims: empty_runs [(first set, count)]"""
    env = pattern_env(Nb)
    parts = [np.zeros(300, np.int64), _split(rng, chunk * 5 // 2, tile), np.zeros(512, np.int64),
             _split(rng, chunk * 3 // 2 + 3, tile), _light(rng, tile), np.zeros(700, np.int64)]
    claims = dict(empty_runs=[])
    s = 0
    for p in parts:
        if len(p) >= 300 and not p.any():
            claims["empty_runs"].append((s, len(p)))
        s += len(p)
    return Layout("L4 empty tiles", fill(np.concatenate(parts), env, rng, p_hit=p_hit), env, claims)


def no_leaves(Nb, n=1000):
    """L4': n empty sets, a store without a leaf"""
    env = pattern_env(Nb)
    z = np.zeros(0)
    return Layout("L4 no leaves", (np.zeros(n + 1, np.uint64), z.astype(np.uint32), z.astype(np.uint64),
                                   z.astype(bool)), env, dict(n_blocks=0))


def stride(Nb, rng, n_sets=700_000, grid_tiles=1184, chunk=CHUNK_LEAVES, tile=TILE_SETS, common_key=8 * 1000):
    """L5: more tiles than one K3 grid holds (`grid_tiles` CTAs stride over them), with multi-chunk tiles at
    t0 + k * grid_tiles for k = 0, 1, 2, so one CTA sweeps three of them.  A heavy tile's first set is giant (1 to 2.5
    chunks of leaves, no hit but at `common_key`); every set, empty ones excepted, has one leaf at `common_key` (a
    class-0 block) with bits outside that block: no hit, until a change adds one of those bits.  claims: heavy
    [tile], giants [set], common_key"""
    env = pattern_env(Nb)
    assert env[common_key] == CLASS_MASKS[0]
    n_tiles = -(-n_sets // tile)
    heavy = sorted({t0 + k * grid_tiles for t0 in (3, 250, 777, grid_tiles - 1) for k in range(3)
                    if t0 + k * grid_tiles < n_tiles - 1})
    sizes = _light(rng, n_sets, mean=4)
    giants = []
    for t in heavy:
        s0 = t * tile
        sizes[s0] = int(rng.integers(chunk, chunk * 5 // 2))
        sizes[s0 + 1:s0 + tile] = rng.integers(60, 200, size=tile - 1)
        giants.append(s0)
    off = np.concatenate([[0], np.cumsum(sizes)])
    n = int(off[-1])
    quiet = np.zeros(n, dtype=bool)
    for s in giants:
        quiet[off[s]:off[s + 1]] = True
    o, keys, bits, hit = fill(sizes, env, rng, p_hit=1 / 30, quiet=quiet)
    # the common leaf: a random leaf of every set, made a miss
    at = off[:-1] + (rng.random(n_sets) * sizes).astype(np.int64)
    odd = np.uint64(0xAAAAAAAAAAAAAAAA)
    keys[keys == common_key] = common_key + 8           # the common leaves are the only ones at that key
    keys[at] = common_key
    bits[at] = rng.integers(0, 2 ** 64, size=n_sets, dtype=np.uint64) & odd
    bits[at[giants]] = odd                              # every giant is a candidate of any change at the common key
    hit[at] = False
    return Layout("L5 stride", (o, keys, bits, hit), env, dict(heavy=heavy, giants=giants, common_key=common_key))
