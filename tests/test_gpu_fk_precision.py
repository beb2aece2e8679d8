"""K1 (`fk_rk4_fp64_kernel<NT, RETRACT>`, csrc/fk.cu) against shapes integrated at 34 digits
(golden/fk_mp_vectors.npz), at the bounds the FP64 oracle meets (tests/test_fk_precision_vectors.py):
p, L, L_i and the tip within TOL_P = 1e-12 L, R within 1e-12, the final strains within 1e-11 relative, the
initial strains within 1e-13 relative of the oracle's, and trip counts, node and step counts and flags equal.

The cells run all 24 <NT, RETRACT> instantiations, every routing branch of the first gap (straight, one pitch,
straight beside helices, two pitches, general polynomial) with and without retraction, rotation, and robots on
both sides of the constant-memory table limit.  Each configuration also runs alone (31 idle lanes: the generic
RtPtr step) and as a full warp of copies (the RtConst step from constant memory); the two give the same bits.

Measured maxima over all cells (B200, 1000 W power limit): not measured yet.
"""
import threading

import numpy as np
import pytest

from tests.golden import make_fk_mp_vectors as mk
from tests.test_fk_precision_vectors import TOL_P_REL, TOL_R, TOL_STRAIN_REL, shape_errors, strain_err

pytestmark = pytest.mark.gpu

TOL_UV0_REL = 1e-13   # initial strains: the same fixed-point iteration as the oracle, rsqrt instead of sqrt / div
ALL = ("p", "R", "t", "npts", "L", "L_i", "tip", "uv", "flags", "iters", "nsteps")


@pytest.fixture(scope="module")
def irt():
    import irt_b200
    return irt_b200


@pytest.fixture(scope="module")
def ctx(irt):
    return irt.Context(0)


@pytest.fixture(scope="module")
def vectors():
    return mk.load()


@pytest.fixture(scope="module")
def robots(irt, ctx, vectors):
    return {name: irt.Robot(ctx, c["spec"]) for name, c in vectors.items()}


def check_accuracy(c, out):
    """every output of a shape_batch over the cell's states against the stored vectors; returns the worst errors"""
    name, L = c["name"], c["spec"]["L"]
    for k in ("npts", "iters", "nsteps", "flags"):
        bad = np.nonzero(out[k] != c[k])[0]
        assert len(bad) == 0, "%s state %d: %s %s != %s" % (name, bad[0], k, out[k][bad[0]], c[k][bad[0]])
    worst = dict(p=0.0, R=0.0, L=0.0, L_i=0.0, tip=0.0, uv0=0.0, uvf=0.0)
    for i in range(len(c["states"])):
        n = c["npts"][i]
        errs = shape_errors(c, i, out["p"][i, :n], out["R"][i, :n], out["L"][i], out["L_i"][i])
        errs["tip"] = (np.abs(out["tip"][i] - c["p"][c["off"][i + 1] - 1]).max() / L, n - 1)
        uv = out["uv"][i]
        errs["uv0"] = (strain_err((uv[6:9], uv[0:3]), (c["v_i"][i], c["u_i"][i]), L), 0)
        errs["uvf"] = (strain_err((uv[9:12], uv[3:6]), (c["v_f"][i], c["u_f"][i]), L), n - 1)
        for k, (err, at) in errs.items():
            tol = dict(R=TOL_R, uv0=TOL_UV0_REL, uvf=TOL_STRAIN_REL).get(k, TOL_P_REL)
            what = "tendon" if k == "L_i" else "node"
            assert err < tol, "%s state %d: %s differs by %.3g (bound %.0e) at %s %d" % (name, i, k, err, tol,
                                                                                          what, at)
            worst[k] = max(worst[k], err)
    return worst


def test_fk_accuracy_per_cell(robots, vectors):
    table = {}
    for name, c in vectors.items():
        rb = robots[name]
        spec = c["spec"]
        K = rb.max_points - 1
        tab = (2 * K - 1) * len(spec["C"]) * 6
        if name.startswith("ct_"):   # the cell is on the side of the constant-table limit its name says
            assert (tab <= mk.FK_CT_DOUBLES) == name.startswith("ct_below"), (name, K, tab)
        table[name] = check_accuracy(c, rb.shape_batch(c["states"], want=ALL))
    keys = ("p", "R", "L", "L_i", "tip", "uv0", "uvf")
    print("\nworst error per cell (p, L, L_i, tip: relative to L; R absolute; strains relative)")
    print("%-28s" % "cell" + "".join("%9s" % k for k in keys))
    for name, w in table.items():
        print("%-28s" % name + "".join("%9.1e" % w[k] for k in keys))
    print("%-28s" % "max" + "".join("%9.1e" % max(w[k] for w in table.values()) for k in keys))


def _same(a, b, label, keys=ALL):
    for k in keys:
        assert np.array_equal(a[k], b[k]), "%s: %s differs" % (label, k)


def test_fast_and_generic_steps_bit_identical(robots, vectors):
    """Alone in a batch, a configuration's warp has 31 idle lanes, so every regular step takes the generic
    rk4_step<RtPtr>; as 32 copies, a full warp of one step count takes rk4_step<RtConst> (constant-memory table,
    where it fits).  Both equal the whole-cell batch of test_fk_accuracy_per_cell bit for bit."""
    for name, c in vectors.items():
        rb = robots[name]
        cell = rb.shape_batch(c["states"], want=ALL)
        for i, st in enumerate(c["states"]):
            one = rb.shape_batch(st[None], want=ALL)
            warp = rb.shape_batch(np.repeat(st[None], 32, axis=0), want=ALL)
            for k in ALL:
                label = "%s state %d" % (name, i)
                assert np.array_equal(one[k][0], cell[k][i]), "%s: %s alone != in the cell batch" % (label, k)
                bad = [j for j in range(32) if not np.array_equal(warp[k][j], one[k][0])]
                assert not bad, "%s: %s of lane %d of a full warp != alone (generic step)" % (label, k, bad[0])


@pytest.mark.parametrize("name", ["nt08_ret_helix", "ct_above_nt06_dl00185", "nt05_ret_two_pitches",
                                  "nt04_full_two_pitches"])
def test_batch_invariance(irt, robots, vectors, wl, name):
    """a configuration's outputs are the same bits whatever batch, position, warp neighbours and API carry it"""
    torch = pytest.importorskip("torch")
    c = vectors[name]
    spec, rb = c["spec"], robots[name]
    L, dL, cap = spec["L"], spec["dL"], rb.max_points
    target = c["states"][0]
    ref = rb.shape_batch(target[None], want=ALL)
    filler = wl.sample_states(spec, 4097, stream=501)

    def check(batch, j, label):
        _same({k: v[j] for k, v in rb.shape_batch(batch, want=ALL).items()}, {k: v[0] for k, v in ref.items()},
              "%s: %s" % (name, label))

    for pos in (0, 5, 31, 32):
        b = filler[:33].copy()
        b[pos] = target
        check(b, pos, "position %d of 33" % pos)
    for n in (1, 31, 32, 33, 4097):
        b = filler[:n].copy()
        b[n // 2] = target
        check(b, n // 2, "batch of %d" % n)
    if spec["enable_retraction"]:
        # one warp: the configuration beside BAD_STATE lanes (NaN, far below 0) and degenerate ones (s >= L)
        b = filler[:32].copy()
        b[1::4, -1] = np.nan
        b[2::4, -1] = L
        b[3::4, -1] = L + 0.01
        b[4::8, -1] = -0.5
        b[0] = target
        out = rb.shape_batch(b, want=ALL)
        assert np.all(out["flags"][1::4] & irt.FLAG_BAD_STATE) and np.all(out["npts"][2::4] == 1)
        check(b, 0, "warp with BAD_STATE and degenerate lanes")
        # every bucket (step count) smaller than a warp: one filler per step count, none with the target's
        b = np.repeat(filler[:1], cap, axis=0)
        b[:, -1] = L - (np.arange(cap) + 0.3) * dL
        steps = rb.shape_batch(b, want=("nsteps",))["nsteps"]
        b = b[steps != ref["nsteps"][0]]
        b = np.concatenate([b[:7], target[None], b[7:]])
        check(b, 7, "batch of %d buckets of one configuration each" % len(b))
    # the device-pointer and packed forms
    b = filler[:33].copy()
    b[7] = target
    n = len(b)
    shapes = dict(p=(n, cap, 3), R=(n, cap, 9), t=(n, cap), npts=(n,), L=(n,), L_i=(n, len(spec["C"])),
                  tip=(n, 3), uv=(n, 12), flags=(n,), iters=(n,), nsteps=(n,))
    d = {k: torch.zeros(s, dtype=torch.int32 if k in ("npts", "flags", "iters", "nsteps") else torch.float64,
                        device="cuda") for k, s in shapes.items()}
    rb.shape_batch_dev(torch.from_numpy(b).cuda(), n, d)
    rb.ctx.synchronize()
    got = {k: v[7].cpu().numpy() for k, v in d.items()}
    got["flags"] = got["flags"].view(np.uint32)
    got["R"] = got["R"].reshape(cap, 3, 3).transpose(0, 2, 1)   # column-major 9-vectors -> [row][col]
    _same(got, {k: v[0] for k, v in ref.items()}, "%s: shape_batch_dev" % name)
    k = rb.shape_batch_packed(b, want=ALL)
    rows = slice(k["row_offsets"][7], k["row_offsets"][8])
    npts = ref["npts"][0]
    assert rows.stop - rows.start == npts
    assert np.array_equal(k["p"][rows], ref["p"][0, :npts])
    assert np.array_equal(k["t"][rows], ref["t"][0, :npts])
    assert np.array_equal(k["R"][rows].reshape(-1, 3, 3).transpose(0, 2, 1), ref["R"][0, :npts])
    for key in ("npts", "L", "L_i", "tip", "uv", "flags", "iters", "nsteps"):
        assert np.array_equal(k[key][7], ref[key][0]), "%s: shape_batch_packed %s" % (name, key)


def test_constant_table_owner_across_robots_and_threads(irt, wl):
    """The constant-memory copy of the routing table is one per device and process: a launch for another robot
    uploads its own.  Robots A and B alternate on one context, then run concurrently from two host threads on
    two contexts of device 0 (ctypes releases the GIL during the calls); every batch is bit-identical to the
    robot's first run."""
    specs = dict(a=wl.robot_a(0.005), b=wl.robot_b(0.005, rotation=True))
    states = {k: wl.sample_states(s, 2000, stream=502 + i) for i, (k, s) in enumerate(specs.items())}
    want = ("p", "L_i", "tip", "uv", "npts", "iters", "flags")
    ctx = irt.Context(0)
    robots = {k: irt.Robot(ctx, s) for k, s in specs.items()}
    first = {}
    for k in "abab":
        out = robots[k].shape_batch(states[k], want=want)
        if k in first:
            _same(out, first[k], "robot %s after a switch" % k, want)
        else:
            first[k] = out
    errors = []

    def worker(k):
        try:
            c = irt.Context(0)
            r = irt.Robot(c, specs[k])
            for it in range(20):
                out = r.shape_batch(states[k], want=want)
                _same(out, first[k], "robot %s, thread run %d" % (k, it), want)
            r.close()
            c.close()
        except Exception as e:   # reported by the main thread
            errors.append(e)
    threads = [threading.Thread(target=worker, args=(k,)) for k in "ab"]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[0]
    for r in robots.values():
        r.close()
    ctx.close()

