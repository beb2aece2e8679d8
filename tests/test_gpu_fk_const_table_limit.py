"""K1's constant-memory routing table (csrc/fk.cu) on both sides of its size limit.

The copy in constant memory holds IRT_CT_WIDTH = 10 doubles per tendon and table row (r, r', r'' and the products
rx^2, ry^2, rx ry, |r|^2) in FK_CT_DOUBLES = 8192 doubles: a 6-tendon robot fits with up to 136 table rows.  Robot B
(L = 0.2) at dL = 0.00295 has K = 68 grid nodes, 135 rows (8100 doubles: the fast path reads the last rows of the
array); at dL = 0.0029 it has K = 69, 137 rows (8220 doubles: generic path only).  On both sides, a configuration
alone in a batch (31 idle lanes: every step takes the generic rk4_step<RtPtr>) and 32 copies of it (a full warp of
one step count: rk4_step<RtConst> where the table fits) give the same bits, and the batch matches the oracle.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CT_DOUBLES, CT_WIDTH = 8192, 10
KEYS = ("p", "npts", "L", "L_i", "flags")


@pytest.mark.parametrize("dL, K, fits", [(0.00295, 68, True), (0.0029, 69, False)])
def test_constant_table_limit(orc, wl, dL, K, fits):
    import irt_b200
    ctx = irt_b200.Context(0)
    spec = wl.robot_b(dL)
    rb = irt_b200.Robot(ctx, spec)
    assert rb.max_points - 1 == K
    assert ((2 * K - 1) * len(spec["C"]) * CT_WIDTH <= CT_DOUBLES) == fits

    states = wl.sample_states(spec, 64, stream=11)
    out = rb.shape_batch(states)
    ref = orc.fk_batch(orc.robot(spec), states, rb.max_points)
    assert np.array_equal(out["npts"], ref["npts"])
    assert np.array_equal(out["flags"], ref["flags"])
    assert np.abs(out["p"] - ref["p"]).max() < 1e-9 * spec["L"]

    for i in range(4):
        one = rb.shape_batch(states[i:i + 1])
        warp = rb.shape_batch(np.repeat(states[i:i + 1], 32, axis=0))
        for k in KEYS:
            assert np.array_equal(one[k][0], out[k][i]), "state %d: %s alone != in the batch" % (i, k)
            for j in range(32):
                assert np.array_equal(warp[k][j], one[k][0]), "state %d: %s of lane %d != alone" % (i, k, j)
