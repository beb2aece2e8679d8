"""The 34-digit FK vectors (golden/fk_mp_vectors.npz, written by golden/make_fk_mp_vectors.py) against the FP64
oracle, at a bound near the real accuracy of an FP64 integration rather than the product's 1e-9 L contract.

Measured maxima of the FP64 oracle over all 27 cells: |dp| 2.2e-14 L, |dR| 1.3e-13, |dL| 5.8e-15 L,
|dL_i| 9.3e-15 L, final u 2.4e-13 and final v 1.6e-15 relative (as TOL_STRAIN_REL measures them).  TOL_P sits 45x above the
worst point error; tests/test_gpu_fk_precision.py holds the CUDA kernel to the same bounds.
"""
import numpy as np
import pytest

from tests.golden import make_fk_mp_vectors as mk

TOL_P_REL = 1e-12     # p, L, L_i: relative to the backbone length L
TOL_R = 1e-12         # R: absolute
TOL_STRAIN_REL = 1e-11  # final v / u: relative to max(|v|), max(|u|, 1 / L)


@pytest.fixture(scope="module")
def vectors():
    return mk.load()


def strain_err(got, want, L):
    """relative error of a final (v, u) pair; u is measured against max(|u|, 1/L) (a bend of one radian over the
    backbone), so a straight shape's u of ~0 does not turn rounding noise into a large relative error"""
    v, u = np.asarray(got[0]), np.asarray(got[1])
    ev = np.abs(v - want[0]).max() / np.abs(want[0]).max()
    eu = np.abs(u - want[1]).max() / max(np.abs(want[1]).max(), 1.0 / L)
    return max(ev, eu)


def shape_errors(c, i, p, R, L_tot, L_i):
    """worst errors of state i of cell c (p, R: all npts nodes of the shape): dict name -> (error, node or tendon)"""
    L = c["spec"]["L"]
    sl = slice(c["off"][i], c["off"][i + 1])
    node = c["node"][sl]
    dp = np.abs(np.asarray(p)[node] - c["p"][sl]).max(axis=1) / L
    dR = np.abs(np.asarray(R)[node].reshape(-1, 9) - c["R"][sl].reshape(-1, 9)).max(axis=1)
    dLi = np.abs(np.asarray(L_i) - c["L_i"][i]) / L
    return dict(p=(dp.max(), int(node[dp.argmax()])), R=(dR.max(), int(node[dR.argmax()])),
                L=(abs(L_tot - c["L"][i]) / L, -1), L_i=(dLi.max(), int(dLi.argmax())))


def test_cells_cover_every_kernel_and_routing_class(vectors):
    assert list(vectors) == [c[0] for c in mk.CELLS]
    for name, nt, retract, _, rot, dL in mk.CELLS:
        spec = vectors[name]["spec"]
        assert (len(spec["C"]), spec["enable_retraction"], spec["enable_rotation"], spec["dL"]) == (nt, retract,
                                                                                                     rot, dL)
        assert len(vectors[name]["states"]) >= 10, name
    assert {(len(c["spec"]["C"]), c["spec"]["enable_retraction"]) for c in vectors.values()} == \
        {(nt, r) for nt in range(1, 13) for r in (False, True)}


def test_fp64_oracle_within_tol(orc, vectors):
    for name, c in vectors.items():
        spec = c["spec"]
        rb = orc.robot(spec)
        for i, st in enumerate(c["states"]):
            a = orc.shape(rb, st)
            assert a["iters"] == c["iters"][i], (name, i)
            assert len(a["t"]) == c["npts"][i], (name, i)
            assert np.array_equal(a["u_i"], c["u_i"][i]) and np.array_equal(a["v_i"], c["v_i"][i]), (name, i)
            for out, (err, at) in shape_errors(c, i, a["p"], a["R"], a["L"], a["L_i"]).items():
                tol = TOL_R if out == "R" else TOL_P_REL
                assert err < tol, "%s state %d: %s differs by %.3g at node/tendon %d" % (name, i, out, err, at)
            err = strain_err((a["v_f"], a["u_f"]), (c["v_f"][i], c["u_f"][i]), spec["L"])
            assert err < TOL_STRAIN_REL, "%s state %d: final strains differ by %.3g" % (name, i, err)


@pytest.mark.parametrize("name,i", [("nt01_full_straight", 0), ("nt02_ret_straight", 14),
                                    ("nt05_full_general", 9)])
def test_generator_reproduces_file(vectors, name, i):
    """three stored shapes recomputed with the generator: the file is what the generator writes"""
    c = vectors[name]
    got = mk.shape_mp(c["spec"], c["states"][i])
    sl = slice(c["off"][i], c["off"][i + 1])
    assert got["iters"] == c["iters"][i] and got["npts"] == c["npts"][i]
    assert np.array_equal(c["node"][sl], mk.stored_nodes(got["npts"]))
    got["p"], got["R"] = got["p"][c["node"][sl]], got["R"][c["node"][sl]]
    for k, want in (("p", c["p"][sl]), ("R", c["R"][sl]), ("L", c["L"][i]), ("L_i", c["L_i"][i]),
                    ("u_f", c["u_f"][i]), ("v_f", c["v_f"][i]), ("u_i", c["u_i"][i]), ("v_i", c["v_i"][i])):
        assert np.array_equal(got[k], want), k
