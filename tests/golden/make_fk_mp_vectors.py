"""Generate tests/golden/fk_mp_vectors.npz: whole FK shapes at 34 significant digits.

    python tests/golden/make_fk_mp_vectors.py          (about a minute on 8 cores)

For every cell (a robot) and every state in it, the FP64 oracle (oracle/tendon_oracle.cpp) runs first; its
fixed-point trip count, initial strains v_i / u_i, node count, RK4 step count and validity flags are stored.
Then oracle/fk_second_opinion.py integrates the same discrete scheme (classic RK4 on the grid
{s} U {L - i dL}) from that initial condition in mpmath at 34 digits; its lengths (L, L_i), final strains
(v, u) and the nodes (p, R) of stored_nodes() are stored rounded to float64.  Starting both from the oracle's
v_i / u_i separates the integrator's rounding error from the fixed-point stop rule, whose last iterate is not the exact fixed point.

The cells cover every compiled K1 kernel (`fk_rk4_fp64_kernel<NT, RETRACT>`, NT = 1..12 with and without
retraction), each routing class of the device's first-gap evaluation with and without retraction, rotation,
and both sides of the constant-memory routing table limit (FK_CT_DOUBLES in csrc/fk.cu).  States whose fixed
point does not converge (1000 iterations) are left out: their last iterate is not a contraction.
tests/test_fk_precision_vectors.py pins this file against the FP64 oracle, tests/test_gpu_fk_precision.py
pins the GPU against it.
"""
import json
import math
import multiprocessing
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import irt_b200.workloads as wl  # noqa: E402

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fk_mp_vectors.npz")
MP_DPS = 34
NODE_STRIDE = 6
MAX_ITERS = 1000
FLAG_BAD_STATE = 32
FK_CT_DOUBLES = 7680      # csrc/fk.cu: doubles of the constant-memory copy of the routing table
MAX_TENDONS = 12
ROUTING = ("straight", "helix", "straight+helix", "two_pitches", "general")
EDGE_TAU = [3.0, 7.5, 1.0, 0.0, 12.0, 4.0]
# first-gap cases of test_fk_edge_cases (robot B, dL = 0.005): s == L, the K == 0 band (L - dL/2 < s < L),
# an exact node, one-step and two-step first gaps, a base slightly before 0
EDGE_S = [0.2, 0.199, 0.1975, 0.195, 0.0131, 0.0169, -1e-4, -0.0014]


def routing(kind, nt, L):
    """(C, D, general) of `nt` tendons of one routing class; every tendon shares the coefficient counts"""
    c0 = [2 * math.pi * j / nt + 0.1 for j in range(nt)]
    w = 2 * math.pi / L                       # one turn over the backbone
    hand = [(-1) ** j for j in range(nt)]
    if kind == "straight":                    # n_c = n_d = 1: on the device c1_abs == 0, no sincos
        return [[c] for c in c0], [[0.008 + 0.0005 * j] for j in range(nt)], False
    if kind == "helix":                       # one pitch, both handednesses: c1_uniform
        return [[c, h * w] for c, h in zip(c0, hand)], [[0.01] for _ in range(nt)], False
    if kind == "straight+helix":              # c1_uniform with c1_sign == 0 for every third tendon
        return ([[c, 0.0 if j % 3 == 0 else hand[j] * w] for j, c in enumerate(c0)],
                [[0.01] for _ in range(nt)], False)
    if kind == "two_pitches":                 # simple routing, !c1_uniform: one sincos per tendon and time
        return ([[c, hand[j] * w * (1.0, 1.5, 0.75)[j % 3]] for j, c in enumerate(c0)],
                [[0.01] for _ in range(nt)], False)
    # general polynomial theta (n_c up to IRT_MAX_COEF) and linear rho: the device's routing_eval
    n_c = 8 if nt % 2 else 4
    C = [[c0[j]] + [0.3 * (-1) ** (i + j) * (1 + 0.1 * j) / (i * L ** i) for i in range(1, n_c)]
         for j in range(nt)]
    D = [[0.008 + 0.0005 * j, 0.01 * (j % 3 - 1)] for j in range(nt)]
    return C, D, True


def make_spec(nt, retract, kind, rotation, dL):
    spec = wl.robot_a(dL)
    L = spec["L"]
    spec["C"], spec["D"], general = routing(kind, nt, L)
    # at most robot B's total tension: with more, most shapes do not converge
    spec["max_tension"] = [20.0 * min(1.0, 6.0 / nt)] * nt
    # general routing has no closed-form home length (reference UB): keep the length limits out of play
    spec["min_length"] = [-1.0 if general else -0.015] * nt
    spec["max_length"] = [1.0 if general else 0.035] * nt
    spec["enable_retraction"] = bool(retract)
    spec["enable_rotation"] = bool(rotation)
    return spec


def _cell_list():
    """(name, NT, retraction, routing class, rotation, dL).  The routing class rotates with NT so that each
    appears with and without retraction."""
    out = []
    for retract in (False, True):
        for nt in range(1, MAX_TENDONS + 1):
            kind = ROUTING[(nt - 1 + 4 * retract) % len(ROUTING)]
            rot = nt % 4 == 3
            name = "nt%02d_%s_%s%s" % (nt, "ret" if retract else "full", kind.replace("+", "_"),
                                       "_rot" if rot else "")
            out.append((name, nt, retract, kind, rot, 0.005))
    # both sides of the constant-table limit, L = 0.2: the table has (2 K - 1) * NT * 6 doubles
    out += [("ct_below_nt06_dl00187", 6, True, "helix", False, 0.00187),            # K = 107: 7668
            ("ct_above_nt06_dl00185", 6, True, "helix", True, 0.00185),             # K = 108: 7740
            ("ct_above_nt12_dl0003", 12, True, "straight+helix", False, 0.003)]     # K = 67: 9576
    return out


CELLS = _cell_list()
# every <NT, RETRACT> instantiation of the FK kernel runs, every routing class with and without retraction
assert {(c[1], c[2]) for c in CELLS} == {(nt, r) for nt in range(1, MAX_TENDONS + 1) for r in (False, True)}
assert {(c[3], c[2]) for c in CELLS} == {(k, r) for k in ROUTING for r in (False, True)}
assert sum(c[4] for c in CELLS) >= 3


def cells():
    """name -> robot spec"""
    return {name: make_spec(nt, r, kind, rot, dL) for name, nt, r, kind, rot, dL in CELLS}


def states(spec, stream):
    nt = len(spec["C"])
    retract, rot = spec["enable_retraction"], spec["enable_rotation"]
    st = wl.sample_states(spec, 6 if retract else 8, stream=stream)

    def row(tau, s, phi):
        return list(tau) + ([phi] if rot else []) + ([s] if retract else [])
    tmax = spec["max_tension"]
    extra = [row(tmax, 0.0, 0.7), row([tmax[0]] + [0.0] * (nt - 1), 0.05, -2.0), row([0.0] * nt, 0.1, 3.0)]
    if retract:
        tau = [EDGE_TAU[j % len(EDGE_TAU)] for j in range(nt)]
        extra += [row(tau, s, 1.0) for s in EDGE_S]
    return np.concatenate([st, np.array(extra)])


_ORC = None


def _oracle():
    global _ORC
    if _ORC is None:
        from oracle.oracle import Oracle, build
        build()
        _ORC = Oracle("canonical")
    return _ORC


def shape_mp(spec, state):
    """The FP64 oracle's initial condition, then the 34-digit integration.  Returns a dict of float64 arrays."""
    import mpmath
    from oracle import fk_second_opinion as so
    orc = _oracle()
    a = orc.shape(orc.robot(spec), state)
    out = dict(iters=a["iters"], v_i=np.array(a["v_i"]), u_i=np.array(a["u_i"]), npts=len(a["t"]))
    if a["iters"] >= MAX_ITERS:
        return out
    mp = mpmath.mp.clone()
    mp.dps = MP_DPS
    b = so.fk(spec, [float(x) for x in state], mp=mp, v0u0=(a["v_i"], a["u_i"]))
    f = np.vectorize(float, otypes=[np.float64])
    out.update(p=f(np.array(b["p"], dtype=object)), R=f(np.array(b["R"], dtype=object)), L=float(b["L"]),
               L_i=f(np.array(b["L_i"], dtype=object)), v_f=f(np.array(b["v_f"], dtype=object)),
               u_f=f(np.array(b["u_f"], dtype=object)))
    assert len(out["p"]) == out["npts"], "grid of the second opinion differs from the oracle's"
    return out


def stored_nodes(n):
    """nodes whose p and R are stored: the base, the end of the first gap and the next node, every
    NODE_STRIDE-th node and the tip (the error of an RK4 integration grows smoothly along the backbone, and all
    nodes would make the file three times larger)"""
    return np.array(sorted({0, 1, 2, n - 1}.union(range(0, n, NODE_STRIDE)).intersection(range(n))))


def _job(args):
    return shape_mp(*args)


def cell_arrays(name, spec, stream, pool_map=map):
    orc = _oracle()
    st = states(spec, stream)
    res = list(pool_map(_job, [(spec, s) for s in st]))
    # the library's outputs hold max_points = the node count of s = 0; it flags a base so far below 0 that its grid
    # has one node more BAD_STATE (test_fk_edge_cases), so such states are left out here
    cap = len(orc.t_range(0.0, spec["L"], spec["dL"]))
    ref = orc.fk_batch(orc.robot(spec), st, cap)
    keep = [i for i, r in enumerate(res) if r["iters"] < MAX_ITERS and r["npts"] <= cap
            and not ref["flags"][i] & FLAG_BAD_STATE]
    res = [res[i] for i in keep]
    npts = np.array([r["npts"] for r in res], dtype=np.int32)
    assert np.array_equal(npts, ref["npts"][keep])
    nodes = [stored_nodes(n) for n in npts]
    for r, k in zip(res, nodes):
        r["p"], r["R"] = r["p"][k], r["R"][k]
    d = {
        "spec": np.array(json.dumps(spec, sort_keys=True)),
        "states": st[keep],
        "npts": npts,
        "off": np.concatenate([[0], np.cumsum([len(k) for k in nodes])]).astype(np.int64),
        "node": np.concatenate(nodes).astype(np.int16),
        "iters": np.array([r["iters"] for r in res], dtype=np.int32),
        "nsteps": ref["nsteps"][keep],
        "flags": ref["flags"][keep],
        "u_i": np.stack([r["u_i"] for r in res]),
        "v_i": np.stack([r["v_i"] for r in res]),
        "p": np.concatenate([r["p"] for r in res]),
        "R": np.concatenate([r["R"] for r in res]),
        "L": np.array([r["L"] for r in res]),
        "L_i": np.stack([r["L_i"] for r in res]),
        "u_f": np.stack([r["u_f"] for r in res]),
        "v_f": np.stack([r["v_f"] for r in res]),
    }
    return {name + "/" + k: v for k, v in d.items()}


def load(path=PATH):
    """cell name -> dict of the stored arrays, with "spec" decoded and "name" added"""
    z = np.load(path)
    out = {}
    for name in z["cells"]:
        d = {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(name + "/")}
        d["spec"] = json.loads(str(d["spec"]))
        d["name"] = str(name)
        out[str(name)] = d
    return out


def main():
    out = {}
    names = []
    with multiprocessing.Pool() as pool:
        for k, (name, spec) in enumerate(cells().items()):
            out.update(cell_arrays(name, spec, 200 + k, pool.map))
            names.append(name)
            print(name, len(out[name + "/npts"]), "states", flush=True)
    out["cells"] = np.array(names)
    np.savez_compressed(PATH, **out)
    print("wrote", PATH, os.path.getsize(PATH), "bytes")


if __name__ == "__main__":
    main()
