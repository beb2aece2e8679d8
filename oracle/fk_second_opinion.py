"""Independent second restatement of the tendon-robot forward kinematics
(TEST INFRASTRUCTURE ONLY -- used to pin oracle/tendon_oracle.cpp, never by the product).

Deliberately written differently from the C++ oracle so that a shared transcription error
is unlikely:
  * vector identities instead of dense hat-matrix products
    (A_i = tau/sigma^3 (sigma^2 I - q q^T), B_i = c3 (s2 r^ - m q^T), H_i = c3 (s2(|r|^2 I - r r^T) - m m^T)),
  * one dense 6x6 solve (Gaussian elimination) instead of the blockwise inverse,
  * the arclength grid built from its closed form {s} U {L - i dL},
  * generic over the scalar type: python float or mpmath.mpf (50 digits).

Model: Rucker & Webster Cosserat-rod tendon robot as restated in SURVEY.md Appendix A
(reference: tendon/tendon_deriv.cpp:95-178, tendon/solve_initial_bending.cpp:15-73,
tendon/TendonRobot.cpp:325-500, tendon/get_r_info.cpp:105-144).
"""
import math


class Num:
    """scalar backend: float64 or mpmath"""

    def __init__(self, mp=None):
        self.mp = mp
        if mp is None:
            self.f = float
            self.sqrt, self.sin, self.cos, self.pi = math.sqrt, math.sin, math.cos, math.pi
        else:
            self.f = mp.mpf
            self.sqrt, self.sin, self.cos, self.pi = mp.sqrt, mp.sin, mp.cos, mp.pi


def cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def add(a, b):
    return [x + y for x, y in zip(a, b)]


def sub(a, b):
    return [x - y for x, y in zip(a, b)]


def scale(s, a):
    return [s * x for x in a]


def solve(M, rhs):
    n = len(rhs)
    A = [list(M[i]) + [rhs[i]] for i in range(n)]
    for c in range(n):
        piv = max(range(c, n), key=lambda r: abs(A[r][c]))
        A[c], A[piv] = A[piv], A[c]
        for r in range(c + 1, n):
            f = A[r][c] / A[c][c]
            for j in range(c, n + 1):
                A[r][j] -= f * A[c][j]
    x = [0] * n
    for r in range(n - 1, -1, -1):
        s = A[r][n] - sum(A[r][j] * x[j] for j in range(r + 1, n))
        x[r] = s / A[r][r]
    return x


def stiffness(nm, rb):
    f = nm.f
    ro, ri, E, nu = f(rb["ro"]), f(rb["ri"]), f(rb["E"]), f(rb["nu"])
    I = nm.pi / 4 * (ro ** 4 - ri ** 4)
    Ar = nm.pi * (ro ** 2 - ri ** 2)
    G = E / (2 * (1 + nu))
    return [E * I, E * I, 2 * I * G], [G * Ar, G * Ar, E * Ar]  # K_bt diag, K_se diag


def routing(nm, rb, t):
    """r, r', r'' for each tendon; r = rho (sin th, cos th, 0)."""
    out = []
    for Cc, Dd in zip(rb["C"], rb["D"]):
        th = sum(nm.f(c) * t ** i for i, c in enumerate(Cc))
        th1 = sum(i * nm.f(c) * t ** (i - 1) for i, c in enumerate(Cc) if i >= 1)
        th2 = sum(i * (i - 1) * nm.f(c) * t ** (i - 2) for i, c in enumerate(Cc) if i >= 2)
        rho = sum(nm.f(d) * t ** i for i, d in enumerate(Dd))
        rho1 = sum(i * nm.f(d) * t ** (i - 1) for i, d in enumerate(Dd) if i >= 1)
        rho2 = sum(i * (i - 1) * nm.f(d) * t ** (i - 2) for i, d in enumerate(Dd) if i >= 2)
        s, c = nm.sin(th), nm.cos(th)
        e = [s, c, 0]          # unit radial
        e1 = [c, -s, 0]        # d e / d theta
        r = scale(rho, e)
        rd = add(scale(rho1, e), scale(rho * th1, e1))
        # d/dt of rd: rho'' e + rho' th' e1 + (rho' th' + rho th'') e1 + rho th' * (-th' e)
        rdd = add(add(scale(rho2, e), scale(2 * rho1 * th1 + rho * th2, e1)),
                  scale(-rho * th1 * th1, e))
        out.append((r, rd, rdd))
    return out


def vu_dot(nm, rb, Kbt, Kse, tau, v, u, t):
    """(v', u', sigma_i) from the tendon/backbone force balance."""
    z = nm.f(0)
    M = [[z] * 6 for _ in range(6)]
    for i in range(3):
        M[i][i] = Kse[i]
        M[i + 3][i + 3] = Kbt[i]
    a = [z, z, z]
    b = [z, z, z]
    sig = []
    for (r, rd, rdd), tj in zip(routing(nm, rb, t), tau):
        tj = nm.f(tj)
        q = add(add(cross(u, r), rd), v)
        s2 = dot(q, q)
        s = nm.sqrt(s2)
        sig.append(s)
        c3 = tj / (s2 * s)
        m = cross(r, q)
        r2 = dot(r, r)
        for i in range(3):
            for j in range(3):
                dij = 1 if i == j else 0
                Aij = c3 * (s2 * dij - q[i] * q[j])
                M[i][j] += Aij
                M[3 + i][3 + j] += c3 * (s2 * (r2 * dij - r[i] * r[j]) - m[i] * m[j])
        # B = c3 (s2 r^ - m q^T) (bottom-left); G = B^T (top-right)
        rh = [[0, -r[2], r[1]], [r[2], 0, -r[0]], [-r[1], r[0], 0]]
        for i in range(3):
            for j in range(3):
                Bij = c3 * (s2 * rh[i][j] - m[i] * q[j])
                M[3 + i][j] += Bij
                M[j][3 + i] += Bij
        w = add(cross(u, add(q, rd)), rdd)
        ai = scale(c3, sub(scale(s2, w), scale(dot(q, w), q)))
        a = add(a, ai)
        b = add(b, cross(r, ai))
    vm = [v[0], v[1], v[2] - 1]
    Kv = [Kse[i] * vm[i] for i in range(3)]
    Ku = [Kbt[i] * u[i] for i in range(3)]
    c = sub(sub(scale(-1, cross(u, Ku)), cross(v, Kv)), b)
    d = sub(scale(-1, cross(u, Kv)), a)
    sol = solve(M, d + c)
    return sol[:3], sol[3:], sig


def initial_bending(nm, rb, Kbt, Kse, tau, s_start, max_iter=1000, thr=5e-6):
    f = nm.f
    v, u = [f(0), f(0), f(1)], [f(0), f(0), f(0)]
    rr = routing(nm, rb, s_start)
    it = 0
    for it in range(max_iter):
        Ft, Lt = [f(0)] * 3, [f(0)] * 3
        for (r, rd, _), tj in zip(rr, tau):
            q = add(add(cross(u, r), rd), v)
            n = scale(1 / nm.sqrt(dot(q, q)), q)
            Ft = sub(Ft, scale(f(tj), n))
            Lt = sub(Lt, scale(f(tj), cross(r, n)))
        res = nm.sqrt(sum((Kse[i] * (v[i] - (1 if i == 2 else 0)) - Ft[i]) ** 2 for i in range(3))
                      + sum((Kbt[i] * u[i] - Lt[i]) ** 2 for i in range(3)))
        if res < thr:
            break
        vn = [Ft[i] / Kse[i] + (1 if i == 2 else 0) for i in range(3)]
        un = [Lt[i] / Kbt[i] for i in range(3)]
        dv = nm.sqrt(dot(sub(vn, v), sub(vn, v)))
        du = nm.sqrt(dot(sub(un, u), sub(un, u)))
        if dv < 1e-9 * nm.sqrt(dot(v, v)) and du < 1e-9 * nm.sqrt(dot(u, u)):
            break
        v, u = vn, un
    else:
        it = max_iter
    return v, u, it


def grid(nm, s, L, dL):
    """{s} U {L - i dL : i = K-1..0}, K = #{i >= 0 : s + i dL <= L - dL/2}."""
    K = int(math.floor(float((L - s) / dL - nm.f(1) / 2))) + 1
    pts = [s] + [L - i * dL for i in range(K - 1, -1, -1)]
    return pts


def fk(rb, state, mp=None, v0u0=None):
    """Returns dict(t, p, R (row-major 3x3 lists), L, L_i, v0, u0, v_f, u_f, iters).  `v0u0` lets the
    caller impose the initial condition (to compare integrators independently of the fixed-point stop rule)."""
    nm = Num(mp)
    f = nm.f
    N = len(rb["C"])
    tau = [f(x) for x in state[:N]]
    idx = N
    rot = f(0)
    if rb.get("enable_rotation"):
        rot = f(state[idx])
        idx += 1
    s = f(state[idx]) if rb.get("enable_retraction") else f(0)
    L, dL = f(rb["L"]), f(rb["dL"])
    Kbt, Kse = stiffness(nm, rb)
    if v0u0 is None:
        v, u, iters = initial_bending(nm, rb, Kbt, Kse, tau, s, thr=f(rb["residual_threshold"]))
    else:
        v, u, iters = [f(x) for x in v0u0[0]], [f(x) for x in v0u0[1]], -1
    p = [f(0)] * 3
    R = [[f(1), f(0), f(0)], [f(0), f(1), f(0)], [f(0), f(0), f(1)]]
    Lb = f(0)
    Li = [f(0)] * N

    def deriv(y, t):
        p, R, v, u, Lb, Li = y
        vd, ud, sig = vu_dot(nm, rb, Kbt, Kse, tau, v, u, t)
        pd = [dot(R[i], v) for i in range(3)]
        # R' = R u^  -> column j of R' = R (u^ e_j) ; row form: R'[i] = R[i] x (-u) ... use direct
        uh = [[0, -u[2], u[1]], [u[2], 0, -u[0]], [-u[1], u[0], 0]]
        Rd = [[sum(R[i][k] * uh[k][j] for k in range(3)) for j in range(3)] for i in range(3)]
        return (pd, Rd, vd, ud, nm.sqrt(dot(v, v)), sig)

    def axpy(y, h, k):
        p, R, v, u, Lb, Li = y
        kp, kR, kv, ku, kL, kLi = k
        return (add(p, scale(h, kp)),
                [[R[i][j] + h * kR[i][j] for j in range(3)] for i in range(3)],
                add(v, scale(h, kv)), add(u, scale(h, ku)), Lb + h * kL,
                [a + h * b for a, b in zip(Li, kLi)])

    y = (p, R, v, u, Lb, Li)
    ts = grid(nm, s, L, dL)
    out_p, out_R = [y[0]], [y[1]]
    eps = f(2.220446049250313e-16)
    for k in range(len(ts) - 1):
        t = ts[k]
        while ts[k + 1] - t > eps:
            h = min(dL, ts[k + 1] - t)
            k1 = deriv(y, t)
            k2 = deriv(axpy(y, h / 2, k1), t + h / 2)
            k3 = deriv(axpy(y, h / 2, k2), t + h / 2)
            k4 = deriv(axpy(y, h, k3), t + h)
            y = axpy(axpy(axpy(axpy(y, h / 6, k1), h / 3, k2), h / 3, k3), h / 6, k4)
            t = t + h
        out_p.append(y[0])
        out_R.append(y[1])
    if rb.get("enable_rotation"):
        c, sn = nm.cos(rot), nm.sin(rot)
        Rz = [[c, -sn, 0], [sn, c, 0], [0, 0, 1]]
        out_p = [[dot(Rz[i], q) for i in range(3)] for q in out_p]
        out_R = [[[sum(Rz[i][k] * Rm[k][j] for k in range(3)) for j in range(3)] for i in range(3)]
                 for Rm in out_R]
    return dict(t=ts, p=out_p, R=out_R, L=y[4], L_i=y[5], v0=v, u0=u, v_f=y[2], u_f=y[3], iters=iters)
