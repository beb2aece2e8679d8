// fk.cu -- K1 `fk_rk4_fp64`: batched forward kinematics of tendon robots on sm_100a.
//
// Replaces TendonRobot::shape -> tension_shape (tendon/TendonRobot.cpp:325-500):
//   solve_initial_bending (tendon/solve_initial_bending.cpp:15-73), RK4 over t_range
//   (TendonRobot.cpp:69-84,458-462) of tendon_deriv (tendon/tendon_deriv.cpp:95-178), the
//   convergence flag (TendonRobot.cpp:188-217,470-474), rotate_z (TendonResult.cpp:13-18) and
//   the length-limit part of is_valid_shape (AbstractValidityChecker.cpp:99-114).
//
// Design (B200-first, not a translation):
//   * one configuration per thread; the whole ODE state lives in registers.
//   * the routing r, r', r'' of every tendon at every RK4 stage time is state-independent
//     because the arclength grid is anchored at L (TendonRobot.cpp:69-84): it is tabulated once
//     per robot on the host (the sin/cos of get_r_info.cpp:133-134 never run in the hot loop)
//     and staged in shared memory; a warp walks the table in lock-step so every read is a
//     broadcast.  Only the irregular first gap next to the retracted base is evaluated per thread.
//   * the per-tendon 3x3 blocks are accumulated in outer-product form
//       A_i = c3 (s2 I - q q^T),  B_i = c3 (s2 r^ - m q^T),  G_i = B_i^T,
//       H_i = c3 (s2 (|r|^2 I - r r^T) - m m^T),   m = r x q, c3 = tau / sigma^3,
//     (algebraically identical to tendon_deriv.cpp:136-157) and the 6x6 system is solved by a
//     symmetric Schur complement (same block elimination as linsubsolve2, tendon_deriv.cpp:60-87)
//     using adjugates, so a derivative evaluation needs 2 reciprocals and N+1 rsqrt only.
//   * configurations are bucketed by node count (retraction) so warps stay converged.
#include <cmath>
#include <mutex>
#include <limits>

#include "common.cuh"

namespace {

constexpr int FK_THREADS = 128;
constexpr int FK_BLOCKS_PER_SM = 2;

// Branch-free reciprocal / reciprocal square root: the hardware FP64 seed (MUFU.RCP64H /
// MUFU.RSQ64H, ~20 bits) refined by two Newton steps (relative error ~1e-16, not correctly
// rounded).  Unlike the library routines they contain no special-case branches, so the compiler
// can interleave the dependency chains of different tendons.  Valid for normal, finite inputs
// (here: |q|^2 ~ 1 and determinants of positive-definite stiffness blocks).
__device__ __forceinline__ double rcp_fast(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double e = fma(-x, y, 1.0);
  y = fma(y, e, y);
  e = fma(-x, y, 1.0);
  return fma(y, e, y);
}
__device__ __forceinline__ double rsqrt_fast(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double hx = 0.5 * x;
  double e = fma(-hx * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-hx * y, y, 0.5);
  return fma(y, e, y);
}

// routing at arbitrary t, per thread (only used inside the irregular first gap); same
// power-sum form as get_poly_vecs / get_r_info2 (tendon/get_r_info.cpp:17-40,105-144), with the
// coefficient loops fully unrolled so S, S', S'' stay in registers
template <int NT>
__device__ __forceinline__ void routing_eval(const RobotDev &rb, double t, double *out) {
  const int Na = rb.n_c, Nm = rb.n_d;
  double S[IRT_MAX_COEF], Sd[IRT_MAX_COEF], Sdd[IRT_MAX_COEF];
  S[0] = 1; Sd[0] = 0; Sdd[0] = 0;
  S[1] = t; Sd[1] = 1; Sdd[1] = 0;
#pragma unroll
  for (int i = 2; i < IRT_MAX_COEF; i++) {
    S[i] = t * S[i - 1];
    Sd[i] = i * S[i - 1];
    Sdd[i] = i * (i - 1) * S[i - 2];
  }
#pragma unroll 1
  for (int j = 0; j < NT; j++) {
    const double *C = rb.C + j * IRT_MAX_COEF, *D = rb.D + j * IRT_MAX_COEF;
    double th = 0, th1 = 0, th2 = 0, rho = 0, rho1 = 0, rho2 = 0;
#pragma unroll
    for (int i = 0; i < IRT_MAX_COEF; i++) {
      if (i < Na) { th += C[i] * S[i]; th1 += C[i] * Sd[i]; th2 += C[i] * Sdd[i]; }
      if (i < Nm) { rho += D[i] * S[i]; rho1 += D[i] * Sd[i]; rho2 += D[i] * Sdd[i]; }
    }
    double sn, cs;
    sincos(th, &sn, &cs);
    double *o = out + 6 * j;
    o[0] = rho * sn;
    o[1] = rho * cs;
    o[2] = rho1 * sn + rho * (cs * th1);
    o[3] = rho1 * cs + rho * (-sn * th1);
    o[4] = ((rho2 * sn + (2 * rho1) * (cs * th1)) - rho * (sn * th1 * th1)) + rho * (cs * th2);
    o[5] = ((rho2 * cs + (2 * rho1) * (-sn * th1)) - rho * (cs * th1 * th1)) + rho * (-sn * th2);
  }
}

// Straight and helical routing (theta of degree <= 1, rho constant: exactly the tendons whose home length has a
// closed form, TendonRobot.cpp:281-310): the power sums of get_r_info2 collapse to theta = C0 + C1 t,
// theta' = C1, theta'' = 0, rho = D0, rho' = rho'' = 0, and every term of the general formulas that is
// multiplied by one of the zeros drops out.  A double-precision sincos is ~200 instructions, and a shape with
// retraction needs the routing of all tendons at 4 head times; when all tendons wind at the same rate |C1|
// (rb.c1_uniform: helices of equal pitch, either handedness, and straight tendons) ONE sincos(|C1| t) per time
// serves every tendon through the angle-addition formulas with sin(C0), cos(C0) tabulated by the host:
// 4 sincos per shape instead of 4 N (within 2 ulp of the direct evaluation).
template <int NT, int NEVAL>
__device__ __forceinline__ void routing_eval_simple(const RobotDev &rb, const double (&t)[NEVAL],
                                                    double *const (&out)[NEVAL]) {
  if (rb.c1_uniform) {
    double sw[NEVAL], cw[NEVAL];
#pragma unroll
    for (int k = 0; k < NEVAL; k++) {
      sw[k] = 0.0; cw[k] = 1.0;
      if (rb.c1_abs != 0.0) sincos(rb.c1_abs * t[k], &sw[k], &cw[k]);
    }
#pragma unroll 1
    for (int j = 0; j < NT; j++) {
      const double s0 = rb.sin_c0[j], c0 = rb.cos_c0[j], sg = rb.c1_sign[j];
      const double c1 = sg * rb.c1_abs, rho = rb.D[j * IRT_MAX_COEF];
#pragma unroll
      for (int k = 0; k < NEVAL; k++) {
        const double ssw = sg * sw[k];
        const double cwk = (sg != 0.0) ? cw[k] : 1.0;   // a straight tendon beside helices does not wind
        const double sn = fma(s0, cwk, c0 * ssw), cs = fma(c0, cwk, -s0 * ssw);
        double *o = out[k] + 6 * j;
        o[0] = rho * sn;
        o[1] = rho * cs;
        o[2] = rho * (cs * c1);
        o[3] = rho * (-sn * c1);
        o[4] = -(rho * (sn * c1 * c1));
        o[5] = -(rho * (cs * c1 * c1));
      }
    }
    return;
  }
#pragma unroll 1
  for (int j = 0; j < NT; j++) {
    const double c0 = rb.C[j * IRT_MAX_COEF], c1 = (rb.n_c > 1) ? rb.C[j * IRT_MAX_COEF + 1] : 0.0;
    const double rho = rb.D[j * IRT_MAX_COEF];
#pragma unroll 1
    for (int k = 0; k < NEVAL; k++) {
      double sn, cs;
      sincos(fma(c1, t[k], c0), &sn, &cs);
      double *o = out[k] + 6 * j;
      o[0] = rho * sn;
      o[1] = rho * cs;
      o[2] = rho * (cs * c1);
      o[3] = rho * (-sn * c1);
      o[4] = -(rho * (sn * c1 * c1));
      o[5] = -(rho * (cs * c1 * c1));
    }
  }
}

// Where a stage reads its routing row from.  RtPtr: a pointer to [NT][6] values (the shared-memory table, or the
// per-thread rows of the irregular first gap); it forms the products of r itself.  RtConst: a row of the wide copy
// of the table in CONSTANT memory ([NT][IRT_CT_WIDTH]: r, r', r'' and the products rx^2, ry^2, rx ry, |r|^2 that the
// host tabulated), named by a warp-uniform index: the values arrive through the uniform datapath (LDCU -> uniform
// registers) and enter the FP64 instructions as uniform-register operands.  That matters because the FP64 pipe's
// issue rate is bounded by register-file reads: a DFMA with three distinct register pairs costs 3 issue cycles
// instead of 2 (irt_measure_fp64_rate mode 2: 0.68 of the DFMA peak), and every routing value that comes from a
// uniform register is one pair less -- and the values of a row occupy no registers of any thread.
constexpr int FK_CT_DOUBLES = 8192;   // the whole 64 KB constant bank: 136 rows of a 6-tendon robot
__constant__ double c_fk_tab[FK_CT_DOUBLES];
struct RtPtr {
  const double *p;
  __device__ __forceinline__ double rx(int j) const { return p[6 * j + 0]; }
  __device__ __forceinline__ double ry(int j) const { return p[6 * j + 1]; }
  __device__ __forceinline__ double dx(int j) const { return p[6 * j + 2]; }
  __device__ __forceinline__ double dy(int j) const { return p[6 * j + 3]; }
  __device__ __forceinline__ double ddx(int j) const { return p[6 * j + 4]; }
  __device__ __forceinline__ double ddy(int j) const { return p[6 * j + 5]; }
  // rounded like the host's table (no contraction), so both paths see the same values
  __device__ __forceinline__ double rxx(int j) const { return __dmul_rn(rx(j), rx(j)); }
  __device__ __forceinline__ double ryy(int j) const { return __dmul_rn(ry(j), ry(j)); }
  __device__ __forceinline__ double rxy(int j) const { return __dmul_rn(rx(j), ry(j)); }
  __device__ __forceinline__ double rr(int j) const { return __dadd_rn(rxx(j), ryy(j)); }
};
struct RtConst {
  int base;
  __device__ __forceinline__ double at(int j, int k) const { return c_fk_tab[base + IRT_CT_WIDTH * j + k]; }
  __device__ __forceinline__ double rx(int j) const { return at(j, 0); }
  __device__ __forceinline__ double ry(int j) const { return at(j, 1); }
  __device__ __forceinline__ double dx(int j) const { return at(j, 2); }
  __device__ __forceinline__ double dy(int j) const { return at(j, 3); }
  __device__ __forceinline__ double ddx(int j) const { return at(j, 4); }
  __device__ __forceinline__ double ddy(int j) const { return at(j, 5); }
  __device__ __forceinline__ double rxx(int j) const { return at(j, 6); }
  __device__ __forceinline__ double ryy(int j) const { return at(j, 7); }
  __device__ __forceinline__ double rxy(int j) const { return at(j, 8); }
  __device__ __forceinline__ double rr(int j) const { return at(j, 9); }
};

// (v', u', sigma_i) at one RK4 stage.  rt: the routing of the NT tendons (RtPtr or RtConst).
template <int NT, typename RT>
__device__ __forceinline__ void vu_dot(const RT &rt, const double (&tau)[NT],
                                       const double (&Kse)[3], const double (&Kbt)[3],
                                       const double (&v)[3], const double (&u)[3],
                                       double (&vd)[3], double (&ud)[3], double (&sig)[NT]) {
  // symmetric A (00,01,02,11,12,22), full B (row-major), symmetric H, a, b.  The stiffness diagonals K_se, K_bt
  // are the start values of the sums they belong to.
  double a00 = 0, a01 = 0, a02 = -0.0, a11 = 0, a12 = -0.0, a22 = Kse[2];
  double b00 = 0, b01 = 0, b02 = 0, b10 = 0, b11 = 0, b12 = 0, b20 = 0, b21 = 0, b22 = 0;
  double h00 = Kbt[0], h01 = 0, h02 = 0, h11 = Kbt[1], h12 = 0, h22 = Kbt[2];
  // sums that are built with plain additions start from -0.0: (-0.0) + x == x for every x, so the first tendon's
  // "0 + x" folds away (with +0.0 it may not: 0 + (-0) is +0), one FP64 instruction less per sum and stage; the
  // value of a sum can differ from the +0.0 start only in the sign of an exact zero
  double av0 = -0.0, av1 = -0.0, av2 = -0.0, bv0 = 0, bv1 = 0, bv2 = 0;
  double esum = -0.0;
#pragma unroll
  for (int j = 0; j < NT; j++) {
    const double rx = rt.rx(j), ry = rt.ry(j);
    const double dx = rt.dx(j), dy = rt.dy(j);
    const double ddx = rt.ddx(j), ddy = rt.ddy(j);
    // q = u x r + r' + v        (r_z = r'_z = r''_z = 0)
    const double qx = fma(-u[2], ry, dx + v[0]);
    const double qy = fma(u[2], rx, dy + v[1]);
    const double qz = fma(u[0], ry, fma(-u[1], rx, v[2]));
    const double s2 = fma(qx, qx, fma(qy, qy, qz * qz));
    const double rs = rsqrt_fast(s2);
    sig[j] = s2 * rs;
    const double e = tau[j] * rs;        // tau / sigma
    const double c3 = e * (rs * rs);     // tau / sigma^3
    // With r_z = 0, m = r x q = (ry qz, -rx qz, mz), and t = c3 qz q, kap = e - c3 qz^2:
    //   A_i = e I - c3 q q^T                 z row: -t (+ e on the diagonal: kap)
    //   B_i = e r^ - c3 m q^T                rows 0, 1: -ry t, rx t (+ e r^: ry kap, -rx kap in column 2);
    //                                        row 2: -c3 mz q (+ e r^: -e ry, e rx)
    //   H_i = e (|r|^2 I - r r^T) - c3 m m^T  = kap [[ry^2, -rx ry], [-rx ry, rx^2]] in the top-left block,
    //                                          -+ r (c3 qz mz) in column 2, e |r|^2 - c3 mz^2 on the diagonal
    // so most accumulations are one register pair against a routing value or product that the fast path reads
    // from a uniform register
    const double mz = fma(rx, qy, -ry * qx);
    const double cqx = c3 * qx, cqy = c3 * qy, cqz = c3 * qz, cmz = c3 * mz;
    const double tx = cqz * qx, ty = cqz * qy, kap = fma(-cqz, qz, e), tzm = cqz * mz;
    a00 = fma(-cqx, qx, a00); a01 = fma(-cqx, qy, a01); a11 = fma(-cqy, qy, a11);
    a02 -= tx; a12 -= ty; a22 += kap;
    esum += e;
    b00 = fma(-ry, tx, b00); b01 = fma(-ry, ty, b01); b02 = fma(ry, kap, b02);
    b10 = fma(rx, tx, b10); b11 = fma(rx, ty, b11); b12 = fma(-rx, kap, b12);
    b20 = fma(-cmz, qx, b20); b21 = fma(-cmz, qy, b21); b22 = fma(-cmz, qz, b22);
    b20 = fma(-e, ry, b20); b21 = fma(e, rx, b21);
    h00 = fma(kap, rt.ryy(j), h00); h01 = fma(-kap, rt.rxy(j), h01); h11 = fma(kap, rt.rxx(j), h11);
    h02 = fma(-ry, tzm, h02); h12 = fma(rx, tzm, h12);
    h22 = fma(e, rt.rr(j), h22); h22 = fma(-cmz, mz, h22);
    // w = u x (q + r') + r''
    const double gx = qx + dx, gy = qy + dy, gz = qz;
    const double wx = fma(u[1], gz, fma(-u[2], gy, ddx));
    const double wy = fma(u[2], gx, fma(-u[0], gz, ddy));
    const double wz = fma(u[0], gy, -u[1] * gx);
    const double qw = fma(qx, wx, fma(qy, wy, qz * wz));
    // a_i = A_i w = e w - c3 q (q.w)
    const double ax = fma(e, wx, -cqx * qw), ay = fma(e, wy, -cqy * qw), az = fma(e, wz, -cqz * qw);
    av0 += ax; av1 += ay; av2 += az;
    // b_i = r x a_i
    bv0 = fma(ry, az, bv0); bv1 = fma(-rx, az, bv1); bv2 = fma(rx, ay, bv2); bv2 = fma(-ry, ax, bv2);
  }
  // A += (sum e) I on the diagonal entries whose sums do not hold it yet, and K_se
  a00 += esum + Kse[0]; a11 += esum + Kse[1];

  // right-hand sides (tendon_deriv.cpp:159-161), K diagonal
  const double kv0 = Kse[0] * v[0], kv1 = Kse[1] * v[1], kv2 = Kse[2] * (v[2] - 1.0);
  const double ku0 = Kbt[0] * u[0], ku1 = Kbt[1] * u[1], ku2 = Kbt[2] * u[2];
  // c = -u x Ku - v x Kv - b ; d = -u x Kv - a
  const double c0 = -(fma(u[1], ku2, -u[2] * ku1)) - (fma(v[1], kv2, -v[2] * kv1)) - bv0;
  const double c1 = -(fma(u[2], ku0, -u[0] * ku2)) - (fma(v[2], kv0, -v[0] * kv2)) - bv1;
  const double c2 = -(fma(u[0], ku1, -u[1] * ku0)) - (fma(v[0], kv1, -v[1] * kv0)) - bv2;
  const double d0 = -(fma(u[1], kv2, -u[2] * kv1)) - av0;
  const double d1 = -(fma(u[2], kv0, -u[0] * kv2)) - av1;
  const double d2 = -(fma(u[0], kv1, -u[1] * kv0)) - av2;

  // solve [[A, B^T],[B, H]] [v'; u'] = [d; c]:  adjugate of symmetric A
  const double C00 = fma(a11, a22, -a12 * a12), C01 = fma(a02, a12, -a01 * a22),
               C02 = fma(a01, a12, -a02 * a11), C11 = fma(a00, a22, -a02 * a02),
               C12 = fma(a01, a02, -a00 * a12), C22 = fma(a00, a11, -a01 * a01);
  const double detA = fma(a00, C00, fma(a01, C01, a02 * C02));
  const double idA = rcp_fast(detA);
  // Y = adj(A) B^T (unscaled):  Y[i][j] = sum_k C[i][k] B[j][k]
  const double y00 = fma(C00, b00, fma(C01, b01, C02 * b02));
  const double y01 = fma(C00, b10, fma(C01, b11, C02 * b12));
  const double y02 = fma(C00, b20, fma(C01, b21, C02 * b22));
  const double y10 = fma(C01, b00, fma(C11, b01, C12 * b02));
  const double y11 = fma(C01, b10, fma(C11, b11, C12 * b12));
  const double y12 = fma(C01, b20, fma(C11, b21, C12 * b22));
  const double y20 = fma(C02, b00, fma(C12, b01, C22 * b02));
  const double y21 = fma(C02, b10, fma(C12, b11, C22 * b12));
  const double y22 = fma(C02, b20, fma(C12, b21, C22 * b22));
  // S = H - idA * B Y   (symmetric)
  const double s00 = fma(-idA, fma(b00, y00, fma(b01, y10, b02 * y20)), h00);
  const double s01 = fma(-idA, fma(b00, y01, fma(b01, y11, b02 * y21)), h01);
  const double s02 = fma(-idA, fma(b00, y02, fma(b01, y12, b02 * y22)), h02);
  const double s11 = fma(-idA, fma(b10, y01, fma(b11, y11, b12 * y21)), h11);
  const double s12 = fma(-idA, fma(b10, y02, fma(b11, y12, b12 * y22)), h12);
  const double s22 = fma(-idA, fma(b20, y02, fma(b21, y12, b22 * y22)), h22);
  // z = A^-1 d
  const double z0 = idA * fma(C00, d0, fma(C01, d1, C02 * d2));
  const double z1 = idA * fma(C01, d0, fma(C11, d1, C12 * d2));
  const double z2 = idA * fma(C02, d0, fma(C12, d1, C22 * d2));
  // y = c - B z
  const double r0 = c0 - fma(b00, z0, fma(b01, z1, b02 * z2));
  const double r1 = c1 - fma(b10, z0, fma(b11, z1, b12 * z2));
  const double r2 = c2 - fma(b20, z0, fma(b21, z1, b22 * z2));
  // u' = S^-1 y
  const double T00 = fma(s11, s22, -s12 * s12), T01 = fma(s02, s12, -s01 * s22),
               T02 = fma(s01, s12, -s02 * s11), T11 = fma(s00, s22, -s02 * s02),
               T12 = fma(s01, s02, -s00 * s12), T22 = fma(s00, s11, -s01 * s01);
  const double detS = fma(s00, T00, fma(s01, T01, s02 * T02));
  const double idS = rcp_fast(detS);
  ud[0] = idS * fma(T00, r0, fma(T01, r1, T02 * r2));
  ud[1] = idS * fma(T01, r0, fma(T11, r1, T12 * r2));
  ud[2] = idS * fma(T02, r0, fma(T12, r1, T22 * r2));
  // v' = z - idA * Y u'
  vd[0] = fma(-idA, fma(y00, ud[0], fma(y01, ud[1], y02 * ud[2])), z0);
  vd[1] = fma(-idA, fma(y10, ud[0], fma(y11, ud[1], y12 * ud[2])), z1);
  vd[2] = fma(-idA, fma(y20, ud[0], fma(y21, ud[1], y22 * ud[2])), z2);
}

// Integration state of one configuration; it lives in registers (255 per thread, 8 warps per SM).
template <int NT>
struct FkState {
  double R[9];  // column-major (R[i + 3 j]) like Eigen
  double v[3], u[3];
  double p[3];
  double L;       // backbone length
  double Li[NT];  // tendon lengths
};

// one classic RK4 step of size h; rt0/rt1/rt2 = routing at t, t+h/2, t+h.
// The four stages are a real loop (not unrolled): the hot loop body is ONE copy of vu_dot, which
// keeps the instruction footprint inside the SM's instruction cache.
template <int NT, typename RT>
__device__ __forceinline__ void rk4_step(FkState<NT> &x, const double (&tau)[NT],
                                         const double (&Kse)[3], const double (&Kbt)[3], double h,
                                         const RT &rt0, const RT &rt1, const RT &rt2) {
  const double hh = 0.5 * h, w1 = h * (1.0 / 6.0), w2 = h * (1.0 / 3.0);
  double sv[3], su[3], sR[9];      // stage values
  double aR[9], av[3], au[3];      // k1 + 2 k2 + 2 k3 + k4
  double vd[3], ud[3], sig[NT], Rd[9];
#pragma unroll
  for (int i = 0; i < 3; i++) { sv[i] = x.v[i]; su[i] = x.u[i]; av[i] = 0.0; au[i] = 0.0; }
#pragma unroll
  for (int i = 0; i < 9; i++) { sR[i] = x.R[i]; aR[i] = 0.0; }

#pragma unroll 1
  for (int stage = 0; stage < 4; stage++) {
    const bool outer = (stage == 0) || (stage == 3);
    const RT rt = (stage == 0) ? rt0 : ((stage == 3) ? rt2 : rt1);
    const double wq = outer ? w1 : w2;     // quadrature weight
    const double wk = outer ? 1.0 : 2.0;   // slope weight
    const double a = (stage == 2) ? h : hh;
    vu_dot<NT, RT>(rt, tau, Kse, Kbt, sv, su, vd, ud, sig);
    // p' = R v ; L' = |v| ; L_i' = sigma_i : pure quadratures, accumulate in place
#pragma unroll
    for (int i = 0; i < 3; i++)
      x.p[i] = fma(wq, fma(sR[i], sv[0], fma(sR[i + 3], sv[1], sR[i + 6] * sv[2])), x.p[i]);
    {
      const double vv = fma(sv[0], sv[0], fma(sv[1], sv[1], sv[2] * sv[2]));
      x.L = fma(wq, vv * rsqrt_fast(vv), x.L);
    }
#pragma unroll
    for (int j = 0; j < NT; j++) x.Li[j] = fma(wq, sig[j], x.Li[j]);
    // R' = R u^
#pragma unroll
    for (int i = 0; i < 3; i++) {
      Rd[i] = fma(sR[i + 3], su[2], -sR[i + 6] * su[1]);
      Rd[i + 3] = fma(sR[i + 6], su[0], -sR[i] * su[2]);
      Rd[i + 6] = fma(sR[i], su[1], -sR[i + 3] * su[0]);
    }
#pragma unroll
    for (int i = 0; i < 9; i++) { aR[i] = fma(wk, Rd[i], aR[i]); sR[i] = fma(a, Rd[i], x.R[i]); }
#pragma unroll
    for (int i = 0; i < 3; i++) {
      av[i] = fma(wk, vd[i], av[i]); au[i] = fma(wk, ud[i], au[i]);
      sv[i] = fma(a, vd[i], x.v[i]); su[i] = fma(a, ud[i], x.u[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < 9; i++) x.R[i] = fma(w1, aR[i], x.R[i]);
#pragma unroll
  for (int i = 0; i < 3; i++) { x.v[i] = fma(w1, av[i], x.v[i]); x.u[i] = fma(w1, au[i], x.u[i]); }
}

struct RotZ {
  double c, s;
  int on;
};

template <int NT>
__device__ __forceinline__ void emit_node(const irt_fk_outputs &o, int64_t row_base, int k,
                                          double t, const FkState<NT> &x, const RotZ &rz) {
  const int64_t row = row_base + k;
  const double p0 = x.p[0], p1 = x.p[1], p2 = x.p[2];
  double px = p0, py = p1;
  if (rz.on) {
    px = rz.c * p0 - rz.s * p1;
    py = rz.s * p0 + rz.c * p1;
  }
  if (o.p) {
    double *dst = o.p + row * 3;
    dst[0] = px; dst[1] = py; dst[2] = p2;
  }
  if (o.t) o.t[row] = t;
  if (o.R) {
    double *dst = o.R + row * 9;
#pragma unroll
    for (int j = 0; j < 3; j++) {
      double r0 = x.R[3 * j], r1 = x.R[3 * j + 1];
      if (rz.on) {
        dst[3 * j] = rz.c * r0 - rz.s * r1;
        dst[3 * j + 1] = rz.s * r0 + rz.c * r1;
      } else {
        dst[3 * j] = r0;
        dst[3 * j + 1] = r1;
      }
      dst[3 * j + 2] = x.R[3 * j + 2];
    }
  }
}

// ---- bucket keys ------------------------------------------------------------------------------
// Configurations are counting-sorted by (RK4 step count, tension bin) before the RK4 kernel so that the lanes
// of a warp run the same number of steps (retraction) and about the same number of fixed-point iterations
// (solve_initial_bending.cpp:41-70: the iteration count grows with the tension; binning sum(tau) brings the
// warp-max of a C2 batch from 33 to 24 iterations at a mean of 17.5).  key = bucket | K << 16, where K is the
// node count of util::range's accumulation (vector_ops.h:67-75) -- evaluated ONCE here, in a memory-bound
// kernel, instead of as a latency-bound chain of dependent additions in front of every shape.
constexpr int FK_TAU_BINS = 8;
constexpr int FK_K_BAD = 0xFFFF;   // the grid would exceed max_points (s < 0 beyond the first gap)

__device__ __forceinline__ int fk_bucket_key(const RobotDev &rb, const double *st, int state_size, int *K_out) {
  int T = 0, K = 0;
  if (rb.enable_retraction) {
    const double s = st[state_size - 1];
    if (s >= -rb.dL && s < rb.L) {
      const double lim = rb.L - (rb.dL / 2);
      for (double p = s; p <= lim; p += rb.dL) K++;
      if (K > rb.Kfull) {
        K = FK_K_BAD;   // flagged IRT_FLAG_BAD_STATE by the FK kernel
      } else if (K >= 1) {
        const double t1 = rb.node_t[K - 1];
        const double h0 = fmin(rb.dL, t1 - s);
        T = K - 1 + ((t1 - (s + h0) > 2.220446049250313e-16) ? 2 : 1);
      }
    }
  } else {
    K = rb.Kfull;
    T = rb.Kfull - 1 + ((rb.n_head == 4) ? 2 : 1);
  }
  double ts = 0.0;
  for (int j = 0; j < rb.n_tendons; j++) ts += st[j];
  int bin = (int)(ts * rb.tau_bin_scale);
  bin = (bin < 0 || !(ts == ts)) ? 0 : (bin >= FK_TAU_BINS ? FK_TAU_BINS - 1 : bin);
  *K_out = K;
  return T * FK_TAU_BINS + bin;
}

struct FkArgs {
  const double *states;   // [.][state_size]; configuration i of this launch is row lo + i
  int state_size;
  int64_t n;              // number of configurations (d_range == nullptr) or an upper bound of it
  const int32_t *range;   // device {lo, hi} or nullptr (lo = 0, hi = n)
  int cap_pts;
  irt_fk_outputs o;       // output arrays are indexed by the absolute row lo + i
  const int32_t *perm;    // [n] bucket order (relative indices)
  const int32_t *keys;    // [n] bucket | K << 16 (relative indices)
  const int64_t *row_off; // packed rows (absolute index) or nullptr
  int32_t *work;          // dynamic work counter (zero at launch)
  int use_const;          // c_fk_tab holds this robot's routing table
};

// Persistent kernel: FK_BLOCKS_PER_SM CTAs per SM stage the routing table once, then every WARP fetches the next
// 32 configurations of the bucket order from a global counter until the batch is done (no CTA-wide barrier after
// the staging, no tail of half-empty CTAs, and the batch size may live in device memory: K2's bisection rounds
// launch this kernel without the host knowing how many samples a round has).
template <int NT, bool RETRACT>
__global__ void __launch_bounds__(FK_THREADS, FK_BLOCKS_PER_SM) fk_rk4_fp64_kernel(const RobotDev rb, const FkArgs a) {
  extern __shared__ double smem[];
  double *tab = smem;                                // [n_table][NT][6]
  double *head = smem + (size_t)rb.n_table * NT * 6; // [4][NT][6]
  int64_t lo = 0, n = a.n;
  if (a.range) { lo = a.range[0]; n = (int64_t)a.range[1] - lo; }
  if (n <= 0 || (int64_t)blockIdx.x * FK_THREADS >= n) return;   // the other CTAs cover the batch
  for (int i = threadIdx.x; i < rb.n_table * NT * 6; i += blockDim.x) tab[i] = rb.table[i];
  for (int i = threadIdx.x; i < 4 * NT * 6; i += blockDim.x) head[i] = rb.head[i];
  __syncthreads();
  const irt_fk_outputs &o = a.o;
  const int state_size = a.state_size, cap_pts = a.cap_pts;
  const double Kse[3] = {rb.Kse[0], rb.Kse[1], rb.Kse[2]};
  const double Kbt[3] = {rb.Kbt[0], rb.Kbt[1], rb.Kbt[2]};
  const int lane = threadIdx.x & 31;

  // every WARP fetches the next 32 configurations of the bucket order from a global counter
#pragma unroll 1
  for (;;) {
  int64_t wbase = 0;
  if (lane == 0) wbase = (int64_t)atomicAdd(a.work, 32);
  wbase = __shfl_sync(0xffffffffu, wbase, 0);
  if (wbase >= n) break;
  const int64_t gi = wbase + lane;
  const bool in_range = gi < n;
  const int64_t rel = in_range ? (a.perm ? (int64_t)a.perm[gi] : gi) : 0;
  const int64_t cfg = lo + rel;
  const double *st = a.states + cfg * state_size;
  // first output row of this configuration: dense [n][cap_pts] layout, or packed rows (row_off[cfg])
  const int64_t row_base = a.row_off ? (in_range ? a.row_off[cfg] : 0) : cfg * cap_pts;

  double tau[NT];
#pragma unroll
  for (int j = 0; j < NT; j++) tau[j] = in_range ? st[j] : 0.0;
  RotZ rz{1.0, 0.0, 0};
  if (rb.enable_rotation) {
    rz.on = 1;
    sincos(in_range ? st[NT] : 0.0, &rz.s, &rz.c);
  }
  double s_start = 0.0;
  if (RETRACT) s_start = in_range ? st[state_size - 1] : 0.0;

  uint32_t flags = 0;
  bool active = in_range;
  // The reference integrates from any s_start (TendonRobot.cpp:345-359 only truncates at L).  A base
  // slightly before 0 is what the finite-difference Jacobians of its IK produce (state - d), so
  // s < 0 is supported as long as the grid still fits max_points (K <= Kfull below; the first gap is
  // always in [dL/2, 3dL/2), so the two head steps suffice); NaN or anything further out is outside the
  // reference's state space (OMPL bounds [0, L]) and is flagged.
  if (RETRACT && !(s_start >= -rb.dL)) {
    flags |= IRT_FLAG_BAD_STATE;
    active = false;
  }
  if (s_start > rb.L) s_start = rb.L;  // TendonRobot.cpp:359

  // number of nodes K: util::range's accumulation (vector_ops.h:67-75), bit-for-bit -- taken from the bucket
  // key (fk_bucket_key ran the accumulation)
  int K = 0;
  if (active) {
    if (RETRACT) {
      K = (int)((uint32_t)a.keys[rel] >> 16);
      if (K == FK_K_BAD) {   // only possible for s < 0: one grid point more than the outputs hold
        flags |= IRT_FLAG_BAD_STATE;
        active = false;
        K = 0;
      }
    } else {
      K = rb.Kfull;
    }
  }
  const bool degenerate = active && (s_start == rb.L);  // TendonRobot.cpp:361-372

  FkState<NT> x;
#pragma unroll
  for (int i = 0; i < 3; i++) { x.p[i] = 0; x.v[i] = 0; x.u[i] = 0; }
#pragma unroll
  for (int i = 0; i < 9; i++) x.R[i] = 0;
  x.R[0] = x.R[4] = x.R[8] = 1.0;
  x.v[2] = 1.0;
  x.L = 0;
#pragma unroll
  for (int j = 0; j < NT; j++) x.Li[j] = 0;

  int iters = 0, nsteps = 0;
  double u0[3] = {0, 0, 0}, v0[3] = {0, 0, 1};
  double rt_local[NT * 6], rt_h1[NT * 6], rt_h2[NT * 6], rt_h3[NT * 6];
  const bool run = active && !degenerate;
  // L - dL/2 < s < L: the grid is the single point {s} (K == 0), nothing to integrate
  const bool integ = run && K >= 1;

  // ---- head: the irregular first gap s -> node K-1 takes one or two steps (h = min(dL, t_next - t),
  // repeated while t_next - t > eps, odeint integrate_times) -------------------------------------
  int nhead = 0;
  double hh0 = 0.0, hh1 = 0.0;
  const double *hd0 = head, *hd1 = head + NT * 6, *hd2 = head + 2 * NT * 6, *hd3 = head + 3 * NT * 6;
  if (RETRACT) {
    double tc = s_start;
    if (integ) {
      const double eps = 2.220446049250313e-16;
      const double t1 = rb.node_t[K - 1];
      hh0 = fmin(rb.dL, t1 - s_start);
      nhead = 1;
      tc = s_start + hh0;
      if (t1 - tc > eps) {
        hh1 = fmin(rb.dL, t1 - tc);
        nhead = 2;
      }
    }
    if (run) {   // routing at s (initial condition) and at the stage times of the head steps
      const double tt[4] = {s_start, s_start + 0.5 * hh0, tc, tc + 0.5 * hh1};
      double *const oo[4] = {rt_local, rt_h1, rt_h2, rt_h3};
      if (rb.simple_routing) {
        routing_eval_simple<NT, 4>(rb, tt, oo);
      } else {
        routing_eval<NT>(rb, tt[0], rt_local);
        if (integ) {
          routing_eval<NT>(rb, tt[1], rt_h1);
          if (nhead == 2) {
            routing_eval<NT>(rb, tt[2], rt_h2);
            routing_eval<NT>(rb, tt[3], rt_h3);
          }
        }
      }
    }
    hd0 = rt_local; hd1 = rt_h1; hd2 = rt_h2; hd3 = rt_h3;
  } else if (integ) {
    nhead = (rb.n_head == 4) ? 2 : 1;
    hh0 = rb.head_h[0];
    hh1 = rb.head_h[1];
  }

  if (run) {
    // ---- initial condition: solve_initial_bending.cpp:15-73 ------------------------------
    const double *rt_s = RETRACT ? rt_local : head;
    double v[3] = {0, 0, 1}, u[3] = {0, 0, 0};
    // Same iteration as the reference; the unit vectors use rsqrt and the three exit tests
    // compare squares (residual < thr <=> residual^2 < thr^2, |dv| < 1e-9 |v| <=> |dv|^2 <
    // 1e-18 |v|^2), which keeps FP64 divisions and square roots out of the loop.
    const double thr2 = rb.residual_threshold * rb.residual_threshold;
    for (iters = 0; iters < 1000; ++iters) {
      double Ft0 = 0, Ft1 = 0, Ft2 = 0, Lt0 = 0, Lt1 = 0, Lt2 = 0;
#pragma unroll
      for (int k = 0; k < NT; k++) {
        const double rx = rt_s[6 * k], ry = rt_s[6 * k + 1], dx = rt_s[6 * k + 2], dy = rt_s[6 * k + 3];
        const double qx = fma(-u[2], ry, dx + v[0]);
        const double qy = fma(u[2], rx, dy + v[1]);
        const double qz = fma(u[0], ry, fma(-u[1], rx, v[2]));
        const double tr = tau[k] * rsqrt_fast(fma(qx, qx, fma(qy, qy, qz * qz)));
        const double fx = tr * qx, fy = tr * qy, fz = tr * qz;  // tau * unit(q)
        Ft0 -= fx; Ft1 -= fy; Ft2 -= fz;
        Lt0 = fma(-ry, fz, Lt0); Lt1 = fma(rx, fz, Lt1); Lt2 -= fma(rx, fy, -ry * fx);
      }
      const double e0 = fma(Kse[0], v[0], -Ft0), e1 = fma(Kse[1], v[1], -Ft1),
                   e2 = fma(Kse[2], v[2] - 1.0, -Ft2);
      const double g0 = fma(Kbt[0], u[0], -Lt0), g1 = fma(Kbt[1], u[1], -Lt1),
                   g2 = fma(Kbt[2], u[2], -Lt2);
      const double res2 = fma(e0, e0, fma(e1, e1, e2 * e2)) + fma(g0, g0, fma(g1, g1, g2 * g2));
      if (res2 < thr2) break;
      const double vn0 = rb.KseInv[0] * Ft0, vn1 = rb.KseInv[1] * Ft1, vn2 = fma(rb.KseInv[2], Ft2, 1.0);
      const double un0 = rb.KbtInv[0] * Lt0, un1 = rb.KbtInv[1] * Lt1, un2 = rb.KbtInv[2] * Lt2;
      const double a0 = vn0 - v[0], a1 = vn1 - v[1], a2 = vn2 - v[2];
      const double b0 = un0 - u[0], b1 = un1 - u[1], b2 = un2 - u[2];
      const double dv2 = fma(a0, a0, fma(a1, a1, a2 * a2)), du2 = fma(b0, b0, fma(b1, b1, b2 * b2));
      const double nv2 = fma(v[0], v[0], fma(v[1], v[1], v[2] * v[2]));
      const double nu2 = fma(u[0], u[0], fma(u[1], u[1], u[2] * u[2]));
      if (dv2 < 1e-18 * nv2 && du2 < 1e-18 * nu2) break;
      v[0] = vn0; v[1] = vn1; v[2] = vn2;
      u[0] = un0; u[1] = un1; u[2] = un2;
    }
#pragma unroll
    for (int i = 0; i < 3; i++) { x.v[i] = v0[i] = v[i]; x.u[i] = u0[i] = u[i]; }

    // ---- convergence flag: calc_point_forces at the base, R = I (TendonRobot.cpp:188-217) --
    {
      double Ft[3] = {0, 0, 0}, Lt[3] = {0, 0, 0};
#pragma unroll
      for (int k = 0; k < NT; k++) {
        const double rx = rt_s[6 * k], ry = rt_s[6 * k + 1], dx = rt_s[6 * k + 2], dy = rt_s[6 * k + 3];
        double qx = (-u[2] * ry + dx) + v[0];
        double qy = (u[2] * rx + dy) + v[1];
        double qz = (u[0] * ry - u[1] * rx) + v[2];
        const double nrm = sqrt(qx * qx + qy * qy + qz * qz);
        const double fx = -tau[k] * (qx / nrm), fy = -tau[k] * (qy / nrm), fz = -tau[k] * (qz / nrm);
        Ft[0] += fx; Ft[1] += fy; Ft[2] += fz;
        Lt[0] += ry * fz; Lt[1] += -rx * fz; Lt[2] += rx * fy - ry * fx;
      }
      const double e0 = Kse[0] * v[0] - Ft[0], e1 = Kse[1] * v[1] - Ft[1], e2 = Kse[2] * (v[2] - 1.0) - Ft[2];
      const double g0 = Kbt[0] * u[0] - Lt[0], g1 = Kbt[1] * u[1] - Lt[1], g2 = Kbt[2] * u[2] - Lt[2];
      const double resid = sqrt((e0 * e0 + e1 * e1 + e2 * e2) + (g0 * g0 + g1 * g1 + g2 * g2));
      if (!(resid <= rb.residual_threshold)) flags |= IRT_FLAG_NONCONVERGED;
    }
  }

  // ---- integrate_times(runge_kutta4) over the grid {s} U {node K-1 .. node 0} --------------
  // Head steps, then the regular steps node q -> node q-1.  All steps run through ONE rk4_step call site in
  // a loop that is end-aligned across the warp, so that every lane is at the same regular step q in the
  // same iteration (table reads are broadcasts).
  if (run) emit_node<NT>(o, row_base, 0, s_start, x, rz);
  {
    const int T = integ ? (K - 1 + nhead) : 0;
    // the warp's step count: every lane runs the loop the same number of times (lanes that do not integrate idle
    // in it), so the warp-wide vote of the fast path below is reached by all 32 lanes, and q is warp-uniform
    const int Tmax = __reduce_max_sync(0xffffffffu, T);
    nsteps = T;
#pragma unroll 1
    for (int j = 0; j < Tmax; j++) {
      const int q = Tmax - j;  // regular step q: node q -> node q-1 (1 <= q <= K-1)
      // every lane of the warp takes the regular step q (the common case: buckets are warps of equal step
      // counts): the routing rows come from constant memory by a warp-uniform index, the step size is uniform
      if (a.use_const && __all_sync(0xffffffffu, integ && q <= K - 1)) {
        const int b0 = 2 * q * NT * IRT_CT_WIDTH;
        rk4_step<NT, RtConst>(x, tau, Kse, Kbt, rb.dL, RtConst{b0}, RtConst{b0 - NT * IRT_CT_WIDTH},
                              RtConst{b0 - 2 * NT * IRT_CT_WIDTH});
        emit_node<NT>(o, row_base, K - q + 1, rb.node_t[q - 1], x, rz);
        continue;
      }
      if (integ && q <= K - 1 + nhead) {
        const double *p0, *p1, *p2;
        double h;
        int emit_idx;
        if (q <= K - 1) {
          p0 = tab + (size_t)(2 * q) * NT * 6;
          p1 = p0 - NT * 6;
          p2 = p0 - 2 * NT * 6;
          h = rb.dL;
          emit_idx = K - q + 1;
        } else if (q == K) {  // the head step that lands on node K-1
          p0 = (nhead == 2) ? hd2 : hd0;
          p1 = (nhead == 2) ? hd3 : hd1;
          p2 = tab + (size_t)(2 * (K - 1)) * NT * 6;
          h = (nhead == 2) ? hh1 : hh0;
          emit_idx = 1;
        } else {  // q == K + 1: first of two head steps, lands between grid points (not observed)
          p0 = hd0; p1 = hd1; p2 = hd2;
          h = hh0;
          emit_idx = -1;
        }
        rk4_step<NT, RtPtr>(x, tau, Kse, Kbt, h, RtPtr{p0}, RtPtr{p1}, RtPtr{p2});
        if (emit_idx >= 0) emit_node<NT>(o, row_base, emit_idx, rb.node_t[K - emit_idx], x, rz);
      }
    }
  }

  if (!in_range) continue;
  int npts = 0;
  if (degenerate) {
    npts = 1;
    emit_node<NT>(o, row_base, 0, s_start, x, rz);  // p = 0, R = I, v = e3, u = 0
  } else if (run) {
    npts = K + 1;
  }
  // length limits: is_within_length_limits(calc_dl(home.L_i, L_i)) -- TendonRobot.h:247-278
  if (active) {
    double sh = s_start < 0.0 ? 0.0 : s_start;  // home_shape clamps both ends
    const double Lhome = degenerate ? 0.0 : (rb.L - sh);
#pragma unroll
    for (int j = 0; j < NT; j++) {
      const double dl = Lhome * rb.home_factor[j] - x.Li[j];
      if (dl < rb.min_length[j] || rb.max_length[j] < dl) flags |= IRT_FLAG_LENGTH_LIMIT;
    }
  }
  if (o.npts) o.npts[cfg] = npts;
  if (o.L) o.L[cfg] = x.L;
  if (o.L_i) {
#pragma unroll
    for (int j = 0; j < NT; j++) o.L_i[cfg * NT + j] = x.Li[j];
  }
  if (o.tip) {
    const double p0 = x.p[0], p1 = x.p[1], p2 = x.p[2];
    double px = p0, py = p1;
    if (rz.on) { px = rz.c * p0 - rz.s * p1; py = rz.s * p0 + rz.c * p1; }
    o.tip[cfg * 3] = px; o.tip[cfg * 3 + 1] = py; o.tip[cfg * 3 + 2] = p2;
  }
  if (o.uv) {
    double *d = o.uv + cfg * 12;
#pragma unroll
    for (int i = 0; i < 3; i++) { d[i] = u0[i]; d[3 + i] = x.u[i]; d[6 + i] = v0[i]; d[9 + i] = x.v[i]; }
  }
  if (o.flags) o.flags[cfg] = flags;
  if (o.iters) o.iters[cfg] = iters;
  if (o.nsteps) o.nsteps[cfg] = nsteps;
  }
}

// ---- bucket configurations by (step count, tension bin), descending, so warps stay converged --------
// grid-stride over the configurations [lo, hi) (device range or [0, n)); block-aggregated histogram
__global__ void fk_count_nodes_kernel(const RobotDev rb, const double *__restrict__ states, int state_size,
                                      int64_t n_host, const int32_t *__restrict__ range, int nb,
                                      int32_t *__restrict__ keys, int32_t *__restrict__ hist) {
  extern __shared__ int32_t sh[];
  int64_t lo = 0, n = n_host;
  if (range) { lo = range[0]; n = (int64_t)range[1] - lo; }
  if ((int64_t)blockIdx.x * blockDim.x >= n) return;
  for (int i = threadIdx.x; i < nb; i += blockDim.x) sh[i] = 0;
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int K;
    const int key = fk_bucket_key(rb, states + (lo + i) * state_size, state_size, &K);
    keys[i] = key | (K << 16);
    atomicAdd(&sh[key], 1);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < nb; k += blockDim.x)
    if (sh[k]) atomicAdd(&hist[k], sh[k]);
}

__global__ void fk_row_count_kernel(const RobotDev rb, const double *__restrict__ states, int state_size,
                                    int64_t n, int64_t *__restrict__ counts) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int npts = rb.Kfull + 1;
  if (rb.enable_retraction) {
    double s = states[i * state_size + state_size - 1];
    if (!(s >= -rb.dL)) {
      npts = 0;
    } else {
      if (s > rb.L) s = rb.L;
      int K = 0;
      const double lim = rb.L - (rb.dL / 2);
      for (double p = s; p <= lim; p += rb.dL) K++;
      npts = (K > rb.Kfull) ? 0 : ((s == rb.L) ? 1 : K + 1);
    }
  }
  counts[i] = npts;
}

// Scatter into buckets in DESCENDING key order.  hist[k] = number of configurations with key k (final: the
// count kernel ran before on the same stream); cursor[k] = slots of bucket k handed out so far (zeroed).
// Every block ranks the configurations of a tile per bucket in shared memory and reserves ONE contiguous run per
// (tile, bucket) with a single global atomic, so the ~n same-address atomics of a naive scatter become
// ~n/256 * (occupied buckets); the bucket starts (an exclusive scan of <= a few hundred counts) are computed
// per block by warp 0 instead of by a kernel of their own.  Which slot inside its bucket a configuration gets
// is arbitrary; results are written at the original index, so they do not depend on it.
__global__ void fk_bucket_scatter_kernel(const int32_t *__restrict__ keys, int64_t n_host,
                                         const int32_t *__restrict__ range,
                                         const int32_t *__restrict__ hist, int32_t *__restrict__ cursor,
                                         int nb, int32_t *__restrict__ perm) {
  extern __shared__ int32_t sh[];
  int32_t *cnt = sh, *base = sh + nb, *start = sh + 2 * nb;   // per bucket: tile count, run start, bucket start
  int64_t n = n_host;
  if (range) n = (int64_t)range[1] - range[0];
  if ((int64_t)blockIdx.x * blockDim.x >= n) return;
  if (threadIdx.x < 32) {   // bucket starts: exclusive scan of hist from the highest key down
    const int lane = threadIdx.x;
    int32_t carry = 0;
    for (int top = nb - 1; top >= 0; top -= 32) {
      const int k = top - lane;
      const int32_t c = (k >= 0) ? hist[k] : 0;
      int32_t incl = c;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int32_t t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
      }
      if (k >= 0) start[k] = carry + incl - c;
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
  }
  for (int64_t t0 = (int64_t)blockIdx.x * blockDim.x; t0 < n; t0 += (int64_t)gridDim.x * blockDim.x) {
    for (int k = threadIdx.x; k < nb; k += blockDim.x) cnt[k] = 0;
    __syncthreads();
    const int64_t i = t0 + threadIdx.x;
    int key = 0, local = 0;
    if (i < n) {
      key = keys[i] & 0xFFFF;
      local = atomicAdd(&cnt[key], 1);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < nb; k += blockDim.x) {
      const int32_t c = cnt[k];
      if (c) base[k] = start[k] + atomicAdd(&cursor[k], c);
    }
    __syncthreads();
    if (i < n) perm[base[key] + local] = (int32_t)i;
    __syncthreads();
  }
}

template <int NT, bool RETRACT>
int launch_k(irt_ctx *ctx, const RobotDev &d, const FkArgs &a, size_t smem, cudaStream_t st) {
  int64_t blocks = (a.n + FK_THREADS - 1) / FK_THREADS;
  const int64_t resident = (int64_t)ctx->sm_count * FK_BLOCKS_PER_SM;
  if (blocks > resident) blocks = resident;
  auto k = fk_rk4_fp64_kernel<NT, RETRACT>;
  IRT_CUDA(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<(unsigned)blocks, FK_THREADS, smem, st>>>(d, a);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  return IRT_OK;
}

template <int NT>
int launch_nt(irt_ctx *ctx, const irt_robot *rb, const FkArgs &a, cudaStream_t st) {
  const RobotDev &d = rb->dev;
  const size_t smem = ((size_t)d.n_table + 4) * NT * 6 * sizeof(double);
  return d.enable_retraction ? launch_k<NT, true>(ctx, d, a, smem, st) : launch_k<NT, false>(ctx, d, a, smem, st);
}

}  // namespace

// Rows (backbone points) every configuration will emit, for the packed output layout: the same node
// count rule as the FK kernel (util::range's accumulation; 1 for the degenerate s == L shape; 0 for a
// state outside the reference's state space).
int fk_row_counts(irt_ctx *ctx, const irt_robot *rb, const double *d_states, int64_t n,
                  int64_t *d_counts, cudaStream_t st) {
  if (n <= 0) return IRT_OK;
  const int T = 256;
  fk_row_count_kernel<<<(unsigned)((n + T - 1) / T), T, 0, st>>>(rb->dev, d_states, rb->state_size, n, d_counts);
  IRT_LAUNCHED(ctx);
  IRT_CUDA(ctx, cudaGetLastError());
  return IRT_OK;
}

static int fk_num_buckets(const irt_robot *rb) { return (rb->dev.Kfull + 2) * FK_TAU_BINS; }

// device scratch one FK launch over up to n configurations needs: keys[n], perm[n], hist / cursor / work counter
size_t fk_work_bytes(const irt_robot *rb, int64_t n) {
  return (((size_t)n * 8 + 255) & ~(size_t)255) + (((size_t)fk_num_buckets(rb) * 8 + 64 + 255) & ~(size_t)255);
}

// K1 over configurations [0, n) of d_states -- or, d_range != nullptr, over rows [lo, hi) of d_states and of the
// output arrays with {lo, hi} read from device memory at run time (n = an upper bound of hi - lo).  work:
// fk_work_bytes(rb, n) bytes of device scratch, or nullptr to use the context's scratch buffer.
int fk_launch(irt_ctx *ctx, const irt_robot *rb, const double *d_states, int64_t n, int cap_pts,
              const irt_fk_outputs &o, cudaStream_t st, const int64_t *d_row_off, const int32_t *d_range,
              void *work) {
  if (n <= 0) return IRT_OK;
  if (n > 0x7ff00000LL) return irt_fail(ctx, IRT_ERR_INVALID_ARGUMENT, "batch too large");
  const RobotDev &d = rb->dev;
  size_t smem = ((size_t)d.n_table + 4) * d.n_tendons * 6 * sizeof(double);
  if (smem > 200 * 1024)
    return irt_fail(ctx, IRT_ERR_CAPACITY, "routing table (%zu B) exceeds shared memory", smem);
  const int nb = fk_num_buckets(rb);
  if (nb > 0xFFFF || (size_t)nb * 12 > 96 * 1024)
    return irt_fail(ctx, IRT_ERR_CAPACITY, "too many step-count buckets (%d)", nb);
  char *scr = (char *)work;
  if (!scr) {
    scr = (char *)ctx_scratch(ctx, fk_work_bytes(rb, n));
    if (!scr) return irt_fail(ctx, IRT_ERR_CUDA, "scratch alloc of %zu bytes failed", fk_work_bytes(rb, n));
  }
  int32_t *keys = (int32_t *)scr;
  int32_t *perm = keys + n;
  int32_t *hist = (int32_t *)(scr + (((size_t)n * 8 + 255) & ~(size_t)255));   // [nb] counts, [nb] cursors, work
  int32_t *cursor = hist + nb;
  int32_t *workctr = cursor + nb;
  IRT_CUDA(ctx, cudaMemsetAsync(hist, 0, (size_t)nb * 8 + 16, st));
  FkArgs a;
  a.states = d_states; a.state_size = rb->state_size; a.n = n; a.range = d_range; a.cap_pts = cap_pts;
  a.o = o; a.perm = nullptr; a.keys = nullptr; a.row_off = d_row_off; a.work = workctr;
  // Bucketing pays when warps would otherwise diverge: with retraction (step counts differ) always; without it
  // only the fixed-point iteration counts differ, which a batch large enough to fill the GPU several times
  // over amortises (small batches skip the two extra launches)
  if (d.enable_retraction) {
    const int T = 256;
    int64_t B = (n + T - 1) / T;
    const int64_t maxB = (int64_t)ctx->sm_count * 8;
    if (B > maxB) B = maxB;
    fk_count_nodes_kernel<<<(unsigned)B, T, nb * sizeof(int32_t), st>>>(d, d_states, rb->state_size, n, d_range, nb,
                                                                     keys, hist);
    IRT_LAUNCHED(ctx);
    if ((size_t)nb * 12 > 48 * 1024)
      IRT_CUDA(ctx, cudaFuncSetAttribute(fk_bucket_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         nb * 12));
    fk_bucket_scatter_kernel<<<(unsigned)B, T, 3 * nb * sizeof(int32_t), st>>>(keys, n, d_range, hist, cursor, nb,
                                                                            perm);
    IRT_LAUNCHED(ctx);
    IRT_CUDA(ctx, cudaGetLastError());
    a.perm = perm;
    a.keys = keys;
  }
  a.use_const = 0;
  // The kernel's fast path reads the routing table from constant memory, which is ONE array per device and process:
  // it is tagged with the robot it holds.  A launch for another robot waits for everything that may still read the
  // old table (device-wide, rare: applications use one robot), uploads, and the lock is held across the launch so
  // that no other host thread swaps the table between the check and the launch.
  static std::mutex ct_mutex;
  static unsigned long long ct_owner[64] = {};
  std::unique_lock<std::mutex> ct_lock(ct_mutex, std::defer_lock);
  const size_t tab_doubles = (size_t)d.n_table * d.n_tendons * IRT_CT_WIDTH;
  if (tab_doubles <= (size_t)FK_CT_DOUBLES && ctx->device >= 0 && ctx->device < 64) {
    ct_lock.lock();
    if (ct_owner[ctx->device] != rb->uid) {
      IRT_CUDA(ctx, cudaDeviceSynchronize());
      IRT_CUDA(ctx, cudaMemcpyToSymbolAsync(c_fk_tab, rb->d_ctab, tab_doubles * sizeof(double), 0,
                                            cudaMemcpyDeviceToDevice, st));
      IRT_CUDA(ctx, cudaStreamSynchronize(st));
      ct_owner[ctx->device] = rb->uid;
    }
    a.use_const = 1;
  }
  switch (d.n_tendons) {
    case 1: return launch_nt<1>(ctx, rb, a, st);
    case 2: return launch_nt<2>(ctx, rb, a, st);
    case 3: return launch_nt<3>(ctx, rb, a, st);
    case 4: return launch_nt<4>(ctx, rb, a, st);
    case 5: return launch_nt<5>(ctx, rb, a, st);
    case 6: return launch_nt<6>(ctx, rb, a, st);
    case 7: return launch_nt<7>(ctx, rb, a, st);
    case 8: return launch_nt<8>(ctx, rb, a, st);
    case 9: return launch_nt<9>(ctx, rb, a, st);
    case 10: return launch_nt<10>(ctx, rb, a, st);
    case 11: return launch_nt<11>(ctx, rb, a, st);
    case 12: return launch_nt<12>(ctx, rb, a, st);
    default:
      return irt_fail(ctx, IRT_ERR_UNSUPPORTED, "no fk kernel for %d tendons (1..%d supported)",
                      d.n_tendons, IRT_MAX_TENDONS);
  }
}
