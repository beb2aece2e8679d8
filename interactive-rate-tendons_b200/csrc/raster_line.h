// raster_line.h -- the voxel traversal of one line segment (VoxelOctree::add_line), shared by the device rasteriser
// (voxel_raster.cu, which includes this file inside its anonymous namespace) and a host harness
// (tests/cpp/test_raster_line_host.cpp) that runs the same text against the oracle on millions of segments without a
// GPU.  Grid: anything with lo[3], hi[3], d[3], inv_d[3], Ng (GridDev on the device).  Sink: cell(ix, iy, iz) and
// finish().  Every floating-point operation is spelled out in the reference's order: compile without FMA contraction
// (nvcc -fmad=false, g++ -ffp-contract=off).
#pragma once
#include <math.h>

#ifdef __CUDACC__
#define RL_HD __device__
#define RL_HDI __device__ __forceinline__
#else
#include <stdlib.h>
#define RL_HD inline
#define RL_HDI inline
#endif
// hooks of the host harness (count which path a segment took); nothing on the device
#ifndef RL_ON_FAST_PATH_DONE
#define RL_ON_FAST_PATH_DONE
#endif
#ifndef RL_ON_LITERAL_PATH
#define RL_ON_LITERAL_PATH
#endif

struct D3 {
  double x, y, z;
};

// collision/collision_primitives.h:62-85, literal operation order
RL_HD bool segment_aabox_intersect(const D3 &A, const D3 &B, const D3 &C, const D3 &D) {
  const D3 AB = {B.x - A.x, B.y - A.y, B.z - A.z};
  const double len = sqrt((AB.x * AB.x + AB.y * AB.y) + AB.z * AB.z) / 2;
  const double l2 = 2 * len;
  const D3 U = {AB.x / l2, AB.y / l2, AB.z / l2};
  const D3 Uabs = {fabs(U.x), fabs(U.y), fabs(U.z)};
  const D3 P = {(A.x + B.x) / 2 - (D.x + C.x) / 2, (A.y + B.y) / 2 - (D.y + C.y) / 2,
                (A.z + B.z) / 2 - (D.z + C.z) / 2};
  const D3 ext = {fabs(D.x - C.x) / 2, fabs(D.y - C.y) / 2, fabs(D.z - C.z) / 2};
  const D3 UxP = {fabs(U.y * P.z - U.z * P.y), fabs(U.z * P.x - U.x * P.z), fabs(U.x * P.y - U.y * P.x)};
  const D3 Pabs = {fabs(P.x), fabs(P.y), fabs(P.z)};
  const bool separated = Pabs.x > ext.x + len * Uabs.x || Pabs.y > ext.y + len * Uabs.y ||
                         Pabs.z > ext.z + len * Uabs.z ||
                         UxP.x > ext.y * Uabs.z + ext.z * Uabs.y ||
                         UxP.y > ext.z * Uabs.x + ext.x * Uabs.z ||
                         UxP.z > ext.x * Uabs.y + ext.y * Uabs.x;
  return !separated;
}

// VoxelOctree::add_line -- collision/VoxelOctree.cpp:325-426, reproduced literally including the
// "voxel index times metric cell size" initial error (:371-373) and the overshoot past B (:423-424).
template <typename Grid, typename Sink>
RL_HD void add_line(const Grid &g, Sink &sink, const D3 &a, const D3 &b) {
  const D3 ll = {g.lo[0], g.lo[1], g.lo[2]}, ur = {g.hi[0], g.hi[1], g.hi[2]};
  // A segment whose endpoints both lie well inside the grid box intersects it: the reference's
  // separating-axis test cannot report otherwise, so it is only evaluated for segments near or outside the faces.
  const D3 A = {(a.x - ll.x) * g.inv_d[0], (a.y - ll.y) * g.inv_d[1], (a.z - ll.z) * g.inv_d[2]};
  const D3 B = {(b.x - ll.x) * g.inv_d[0], (b.y - ll.y) * g.inv_d[1], (b.z - ll.z) * g.inv_d[2]};
  const int Axi = (int)A.x - (A.x < 0), Ayi = (int)A.y - (A.y < 0), Azi = (int)A.z - (A.z < 0);
  const int Bxi = (int)B.x - (B.x < 0), Byi = (int)B.y - (B.y < 0), Bzi = (int)B.z - (B.z < 0);
  const int N = g.Ng;
  {
    // both endpoints in INTERIOR cells (not the outermost layer): the segment lies inside the grid box by a
    // whole cell, so it intersects it (integer compares instead of 12 FP64 ones)
    const unsigned lim = (unsigned)(N - 2);
    const bool inside = (unsigned)(Axi - 1) < lim && (unsigned)(Ayi - 1) < lim && (unsigned)(Azi - 1) < lim &&
                        (unsigned)(Bxi - 1) < lim && (unsigned)(Byi - 1) < lim && (unsigned)(Bzi - 1) < lim;
    if (!inside && !segment_aabox_intersect(a, b, ll, ur)) return;
  }
#define IDX_IN(v) (0 <= (v) && (v) < N)
#define VOX_IN(x, y, z) (IDX_IN(x) && IDX_IN(y) && IDX_IN(z))
  // cells are emitted in path order A, steps, B (the result is a set; the reference adds B, A, steps): along a
  // monotone path the 4x4x4 block only changes when a block face is crossed, which keeps the sinks' block
  // accumulators in registers
  const bool entered = VOX_IN(Axi, Ayi, Azi);
  const bool b_in = VOX_IN(Bxi, Byi, Bzi);
  if (entered) sink.cell(Axi, Ayi, Azi);
  D3 U = {B.x - A.x, B.y - A.y, B.z - A.z};
  const double z = (U.x * U.x + U.y * U.y) + U.z * U.z;  // Eigen normalized()
  // Division-free traversal.  The reference's ray parameters are t_axis(k) = (e_axis + k) * n / |U_axis| (U the
  // un-normalised direction, n its norm, k the steps already taken on that axis), so every comparison between
  // two of them is a comparison of cross products (e_x + k_x) |U_y| <> (e_y + k_y) |U_x|: no square root, no
  // division (1 sqrt + 6 divisions per segment otherwise: ~200 of ~300 FP64 instructions).  The reference's
  // own values carry a few ulp of rounding, so a decision is only taken here when the two sides differ by more
  // than 1e-12 relative; a closer call or a direction component near the reference's 1e-10 validity threshold
  // hands the segment to the literal code below.  Cells are emitted as the path advances: up to a close call the
  // decisions are the reference's, so the cells emitted before a hand-over are cells the literal code adds too.
  {
    const double adx = fabs(U.x), ady = fabs(U.y), adz = fabs(U.z);
    const double zhi = 1.0001e-20 * z;   // |U_axis| / n > 1e-10 with margin
    if (z > 0.0 && adx * adx > zhi && ady * ady > zhi && adz * adz > zhi) {
      const int sx = 1 - 2 * (U.x < 0), sy = 1 - 2 * (U.y < 0), sz = 1 - 2 * (U.z < 0);
      double Nx = fabs(A.x - (Axi + sx) * g.d[0]);
      double Ny = fabs(A.y - (Ayi + sy) * g.d[1]);
      double Nz = fabs(A.z - (Azi + sz) * g.d[2]);
      int xi = Axi, yi = Ayi, zi = Azi;
      // steps left on every axis until the path has passed B's cell (the loop runs while none is negative)
      int rx = sx * (Bxi - Axi), ry = sy * (Byi - Ayi), rz = sz * (Bzi - Azi);
      bool ent = entered, ok = true;
      while ((rx | ry | rz) >= 0) {
        const double xy_l = Nx * ady, xy_r = Ny * adx, xz_l = Nx * adz, xz_r = Nz * adx, yz_l = Ny * adz, yz_r = Nz * ady;
        const double tol = 1e-12;
        if (fabs(xy_l - xy_r) <= tol * (xy_l + xy_r) || fabs(xz_l - xz_r) <= tol * (xz_l + xz_r) ||
            fabs(yz_l - yz_r) <= tol * (yz_l + yz_r)) {
          ok = false;
          break;
        }
        const bool ax0 = (xy_l < xy_r) && (xz_l < xz_r);            // tx is the minimum
        const bool ax1 = !ax0 && !(xy_l < xy_r) && (yz_l < yz_r);   // ty is
        const bool ax2 = !ax0 && !ax1;
        xi += ax0 ? sx : 0; yi += ax1 ? sy : 0; zi += ax2 ? sz : 0;
        rx -= ax0 ? 1 : 0; ry -= ax1 ? 1 : 0; rz -= ax2 ? 1 : 0;
        const int moved = ax0 ? xi : (ax1 ? yi : zi);
        if (ent && !IDX_IN(moved)) break;
        Nx = ax0 ? Nx + 1.0 : Nx; Ny = ax1 ? Ny + 1.0 : Ny; Nz = ax2 ? Nz + 1.0 : Nz;
        if (!ent) ent = VOX_IN(xi, yi, zi);
        if (ent) sink.cell(xi, yi, zi);
      }
      if (ok) {
        if (b_in) sink.cell(Bxi, Byi, Bzi);
        sink.finish();
        RL_ON_FAST_PATH_DONE
        return;
      }
    }
  }
  RL_ON_LITERAL_PATH
  bool entered_l = entered;
  if (z > 0.0) {
    const double n = sqrt(z);
    U.x /= n; U.y /= n; U.z /= n;
  }
  const int step_x = 1 - 2 * (U.x < 0), step_y = 1 - 2 * (U.y < 0), step_z = 1 - 2 * (U.z < 0);
  const double ex = fabs(A.x - (Axi + step_x) * g.d[0]);
  const double ey = fabs(A.y - (Ayi + step_y) * g.d[1]);
  const double ez = fabs(A.z - (Azi + step_z) * g.d[2]);
  const double ux = fabs(U.x), uy = fabs(U.y), uz = fabs(U.z);
  const double threshold = 1e-10;
  const double tx_delta = (ux > threshold) ? 1 / ux : 1 / threshold;
  const double ty_delta = (uy > threshold) ? 1 / uy : 1 / threshold;
  const double tz_delta = (uz > threshold) ? 1 / uz : 1 / threshold;
  double tx = fabs(ex * tx_delta), ty = fabs(ey * ty_delta), tz = fabs(ez * tz_delta);
  int xi = Axi, yi = Ayi, zi = Azi;
  while (step_x * (Bxi - xi) >= 0 && step_y * (Byi - yi) >= 0 && step_z * (Bzi - zi) >= 0) {
    const bool tx_is_min = (tx < ty) && (tx < tz);
    const bool ty_is_min = !(tx < ty) && (ty < tz);
    if (tx_is_min) {
      xi += step_x;
      if (entered_l && !IDX_IN(xi)) break;
      tx += tx_delta;
    } else if (ty_is_min) {
      yi += step_y;
      if (entered_l && !IDX_IN(yi)) break;
      ty += ty_delta;
    } else {
      zi += step_z;
      if (entered_l && !IDX_IN(zi)) break;
      tz += tz_delta;
    }
    if (!entered_l && VOX_IN(xi, yi, zi)) entered_l = true;
    if (entered_l) sink.cell(xi, yi, zi);
  }
  if (b_in) sink.cell(Bxi, Byi, Bzi);
  sink.finish();
#undef IDX_IN
#undef VOX_IN
}

// find_cell -- collision/VoxelOctree.cpp:309-317 (+domain_check :1511-1521); false = domain error
template <typename Grid>
RL_HDI bool find_cell(const Grid &g, const D3 &p, long long *c) {
  if (p.x < g.lo[0] || g.hi[0] < p.x) return false;
  if (p.y < g.lo[1] || g.hi[1] < p.y) return false;
  if (p.z < g.lo[2] || g.hi[2] < p.z) return false;
  // the quotient by the reciprocal differs from the reference's division by a few ulp (< 1e-13 cells): the
  // truncation is the same unless the point is within 1e-9 of a cell face, where the division itself decides
  const double qx = (p.x - g.lo[0]) * g.inv_d[0], qy = (p.y - g.lo[1]) * g.inv_d[1], qz = (p.z - g.lo[2]) * g.inv_d[2];
  const double fx = qx - floor(qx), fy = qy - floor(qy), fz = qz - floor(qz);
  const double m = 1e-9;
  if (fx > m && fx < 1.0 - m && fy > m && fy < 1.0 - m && fz > m && fz < 1.0 - m) {
    c[0] = (long long)qx; c[1] = (long long)qy; c[2] = (long long)qz;
    return true;
  }
  c[0] = (long long)((p.x - g.lo[0]) / g.d[0]);
  c[1] = (long long)((p.y - g.lo[1]) / g.d[1]);
  c[2] = (long long)((p.z - g.lo[2]) / g.d[2]);
  return true;
}

// event of one point pair of should_subdivide (VoxelEnvironment.cpp:304-341), points already in grid coordinates:
// 0 = cells at most 1 apart, 1 = far apart, 2 = domain error (a point outside the grid: find_cell would throw)
template <typename Grid>
RL_HDI int pair_event_core(const Grid &g, const D3 &qa, const D3 &qb) {
  const bool in_a = !(qa.x < g.lo[0] || g.hi[0] < qa.x || qa.y < g.lo[1] || g.hi[1] < qa.y || qa.z < g.lo[2] || g.hi[2] < qa.z);
  const bool in_b = !(qb.x < g.lo[0] || g.hi[0] < qb.x || qb.y < g.lo[1] || g.hi[1] < qb.y || qb.z < g.lo[2] || g.hi[2] < qb.z);
  const double tight = 1.0 - 1e-9;
  if (!in_a || !in_b) return 2;
  // two points less than one cell apart on every axis: their cells differ by at most 1 (the common case at the
  // last bisection level) -- no need to locate them
  if (fabs(qa.x - qb.x) < g.d[0] * tight && fabs(qa.y - qb.y) < g.d[1] * tight && fabs(qa.z - qb.z) < g.d[2] * tight)
    return 0;
#ifdef __CUDACC__
  long long s[3], e[3];
#else
  long long s[3] = {0, 0, 0}, e[3] = {0, 0, 0};   // both points are in the domain here: find_cell fills them (gcc cannot see it)
#endif
  find_cell(g, qa, s);
  find_cell(g, qb, e);
  const long long dx = llabs(s[0] - e[0]), dy = llabs(s[1] - e[1]), dz = llabs(s[2] - e[2]);
  return (dx > 1 || dy > 1 || dz > 1) ? 1 : 0;
}
