// kino_smooth.cuh -- smooth-step terrains for the contact kernels.
//
// Restates, with runtime parameters instead of baked constants,
//   SmoothTerrain.create_height_function   utilities/smooth_terrain.py:201-227
//   SmoothTerrain.step                     utilities/smooth_terrain.py:235-336
//   TerrainSum.create_height_function      utilities/terrain_sum.py:19-38
//   TerrainDescriptor normal / orientation utilities/terrain_descriptor.py:45-80
// and the terrain-dependent rows/costs of the contact block (complementarity.py:24-32, 68-89;
// contacts.py:24, 54-66, 158-166) including their first and second derivatives, obtained from
// truncated Taylor series of the surface (hb_jet.cuh) instead of CasADi's graph AD.
//
// Kernel terrain 1, the stairs (BASELINE config 5): two axis-aligned flat steps with origins at z = 0,
//   h(p) = z - sum_i exp(-g_i^20) height_i,   g_i = (2 (x - ox_i) / l_i)^10 + (2 (y - oy_i) / w_i)^10
// terrain parameters tp[10] = (l, w, height, ox, oy) x 2.
//
// Kernel terrain 2, K general steps (the ramp's terrain): yaw theta, origin o and a top tilted to the normal n,
//   (x_t, y_t) = R_z(theta)^T (p - o),   g = (2 x_t / l)^10 + (2 y_t / w)^10,
//   h(p) = z - sum_i [exp(-g_i^20) pi_i(x_t, y_t) + oz_i],   pi = height - n_x / n_z x_t - n_y / n_z y_t
// terrain parameters tp[10 K] = (l, w, height, ox, oy, oz, yaw, n_x, n_y, n_z) x K.
#pragma once
#include "hb_jet.cuh"

namespace hb {

// exp(-g^20) of one step as a series, from the series of g.  Far outside the step exp(-g^20) underflows to exactly 0
// while the powers of g overflow; the reference's graph then evaluates 0 * inf = NaN in the high derivatives.  The limit
// is 0, so callers skip the step where g0 > STEP_CUTOFF (identical wherever the reference is finite, finite where it is
// not): g^20 > 1100 > -log(DBL_TRUE_MIN), so exp(-G) == 0 in fp64.
constexpr double STEP_CUTOFF = 1.42;
__device__ __forceinline__ BJ<4> step_bump(const BJ<4>& g) {
  // G = g^20: C(20,k) g0^(20-k)
  const double g0 = g.c[0];
  const double g2 = g0 * g0, g4 = g2 * g2, g8 = g4 * g4, g16 = g8 * g8;
  double fp[5];
  fp[4] = 4845.0 * g16;
  fp[3] = 1140.0 * g16 * g0;
  fp[2] = 190.0 * g16 * g2;
  fp[1] = 20.0 * g16 * g2 * g0;
  fp[0] = g16 * g4;
  const BJ<4> G = bj_compose<4>(g, fp);
  // E = exp(-G)
  const double e0 = exp(-G.c[0]);
  const double fe[5] = {e0, e0, e0 / 2.0, e0 / 6.0, e0 / 24.0};
  return bj_compose<4>(-G, fe);
}

__device__ __forceinline__ BJ<4> smooth_steps_surface(const double* __restrict__ tp, double x, double y) {
  BJ<4> T = bj_const<4>(0.0);
#pragma unroll 1
  for (int s = 0; s < 2; ++s) {
    const double l = tp[5 * s], w = tp[5 * s + 1], height = tp[5 * s + 2], ox = tp[5 * s + 3], oy = tp[5 * s + 4];
    const double dX = 2.0 / l, dY = 2.0 / w;
    const double X0 = dX * (x - ox), Y0 = dY * (y - oy);
    // X^10 and Y^10 expanded to fourth order: C(10,k) X0^(10-k) dX^k
    const double X2 = X0 * X0, X4 = X2 * X2, X6 = X4 * X2, Y2 = Y0 * Y0, Y4 = Y2 * Y2, Y6 = Y4 * Y2;
    BJ<4> g = bj_const<4>(X6 * X4 + Y6 * Y4);
    g.c[bidx(1, 0)] = 10.0 * X6 * X2 * X0 * dX;
    g.c[bidx(2, 0)] = 45.0 * X6 * X2 * dX * dX;
    g.c[bidx(3, 0)] = 120.0 * X6 * X0 * dX * dX * dX;
    g.c[bidx(4, 0)] = 210.0 * X6 * dX * dX * dX * dX;
    g.c[bidx(0, 1)] = 10.0 * Y6 * Y2 * Y0 * dY;
    g.c[bidx(0, 2)] = 45.0 * Y6 * Y2 * dY * dY;
    g.c[bidx(0, 3)] = 120.0 * Y6 * Y0 * dY * dY * dY;
    g.c[bidx(0, 4)] = 210.0 * Y6 * dY * dY * dY * dY;
    const double g0 = g.c[0];
    if (g0 > STEP_CUTOFF) continue;
    const BJ<4> E = step_bump(g);
    T = T + height * E;
  }
  return T;
}

// t^10 of a linear series t: C(10,k) t0^(10-k) composed with t - t0
__device__ __forceinline__ BJ<4> bj_pow10(const BJ<4>& t) {
  const double t0 = t.c[0], t2 = t0 * t0, t4 = t2 * t2, t6 = t4 * t2;
  const double f[5] = {t6 * t4, 10.0 * t6 * t2 * t0, 45.0 * t6 * t2, 120.0 * t6 * t0, 210.0 * t6};
  return bj_compose<4>(t, f);
}
// a + bx (x - x0) + by (y - y0) as a series at (x0, y0)
__device__ __forceinline__ BJ<4> bj_linear(double a, double bx, double by) {
  BJ<4> r = bj_const<4>(a);
  r.c[bidx(1, 0)] = bx;
  r.c[bidx(0, 1)] = by;
  return r;
}

__device__ __forceinline__ BJ<4> tilted_steps_surface(const double* __restrict__ tp, int n_steps, double x, double y) {
  BJ<4> T = bj_const<4>(0.0);
#pragma unroll 1
  for (int s = 0; s < n_steps; ++s) {
    const double* q = tp + 10 * s;
    const double l = q[0], w = q[1], height = q[2], ox = q[3], oy = q[4], oz = q[5], yaw = q[6];
    const double nx = q[7], ny = q[8], nz = q[9];
    T.c[0] += oz;  // the origin height counts everywhere, also past the cut-off
    double sn, cs;
    sincos(yaw, &sn, &cs);
    const double dx = x - ox, dy = y - oy;
    const double xt = cs * dx + sn * dy, yt = cs * dy - sn * dx;
    // X = 2 x_t / l, Y = 2 y_t / w: linear in (x, y)
    const BJ<4> X = bj_linear(2.0 * xt / l, 2.0 * cs / l, 2.0 * sn / l);
    const BJ<4> Y = bj_linear(2.0 * yt / w, -2.0 * sn / w, 2.0 * cs / w);
    const BJ<4> g = bj_pow10(X) + bj_pow10(Y);
    if (g.c[0] > STEP_CUTOFF) continue;
    const BJ<4> E = step_bump(g);
    // tilted top pi = height + a x_t + b y_t
    const double a = -nx / nz, b = -ny / nz;
    T = T + E * bj_linear(height + a * xt + b * yt, a * cs - b * sn, a * sn + b * cs);
  }
  return T;
}

// the surface of kernel terrain 1 or 2; n_steps is read by terrain 2 only
template <int TERRAIN>
__device__ __forceinline__ BJ<4> terrain_surface(const double* __restrict__ tp, int n_steps, double x, double y) {
  static_assert(TERRAIN == 1 || TERRAIN == 2, "smooth terrains are 1 and 2");
  if constexpr (TERRAIN == 1) return smooth_steps_surface(tp, x, y);
  else return tilted_steps_surface(tp, n_steps, x, y);
}

struct TFrame {
  TJ h, gx, gy;      // height and the x, y components of its gradient (the z component is 1)
  TJ n[3], xh[3], yh[3];
  TJ Dn[3][2];       // d n_a / d x, d n_a / d y  (d / d z = 0)
};

template <int TERRAIN>
__device__ __forceinline__ void terrain_frame(const double* __restrict__ tp, int n_steps, double x, double y, double z,
                                              TFrame& F) {
  const BJ<4> T = terrain_surface<TERRAIN>(tp, n_steps, x, y);
  const BJ<3> gx3 = -bj_ddx<4>(T), gy3 = -bj_ddy<4>(T);
  const BJ<3> inv3 = bj_invsqrt<3>(gx3 * gx3 + gy3 * gy3 + 1.0);
  BJ<3> n3[3];
  n3[0] = gx3 * inv3;
  n3[1] = gy3 * inv3;
  n3[2] = inv3;
  BJ<2> n2[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    F.Dn[a][0] = tj_from(bj_ddx<3>(n3[a]));
    F.Dn[a][1] = tj_from(bj_ddy<3>(n3[a]));
    n2[a] = bj_trunc<3, 2>(n3[a]);
    F.n[a] = tj_from(n2[a]);
  }
  // y0 = n x e_x, x0 = y0 x n, x = x0 / |x0|, y = n x x   (terrain_descriptor.py:66-71)
  BJ<2> x0[3];
  x0[0] = n2[2] * n2[2] + n2[1] * n2[1];
  x0[1] = -(n2[0] * n2[1]);
  x0[2] = -(n2[0] * n2[2]);
  const BJ<2> xi = bj_invsqrt<2>(x0[0] * x0[0] + x0[1] * x0[1] + x0[2] * x0[2]);
  BJ<2> xh[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    xh[a] = x0[a] * xi;
    F.xh[a] = tj_from(xh[a]);
  }
  F.yh[0] = tj_from(n2[1] * xh[2] - n2[2] * xh[1]);
  F.yh[1] = tj_from(n2[2] * xh[0] - n2[0] * xh[2]);
  F.yh[2] = tj_from(n2[0] * xh[1] - n2[1] * xh[0]);
  F.h = tj_from(-bj_trunc<4, 2>(T));
  F.h.c[0] += z;
  F.h.c[3] = 1.0;
  F.gx = tj_from(bj_trunc<3, 2>(gx3));
  F.gy = tj_from(bj_trunc<3, 2>(gy3));
}

__device__ __forceinline__ TJ tj_dot(const TJ* a, D3 b) { return b.x * a[0] + b.y * a[1] + b.z * a[2]; }
__device__ __forceinline__ double comp(D3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }

// A contact force in the terrain frame at the point, as series in the point position: its normal component
// N = n.f (contacts.py:24), its tangential components X = x.f, Y = y.f, and the friction-cone margin
// mu^2 N^2 - X^2 - Y^2 (contacts.py:54-66), as the pose-finder contact kernel uses them.  kino_contact.cu spells the
// same expressions inline: routed through these helpers its smooth-terrain Hessian changes in the last bits.
struct FrameForce {
  TJ N, X, Y, fric;
};
__device__ __forceinline__ FrameForce frame_force(const TFrame& F, D3 f, double mu) {
  FrameForce r;
  r.N = tj_dot(F.n, f);
  r.X = tj_dot(F.xh, f);
  r.Y = tj_dot(F.yh, f);
  r.fric = (mu * mu) * (r.N * r.N) - r.X * r.X - r.Y * r.Y;
  return r;
}
// d (friction-cone margin) / d f_d, as a series in the point position
__device__ __forceinline__ TJ frame_force_fric_df(const TFrame& F, const FrameForce& r, double mu, int d) {
  return (2.0 * mu * mu) * (r.N * F.n[d]) - 2.0 * (r.X * F.xh[d]) - 2.0 * (r.Y * F.yh[d]);
}
// d2 (friction-cone margin) / d f_a d f_b at the point
__device__ __forceinline__ double frame_force_fric_dff(const TFrame& F, double mu, int a, int b) {
  return 2.0 * mu * mu * F.n[a].c[0] * F.n[b].c[0] - 2.0 * F.xh[a].c[0] * F.xh[b].c[0] -
         2.0 * F.yh[a].c[0] * F.yh[b].c[0];
}

// Values and derivatives of every terrain-dependent row / cost of one contact point.
struct SmoothPoint {
  // rows (Taylor series in the point position, all other variables frozen)
  TJ planar[3], dcc, fric, swing, N;
  TFrame F;
  TJ tau;
};

}  // namespace hb
