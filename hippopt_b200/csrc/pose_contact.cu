// pose_contact.cu -- contact constraints, static balance and regularisation costs of the humanoid
// pose finder (BASELINE config 2): one warp per instance (single knot).
//
// Rows / costs (reference file:line restated):
//   relaxed complementarity  eps - h(p) n.(f mass) >= 0   humanoid_pose_finder/planner.py:704-726,
//                                                          expressions/complementarity.py:131-138
//   height / normal force / friction cone                  planner.py:728-749, expressions/contacts.py:24,54-66
//   static balance  g + sum_i [f_i; (p_i - x) x f_i] = 0   planner.py:482-511, expressions/centroidal.py:62-64
//   joint position bounds                                  planner.py:513-521
//   com position, average force, point position, force regularisation costs   planner.py:566-575, 751-788
// The kinematic rows (FK consistency, CoM consistency, unit quaternion) and the base-quaternion / frame /
// joint costs come from kino_kin_kernel, which runs on a virtual knot (KinoConst::zmap).
//
// Local Jacobian order: hippopt_b200/pose_layout.py::_enumerate_jp.  Cost weights reuse KinoConst
// slots: w_centroid = com, w_ratio = average force, w_swing = point position, w_fd = force.
//
// TERRAIN: 0 = PlanarTerrain (h = p_z, n = e_z, R_t = I), 1 = the two smooth steps of the stairs (BASELINE config 5,
// kino_smooth.cuh) with their ten parameters at p + po_terrain, 2 = K general smooth steps (kino_smooth.cuh) with their
// 10 K parameters closing p.  On the steps h depends on the whole point position and
// n, R_t on (x, y): lane i < 8 evaluates the terrain frame of point i as order-2 series in its position and forms the
// four terrain rows, their 25 Jacobian entries and the multiplier-weighted second derivatives from them.
#include "kino_const.cuh"
#include "kino_smooth.cuh"

namespace hb {

// Terrain rows of contact point i on the smooth steps: relaxed complementarity eps - h n.(f mass), height h, normal
// force n.f and friction-cone margin mu^2 (n.f)^2 - (x.f)^2 - (y.f)^2 (g rows, local Jacobian entries 25 i .. 25 i + 18
// in pose_layout.py::_enumerate_jp order, and the multiplier-weighted (p, p), (p, f), (f, f) second derivatives).
template <int TERRAIN, class JPut, class HAdd, class LamRow>
__device__ __forceinline__ void smooth_point_rows(const KinoConst& C, const double* __restrict__ tp, int n_steps, int i,
                                                  D3 ppos, D3 pf,
                                                  double mass, double eps, double mu, bool want_g, bool want_jac,
                                                  bool want_hess, double* __restrict__ gb, JPut& jput, HAdd& hadd,
                                                  LamRow& lamrow) {
  const int fb_ = i * HB_KF_PT_COUNT, o = 15 * i;
  TFrame F;
  terrain_frame<TERRAIN>(tp, n_steps, ppos.x, ppos.y, ppos.z, F);
  const FrameForce ff = frame_force(F, pf, mu);
  const TJ hN = F.h * ff.N;  // h n.f: the complementarity row is eps - mass h n.f
  if (want_g) {
    int r = grow(C, fb_ + HB_KF_PT_DCC, 0, 0);
    if (r >= 0) gb[r] = eps - mass * hN.c[0];
    r = grow(C, fb_ + HB_KF_PT_HEIGHT, 0, 0);
    if (r >= 0) gb[r] = F.h.c[0];
    r = grow(C, fb_ + HB_KF_PT_NORMAL, 0, 0);
    if (r >= 0) gb[r] = ff.N.c[0];
    r = grow(C, fb_ + HB_KF_PT_FRICTION, 0, 0);
    if (r >= 0) gb[r] = ff.fric.c[0];
  }
  if (want_jac) {
    // complementarity (p, f), height (p), normal (p_xy, f), friction (p_xy, f): n and R_t do not depend on z
    const int b0 = 25 * i;
    const double h0 = F.h.c[0];
    for (int d = 0; d < 3; ++d) {
      jput(b0 + d, -mass * hN.c[1 + d]);
      jput(b0 + 3 + d, -mass * h0 * F.n[d].c[0]);
      jput(b0 + 6 + d, F.h.c[1 + d]);
      jput(b0 + 11 + d, F.n[d].c[0]);
      jput(b0 + 16 + d, frame_force_fric_df(F, ff, mu, d).c[0]);
    }
    jput(b0 + 9, ff.N.c[1]);
    jput(b0 + 10, ff.N.c[2]);
    jput(b0 + 14, ff.fric.c[1]);
    jput(b0 + 15, ff.fric.c[2]);
  }
  if (want_hess) {
    const double lc = lamrow(fb_ + HB_KF_PT_DCC, 0), lh = lamrow(fb_ + HB_KF_PT_HEIGHT, 0);
    const double ln = lamrow(fb_ + HB_KF_PT_NORMAL, 0), lf = lamrow(fb_ + HB_KF_PT_FRICTION, 0);
    const double lcm = -lc * mass;
    // the four rows weighted by their multipliers, as one series in the point position
    const TJ Lp = lcm * hN + lh * F.h + ln * ff.N + lf * ff.fric;
    int e = 0;
    for (int a = 0; a < 3; ++a)
      for (int bb = a; bb < 3; ++bb) hadd(o + Z_P + a, o + Z_P + bb, tj_hess(Lp, e++));
    for (int d = 0; d < 3; ++d) {
      const TJ Gf = lcm * (F.h * F.n[d]) + ln * F.n[d] + lf * frame_force_fric_df(F, ff, mu, d);  // d Lp / d f_d
      for (int a = 0; a < 3; ++a) hadd(o + Z_P + a, o + Z_F + d, Gf.c[1 + a]);
    }
    for (int a = 0; a < 3; ++a)
      for (int bb = a; bb < 3; ++bb) hadd(o + Z_F + a, o + Z_F + bb, lf * frame_force_fric_dff(F, mu, a, bb));
  }
}

template <int TERRAIN>
__global__ void __launch_bounds__(128) pose_contact_kernel(const KinoConst* __restrict__ Cp, unsigned mask,
                                                           const double* __restrict__ x, const double* __restrict__ p,
                                                           long p_stride, const double* __restrict__ lam,
                                                           const double* __restrict__ sigma, double* __restrict__ fpart,
                                                           double* __restrict__ grad_f, double* __restrict__ g,
                                                           double* __restrict__ jac, double* __restrict__ hess,
                                                           long batch) {
  extern __shared__ double smem[];
  const KinoConst& C = *Cp;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const long b = (long)blockIdx.x * (blockDim.x >> 5) + warp;
  if (b >= batch) return;
  const ContactSmem L = pose_contact_smem_layout(C.n_hc);
  double* sm = smem + (size_t)warp * L.total;
  double* zs = sm + L.z;
  double* hbuf = sm + L.hbuf;
  double* gbuf = sm + L.gbuf;
  double* ls_coef = sm + L.ls_coef;
  double* ls_w = sm + L.ls_w;
  double* ls_r = sm + L.ls_r;
  int* ls_var = reinterpret_cast<int*>(sm + L.ls_var);
  const double* xb = x + b * C.n_x;
  const double* pp = p + b * p_stride;
  const bool want_f = mask & HB_EVAL_F, want_grad = mask & HB_EVAL_GRAD_F, want_g = mask & HB_EVAL_G;
  const bool want_jac = mask & HB_EVAL_JAC_G, want_hess = mask & HB_EVAL_HESS_L;
  for (int i = lane; i < NZ; i += 32) {
    const int zi = C.zmap[i];
    zs[i] = zi >= 0 ? xb[zi] : 0.0;
  }
  for (int i = lane; i < C.n_hc; i += 32) hbuf[i] = 0.0;
  for (int i = lane; i < NCV; i += 32) gbuf[i] = 0.0;
  __syncwarp();
  const double mass = pp[C.po_mass], eps = pp[C.po_eps], mu = pp[C.po_mu];
  // local Jacobian entries per contact point (complementarity, height, normal, friction, FK) and of the robot rows
  constexpr int JC_PT = TERRAIN == 0 ? 13 : 25, JC_ROBOT = 8 * JC_PT;
  const double* refst = pp + C.po_init;  // references.state: per point (p, f, descriptor), pb, q, s, com
  double* gb = g + b * C.m;
  const double* lb = lam + b * C.m;
  const double sg = want_hess ? sigma[b] : 0.0;
  double* jb = jac + b * C.nnz_j + C.knot_maps[0].jc_base;  // single knot: one knot-relative table
  auto jput = [&](int e, double v) {
    const int slot = C.jc_map[e];
    if (slot >= 0) jb[slot] = v;
  };
  auto hadd = [&](int vi, int vj, double v) {
    const int e = C.hc_index[vi * NCV + vj];
    if (e >= 0) hbuf[e] += v;
  };
  auto lamrow = [&](int fam, int r) -> double {
    const int row = grow(C, fam, 0, r);
    return row >= 0 ? lb[row] : 0.0;
  };
  const int pi_ = lane & 7;
  const D3 ppos = ld3(zs + 15 * pi_ + Z_P), pf = ld3(zs + 15 * pi_ + Z_F);
  const D3 comv = ld3(zs + Z_COM);
  double cost = 0.0;
  // static balance sums
  D3 lin = pf, ang = cross(ppos - comv, pf);
  if (lane >= 8) lin = ang = v3<double>(0.0, 0.0, 0.0);
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) {
    lin.x += __shfl_xor_sync(0xffffffffu, lin.x, o);
    lin.y += __shfl_xor_sync(0xffffffffu, lin.y, o);
    lin.z += __shfl_xor_sync(0xffffffffu, lin.z, o);
    ang.x += __shfl_xor_sync(0xffffffffu, ang.x, o);
    ang.y += __shfl_xor_sync(0xffffffffu, ang.y, o);
    ang.z += __shfl_xor_sync(0xffffffffu, ang.z, o);
  }
  const D3 fsum = v3<double>(__shfl_sync(0xffffffffu, lin.x, 0), __shfl_sync(0xffffffffu, lin.y, 0),
                             __shfl_sync(0xffffffffu, lin.z, 0));
  const D3 asum = v3<double>(__shfl_sync(0xffffffffu, ang.x, 0), __shfl_sync(0xffffffffu, ang.y, 0),
                             __shfl_sync(0xffffffffu, ang.z, 0));
  if constexpr (TERRAIN != 0) {
    const int n_steps = TERRAIN == 2 ? (C.n_p - C.po_terrain) / 10 : 0;  // the step records close p
    if (lane < 8 && (want_g || want_jac || want_hess))
      smooth_point_rows<TERRAIN>(C, pp + C.po_terrain, n_steps, lane, ppos, pf, mass, eps, mu, want_g, want_jac, want_hess,
                        gb, jput, hadd, lamrow);
  }
  if (want_g) {
    if (TERRAIN == 0 && lane < 8) {
      const int fb_ = lane * HB_KF_PT_COUNT;
      int r = grow(C, fb_ + HB_KF_PT_DCC, 0, 0);
      if (r >= 0) gb[r] = eps - ppos.z * (pf.z * mass);
      r = grow(C, fb_ + HB_KF_PT_HEIGHT, 0, 0);
      if (r >= 0) gb[r] = ppos.z;
      r = grow(C, fb_ + HB_KF_PT_NORMAL, 0, 0);
      if (r >= 0) gb[r] = pf.z;
      r = grow(C, fb_ + HB_KF_PT_FRICTION, 0, 0);
      if (r >= 0) gb[r] = -(pf.x * pf.x) - pf.y * pf.y + mu * mu * (pf.z * pf.z);
    }
    if (lane < 6) {
      const int r = grow(C, HB_KF_H_DYN, 0, lane);
      const double s = lane < 3 ? comp(fsum, lane) : comp(asum, lane - 3);
      if (r >= 0) gb[r] = pp[C.po_gravity + lane] + s;
    }
    if (lane < HB_N_JOINTS) {
      const int r = grow(C, HB_KF_S_BOUNDS, 0, lane);
      if (r >= 0) gb[r] = zs[Z_S + lane];
    }
  }
  // ---- costs: com position, point position, force regularisation
  if (lane < 3) {
    const double e = zs[Z_COM + lane] - refst[102 + lane];
    cost += C.w_centroid * e * e;
    gbuf[CV_COM + lane] += 2.0 * C.w_centroid * e;
    if (want_hess) hadd(CV_COM + lane, CV_COM + lane, 2.0 * sg * C.w_centroid);
  }
  if (lane < 8) {
    const int o = 15 * lane;
    for (int c = 0; c < 3; ++c) {
      const double ep = zs[o + Z_P + c] - refst[9 * lane + c];
      const double ef = zs[o + Z_F + c] - refst[9 * lane + 3 + c];
      cost += C.w_swing * ep * ep + C.w_fd * ef * ef;
      gbuf[o + Z_P + c] += 2.0 * C.w_swing * ep;
      gbuf[o + Z_F + c] += 2.0 * C.w_fd * ef;
      if (want_hess) {
        hadd(o + Z_P + c, o + Z_P + c, 2.0 * sg * C.w_swing);
        hadd(o + Z_F + c, o + Z_F + c, 2.0 * sg * C.w_fd);
      }
    }
  }
  __syncwarp();
  // ---- average-force least-squares rows: foot (2) x point (4) x component (3)
  if (lane < 24) {
    const int foot = lane / 12, i = (lane % 12) / 3, c = lane % 3;
    int* var = ls_var + lane * LS_MAXV;
    double* cf = ls_coef + lane * LS_MAXV;
    double ssum = 0.0;
    for (int j = 0; j < 4; ++j) {
      var[j] = 15 * (4 * foot + j) + Z_F + c;
      cf[j] = (j == i ? 1.0 : 0.0) - 0.25;
      ssum += zs[var[j]];
    }
    const double r = zs[var[i]] - 0.25 * ssum;
    ls_w[lane] = C.w_ratio;
    ls_r[lane] = r;
    cost += C.w_ratio * r * r;
  }
  __syncwarp();
  for (int row = 0; row < 24; ++row) {
    const int* var = ls_var + row * LS_MAXV;
    const double* cf = ls_coef + row * LS_MAXV;
    const double w = ls_w[row];
    if (lane < 4) gbuf[var[lane]] += 2.0 * w * ls_r[row] * cf[lane];
    if (want_hess && lane < 10) {
      int a = 0, tt = lane;
      while (tt >= 4 - a) {
        tt -= 4 - a;
        ++a;
      }
      hadd(var[a], var[a + tt], 2.0 * sg * w * cf[a] * cf[a + tt]);
    }
    __syncwarp();
  }
  if (want_f || want_grad) {
    const double total = warp_sum(cost);
    if (lane == 0 && want_f) fpart[b * 2] = total;
  }
  if (want_grad) {
    double* gf = grad_f + b * C.n_x;
    for (int i = lane; i < NCV; i += 32) {
      const int off = i < 120 ? i : (i < CV_H ? Z_COM + i - CV_COM : Z_H + i - CV_H);
      if (C.zmap[off] >= 0) gf[C.zmap[off]] = gbuf[i];
    }
  }
  // ---- Jacobian
  if (want_jac) {
    if (TERRAIN == 0 && lane < 8) {
      const int b0 = 13 * lane;
      jput(b0 + 0, -pf.z * mass);
      jput(b0 + 1, -ppos.z * mass);
      jput(b0 + 2, 1.0);
      jput(b0 + 3, 1.0);
      jput(b0 + 4, -2.0 * pf.x);
      jput(b0 + 5, -2.0 * pf.y);
      jput(b0 + 6, 2.0 * mu * mu * pf.z);
      for (int c = 0; c < 3; ++c) {
        jput(b0 + 7 + c, 1.0);
        jput(b0 + 10 + c, -1.0);
      }
    }
    if (TERRAIN != 0 && lane < 8) {
      const int b0 = JC_PT * lane + 19;  // the FK entries follow the point's 19 terrain-row entries
      for (int c = 0; c < 3; ++c) {
        jput(b0 + c, 1.0);
        jput(b0 + 3 + c, -1.0);
      }
    }
    if (lane < 6) jput(JC_ROBOT + lane, lane < 3 ? 1.0 : -1.0);
    for (int e = lane; e < 126; e += 32) {
      double v;
      if (e < 24) v = 1.0;
      else {
        const int q = e < 72 ? e - 24 : (e < 120 ? e - 72 : e - 120);
        const int i = q / 6, pr = q % 6, a = pr >> 1;
        const int bcol = a == 0 ? (pr & 1) + 1 : (a == 1 ? ((pr & 1) ? 2 : 0) : (pr & 1));
        const int c = 3 - a - bcol;
        if (e < 72) v = eps3(a, bcol) * zs[15 * i + Z_F + c];
        else if (e < 120) v = -eps3(a, bcol) * (zs[15 * i + Z_P + c] - zs[Z_COM + c]);
        else v = -eps3(a, bcol) * comp(fsum, c);
      }
      jput(JC_ROBOT + 6 + e, v);
    }
    if (lane < HB_N_JOINTS) jput(JC_ROBOT + 132 + lane, 1.0);
  }
  // ---- Hessian
  if (want_hess) {
    if (lane < 8) {
      const int o = 15 * lane;
      if constexpr (TERRAIN == 0) {
        const int fb_ = lane * HB_KF_PT_COUNT;
        const double lc = lamrow(fb_ + HB_KF_PT_DCC, 0), lf = lamrow(fb_ + HB_KF_PT_FRICTION, 0);
        hadd(o + Z_P + 2, o + Z_F + 2, -lc * mass);
        hadd(o + Z_F, o + Z_F, -2.0 * lf);
        hadd(o + Z_F + 1, o + Z_F + 1, -2.0 * lf);
        hadd(o + Z_F + 2, o + Z_F + 2, 2.0 * mu * mu * lf);
      }
      double La[3];
      for (int c = 0; c < 3; ++c) La[c] = lamrow(HB_KF_H_DYN, 3 + c);
      for (int a = 0; a < 3; ++a)
        for (int bb = 0; bb < 3; ++bb) {
          if (a == bb) continue;
          const int c = 3 - a - bb;
          const double v = eps3(a, bb) * La[c];
          hadd(o + Z_P + a, o + Z_F + bb, v);
          hadd(CV_COM + a, o + Z_F + bb, -v);
        }
    }
    __syncwarp();
    double* hb_ = hess + b * C.nnz_h + C.knot_maps[0].hc_base;
    for (int e = lane; e < C.n_hc; e += 32) {
      const int slot = C.hc_map[e];
      if (slot >= 0) hb_[slot] = hbuf[e];
    }
  }
}

}  // namespace hb
