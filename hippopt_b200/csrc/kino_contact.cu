// kino_contact.cu -- integrator defects, contact-point constraints, bounds and contact-space costs of the
// kinodynamic NLP: one warp per (instance, knot); planar terrain.
//
// Rows / costs evaluated here (reference file:line restated):
//   ImplicitTrapezoid defects + initial conditions   integrators/implicit_trapezoid.py:31-37,
//                                                    base/multiple_shooting_solver.py:703-742
//     for f_i, p_i (planner.py:721-744), pb, qb, s, com (planner.py:522-564)
//   centroidal momentum dynamics                     planner.py:566-588, expressions/centroidal.py:62-64
//   planar DCC complementarity                       planner.py:646-654, expressions/complementarity.py:24-32
//   DCC margin                                       planner.py:656-669, complementarity.py:68-89
//   height / normal force / friction cone            planner.py:671-697, expressions/contacts.py:24,54-66
//   control bounds                                   planner.py:699-719
//   angular momentum / CoM height / joint bounds     planner.py:341-358, 385-405
//   feet relative height, centroid cost              planner.py:215-264
//   final state / periodicity                        planner.py:407-425, 897-930
//   swing heuristic, control regularisations         planner.py:855-895, contacts.py:158-166
//   force ratio and foot yaw costs                   planner.py:746-853, contacts.py:132
//   CoM velocity cost                                planner.py:432-447
// Terrain: PlanarTerrain (utilities/planar_terrain.py:13,25,37): h = p_z, n = e_z, R = I.
//
// Local Jacobian order: hippopt_b200/kino_layout.py::_enumerate_jc.  Hessian contributions are routed
// through the (variable, variable) -> local entry table hc_index and accumulated per warp in shared
// memory in a fixed order (deterministic), then scattered once.
#include "kino_const.cuh"
#include "contact_jac_desc.h"
#include "kino_smooth.cuh"

namespace hb {

enum { NCV = 129, CV_COM = 120, CV_H = 123, LS_ROWS = 31, LS_MAXV = 8 };
// Hessian-phase inputs of contact point i, parked at park[8 q + i] of the kinodynamic kernel's shared block as soon
// as they are known: multipliers of the planar (x, y), DCC and friction rows, of the angular momentum dynamics (3),
// and d tau / d p_z, d2 tau / d p_z2
enum { PK_L0, PK_L1, PK_LD, PK_LF, PK_LA, PK_DTAU = PK_LA + 3, PK_DDTAU, PK_COUNT };

// Per-warp shared block.  The least-squares row tables (ls_*) are used by the pose-finder kernel only; the
// kinodynamic kernel sums its least-squares rows in closed form and has the parked Hessian inputs instead
// (968 doubles per warp at config 3: 7 CTAs of 4 warps fit an SM's shared memory).
struct ContactSmem {
  int z, zp, hbuf, gbuf, ls_coef, ls_w, ls_r, ls_var, ls_n, park, total;
};
__host__ __device__ inline ContactSmem contact_smem_layout_(int n_hc, bool ls_tables) {
  ContactSmem s;
  int o = 0;
  s.z = o;
  o += NZ + 1;
  s.zp = o;
  o += NZ + 1;
  s.hbuf = o;
  o += (n_hc + 1) & ~1;
  s.gbuf = o;
  o += NCV + 1;
  s.ls_coef = s.ls_w = s.ls_r = s.ls_var = s.ls_n = s.park = -1;
  if (!ls_tables) {
    s.park = o;
    o += 8 * PK_COUNT;
  } else {
    s.ls_coef = o;
    o += LS_ROWS * LS_MAXV;
    s.ls_w = o;
    o += LS_ROWS + 1;
    s.ls_r = o;
    o += LS_ROWS + 1;
    s.ls_var = o;  // ints, two per double slot
    o += (LS_ROWS * LS_MAXV) / 2 + 1;
    s.ls_n = o;
    o += LS_ROWS / 2 + 1;
  }
  s.total = o;
  return s;
}
// one layout per kernel, so that a launch cannot size the block of the other kernel
__host__ __device__ inline ContactSmem kino_contact_smem_layout(int n_hc) { return contact_smem_layout_(n_hc, false); }
__host__ __device__ inline ContactSmem pose_contact_smem_layout(int n_hc) { return contact_smem_layout_(n_hc, true); }

__device__ __forceinline__ double eps3(int a, int b) { return ((b - a + 3) % 3 == 1) ? 1.0 : -1.0; }

// state scalars with linear dynamics, in family emission order (kino_layout.py::linear_states)
__device__ __forceinline__ void linear_state(int j, int& so, int& ro, int& fam_dyn, int& fam_ic, int& comp) {
  if (j < 48) {
    const int i = j / 6, w = (j % 6) / 3;
    comp = j % 3;
    so = 15 * i + (w == 0 ? Z_F : Z_P) + comp;
    ro = 15 * i + (w == 0 ? Z_FD : Z_V) + comp;
    fam_dyn = i * HB_KF_PT_COUNT + (w == 0 ? HB_KF_PT_F_DYN : HB_KF_PT_P_DYN);
    fam_ic = i * HB_KF_PT_COUNT + (w == 0 ? HB_KF_PT_F_IC : HB_KF_PT_P_IC);
  } else if (j < 51) {
    comp = j - 48;
    so = Z_PB + comp;
    ro = Z_VB + comp;
    fam_dyn = HB_KF_PB_DYN;
    fam_ic = HB_KF_PB_IC;
  } else if (j < 55) {
    comp = j - 51;
    so = Z_Q + comp;
    ro = Z_QD + comp;
    fam_dyn = HB_KF_Q_DYN;
    fam_ic = HB_KF_Q_IC;
  } else if (j < 78) {
    comp = j - 55;
    so = Z_S + comp;
    ro = Z_SD + comp;
    fam_dyn = HB_KF_S_DYN;
    fam_ic = HB_KF_S_IC;
  } else {
    comp = j - 78;
    so = Z_COM + comp;
    ro = Z_H + comp;
    fam_dyn = HB_KF_COM_DYN;
    fam_ic = HB_KF_COM_IC;
  }
}

// TERRAIN: 0 = PlanarTerrain, 1 = sum of two smooth steps, 2 = sum of K general (rotated, raised, tilted) smooth steps
// (kino_smooth.cuh)
// CTAs per SM of the planar kernel, kernel time per bench step (config 3, NVIDIA B200 at 1000 W, 1965 MHz, three
// alternated runs): 5 (96 registers, no spill) 0.241 ms, 6 (80, 12 B spill) 0.224 ms, 7 (72, 8 B spill) 0.213 ms.
// Shared memory allows 7: 30 976 B per CTA.
constexpr int CONTACT_MIN_BLOCKS = 7;
template <int TERRAIN>
__global__ void __launch_bounds__(128, TERRAIN == 0 ? CONTACT_MIN_BLOCKS : 1) kino_contact_kernel(const __grid_constant__ KinTopo T,
                                                           const KinoConst* __restrict__ Cp, unsigned mask,
                                                           const double* __restrict__ x, const double* __restrict__ p,
                                                           long p_stride, const double* __restrict__ lam,
                                                           const double* __restrict__ sigma, double* __restrict__ fpart,
                                                           double* __restrict__ grad_f, double* __restrict__ g,
                                                           double* __restrict__ jac, double* __restrict__ hess,
                                                           long batch) {
  extern __shared__ double smem[];
  // C: warp-uniform scalars and tables from the constant bank (kernel parameter); G: the global copy, for
  // row families indexed by the lane (one coalesced 16-byte load instead of a serialised constant fetch)
  const KinTopo& C = T;
  const KinoConst& G = *Cp;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const long wid = (long)blockIdx.x * (blockDim.x >> 5) + warp;
  const int N = C.N;
  if (wid >= batch * N) return;
  const long b = wid / N;
  const int k = (int)(wid % N);
  const ContactSmem L = kino_contact_smem_layout(C.n_hc);
  double* sm = smem + (size_t)warp * L.total;
  double* zs = sm + L.z;
  double* zp = sm + L.zp;
  double* hbuf = sm + L.hbuf;
  double* gbuf = sm + L.gbuf;
  double* park = sm + L.park;
  const double* xinst = x + b * C.n_x;
  const double* xb = xinst + (long)k * NZ;
  const double* pp = p + b * p_stride;
  HB_PHASE_INIT
  const bool k1 = k >= 1;
  const bool want_f = mask & HB_EVAL_F, want_grad = mask & HB_EVAL_GRAD_F, want_g = mask & HB_EVAL_G;
  const bool want_jac = mask & HB_EVAL_JAC_G, want_hess = mask & HB_EVAL_HESS_L;
  // solution report (hb_eval_cost_terms): fpart is the [batch][N][HB_COST_TERMS] table of named cost values
  const bool want_terms = mask & HB_EVAL_COST_TERMS_BIT;
  // (the row address is formed where a value is written: kept from here it is a 64-bit value spilled at 72 registers)
  auto ct = [&](int i) -> double& { return fpart[(b * N + k) * HB_COST_TERMS + i]; };
  double c_swing = 0.0;  // swing-height cost of this lane's point (terrain-dependent block below)

  // every global input is requested before the first shared-memory store: a store waits for its load and,
  // in program order, would hold back the loads behind it (x, the parameters and the multipliers would
  // each pay their DRAM latency in turn)
  double xs_[6], xp_[6];
#pragma unroll
  for (int u = 0; u < 6; ++u) {
    const int i = lane + 32 * u;
    xs_[u] = i < NZ ? xb[i] : 0.0;
    xp_[u] = (i < NZ && k1) ? xb[i - NZ] : 0.0;
  }

  const double dt = pp[C.po_dt];
  const double hdt = 0.5 * dt;
  const double mass = pp[C.po_mass];
  const double kt = pp[C.po_kt], kbs = pp[C.po_kbs], eps = pp[C.po_eps], mu = pp[C.po_mu];
  const double* ref = pp + C.po_refs0 + R_COUNT * k;
  double* gb = g + b * C.m;
  const double* lb = lam + b * C.m;
  const double sg = want_hess ? sigma[b] : 0.0;
  // {jc_base, jc_off, jc_cnt, hc_base} of the knot class: re-read (L1) by each phase that scatters rather than held
  // in registers from here
  auto knot_maps = [&]() { return *reinterpret_cast<const int4*>(&C.knot_maps[k].jc_base); };
  auto jput = [&](int e, double v) {
    const int4 km = knot_maps();
    const int slot = C.jc_map[km.y + e];
    if (slot >= 0) jac[b * C.nnz_j + km.x + slot] = v;
  };
  auto hadd = [&](int vi, int vj, double v) {
    const int e = C.hc_index[vi * NCV + vj];
    if (e >= 0) hbuf[e] += v;
  };
  auto lamrow = [&](int fam, int kk, int r) -> double {
    const int row = grow(G, fam, kk, r);
    return row >= 0 ? lb[row] : 0.0;
  };
  // Multipliers of this lane's contact-point rows and of the momentum dynamics, requested here so that
  // their DRAM latency overlaps the g / Jacobian work (they are consumed in the Hessian section).
  double lam_pl[3] = {0.0, 0.0, 0.0}, lam_dcc = 0.0, lam_h = 0.0, lam_n = 0.0, lam_fr = 0.0, La[3] = {0.0, 0.0, 0.0};
  if (want_hess && lane < 8) {
    const int fb_ = lane * HB_KF_PT_COUNT;
    const int rp = grow(G, fb_ +HB_KF_PT_PLANAR, k, 0), rd = grow(G, fb_ +HB_KF_PT_DCC, k, 0);
    const int rf = grow(G, fb_ +HB_KF_PT_FRICTION, k, 0);
    const int ra = grow(C, HB_KF_H_DYN, k, 3), rb = grow(C, HB_KF_H_DYN, k + 1, 3);
    if (rp >= 0) {
      lam_pl[0] = lb[rp];
      lam_pl[1] = lb[rp + 1];
      lam_pl[2] = lb[rp + 2];
    }
    if (rd >= 0) lam_dcc = lb[rd];
    if (rf >= 0) lam_fr = lb[rf];
    if constexpr (TERRAIN != 0) {
      lam_h = lamrow(fb_ + HB_KF_PT_HEIGHT, k, 0);
      lam_n = lamrow(fb_ + HB_KF_PT_NORMAL, k, 0);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) La[c] = (ra >= 0 ? lb[ra + c] : 0.0) + (rb >= 0 ? lb[rb + c] : 0.0);
  }
#pragma unroll
  for (int u = 0; u < 6; ++u) {
    const int i = lane + 32 * u;
    if (i < NZ) {
      zs[i] = xs_[u];
      zp[i] = xp_[u];
    }
  }
  if (want_hess && lane < 8) {
    double* pk = park + lane;
    pk[8 * PK_L0] = lam_pl[0];
    pk[8 * PK_L1] = lam_pl[1];
    pk[8 * PK_LD] = lam_dcc;
    pk[8 * PK_LF] = lam_fr;
#pragma unroll
    for (int c = 0; c < 3; ++c) pk[8 * (PK_LA + c)] = La[c];
  }
  for (int i = lane; i < C.n_hc; i += 32) hbuf[i] = 0.0;
  for (int i = lane; i < NCV; i += 32) gbuf[i] = 0.0;
  __syncwarp();
  HB_PHASE(1, 0);  // inputs loaded and staged

  // ------------------------------------------------------------------ per-point quantities (lanes 0..7)
  const int pi_ = lane & 7;
  double cost = 0.0;

  // ------------------------------------------------------------------ g rows
  if (want_g) {
    // linear defects / initial conditions
    for (int j = lane; j < 81; j += 32) {
      int so, ro, fd, fi, comp;
      linear_state(j, so, ro, fd, fi, comp);
      if (k1) {
        const int r = grow(G, fd, k, comp);
        if (r >= 0) gb[r] = zs[so] - (zp[so] + hdt * (zp[ro] + zs[ro]));
      } else {
        const int r = grow(G, fi, 0, comp);
        if (r >= 0) gb[r] = zs[so];
      }
    }
    if (!k1 && lane < 6) {
      const int r = grow(C, HB_KF_H_IC, 0, lane);
      if (r >= 0) gb[r] = zs[Z_H + lane] - xinst[C.h_init + lane];
    }
  }
  // centroidal momentum dynamics: F(z) = g + sum_i [f_i; (p_i - x) x f_i] at knots k (lanes 0..7) and k-1 (8..15)
  {
    const double* zz = (lane & 8) ? zp : zs;
    const D3 pos = ld3(zz + 15 * pi_ + Z_P), frc = ld3(zz + 15 * pi_ + Z_F), com = ld3(zz + Z_COM);
    D3 lin = frc, ang = cross(pos - com, frc);
    if (lane >= 16) lin = ang = v3<double>(0.0, 0.0, 0.0);
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
      lin.x += __shfl_xor_sync(0xffffffffu, lin.x, o);
      lin.y += __shfl_xor_sync(0xffffffffu, lin.y, o);
      lin.z += __shfl_xor_sync(0xffffffffu, lin.z, o);
      ang.x += __shfl_xor_sync(0xffffffffu, ang.x, o);
      ang.y += __shfl_xor_sync(0xffffffffu, ang.y, o);
      ang.z += __shfl_xor_sync(0xffffffffu, ang.z, o);
    }
    // lanes 0..7 hold F(z_k) sums, lanes 8..15 F(z_{k-1}); bring both to lanes 0..5
    const double Fk[6] = {lin.x, lin.y, lin.z, ang.x, ang.y, ang.z};
    double fa = 0.0, fb = 0.0;
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const double vb_ = __shfl_sync(0xffffffffu, Fk[c], 0);
      const double va_ = __shfl_sync(0xffffffffu, Fk[c], 8);
      if (lane == c) {
        fb = vb_;
        fa = va_;
      }
    }
    if (want_g && k1 && lane < 6) {
      const double gr = pp[C.po_gravity + lane];
      const int r = grow(C, HB_KF_H_DYN, k, lane);
      if (r >= 0) gb[r] = zs[Z_H + lane] - (zp[Z_H + lane] + hdt * ((gr + fa) + (gr + fb)));
    }
  }
  const D3 fsum = v3<double>(
      zs[Z_F] + zs[15 + Z_F] + zs[30 + Z_F] + zs[45 + Z_F] + zs[60 + Z_F] + zs[75 + Z_F] + zs[90 + Z_F] + zs[105 + Z_F],
      zs[Z_F + 1] + zs[16 + Z_F] + zs[31 + Z_F] + zs[46 + Z_F] + zs[61 + Z_F] + zs[76 + Z_F] + zs[91 + Z_F] + zs[106 + Z_F],
      zs[Z_F + 2] + zs[17 + Z_F] + zs[32 + Z_F] + zs[47 + Z_F] + zs[62 + Z_F] + zs[77 + Z_F] + zs[92 + Z_F] + zs[107 + Z_F]);
  const D3 comv = ld3(zs + Z_COM);
  // the point's variables, read here (after the defect and momentum rows) so that they are not live through them
  const double* zpt = zs + 15 * pi_;
  const D3 pv = ld3(zpt + Z_V), pfd = ld3(zpt + Z_FD), ppos = ld3(zpt + Z_P), pf = ld3(zpt + Z_F), pu = ld3(zpt + Z_U);
  const double tau = tanh(kt * ppos.z);

  if constexpr (TERRAIN != 0) {
    // ---------------------------------------------------------------- smooth-step terrains (config 5, the ramp)
    const double* tp = pp + C.po_terrain;
    const int n_steps = TERRAIN == 2 ? (G.n_p - C.po_terrain) / 10 : 0;  // the step records close p
    if (lane < 8) {
      const int fb_ = lane * HB_KF_PT_COUNT;
      const int o = 15 * lane;
      TFrame F;
      terrain_frame<TERRAIN>(tp, n_steps, ppos.x, ppos.y, ppos.z, F);
      const double t0 = tanh(kt * F.h.c[0]);
      const double t1 = kt * (1.0 - t0 * t0);
      const TJ tauj = tj_compose(F.h, t0, t1, -kt * t0 * t1);
      const TJ Nn = tj_dot(F.n, pf), Nd = tj_dot(F.n, pfd), X = tj_dot(F.xh, pf), Y = tj_dot(F.yh, pf);
      const TJ Xv = tj_dot(F.xh, pv), Yv = tj_dot(F.yh, pv);
      const TJ hv = pv.x * F.gx + pv.y * F.gy + pv.z;  // grad h . v
      TJ Dnv[3], planar[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        Dnv[a] = pv.x * F.Dn[a][0] + pv.y * F.Dn[a][1];
        planar[a] = -(pu.x * (tauj * F.xh[a]) + pu.y * (tauj * F.yh[a]) + pu.z * F.n[a]) + comp(pv, a);
      }
      const TJ fDnv = tj_dot(Dnv, pf);
      const TJ margin = -(kbs * (F.h * Nn)) - (hv * Nn + F.h * fDnv + F.h * Nd) + eps;
      const TJ fric = (mu * mu) * (Nn * Nn) - X * X - Y * Y;
      const double hd = ref[R_SWING];
      const TJ dh = F.h + (-hd);
      const TJ swing = 0.5 * (dh * dh + Xv * Xv + Yv * Yv);
      const TJ DnTf0 = pf.x * F.Dn[0][0] + pf.y * F.Dn[1][0] + pf.z * F.Dn[2][0];
      const TJ DnTf1 = pf.x * F.Dn[0][1] + pf.y * F.Dn[1][1] + pf.z * F.Dn[2][1];
      if (want_g) {
        int r = grow(G, fb_ +HB_KF_PT_PLANAR, k, 0);
        if (r >= 0) {
          gb[r] = planar[0].c[0];
          gb[r + 1] = planar[1].c[0];
          gb[r + 2] = planar[2].c[0];
        }
        r = grow(G, fb_ +HB_KF_PT_DCC, k, 0);
        if (r >= 0) gb[r] = margin.c[0];
        r = grow(G, fb_ +HB_KF_PT_HEIGHT, k, 0);
        if (r >= 0) gb[r] = F.h.c[0];
        r = grow(G, fb_ +HB_KF_PT_NORMAL, k, 0);
        if (r >= 0) gb[r] = Nn.c[0];
        r = grow(G, fb_ +HB_KF_PT_FRICTION, k, 0);
        if (r >= 0) gb[r] = fric.c[0];
      }
      if (k1) {
        c_swing = C.w_swing * swing.c[0];
        cost += c_swing;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          gbuf[o + Z_P + a] += C.w_swing * swing.c[1 + a];
          gbuf[o + Z_V + a] += C.w_swing * (Xv.c[0] * F.xh[a].c[0] + Yv.c[0] * F.yh[a].c[0]);
        }
      }
      if (want_jac) {
        // the 58 entries of this point are listed first and their scatter slots loaded together: one
        // jput() per entry waited for its own map load (19 % of this kernel's stall samples)
        const int pb0 = 846 + 58 * lane;
        const int4 kmaps = knot_maps();
        const int* jmap = C.jc_map + kmaps.y;
        double* jb = jac + b * C.nnz_j + kmaps.x;
        double jv[58];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          jv[c] = 1.0;
          jv[3 + 3 * c + 0] = -t0 * F.xh[c].c[0];
          jv[3 + 3 * c + 1] = -t0 * F.yh[c].c[0];
          jv[3 + 3 * c + 2] = -F.n[c].c[0];
#pragma unroll
          for (int d = 0; d < 3; ++d) jv[12 + 3 * c + d] = planar[c].c[1 + d];
        }
        const double h0 = F.h.c[0], N0 = Nn.c[0];
        jv[21] = -(F.gx.c[0] * N0 + h0 * DnTf0.c[0]);
        jv[22] = -(F.gy.c[0] * N0 + h0 * DnTf1.c[0]);
        jv[23] = -N0;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          jv[24 + d] = -h0 * F.n[d].c[0];
          jv[27 + d] = margin.c[1 + d];
          jv[30 + d] = -kbs * h0 * F.n[d].c[0] - hv.c[0] * F.n[d].c[0] - h0 * Dnv[d].c[0];
          jv[33 + d] = F.h.c[1 + d];
          jv[38 + d] = F.n[d].c[0];
          jv[43 + d] = 2.0 * mu * mu * N0 * F.n[d].c[0] - 2.0 * X.c[0] * F.xh[d].c[0] - 2.0 * Y.c[0] * F.yh[d].c[0];
          jv[46 + d] = 1.0;
          jv[49 + d] = mass;
          jv[52 + d] = 1.0;
          jv[55 + d] = -1.0;
        }
        jv[36] = Nn.c[1];
        jv[37] = Nn.c[2];
        jv[41] = fric.c[1];
        jv[42] = fric.c[2];
#pragma unroll
        for (int c0 = 0; c0 < 58; c0 += 29) {
          int sl[29];
#pragma unroll
          for (int u = 0; u < 29; ++u) sl[u] = jmap[pb0 + c0 + u];
#pragma unroll
          for (int u = 0; u < 29; ++u)
            if (sl[u] >= 0) jb[sl[u]] = jv[c0 + u];
        }
      }
      if (want_hess) {
        const double lpl[3] = {lam_pl[0], lam_pl[1], lam_pl[2]};
        const D3 lplv = v3<double>(lpl[0], lpl[1], lpl[2]);
        const double ld = lam_dcc, lh = lam_h, ln = lam_n, lfr = lam_fr;
        const double sws = k1 ? sg * C.w_swing : 0.0;
        const TJ Lp = lpl[0] * planar[0] + lpl[1] * planar[1] + lpl[2] * planar[2] + ld * margin + lh * F.h + ln * Nn +
                      lfr * fric + sws * swing;
        // 63 contributions of this point: listed, their table entries loaded together, then accumulated
        int ti[63], nterm = 0;
        double tv[63];
        auto term = [&](int vi, int vj, double v) {
          ti[nterm] = vi * NCV + vj;
          tv[nterm] = v;
          ++nterm;
        };
        {
          int e = 0;
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int bb = a; bb < 3; ++bb) term(o + Z_P + a, o + Z_P + bb, tj_hess(Lp, e++));
        }
        const TJ Gu[3] = {-(tauj * tj_dot(F.xh, lplv)), -(tauj * tj_dot(F.yh, lplv)), -tj_dot(F.n, lplv)};
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          const TJ gd = d == 0 ? F.gx * Nn + F.h * DnTf0 : (d == 1 ? F.gy * Nn + F.h * DnTf1 : Nn);
          const TJ Gv = (-ld) * gd + sws * (Xv * F.xh[d] + Yv * F.yh[d]);
          const TJ Gfd = (-ld) * (F.h * F.n[d]);
          const TJ Gf = (-ld) * (kbs * (F.h * F.n[d]) + hv * F.n[d] + F.h * Dnv[d]) + ln * F.n[d] +
                        lfr * ((2.0 * mu * mu) * (Nn * F.n[d]) - 2.0 * (X * F.xh[d]) - 2.0 * (Y * F.yh[d]));
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            term(o + Z_P + a, o + Z_U + d, Gu[d].c[1 + a]);
            term(o + Z_P + a, o + Z_V + d, Gv.c[1 + a]);
            term(o + Z_P + a, o + Z_FD + d, Gfd.c[1 + a]);
            term(o + Z_P + a, o + Z_F + d, Gf.c[1 + a]);
          }
        }
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
          for (int bb = 0; bb < 3; ++bb) {
            const double ga = a == 0 ? F.gx.c[0] : (a == 1 ? F.gy.c[0] : 1.0);
            const double dnba = a < 2 ? F.Dn[bb][a].c[0] : 0.0;
            term(o + Z_V + a, o + Z_F + bb, -ld * (ga * F.n[bb].c[0] + F.h.c[0] * dnba));
            if (bb >= a) {
              term(o + Z_F + a, o + Z_F + bb,
                   lfr * (2.0 * mu * mu * F.n[a].c[0] * F.n[bb].c[0] - 2.0 * F.xh[a].c[0] * F.xh[bb].c[0] -
                          2.0 * F.yh[a].c[0] * F.yh[bb].c[0]));
              term(o + Z_V + a, o + Z_V + bb, sws * (F.xh[a].c[0] * F.xh[bb].c[0] + F.yh[a].c[0] * F.yh[bb].c[0]));
            }
          }
#pragma unroll
        for (int c0 = 0; c0 < 63; c0 += 21) {
          int te[21];
#pragma unroll
          for (int u = 0; u < 21; ++u) te[u] = C.hc_index[ti[c0 + u]];
#pragma unroll
          for (int u = 0; u < 21; ++u)
            if (te[u] >= 0) hbuf[te[u]] += tv[c0 + u];
        }
      }
    }
    if (lane == 8) {
      // minimum CoM height: h(com) = com_z - T(com_x, com_y)
      const BJ<2> T2 = bj_trunc<4, 2>(terrain_surface<TERRAIN>(tp, n_steps, comv.x, comv.y));
      if (want_g) {
        const int r = grow(C, HB_KF_COM_HEIGHT, k, 0);
        if (r >= 0) gb[r] = comv.z - T2.c[0];
      }
      if (want_jac) {
        jput(1310 + 12, -T2.c[bidx(1, 0)]);
        jput(1310 + 13, -T2.c[bidx(0, 1)]);
        jput(1310 + 14, 1.0);
      }
      if (want_hess) {
        const double lc = lamrow(HB_KF_COM_HEIGHT, k, 0);
        hadd(CV_COM, CV_COM, -2.0 * lc * T2.c[bidx(2, 0)]);
        hadd(CV_COM, CV_COM + 1, -lc * T2.c[bidx(1, 1)]);
        hadd(CV_COM + 1, CV_COM + 1, -2.0 * lc * T2.c[bidx(0, 2)]);
      }
    }
  }
  if (lane < 8) {
    const int fb_ = lane * HB_KF_PT_COUNT;
    if (want_g) {
      int r;
      if constexpr (TERRAIN == 0) {
        r = grow(G, fb_ +HB_KF_PT_PLANAR, k, 0);
        if (r >= 0) {
          gb[r] = pv.x - tau * pu.x;
          gb[r + 1] = pv.y - tau * pu.y;
          gb[r + 2] = pv.z - pu.z;
        }
        r = grow(G, fb_ +HB_KF_PT_DCC, k, 0);
        if (r >= 0) gb[r] = eps - kbs * (ppos.z * pf.z) - (pv.z * pf.z + ppos.z * pfd.z);
        r = grow(G, fb_ +HB_KF_PT_HEIGHT, k, 0);
        if (r >= 0) gb[r] = ppos.z;
        r = grow(G, fb_ +HB_KF_PT_NORMAL, k, 0);
        if (r >= 0) gb[r] = pf.z;
        r = grow(G, fb_ +HB_KF_PT_FRICTION, k, 0);
        if (r >= 0) gb[r] = -(pf.x * pf.x) - pf.y * pf.y + mu * mu * (pf.z * pf.z);
      }
      r = grow(G, fb_ +HB_KF_PT_U_BOUNDS, k, 0);
      if (r >= 0) {
        gb[r] = pu.x;
        gb[r + 1] = pu.y;
        gb[r + 2] = pu.z;
      }
      r = grow(G, fb_ +HB_KF_PT_FD_BOUNDS, k, 0);
      if (r >= 0) {
        gb[r] = pfd.x * mass;
        gb[r + 1] = pfd.y * mass;
        gb[r + 2] = pfd.z * mass;
      }
    }
    // per-point costs (k >= 1): swing heuristic, control regularisations
    if (k1) {
      double* gp = gbuf + 15 * lane;
      if constexpr (TERRAIN == 0) {
        const double hd = ref[R_SWING];
        const double dh = ppos.z - hd;
        c_swing = C.w_swing * 0.5 * (dh * dh + (pv.x * pv.x + pv.y * pv.y));
        cost += c_swing;
        gp[Z_P + 2] += C.w_swing * dh;
        gp[Z_V] += C.w_swing * pv.x;
        gp[Z_V + 1] += C.w_swing * pv.y;
      }
      const double c_u = C.w_u * (pu.x * pu.x + pu.y * pu.y + pu.z * pu.z);
      const double c_fd = C.w_fd * (pfd.x * pfd.x + pfd.y * pfd.y + pfd.z * pfd.z);
      cost += c_u;
      cost += c_fd;
      if (want_terms) {
        ct(HB_CT_SWING0 + lane) = c_swing;
        ct(HB_CT_UV0 + lane) = c_u;
        ct(HB_CT_FDOT0 + lane) = c_fd;
      }
      gp[Z_U] += 2.0 * C.w_u * pu.x;
      gp[Z_U + 1] += 2.0 * C.w_u * pu.y;
      gp[Z_U + 2] += 2.0 * C.w_u * pu.z;
      gp[Z_FD] += 2.0 * C.w_fd * pfd.x;
      gp[Z_FD + 1] += 2.0 * C.w_fd * pfd.y;
      gp[Z_FD + 2] += 2.0 * C.w_fd * pfd.z;
    }
  }
  if (want_terms && !k1)  // expressions with apply_to_first_elements = False do not exist at knot 0
    for (int i = lane; i < HB_CT_FRAME_QUAT; i += 32) ct(i) = 0.0;
  __syncwarp();
  // CoM velocity cost (all knots): sum_c w_c (h_c - ref_c)^2
  {
    double c_cv = 0.0;
    if (lane < 3) {
      const double e = zs[Z_H + lane] - ref[R_COMV + lane];
      c_cv = C.w_comvel[lane] * e * e;
    }
    if (want_terms) {
      const double t = warp_sum(c_cv);
      if (lane == 0) ct(HB_CT_COM_VELOCITY) = t;
    }
  }
  if (lane < 3) {
    const double e = zs[Z_H + lane] - ref[R_COMV + lane];
    cost += C.w_comvel[lane] * e * e;
    gbuf[CV_H + lane] += 2.0 * C.w_comvel[lane] * e;
    if (want_hess) hadd(CV_H + lane, CV_H + lane, 2.0 * sg * C.w_comvel[lane]);
  }
  if (want_g) {
    if (lane < 3) {
      const int r = grow(C, HB_KF_L_BOUNDS, k, lane);
      if (r >= 0) gb[r] = zs[Z_H + 3 + lane] * mass;
    }
    if (lane == 3) {
      int r = -1;
      if constexpr (TERRAIN == 0) {
        r = grow(C, HB_KF_COM_HEIGHT, k, 0);
        if (r >= 0) gb[r] = comv.z;
      }
      r = grow(C, HB_KF_FEET_RELH, k, 0);
      if (r >= 0) {
        const double lc = (((zs[Z_P + 2] + zs[15 + Z_P + 2]) + zs[30 + Z_P + 2]) + zs[45 + Z_P + 2]) / 4.0;
        const double rc = (((zs[60 + Z_P + 2] + zs[75 + Z_P + 2]) + zs[90 + Z_P + 2]) + zs[105 + Z_P + 2]) / 4.0;
        gb[r] = lc - rc;
      }
    }
    if (lane < HB_N_JOINTS) {
      int r = grow(C, HB_KF_S_BOUNDS, k, lane);
      if (r >= 0) gb[r] = zs[Z_S + lane];
      r = grow(C, HB_KF_SD_BOUNDS, k, lane);
      if (r >= 0) gb[r] = zs[Z_SD + lane];
    }
    // final state rows (alphabetical leaf order, optimization_object.py:305-306) / periodicity
    if (C.has_final && k == N - 1) {
      const int r0 = grow(C, HB_KF_FINAL, k, 0);
      for (int r = lane; r < 105; r += 32) {
        double v;
        if (r < 3) v = zs[Z_COM + r];
        else if (r < 75) {
          const int i = (r - 3) / 9, w = ((r - 3) % 9) / 3, c = (r - 3) % 3;
          v = w == 0 ? pp[C.po_desc0 + 24 * k + 3 * i + c] : (w == 1 ? zs[15 * i + Z_F + c] : zs[15 * i + Z_P + c]);
        } else if (r < 78) v = zs[Z_PB + r - 75];
        else if (r < 82) v = zs[Z_Q + r - 78];
        else v = zs[Z_S + r - 82];
        gb[r0 + r] = v;
      }
    }
    if (C.has_per && k == 0) {
      const int r0 = grow(C, HB_KF_PERIODICITY, 0, 0);
      const double* xl = xinst + (long)(N - 1) * NZ;
      for (int r = lane; r < 84; r += 32) {
        int off;
        if (r < 48) off = 15 * (r / 6) + ((r % 6) < 3 ? Z_U + r % 3 : Z_FD + r % 3);
        else if (r < 54) off = Z_H + r - 48;
        else if (r < 57) off = Z_VB + r - 54;
        else if (r < 61) off = Z_QD + r - 57;
        else off = Z_SD + r - 61;
        gb[r0 + r] = zs[off] - xl[off];
      }
    }
  }

  // The previous knot's variables are dead after the defect rows (last read before the __syncwarp above): the
  // Jacobian's derived sources and coefficient table take their place here, so that what the Jacobian phase needs
  // of this lane's point is in shared memory, not held in registers through the least-squares rows.
  // The point's values are re-read from zs, k_t and k_bs from the parameters (L1): held from the per-point rows to
  // here and on to the Hessian terms, they were spilled at 72 registers.
  const double kt_ = pp[C.po_kt], kbs_ = pp[C.po_kbs];
  const double dtau = kt_ * (1.0 - tau * tau);  // d tau / d p_z
  const double ddtau = -2.0 * kt_ * tau * dtau;  // d2 tau / d p_z2
  if (want_jac) {
    if (lane < 8) {
      zs[JX_TAU + lane] = tau;
      zs[JX_DTAU_U + 2 * lane] = dtau * zpt[Z_U];
      zs[JX_DTAU_U + 2 * lane + 1] = dtau * zpt[Z_U + 1];
      zs[JX_KF + lane] = kbs_ * zpt[Z_F + 2] + zpt[Z_FD + 2];
      zs[JX_KP + lane] = kbs_ * zpt[Z_P + 2] + zpt[Z_V + 2];
    }
    if (lane < 24) zs[JX_PC + lane] = zs[15 * (lane / 3) + Z_P + lane % 3] - zs[Z_COM + lane % 3];
    if (lane >= 24 && lane < 27) zs[JX_FSUM + lane - 24] = lane == 24 ? fsum.x : (lane == 25 ? fsum.y : fsum.z);
    if (lane == 27) zs[JX_ONE] = 1.0;
    if (lane < JC_COUNT) {  // coefficient table, order of the JC_* codes
      const double cv = lane == JC_ONE ? 1.0 : lane == JC_MONE ? -1.0 : lane == JC_HDT ? hdt : lane == JC_MHDT ? -hdt
                      : lane == JC_MASS ? mass : lane == JC_QUARTER ? 0.25 : lane == JC_MQUARTER ? -0.25
                      : lane == JC_PERIODIC ? (k == 0 ? 1.0 : -1.0) : lane == JC_MTWO ? -2.0 : 2.0 * mu * mu;
      zs[JX_COEF + lane] = cv;
    }
  }
  if (want_hess && lane < 8) {
    park[8 * PK_DTAU + lane] = dtau;
    park[8 * PK_DDTAU + lane] = ddtau;
  }

  HB_PHASE(1, 1);  // g rows, per-point terms
  // ------------------------------------------------------------------ least-squares cost rows (k >= 1)
  // 31 linear residuals r = c^T z - ref, each with cost w r^2:
  //   row 0..2    contacts centroid, component c: coefficient -1/8 on the eight p_c
  //   row 3..6    foot yaw, 3 + 2 foot + side: (sin, -cos) on (p_x, p_y) of point pa, (-sin, cos) on point pb,
  //               where (pa, pb) = yaw points (yaw[side], yaw[side + 1]) of the foot
  //   row 7..30   force ratio, 7 + 12 foot + 3 i + c: delta_ij - alpha_i on the four f_c of the foot
  // Lane `row` evaluates one residual.  The gradient 2 w r c and the Hessian 2 sigma w c c^T are summed in closed
  // form: lane v < 24 owns the variables p_c and f_c of point v / 3, c = v % 3, and the Hessian entries of lane l
  // are C.hc_ls[8 l .. 8 l + 6] (hb_kino_create builds them in the order of the slots below).  Every gradient
  // element and every entry is written by one lane, once: no row tables, no rounds, a fixed summation order.
  if (k1 && (want_f || want_grad || want_hess || want_terms)) {
    double w = 0.0, r = 0.0, sn = 0.0, cs = 0.0;
    if (lane < 3) {
      double acc = 0.0;
      for (int i = 0; i < 8; ++i) acc += zs[15 * i + Z_P + lane];
      r = ref[R_CC + lane] - 0.125 * acc;
      w = C.w_centroid * ref[R_CW + lane];
    } else if (lane < 7) {
      const int foot = (lane - 3) >> 1, side = (lane - 3) & 1;
      const double yaw = ref[foot == 0 ? R_YAW_L : R_YAW_R] + (side ? 1.5707963267948966 : 0.0);
      sincos(yaw, &sn, &cs);
      const int pa = 15 * (4 * foot + C.yaw[side]) + Z_P, pb = 15 * (4 * foot + C.yaw[side + 1]) + Z_P;
      r = -sn * (zs[pb] - zs[pa]) + cs * (zs[pb + 1] - zs[pa + 1]);
      w = 0.5 * C.w_yaw;
    } else if (lane < LS_ROWS) {
      const int t = lane - 7;
      const int foot = t / 12, i = (t % 12) / 3, c = t % 3;
      const double alpha = ref[(foot == 0 ? R_RATIO_L : R_RATIO_R) + i];
      const double* zf = zs + 60 * foot + Z_F + c;
      r = zf[15 * i] - alpha * (((zf[0] + zf[15]) + zf[30]) + zf[45]);
      w = C.w_ratio;
    }
    const double cr = w * r * r;
    cost += cr;
    if (want_terms) {  // lane 0: centroid (rows 0..2); 1, 2: yaw left / right; 3 + 4 foot + i: force ratio of (foot, i)
      const int r0 = lane == 0 ? 0 : (lane < 3 ? 3 + 2 * (lane - 1) : 7 + 3 * (lane - 3));
      const int n = lane == 0 ? 3 : (lane < 3 ? 2 : 3);
      double t = 0.0;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const double v = __shfl_sync(0xffffffffu, cr, (r0 + i) & 31);
        if (i < n) t += v;
      }
      if (lane < 11)
        ct(lane == 0 ? HB_CT_CENTROID : (lane == 1 ? HB_CT_YAW_LEFT : (lane == 2 ? HB_CT_YAW_RIGHT : HB_CT_FRATIO0 + lane - 3))) = t;
    }
    // sine and cosine of the two yaw rows of `foot`; sign of point pt in yaw row (foot, side): +1 on pa, -1 on pb, else 0
    double ysn[4], ycs[4];
#pragma unroll
    for (int y = 0; y < 4; ++y) {
      ysn[y] = __shfl_sync(0xffffffffu, sn, 3 + y);
      ycs[y] = __shfl_sync(0xffffffffu, cs, 3 + y);
    }
    auto ysgn = [&](int pt, int side) {
      const int q = pt & 3;
      return q == C.yaw[side] ? 1.0 : (q == C.yaw[side + 1] ? -1.0 : 0.0);
    };
    const double wy = 0.5 * C.w_yaw;
    if (want_grad) {
      const int pt = lane / 3, c = lane % 3, foot = (pt >> 2) & 1;
      const double rc = __shfl_sync(0xffffffffu, r, c), wc = __shfl_sync(0xffffffffu, w, c);
      double ry[2], rf[4];
#pragma unroll
      for (int s = 0; s < 2; ++s) ry[s] = __shfl_sync(0xffffffffu, r, 3 + 2 * foot + s);
#pragma unroll
      for (int i = 0; i < 4; ++i) rf[i] = __shfl_sync(0xffffffffu, r, (7 + 12 * foot + 3 * i + c) & 31);
      if (lane < 24) {
        double gp = 2.0 * wc * rc * -0.125;
        if (c < 2) {
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const double kk = c == 0 ? (foot ? ysn[2 + s] : ysn[s]) : -(foot ? ycs[2 + s] : ycs[s]);
            gp += 2.0 * wy * ry[s] * (ysgn(pt, s) * kk);
          }
        }
        gbuf[15 * pt + Z_P + c] += gp;
        const double* al = ref + (foot ? R_RATIO_R : R_RATIO_L);
        double gf = 0.0;
#pragma unroll
        for (int i = 0; i < 4; ++i) gf += 2.0 * C.w_ratio * rf[i] * ((i == (pt & 3) ? 1.0 : 0.0) - al[i]);
        gbuf[15 * pt + Z_F + c] += gf;
      }
    }
    if (want_hess) {
      const int4 q4 = *reinterpret_cast<const int4*>(C.hc_ls + 8 * lane);
      const int wv[4] = {q4.x, q4.y, q4.z, q4.w};
      const double tw = 2.0 * sg;
      double hv[7];
      // slots 0..3: p_c of points (i, j), component c = t / 36, pair q = t % 36 = 8 d + a -> {a, (a + d) mod 8}:
      // centroid row c, then (c = x, y, both points on one foot) the yaw rows of that foot
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int t = lane + 32 * u, c = t / 36, q = t % 36;
        const int a = q & 7, a2 = (a + (q >> 3)) & 7, i = min(a, a2), j = max(a, a2), foot = i >> 2;
        double v = tw * __shfl_sync(0xffffffffu, w, c & 3) * -0.125 * -0.125;
        if (c < 2 && foot == (j >> 2)) {
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const double kk = c == 0 ? (foot ? ysn[2 + s] : ysn[s]) : -(foot ? ycs[2 + s] : ycs[s]);
            v += tw * wy * (ysgn(i, s) * kk) * (ysgn(j, s) * kk);
          }
        }
        hv[u] = v;
      }
      {  // slot 4: (p_x of point 4 foot + i, p_y of point 4 foot + j), yaw rows only; lane = 16 foot + 4 i + j
        const int foot = lane >> 4, i = (lane >> 2) & 3, j = lane & 3;
        double v = 0.0;
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const double ks = foot ? ysn[2 + s] : ysn[s], kc = -(foot ? ycs[2 + s] : ycs[s]);
          v += tw * wy * (ysgn(i, s) * ks) * (ysgn(j, s) * kc);
        }
        hv[4] = v;
      }
      // slots 5, 6: f_c of points (i, j) of one foot, t = 10 (3 foot + c) + q, q = 4 d + a -> {a, (a + d) mod 4}:
      // the four force-ratio rows of (foot, c)
#pragma unroll
      for (int u = 5; u < 7; ++u) {
        const int t = lane + 32 * (u - 5), foot = (t / 30) & 1, q = t % 10;
        const int a = q & 3, a2 = (a + (q >> 2)) & 3, i = min(a, a2), j = max(a, a2);
        const double* al = ref + (foot ? R_RATIO_R : R_RATIO_L);
        double v = 0.0;
#pragma unroll
        for (int m = 0; m < 4; ++m) v += tw * C.w_ratio * ((m == i ? 1.0 : 0.0) - al[m]) * ((m == j ? 1.0 : 0.0) - al[m]);
        hv[u] = v;
      }
      // the entries of the warp are distinct: old values are read together, then written
      int te[7];
      double old[7];
#pragma unroll
      for (int u = 0; u < 7; ++u) te[u] = (int)(short)((u & 1) ? (wv[u >> 1] >> 16) : (wv[u >> 1] & 0xffff));
#pragma unroll
      for (int u = 0; u < 7; ++u) old[u] = te[u] >= 0 ? hbuf[te[u]] : 0.0;
#pragma unroll
      for (int u = 0; u < 7; ++u)
        if (te[u] >= 0) hbuf[te[u]] = old[u] + hv[u];
    }
  }

  HB_PHASE(1, 2);  // least-squares rows
  // ------------------------------------------------------------------ f partial + grad_f
  if (want_f || want_grad) {
    const double total = warp_sum(cost);
    if (lane == 0 && want_f && !want_terms) fpart[(b * N + k) * 2] = total;
  }
  __syncwarp();
  if (want_grad) {
    double* gf = grad_f + b * C.n_x + (long)k * NZ;
    for (int i = lane; i < NCV; i += 32) {
      const int off = i < 120 ? i : (i < CV_H ? Z_COM + i - CV_COM : Z_H + i - CV_H);
      gf[off] = gbuf[i];
    }
    if (k == 0 && lane < 6) grad_f[b * C.n_x + C.h_init + lane] = 0.0;
  }

  HB_PHASE(1, 3);  // f, grad_f
  // ------------------------------------------------------------------ Jacobian values
  // Every entry is coefficient x source (contact_jac_desc.h): the knot class's destination-sorted list is
  // streamed, {slot, descriptor} pairs, coalesced stores, no per-entry branching.
  if (want_jac) {
    __syncwarp();
    const int4 kmaps = knot_maps();
    double* jb = jac + b * C.nnz_j + kmaps.x;
    const int2* lst = C.jc_list + kmaps.y;
    const int n = kmaps.z;
    for (int eb = lane; eb < n; eb += 256) {
      int2 w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w[u] = (eb + 32 * u) < n ? lst[eb + 32 * u] : make_int2(-1, 0);
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (w[u].x >= 0) jb[w[u].x] = zs[JX_COEF + (w[u].y >> 16)] * zs[w[u].y & 0xffff];
    }
  }

  HB_PHASE(1, 4);  // Jacobian values + scatter
  // ------------------------------------------------------------------ Hessian of the Lagrangian, contact block
  if (want_hess) {
    if (lane < 8) {
      const int o = 15 * lane;
      const double* pk = park + lane;
      const double kk1 = k1 ? 1.0 : 0.0;  // cost terms and the friction row exist from knot 1 on
      // centroidal momentum dynamics: -(dt/2) (lam_k + lam_{k+1})_ang . ((p - x) x f), pair m = 0..5 of (a, b), a != b
      auto mom = [&](int m) {
        const int a = m / 2, bb = a == 0 ? 1 + m % 2 : (a == 1 ? 2 * (m % 2) : m % 2);
        return -hdt * eps3(a, bb) * pk[8 * (PK_LA + 3 - a - bb)];
      };
      if constexpr (TERRAIN == 0) {
        // The 29 terms of this point, in the order of their local entries in the per-point table C.hc_pt (64 bytes
        // per lane, four 16-byte loads that every warp shares in L1): 11 complementarity / friction / swing terms,
        // 6 control regularisations, 12 momentum cross terms.  The entries of one lane are distinct and no other
        // lane touches them, so old values are read, updated and written in batches of 10, each batch computing its
        // own values (the 29 values are never live at once).
        const int4* tq = reinterpret_cast<const int4*>(C.hc_pt + 32 * lane);
        const int4 q4[4] = {tq[0], tq[1], tq[2], tq[3]};
        const int wv[16] = {q4[0].x, q4[0].y, q4[0].z, q4[0].w, q4[1].x, q4[1].y, q4[1].z, q4[1].w,
                            q4[2].x, q4[2].y, q4[2].z, q4[2].w, q4[3].x, q4[3].y, q4[3].z, q4[3].w};
        constexpr int NT = 29;
        auto tval = [&](int t) -> double {
          const double ld = pk[8 * PK_LD], lf = kk1 * pk[8 * PK_LF];
          switch (t) {
            case 0: return -(pk[8 * PK_L0] * zs[o + Z_U] + pk[8 * PK_L1] * zs[o + Z_U + 1]) * pk[8 * PK_DDTAU] + kk1 * sg * C.w_swing;  // (p_z, p_z)
            case 1: return -pk[8 * PK_L0] * pk[8 * PK_DTAU];                                         // (p_z, u_x)
            case 2: return -pk[8 * PK_L1] * pk[8 * PK_DTAU];                                         // (p_z, u_y)
            case 3: return -ld * pp[C.po_kbs];                                                              // (p_z, f_z)
            case 4: return -ld;                                                                      // (v_z, f_z)
            case 5: return -ld;                                                                      // (fdot_z, p_z)
            case 6: case 7: return kk1 * sg * C.w_swing;                                             // (v_x, v_x), (v_y, v_y)
            case 8: case 9: return -2.0 * lf;                                                        // (f_x, f_x), (f_y, f_y)
            case 10: return 2.0 * mu * mu * lf;                                                      // (f_z, f_z)
            default: break;
          }
          if (t < 17) return (t & 1) ? kk1 * 2.0 * sg * C.w_u : kk1 * 2.0 * sg * C.w_fd;          // (u_c, u_c), (fdot_c, fdot_c)
          return ((t - 17) & 1) ? -mom((t - 17) >> 1) : mom((t - 17) >> 1);                       // (p_a, f_b), (com_a, f_b)
        };
#pragma unroll
        for (int c0 = 0; c0 < NT; c0 += 10) {
          int te[10];
          double old[10];
#pragma unroll
          for (int u = 0; u < 10; ++u) {
            const int t = c0 + u;
            te[u] = t < NT ? (int)(short)((t & 1) ? (wv[t >> 1] >> 16) : (wv[t >> 1] & 0xffff)) : -1;
          }
#pragma unroll
          for (int u = 0; u < 10; ++u) old[u] = te[u] >= 0 ? hbuf[te[u]] : 0.0;
#pragma unroll
          for (int u = 0; u < 10; ++u)
            if (c0 + u < NT && te[u] >= 0) hbuf[te[u]] = old[u] + tval(c0 + u);
        }
      } else {
        // The contributions of this point are listed first, their local entries loaded together, and only
        // then accumulated: a hadd() per term serialises "index load -> shared read-modify-write" (the
        // compiler cannot move the next index load above the previous shared store).
        constexpr int NT = 6 + 12;
        int ti[NT];
        double tv[NT];
        int n = 0;
        auto term = [&](int vi, int vj, double v) {
          ti[n] = vi * NCV + vj;
          tv[n] = v;
          ++n;
        };
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          term(o + Z_U + c, o + Z_U + c, kk1 * 2.0 * sg * C.w_u);
          term(o + Z_FD + c, o + Z_FD + c, kk1 * 2.0 * sg * C.w_fd);
        }
#pragma unroll
        for (int m = 0; m < 6; ++m) {
          const int a = m / 2, bb = a == 0 ? 1 + m % 2 : (a == 1 ? 2 * (m % 2) : m % 2);
          const double v = mom(m);
          term(o + Z_P + a, o + Z_F + bb, v);
          term(CV_COM + a, o + Z_F + bb, -v);
        }
        int te[NT];
#pragma unroll
        for (int u = 0; u < NT; ++u) te[u] = C.hc_index[ti[u]];
#pragma unroll
        for (int u = 0; u < NT; ++u)
          if (te[u] >= 0) hbuf[te[u]] += tv[u];
      }
    }
    HB_PHASE(1, 5);  // Hessian terms
    __syncwarp();
    const int2 hcm_ = *reinterpret_cast<const int2*>(&C.knot_maps[k].hc_off);  // {hc_off, hc_cnt}
    const int2 hcm = make_int2(C.knot_maps[k].hc_base, hcm_.x);
    const unsigned* hlst = C.hc_list + hcm.y;  // destination-sorted: entry << 16 | slot
    double* hb_ = hess + b * C.nnz_h + hcm.x;
    const int n_l = hcm_.y;
    for (int eb = lane; eb < n_l; eb += 256) {  // 8 list loads in flight before the dependent stores
      unsigned w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) w[u] = (eb + 32 * u) < n_l ? hlst[eb + 32 * u] : 0xffffffffu;
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (w[u] != 0xffffffffu) hb_[w[u] & 0xffffu] = hbuf[w[u] >> 16];
    }
  }
}

}  // namespace hb
