// kino_kin.cu -- floating-base kinematics block of the kinodynamic NLP: one warp per (instance, knot).
//
// Rows evaluated here (reference file:line of the expression each one restates):
//   unit quaternion            planner.py:276-282
//   contact FK consistency     planner.py:590-632  (expressions/kinematics.py:217-308)
//   CoM consistency            planner.py:284-306  (expressions/kinematics.py:134-214)
//   angular momentum consist.  planner.py:308-339  (expressions/kinematics.py:11-131, quaternion.py:25-51)
//   minimum feet distance      planner.py:360-383  (expressions/kinematics.py:311-394)
// Costs: frame orientation (planner.py:449-477, kinematics.py:397-491), base quaternion (:479-491,
// quaternion.py:54-85), quaternion velocity (:493-503), joint regularisation (:505-520).
//
// Algorithm (not the reference's: CasADi differentiates an expression graph; here the tree structure
// is used directly).
//   1. primal forward kinematics by depth level (lane = body), world transforms, twists, world
//      inertias staged in shared memory; CoM / momentum sums by warp shuffles;
//   2. Jacobian by forward mode: lane j carries the unit tangent of variable j (4 quaternion + 23 joint
//      directions).  A direction rotates one sub-tree rigidly about its joint, so the tangents of the
//      contact points, of the CoM, of P_dot and of the angular momentum are closed-form in the staged
//      primal state and in the composite (sub-tree) moments -- column j of the kinematic rows, no sweep;
//   3. Hessian: the adjoints of the Lagrangian (true multipliers as seeds) once per warp, lane = body
//      (primal_adjoint_pass); then only the TANGENT of those adjoints along every direction, as
//      (direction, body) tasks packed on the lanes by a host-built schedule (kin_tangent_sweep_packed):
//      column j of the Lagrangian Hessian restricted to (q, s) x (vb, qd, sd, q, s).
//   The lean kernel (f and g) also holds the first algorithm for the Jacobian -- a row-per-lane adjoint sweep in
//   fp64 (kin_backward: 32 rows = 24 FK, 3 CoM, 3 momentum, feet distance, frame-orientation trace) -- selected by
//   hb_set_option(HB_OPT_JAC_ADJOINT): an independent cross-check of the forward-mode Jacobian.
#include "kino_const.cuh"

namespace hb {

// per-body staging in shared memory (doubles): origin, CoM arm, twist, world axis, world inertia, rotation,
// I.w, I.hbar, rho = o - o_parent, and (Hessian pass) the primal adjoint totals (n, F, wbar, vbar) plus the
// local primal adjoints cbar, cdbar
enum {
  SB_O = 0, SB_D = 3, SB_W = 6, SB_V = 9, SB_AX = 12, SB_I = 15, SB_R = 21, SB_L = 30, SB_IH = 33, SB_RHO = 36,
  SB_ACC = 39, SB_STRIDE = 51,
  SB_CB = SB_R, SB_CDB = SB_R + 3  // alias the rotation: it is dead once the frames have been staged
};
enum { HSTAGE = 27 * 57 };  // per-warp staging of the Hessian columns (and, before that, the Jacobian rows)
constexpr int KIN_SCAT = 17;  // scatter-map loads in flight per lane in the Hessian kernel's two scatters (8: 5.3 k -> see DESIGN.md)

struct KinSmem {
  int bodies, arms, fdu, fdal, fdar, G, z, gbuf, lamk, slot, stage, total;
};
__host__ __device__ inline KinSmem kin_smem_layout(int nb, int n_slots, bool with_hess) {
  KinSmem s;
  int o = 0;
  s.bodies = o;
  o += nb * SB_STRIDE;
  s.arms = o;
  o += 24;
  s.fdu = o;
  o += 3;
  s.fdal = o;
  o += 3;
  s.fdar = o;
  o += 3;
  s.G = o;
  o += 9;
  s.z = o;
  o += NZ + 1;
  s.gbuf = o;
  o += 58;
  s.lamk = o;  // multipliers of the 32 kinematic rows of the knot (Hessian variant)
  o += with_hess ? 32 : 0;
  s.slot = o;
  o += n_slots * 32 * 12;  // fp64 sweep: adjoints; Hessian sweep: their tangents (primal totals are per body)
  s.stage = o;
  // The Hessian kernel stages its values per warp and scatters them after the sweep with batched map loads.
  // Measured on B200 (config 3): direct stores from the sweep 2.47 ms (17 % of the stall samples sat on
  // the store waiting for its own map load); staging with a naive scatter loop 2.54 ms; staging with
  // the batched scatter 2.25 ms.  The lean kernel stores straight through the map: a stage would cost it
  // a CTA per SM.
  o += with_hess ? HSTAGE : 0;
  s.total = o;
  return s;
}

// direction data of one Hessian lane: every link state tangent is closed-form in these
struct Dir {
  D3 alpha, pi, wpi, vpi, u;
  unsigned mask;
};

template <class T>
struct St {
  V3<T> o, d, w, v, ax;
};

__device__ __forceinline__ St<double> load_state(const double* sb, int l) {
  const double* b = sb + l * SB_STRIDE;
  St<double> s;
  s.o = ld3(b + SB_O);
  s.d = ld3(b + SB_D);
  s.w = ld3(b + SB_W);
  s.v = ld3(b + SB_V);
  s.ax = ld3(b + SB_AX);
  return s;
}
__device__ __forceinline__ St<Dual> load_state(const double* sb, int l, const Dir& dir, Dual) {
  const double* b = sb + l * SB_STRIDE;
  const D3 o = ld3(b + SB_O), d = ld3(b + SB_D), w = ld3(b + SB_W), v = ld3(b + SB_V), ax = ld3(b + SB_AX);
  const double in = ((dir.mask >> l) & 1u) ? 1.0 : 0.0;
  const D3 a = scale(in, dir.alpha);
  const D3 uu = scale(in, dir.u);
  const D3 r = o - dir.pi;
  const D3 to = cross(a, r);
  const D3 tw = cross(a, w - dir.wpi) + uu;
  const D3 tv = cross(dir.wpi, to) + cross(a, (v - dir.vpi) - cross(dir.wpi, r)) + cross(uu, r);
  St<Dual> s;
  s.o = lift<Dual>(o, to);
  s.d = lift<Dual>(d, cross(a, d));
  s.w = lift<Dual>(w, tw);
  s.v = lift<Dual>(v, tv);
  s.ax = lift<Dual>(ax, cross(a, ax));
  return s;
}

// I^w w_l with the primal product staged in shared memory (SB_L), and I^w hbar
__device__ __forceinline__ D3 iw_omega(const double* sb, int l) {
  return ld3(sb + l * SB_STRIDE + SB_L);
}
__device__ __forceinline__ D3 iw_hbar(const double* sb, int l, D3 hb) {
  return symmul(sb + l * SB_STRIDE + SB_I, hb);  // seeds differ per lane in the fp64 sweep
}
// rho_l = o_l - o_parent and the parent's angular velocity, without rebuilding the parent state
__device__ __forceinline__ void parent_link(const double* sb, int l, int p, D3& rho, D3& wp) {
  rho = ld3(sb + l * SB_STRIDE + SB_RHO);
  wp = ld3(sb + p * SB_STRIDE + SB_W);
}
// branch accumulators in shared memory, component-major and lane-minor
__device__ __forceinline__ void slot_get(D3& v, const double* sl, int c) {
  v.x += sl[(c)*32];
  v.y += sl[(c + 1) * 32];
  v.z += sl[(c + 2) * 32];
}
__device__ __forceinline__ void slot_add(double* sl, int c, D3 v) {
  sl[(c)*32] += v.x;
  sl[(c + 1) * 32] += v.y;
  sl[(c + 2) * 32] += v.z;
}

template <class T>
struct Seeds {
  D3 wc;            // d Phi / d (sum_l m_l c_l)   (constant along every direction)
  D3 hb;            // d Phi / d h_ang             (constant along every direction)
  V3<T> footF[2];   // force / torque (about the foot body origin) applied on the two foot bodies
  V3<T> footN[2];
  V3<T> chestN;     // torque on the frame-orientation body
};

// Right-trivialised angular velocity map Omega(a, b) = 2(-b_w a_v + a_w b_v - b_v x a_v)
// (expressions/quaternion.py:42), bilinear in (quaternion a, its rate b).
template <class A, class B>
__device__ __forceinline__ V3<typename Prom<A, B>::type> omega_map(const A* a, const B* b) {
  typedef typename Prom<A, B>::type T;
  V3<A> av = v3<A>(a[0], a[1], a[2]);
  V3<B> bv = v3<B>(b[0], b[1], b[2]);
  V3<T> c = cross(bv, av);
  return v3<T>(2.0 * (a[3] * b[0] - b[3] * a[0] - c.x), 2.0 * (a[3] * b[1] - b[3] * a[1] - c.y),
               2.0 * (a[3] * b[2] - b[3] * a[2] - c.z));
}

struct JacEmit {
  const int* map;  // jk_map row of this knot
  double* jac;     // instance base
  double* gbuf;    // shared: grad_f accumulation for the kinematic variables
  int lane;
  double gscale;   // chest lane: 2 w_frame (phi - 3)
  bool write;
  // local bases inside JK (kino_layout.py::_enumerate_jk)
  __device__ __forceinline__ int base_q() const {
    if (lane < 24) return 4 + lane * 27;
    if (lane < 27) return 4 + 648 + (lane - 24) * 27;
    if (lane < 30) return 4 + 648 + 81 + (lane - 27) * 57 + 7;  // after vb(3), qd(4)
    return -1;
  }
  __device__ __forceinline__ void put(int e, double v) const {
    const int slot = map[e];
    if (slot >= 0) jac[slot] = v;
  }
  // Scatter slots of the two entries the sweep emits at body l, loaded one step ahead (prefetch(l) is
  // called at the top of the iteration) so that the stores do not wait for their own map loads.
  int sbase, sdbase, pre_s, pre_sd;
  __device__ __forceinline__ void init_bases() {
    sdbase = -1;
    if (lane < 27) sbase = base_q() + 4;
    else if (lane < 30) {
      const int b = 4 + 648 + 81 + (lane - 27) * 57;
      sdbase = b + 11;
      sbase = b + 34;
    } else sbase = lane == 30 ? 4 + 648 + 81 + 171 : -1;
    pre_s = pre_sd = -1;
  }
  __device__ __forceinline__ void prefetch(int l) {
    if (!write || l < 1) return;
    pre_s = sbase >= 0 ? map[sbase + l - 1] : -1;
    pre_sd = sdbase >= 0 ? map[sdbase + l - 1] : -1;
  }
  __device__ __forceinline__ void joint(int l, double sbar, double sdbar) const {
    const int j = l - 1;
    if (lane == 31) {
      gbuf[34 + j] += gscale * sbar;  // gbuf order: vb3 qd4 q4 sd23 s23 -> s at 34
      return;
    }
    if (!write) return;
    if (pre_s >= 0) jac[pre_s] = sbar;
    if (pre_sd >= 0) jac[pre_sd] = sdbar;
  }
};

// One adjoint sweep over the tree.  `emit.joint(l, sbar, sdbar)` receives d Phi / d s_{l-1} and
// d Phi / d s_dot_{l-1}; the totals at the root are returned for the base chain rule.
__device__ __forceinline__ void kin_backward(const KinTopo& C, const double* sb, const double* zs,
                                             const Seeds<double>& S, const D3& xc, const D3& xd, double* slot,
                                             JacEmit& emit, D3& n0, D3& w0, D3& v0) {
  const int nb = C.nb;
  const int lane = threadIdx.x & 31;
  for (int i = 0; i < C.n_slots * 12; ++i) slot[i * 32 + lane] = 0.0;
  D3 cn = vzero<double>(), cF = vzero<double>(), cw = vzero<double>(), cv = vzero<double>();
  D3 An = vzero<double>(), AF = vzero<double>(), Aw = vzero<double>(), Av = vzero<double>();
  for (int l = nb - 1; l >= 0; --l) {
    emit.prefetch(l);
    if (!C.carry[l]) {
      cn = vzero<double>();
      cF = vzero<double>();
      cw = vzero<double>();
      cv = vzero<double>();
    }
    if (l == 0) {
      cn = cn + An;
      cF = cF + AF;
      cw = cw + Aw;
      cv = cv + Av;
    }
    const St<double> s = load_state(sb, l);
    // ---- local adjoints of body l
    {
      const double m = C.mass[l];
      const D3 c = s.o + s.d;
      const D3 cd = s.v + cross(s.w, s.d);
      const D3 cbar = scale(m, cross(cd - xd, S.hb) + S.wc);
      const D3 cdbar = scale(m, cross(S.hb, c - xc));
      const D3 Iw = iw_omega(sb, l);
      const D3 Ih = iw_hbar(sb, l, S.hb);
      cF = cF + cbar;
      cn = cn + cross(s.d, cbar) + cross(s.d, cross(cdbar, s.w)) + cross(Iw, S.hb) + cross(Ih, s.w);
      cv = cv + cdbar;
      cw = cw + cross(s.d, cdbar) + Ih;
      if (l == C.foot_body[0]) {
        cF = cF + S.footF[0];
        cn = cn + S.footN[0];
      }
      if (l == C.foot_body[1]) {
        cF = cF + S.footF[1];
        cn = cn + S.footN[1];
      }
      if (l == C.chest_body) cn = cn + S.chestN;
    }
    if (C.slot[l] >= 0) {
      const double* sl = slot + C.slot[l] * 12 * 32 + lane;
      slot_get(cn, sl, 0);
      slot_get(cF, sl, 3);
      slot_get(cw, sl, 6);
      slot_get(cv, sl, 9);
    }
    if (l == 0) break;
    // ---- joint outputs
    emit.joint(l, dot(s.ax, cn), dot(s.ax, cw));
    // ---- contribution to the parent
    const int p = C.parent[l];
    D3 rho, wpar;
    parent_link(sb, l, p, rho, wpar);
    const double sd = zs[Z_SD + l - 1];
    const D3 pn = cn + cross(rho, cF) + scale(sd, cross(s.ax, cw)) + cross(rho, cross(cv, wpar));
    const D3 pw = cw + cross(rho, cv);
    if (p == l - 1) {
      cn = pn;
      cw = pw;  // cF, cv carry unchanged
    } else if (p == 0) {
      An = An + pn;
      AF = AF + cF;
      Aw = Aw + pw;
      Av = Av + cv;
    } else {
      double* sl = slot + C.slot[p] * 12 * 32 + lane;
      slot_add(sl, 0, pn);
      slot_add(sl, 3, cF);
      slot_add(sl, 6, pw);
      slot_add(sl, 9, cv);
    }
  }
  n0 = cn;
  w0 = cw;
  v0 = cv;
}

// ---------------------------------------------------------------------------------------------------
// Hessian pass, split in two so that no lane recomputes what is identical for all of them:
//   (1) primal_adjoint_pass: the adjoints of the Lagrangian (true multipliers as seeds) are the same
//       for every direction; they are computed ONCE per warp, lane = body, accumulated leaf-to-root by
//       depth level, and left in shared memory (SB_ACC totals, SB_CB / SB_CDB local terms);
//   (2) kin_tangent_sweep_packed: only the TANGENT of those adjoints is propagated along every
//       direction (product rule with the staged primal values) -- 2/3 of the arithmetic of a sweep in
//       dual numbers and half of its registers.
struct SeedsP {
  D3 wc, hb, footF[2], footN[2], chestN;
};
struct SeedsT {
  D3 footF[2], footN[2], chestN;  // wc and hb are constants: zero tangent
};

__device__ __forceinline__ void primal_adjoint_pass(const KinTopo& T, double* sb, const double* zs, const SeedsP& S,
                                                    D3 xc, D3 xd, int my_depth, int my_rank, int my_parent,
                                                    double my_mass) {
  const int lane = threadIdx.x & 31;
  const int nb = T.nb;
  if (lane < nb) {
    double* bl = sb + lane * SB_STRIDE;
    const D3 o = ld3(bl + SB_O), d = ld3(bl + SB_D), w = ld3(bl + SB_W), v = ld3(bl + SB_V);
    const double m = my_mass;
    const D3 c = o + d;
    const D3 cd = v + cross(w, d);
    const D3 cbar = scale(m, cross(cd - xd, S.hb) + S.wc);
    const D3 cdbar = scale(m, cross(S.hb, c - xc));
    const D3 Iw = ld3(bl + SB_L), Ih = ld3(bl + SB_IH);
    D3 F = cbar;
    D3 n = cross(d, cbar) + cross(d, cross(cdbar, w)) + cross(Iw, S.hb) + cross(Ih, w);
    const D3 wb = cross(d, cdbar) + Ih;
    if (lane == T.foot_body[0]) {
      F = F + S.footF[0];
      n = n + S.footN[0];
    }
    if (lane == T.foot_body[1]) {
      F = F + S.footF[1];
      n = n + S.footN[1];
    }
    if (lane == T.chest_body) n = n + S.chestN;
    st3(bl + SB_ACC, n);
    st3(bl + SB_ACC + 3, F);
    st3(bl + SB_ACC + 6, wb);
    st3(bl + SB_ACC + 9, cdbar);
    st3(bl + SB_CB, cbar);
    st3(bl + SB_CDB, cdbar);
  }
  __syncwarp();
  // (depth, sibling rank) steps that have at least one body, deepest first: children of one parent are
  // serialised by rank so that the read-modify-write of the parent's totals needs no atomics
  for (int st = 0; st < T.n_steps; ++st) {
    if (my_depth == T.step_depth[st] && my_rank == T.step_rank[st]) {
      const double* bl = sb + lane * SB_STRIDE;
      double* bp = sb + my_parent * SB_STRIDE;
      const D3 n = ld3(bl + SB_ACC), F = ld3(bl + SB_ACC + 3), wb = ld3(bl + SB_ACC + 6), vb = ld3(bl + SB_ACC + 9);
      const D3 ax = ld3(bl + SB_AX), rho = ld3(bl + SB_RHO), wpar = ld3(bp + SB_W);
      const double sd = zs[Z_SD + lane - 1];
      const D3 pn = n + cross(rho, F) + scale(sd, cross(ax, wb)) + cross(rho, cross(vb, wpar));
      const D3 pw = wb + cross(rho, vb);
      st3(bp + SB_ACC, ld3(bp + SB_ACC) + pn);
      st3(bp + SB_ACC + 3, ld3(bp + SB_ACC + 3) + F);
      st3(bp + SB_ACC + 6, ld3(bp + SB_ACC + 6) + pw);
      st3(bp + SB_ACC + 9, ld3(bp + SB_ACC + 9) + vb);
    }
    __syncwarp();
  }
}

__device__ __forceinline__ D3 tangent_of(const V3<Dual>& a) { return v3<double>(a.x.d, a.y.d, a.z.d); }
__device__ __forceinline__ D3 primal_of(const V3<Dual>& a) { return v3<double>(a.x.v, a.y.v, a.z.v); }

// ---------------------------------------------------------------------------------------------------
// Packed tangent sweep.  In a plain sweep lane d would walk all the bodies although direction d only
// moves its own sub-tree: of the 27 x 23 body steps 188 carry non-zero state tangents and 92 more are
// pure propagation through the ancestors of the joint.  Here those (direction, body) steps are TASKS,
// list-scheduled by the host (api.cu::build_sweep_schedule) on the 32 lanes in ~12 rounds instead of
// 23: in every round a lane executes the task sched[round][lane] -- whatever direction it belongs to.
// The four quaternion directions are left out of the schedule (their columns are closed-form, see the
// quaternion columns in kino_kin_kernel): 256 tasks, 92 of them in a sub-tree, in 13 rounds.
//   * direction data (alpha, pivot, ...) and seed tangents stay in the registers of the OWNER lane d and
//     are fetched with warp shuffles by the lane that executes a task of direction d;
//   * a lane keeps the running adjoint of its chain in registers; where a chain ends it is added to a
//     shared-memory slot of the body it feeds (the schedule never lets two chains hit one slot in the
//     same round, so the order of the additions is fixed);
//   * the coupling of ALL bodies through the total momentum, -hb.(P x Pdot)/M, is what would make every
//     step non-zero; its Hessian is the rank-structured term -(1/M) hb.(dP_i x dPdot_j + dP_j x dPdot_i),
//     written into the stage beforehand (cross_terms), and the sweep runs with d xc = d xdot_c = 0.
struct DirData {
  D3 alpha, pi, wpi, vpi;
};
__device__ __forceinline__ D3 shfl3(const D3& v, int src) {
  return v3<double>(__shfl_sync(0xffffffffu, v.x, src), __shfl_sync(0xffffffffu, v.y, src),
                    __shfl_sync(0xffffffffu, v.z, src));
}

__device__ __forceinline__ void kin_tangent_sweep_packed(const KinTopo& T, const double* sb, const double* zs,
                                                         const double* massv, const SeedsT& ownS, D3 hb, double* pslot,
                                                         double* stage) {
  const int lane = threadIdx.x & 31;
  const D3 zero = v3<double>(0.0, 0.0, 0.0);
  for (int i = lane; i < T.n_pslots * 12; i += 32) pslot[i] = 0.0;
  __syncwarp();
  D3 cn = zero, cF = zero, cw = zero, cv = zero;
  unsigned t_next = (unsigned)T.sched[lane];
  for (int r = 0; r < T.n_rounds; ++r) {
    const unsigned t = t_next;
    if (r + 1 < T.n_rounds) t_next = (unsigned)T.sched[(r + 1) * 32 + lane];
    const bool valid = (t & KT_VALID) != 0;
    const int l = (t >> KT_L_SHIFT) & 31, p = (t >> KT_P_SHIFT) & 31, d = (t >> KT_D_SHIFT) & 31;
    const int src = valid ? d : lane;
    const bool heavy = (T.round_heavy_mask >> r) & 1u;  // warp-uniform (constant bank): typed rounds, sweep_schedule.h
    SeedsT S;
    S.footF[0] = S.footF[1] = S.footN[0] = S.footN[1] = S.chestN = zero;
    if ((T.round_seed_mask >> r) & 1u) {  // warp-uniform
      S.footF[0] = shfl3(ownS.footF[0], src);
      S.footF[1] = shfl3(ownS.footF[1], src);
      S.footN[0] = shfl3(ownS.footN[0], src);
      S.footN[1] = shfl3(ownS.footN[1], src);
      S.chestN = shfl3(ownS.chestN, src);
    }
    if (valid) {
      if (t & KT_START) cn = cF = cw = cv = zero;
      const double* bl = sb + l * SB_STRIDE;
      const D3 ax = ld3(bl + SB_AX);
      D3 tax = zero, trho = zero, twpar = zero;
      const D3 rho = ld3(bl + SB_RHO), wpar = ld3(sb + p * SB_STRIDE + SB_W);
      if (heavy) {
        // direction data: the axis / origin / twist of the joint's body, already in shared memory.  The schedule
        // holds joint directions only (SweepTopo::n_base = 0): the quaternion columns are closed-form
        DirData dir;
        {
          const double* bd = sb + (d - 3) * SB_STRIDE;
          dir.wpi = ld3(bd + SB_W);
          dir.vpi = ld3(bd + SB_V);
          dir.alpha = ld3(bd + SB_AX);
          dir.pi = ld3(bd + SB_O);
        }
        const double m = massv[l];
        // with typed rounds every task of a heavy round lies in the sub-tree of its direction (KT_IN_L set); the
        // untyped fallback schedule mixes both kinds, hence the select
        const bool in = (t & KT_IN_L) != 0;
        const D3 a = in ? dir.alpha : zero;
        const D3 d_ = ld3(bl + SB_D), w = ld3(bl + SB_W);
        const D3 rr = ld3(bl + SB_O) - dir.pi;
        const D3 to = cross(a, rr);
        const D3 td = cross(a, d_);
        const D3 tw = cross(a, w - dir.wpi);
        const D3 tv = cadd(cross(dir.wpi, to), a, (ld3(bl + SB_V) - dir.vpi) - cross(dir.wpi, rr));
        tax = cross(a, ax);
        if (in) {  // local adjoints of body l move with the sub-tree of the direction
          const double* I = bl + SB_I;
          const D3 cbar = ld3(bl + SB_CB), cdbar = ld3(bl + SB_CDB), Ih = ld3(bl + SB_IH), Iw = ld3(bl + SB_L);
          const D3 tc = to + td;
          const D3 tcd = cadd(cadd(tv, tw, d_), w, td);
          const D3 tcbar = scale(m, cross(tcd, hb));
          const D3 tcdbar = scale(m, cross(hb, tc));
          const D3 tIw = cadd(symmul(I, tw - cross(a, w)), a, Iw);
          const D3 tIh = csub(cross(a, Ih), I, cross(a, hb));
          cF = cF + tcbar;
          // two accumulators keep the dependent chains short
          D3 n1 = cadd(cadd(cadd(cn, td, cbar), d_, tcbar), td, cross(cdbar, w));
          D3 n2 = cadd(cadd(cadd(cross(d_, cadd(cross(tcdbar, w), cdbar, tw)), tIw, hb), tIh, w), Ih, tw);
          cn = n1 + n2;
          cv = cv + tcdbar;
          cw = cadd(cadd(cw, td, cdbar), d_, tcdbar) + tIh;
        }
        if (t & KT_IN_P) {  // the parent moves with the direction as well
          trho = cross(dir.alpha, rho);
          twpar = cross(dir.alpha, wpar - dir.wpi);
        }
      }
      // seed tangents (zero where they do not apply).  The feet-distance row couples the two feet: a
      // direction that moves one foot also changes the seed on the OTHER foot, which is why the schedule
      // visits the other leg for such a direction
      if (l == T.foot_body[0]) {
        cF = cF + S.footF[0];
        cn = cn + S.footN[0];
      }
      if (l == T.foot_body[1]) {
        cF = cF + S.footF[1];
        cn = cn + S.footN[1];
      }
      if (l == T.chest_body) cn = cn + S.chestN;
      const int ls = (t >> KT_LOAD_SHIFT) & 63;
      if (ls) {
        const double* sl = pslot + (ls - 1) * 12;
        cn = cn + ld3(sl);
        cF = cF + ld3(sl + 3);
        cw = cw + ld3(sl + 6);
        cv = cv + ld3(sl + 9);
      }
      if (l != 0) {
        double* col = stage + d * 57;
        const double sd = zs[Z_SD + l - 1];
        if (heavy) {
          const D3 np = ld3(bl + SB_ACC), Fp = ld3(bl + SB_ACC + 3), wp = ld3(bl + SB_ACC + 6), vp = ld3(bl + SB_ACC + 9);
          col[7 + l - 1] += dot(tax, wp) + dot(ax, cw);   // rows: vb3 qd4 sd23 q4 s23
          col[34 + l - 1] += dot(tax, np) + dot(ax, cn);
          D3 n1 = cadd(cadd(cn, trho, Fp), rho, cF);
          D3 n2 = cadd(scale(sd, cadd(cross(tax, wp), ax, cw)), trho, cross(vp, wpar));
          cn = cadd(n1 + n2, rho, cadd(cross(cv, wpar), vp, twpar));
          cw = cadd(cadd(cw, trho, vp), rho, cv);
        } else {
          // propagation through an ancestor of the joint: every state tangent is zero, the adjoint tangent moves
          // towards the root with the primal coefficients only
          col[7 + l - 1] += dot(ax, cw);
          col[34 + l - 1] += dot(ax, cn);
          cn = cadd(cadd(cn, rho, cF) + scale(sd, cross(ax, cw)), rho, cross(cv, wpar));
          cw = cadd(cw, rho, cv);
        }
      }
      const int fs = (t >> KT_FLUSH_SHIFT) & 63;
      if (fs) {
        double* sl = pslot + (fs - 1) * 12;
        if (t & KT_STORE) {
          st3(sl, cn);
          st3(sl + 3, cF);
          st3(sl + 6, cw);
          st3(sl + 9, cv);
        } else {
          st3(sl, ld3(sl) + cn);
          st3(sl + 3, ld3(sl + 3) + cF);
          st3(sl + 6, ld3(sl + 6) + cw);
          st3(sl + 9, ld3(sl + 9) + cv);
        }
      }
    }
    __syncwarp();
  }
}

// quaternion maps of component a: g_a (rotation tangent of R(q/|q|) along q_a), u_a = d omega_0 / d q_a,
// w_a = d omega_0 / d q_dot_a.
template <class T>
__device__ __forceinline__ void quat_map(const T* q, const double* qd, int a, V3<T>& g, V3<T>& u, V3<T>& w) {
  const T r2 = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  const T r = dsqrt(r2);
  const T ir = 1.0 / r;
  T qh[4], t[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) qh[i] = q[i] * ir;
  T qha = qh[0];  // qh[a] by selects: a may be lane-dependent, and an indexed qh[a] would go to local memory
#pragma unroll
  for (int i = 1; i < 4; ++i)
    if (i == a) qha = qh[i];
#pragma unroll
  for (int i = 0; i < 4; ++i) t[i] = ((i == a ? 1.0 : 0.0) - qh[i] * qha) * ir;
  g = omega_map(qh, t);
  u = omega_map(t, qd);
  double e[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
  for (int i = 0; i < 4; ++i) e[i] = i == a ? 1.0 : 0.0;
  w = omega_map(qh, e);
}
__device__ __forceinline__ void quat_maps(const double* q, const double* qd, D3* g, D3* u, D3* w) {
#pragma unroll
  for (int a = 0; a < 4; ++a) quat_map(q, qd, a, g[a], u[a], w[a]);
}

struct HessEmit {
  const int* map;  // hk_map row of this knot
  double* hess;    // instance base
  int dirj;        // direction index 0..26, or -1 (idle lane)
  double add_sd, add_s;  // joint-regularisation terms on (sd_j, s_j), (s_j, s_j) for joint lanes
  double* stage;   // per-warp staging (HSTAGE doubles); scattered after the sweep
  bool acc = false;  // the stage already holds the cross terms, entries are added
  // stage is never null.  The direct-store branch and the `if (em.stage)` guard of the scatter stay because
  // without them ptxas allocates the kernel differently and spills 12 bytes per thread.
  __device__ __forceinline__ void put(int row, double v) const {
    if (stage) {
      if (acc) stage[dirj * 57 + row] += v;
      else stage[dirj * 57 + row] = v;
      return;
    }
    const int slot = map[dirj * 57 + row];
    if (slot >= 0) hess[slot] = v;
  }
};

// Launch bounds, measured on B200 (tools/time_kino.py): the Hessian kernel is fastest with the full 255 registers
// (2 CTAs/SM; 168 registers spill 1 KB/thread and lose 12%), the lean kernel with 168 registers (3 CTAs/SM, -19%).
constexpr int KIN_H_THREADS = 128, KIN_H_MIN_BLOCKS = 2;
template <bool WITH_HESS>
__global__ void __launch_bounds__(WITH_HESS ? KIN_H_THREADS : 128, WITH_HESS ? KIN_H_MIN_BLOCKS : 3) kino_kin_kernel(
    const __grid_constant__ KinTopo T,
                                                       const KinoConst* __restrict__ Cp, unsigned mask,
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
  const long wid = (long)blockIdx.x * (blockDim.x >> 5) + warp;
  const int N = T.N;
  if (wid >= batch * N) return;
  const long b = wid / N;
  const int k = (int)(wid % N);
  const KinSmem L = kin_smem_layout(T.nb, T.n_slots, WITH_HESS);
  double* sm = smem + (size_t)warp * L.total;
  double* sb = sm + L.bodies;
  double* zs = sm + L.z;
  double* gbuf = sm + L.gbuf;
  double* lamk = sm + L.lamk;
  const double* xb = x + b * T.n_x + (long)k * T.x_stride;
  const double* pb_ = p + b * p_stride;
  const int nb = T.nb;
  const bool k1 = k >= T.cost_k0;  // knots on which the "apply_to_first_elements=False" expressions exist
  HB_PHASE_INIT

  // ---- every global input of this warp is requested here, addresses from the constant bank: the DRAM
  // latencies of x, the parameter slices, the multipliers and the joint frames overlap each other and
  // the forward kinematics instead of being exposed one by one at their points of use
  // (loads first, shared-memory stores last: a store that waits for its load would hold back, in program
  // order, every load behind it)
  // of the 189 variables of the knot this kernel reads the 24 contact-point positions (FK rows) and the robot block
  // [Z_VB, NZ): 93 doubles in 4 coalesced requests (the contact kernel owns the rest of the point variables)
  double xr[4];
  int xi[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    xi[u] = u == 0 ? (lane < 24 ? 15 * (lane / 3) + Z_P + lane % 3 : -1) : Z_VB + lane + 32 * (u - 1);
    if (xi[u] >= NZ) xi[u] = -1;
    xr[u] = 0.0;
    if (xi[u] >= 0) {
      if (T.zmap_identity) xr[u] = xb[xi[u]];
      else {
        const int zi = C.zmap[xi[u]];
        if (zi >= 0) xr[u] = xb[zi];
      }
    }
  }
  const double* rfq = pb_ + T.po_fq + T.ref_stride * k;
  const double* rbq = pb_ + T.po_bq + T.ref_stride * k;
  const double* rbqv = pb_ + T.po_bqv + T.ref_stride * k;
  const double* rjr = pb_ + T.po_jr + T.ref_stride * k;
  const D3 pre_desc = lane < 8 ? ld3(pb_ + T.po_desc0 + 24 * k + 3 * lane) : v3<double>(0.0, 0.0, 0.0);
  double pre_fq[4] = {0.0, 0.0, 0.0, 1.0};
  if (lane == 8) {
#pragma unroll
    for (int i = 0; i < 4; ++i) pre_fq[i] = rfq[i];
  }
  const double pre_bq[4] = {rbq[0], rbq[1], rbq[2], rbq[3]};
  const double pre_bqv = lane < 4 ? rbqv[lane] : 0.0;
  const double pre_jr = lane < HB_N_JOINTS ? rjr[lane] : 0.0;
  const double mass_p = pb_[T.po_mass];
  const bool with_l = WITH_HESS && (mask & HB_EVAL_HESS_L);
  double sg = 0.0, lam_reg = 0.0;
  if (with_l) {
    // multipliers of the 32 kinematic rows of this knot, one per lane, parked in shared memory
    int row;
    if (lane < 24) row = grow(C, (lane / 3) * HB_KF_PT_COUNT + HB_KF_PT_FK, k, lane % 3);
    else if (lane < 27) row = grow(T, HB_KF_COM_KIN, k, lane - 24);
    else if (lane < 30) row = grow(T, HB_KF_MOM_KIN, k, lane - 27);
    else row = grow(T, lane == 30 ? HB_KF_FEET_DIST : HB_KF_UNIT_QUAT, k, 0);
    lam_reg = row >= 0 ? lam[b * T.m + row] : 0.0;
    sg = sigma[b];
  }
  // joint frame constants of this lane's body
  const bool is_link = lane > 0 && lane < nb;
  const int my_depth = is_link ? C.body[lane].depth : -1;
  const int my_parent = is_link ? C.body[lane].parent : 0;
  const int my_rank = is_link ? C.body[lane].sib_rank : -1;
  const double my_mass = lane < nb ? C.body[lane].mass : 0.0;
  D3 b_com = v3<double>(0.0, 0.0, 0.0);
  double b_I[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  if (lane < nb) {
    b_com = ld3(C.body[lane].com);
#pragma unroll
    for (int i = 0; i < 6; ++i) b_I[i] = C.body[lane].inertia[i];
  }
  double bE[9], bEA[9], bEA2[9];
  D3 b_r = v3<double>(0.0, 0.0, 0.0), b_axis = b_r;
  if (is_link) {
    const BodyC& bc = C.body[lane];
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      bE[i] = bc.E[i];
      bEA[i] = bc.EA[i];
      bEA2[i] = bc.EA2[i];
    }
    b_r = ld3(bc.r);
    b_axis = ld3(bc.axis);
  }
  const unsigned my_submask = lane < nb ? C.sub_mask[lane] : 0u;
#pragma unroll
  for (int u = 0; u < 4; ++u)
    if (xi[u] >= 0) zs[xi[u]] = xr[u];
  if (WITH_HESS) lamk[lane] = lam_reg;
  for (int i = lane; i < 58; i += 32) gbuf[i] = 0.0;
  __syncwarp();
  HB_PHASE(0, 0);  // inputs loaded and staged

  // ------------------------------------------------------------------ base
  const double q0 = zs[Z_Q], q1 = zs[Z_Q + 1], q2 = zs[Z_Q + 2], q3 = zs[Z_Q + 3];
  const double qq = q0 * q0 + q1 * q1 + q2 * q2 + q3 * q3;
  const double qn = sqrt(qq);
  const double qh[4] = {q0 / qn, q1 / qn, q2 / qn, q3 / qn};
  const double qdv[4] = {zs[Z_QD], zs[Z_QD + 1], zs[Z_QD + 2], zs[Z_QD + 3]};
  if (lane == 0) {
    // R = I + 2 w [v]x + 2 [v]x^2 (liecasadi SO3.from_quat().as_matrix() [ext])
    const double vx = qh[0], vy = qh[1], vz = qh[2], w = qh[3];
    double* R = sb + SB_R;
    R[0] = 1.0 - 2.0 * (vy * vy + vz * vz);
    R[1] = 2.0 * (vx * vy - w * vz);
    R[2] = 2.0 * (vx * vz + w * vy);
    R[3] = 2.0 * (vx * vy + w * vz);
    R[4] = 1.0 - 2.0 * (vx * vx + vz * vz);
    R[5] = 2.0 * (vy * vz - w * vx);
    R[6] = 2.0 * (vx * vz - w * vy);
    R[7] = 2.0 * (vy * vz + w * vx);
    R[8] = 1.0 - 2.0 * (vx * vx + vy * vy);
    st3(sb + SB_O, v3<double>(0.0, 0.0, 0.0));  // positions are relative to the base origin
    st3(sb + SB_W, omega_map(qh, qdv));
    st3(sb + SB_V, ld3(zs + Z_VB));
    st3(sb + SB_AX, v3<double>(0.0, 0.0, 0.0));
  }
  __syncwarp();
  // ------------------------------------------------------------------ forward kinematics by depth
  // the joint rotations do not depend on the parents: computed by all link lanes at once
  double Rl[9];
  double my_sd = 0.0;
  if (is_link) {
    const double s = zs[Z_S + lane - 1];
    my_sd = zs[Z_SD + lane - 1];
    double sn, cs;
    sincos(s, &sn, &cs);
    const double oc = 1.0 - cs;
#pragma unroll
    for (int i = 0; i < 9; ++i) Rl[i] = bE[i] + sn * bEA[i] + oc * bEA2[i];
  }
  for (int d = 1; d <= T.max_depth; ++d) {
    if (my_depth == d) {
      const double* bp = sb + my_parent * SB_STRIDE;
      double* bl = sb + lane * SB_STRIDE;
      const double sd = my_sd;
      const double* Rp = bp + SB_R;
      double R[9];
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) R[3 * i + j] = Rp[3 * i] * Rl[j] + Rp[3 * i + 1] * Rl[3 + j] + Rp[3 * i + 2] * Rl[6 + j];
#pragma unroll
      for (int i = 0; i < 9; ++i) bl[SB_R + i] = R[i];
      const D3 op = ld3(bp + SB_O), wp = ld3(bp + SB_W), vp = ld3(bp + SB_V);
      const D3 rho = matvec(Rp, b_r);
      const D3 ax = matvec(R, b_axis);
      st3(bl + SB_O, op + rho);
      st3(bl + SB_AX, ax);
      st3(bl + SB_W, wp + scale(sd, ax));
      st3(bl + SB_V, vp + cross(wp, rho));
      st3(bl + SB_RHO, rho);
    }
    __syncwarp();
  }
  HB_PHASE(0, 1);  // forward kinematics by depth
  // ------------------------------------------------------------------ per-body derived quantities + sums
  D3 mc = v3<double>(0.0, 0.0, 0.0), mcd = mc, hl = mc;
  if (lane < nb) {
    double* bl = sb + lane * SB_STRIDE;
    const double* R = bl + SB_R;
    const D3 d = matvec(R, b_com);
    st3(bl + SB_D, d);
    // I^w = R I R^T
    double RI[9];
    const double* I = b_I;
    const double Im[9] = {I[0], I[1], I[2], I[1], I[3], I[4], I[2], I[4], I[5]};
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) RI[3 * i + j] = R[3 * i] * Im[j] + R[3 * i + 1] * Im[3 + j] + R[3 * i + 2] * Im[6 + j];
    double Iw[6];
    const int ii[6] = {0, 0, 0, 1, 1, 2}, jj[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
    for (int e = 0; e < 6; ++e)
      Iw[e] = RI[3 * ii[e]] * R[3 * jj[e]] + RI[3 * ii[e] + 1] * R[3 * jj[e] + 1] + RI[3 * ii[e] + 2] * R[3 * jj[e] + 2];
#pragma unroll
    for (int e = 0; e < 6; ++e) bl[SB_I + e] = Iw[e];
    const D3 o = ld3(bl + SB_O), w = ld3(bl + SB_W), v = ld3(bl + SB_V);
    const D3 c = o + d;
    const D3 cd = v + cross(w, d);
    mc = scale(my_mass, c);
    mcd = scale(my_mass, cd);
    const D3 Lw = symmul(Iw, w);
    st3(bl + SB_L, Lw);
    hl = cross(mc, cd) + Lw;
  }
  const double M = T.total_mass;
  const D3 Pm = v3<double>(warp_sum(mc.x), warp_sum(mc.y), warp_sum(mc.z));
  const D3 Pd = v3<double>(warp_sum(mcd.x), warp_sum(mcd.y), warp_sum(mcd.z));
  D3 hang = v3<double>(warp_sum(hl.x), warp_sum(hl.y), warp_sum(hl.z));
  hang = hang - scale(1.0 / M, cross(Pm, Pd));
  const D3 xc = scale(1.0 / M, Pm), xcd = scale(1.0 / M, Pd);
  // ------------------------------------------------------------------ frames
  if (lane < 8) {
    const int f = lane >> 2;
    const double* Rf = C.foot_R[f];
    const D3 r = pre_desc;
    const D3 bf = matvec(Rf, r) + ld3(C.foot_t[f]);
    const D3 a = matvec(sb + T.foot_body[f] * SB_STRIDE + SB_R, bf);
    st3(sm + L.arms + 3 * lane, a);
  }
  if (lane == 8) {
    // G = R_chest_body * (R_c * R(qd)^T), qd = desired frame quaternion (not normalised, kinematics.py:447)
    const double vx = pre_fq[0], vy = pre_fq[1], vz = pre_fq[2], w = pre_fq[3];
    double Rd[9];
    Rd[0] = 1.0 - 2.0 * (vy * vy + vz * vz);
    Rd[1] = 2.0 * (vx * vy - w * vz);
    Rd[2] = 2.0 * (vx * vz + w * vy);
    Rd[3] = 2.0 * (vx * vy + w * vz);
    Rd[4] = 1.0 - 2.0 * (vx * vx + vz * vz);
    Rd[5] = 2.0 * (vy * vz - w * vx);
    Rd[6] = 2.0 * (vx * vz - w * vy);
    Rd[7] = 2.0 * (vy * vz + w * vx);
    Rd[8] = 1.0 - 2.0 * (vx * vx + vy * vy);
    double Kc[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        Kc[3 * i + j] = C.chest_R[3 * i] * Rd[3 * j] + C.chest_R[3 * i + 1] * Rd[3 * j + 1] + C.chest_R[3 * i + 2] * Rd[3 * j + 2];
    const double* Rb = sb + T.chest_body * SB_STRIDE + SB_R;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) sm[L.G + 3 * i + j] = Rb[3 * i] * Kc[j] + Rb[3 * i + 1] * Kc[3 + j] + Rb[3 * i + 2] * Kc[6 + j];
  }
  if (lane == 9) {
    const double* RR = sb + T.foot_body[1] * SB_STRIDE + SB_R;
    const double* RL = sb + T.foot_body[0] * SB_STRIDE + SB_R;
    const double* Rf = C.foot_R[1];
    st3(sm + L.fdu, matvec(RR, v3<double>(Rf[1], Rf[4], Rf[7])));  // y axis of the reference sole frame
    st3(sm + L.fdal, matvec(RL, ld3(C.foot_t[0])));
    st3(sm + L.fdar, matvec(RR, ld3(C.foot_t[1])));
  }
  __syncwarp();
  const double* G = sm + L.G;
  const double phi = G[0] + G[4] + G[8];
  const D3 mG = v3<double>(G[5] - G[7], G[6] - G[2], G[1] - G[3]);
  const D3 fdu = ld3(sm + L.fdu), fdal = ld3(sm + L.fdal), fdar = ld3(sm + L.fdar);
  const D3 oL = ld3(sb + T.foot_body[0] * SB_STRIDE + SB_O), oR = ld3(sb + T.foot_body[1] * SB_STRIDE + SB_O);
  const D3 fdDelta = (oL + fdal) - (oR + fdar);
  const double feet_y = dot(fdu, fdDelta);

  HB_PHASE(0, 2);  // per-body quantities, sums, frames
  // ------------------------------------------------------------------ values: g rows, costs, grad_f (simple terms)
  const bool want_g = (mask & HB_EVAL_G) != 0;
  double* gb = g + b * T.m;
  if (want_g) {
    if (lane < 8 && k1) {
      const int f = lane >> 2;
      const D3 a = ld3(sm + L.arms + 3 * lane);
      const D3 o = ld3(sb + T.foot_body[f] * SB_STRIDE + SB_O);
      const int r0 = grow(C, lane * HB_KF_PT_COUNT + HB_KF_PT_FK, k, 0);  // lane-indexed family: global table
      const double* pp = zs + 15 * lane + Z_P;
      if (r0 >= 0) {
        gb[r0] = pp[0] - (zs[Z_PB] + o.x + a.x);
        gb[r0 + 1] = pp[1] - (zs[Z_PB + 1] + o.y + a.y);
        gb[r0 + 2] = pp[2] - (zs[Z_PB + 2] + o.z + a.z);
      }
    }
    if (lane == 8) {
      int r0 = grow(T, HB_KF_UNIT_QUAT, k, 0);
      if (r0 >= 0) gb[r0] = qq;
      r0 = grow(T, HB_KF_COM_KIN, k, 0);
      if (r0 >= 0) {
        gb[r0] = zs[Z_COM] - (zs[Z_PB] + xc.x);
        gb[r0 + 1] = zs[Z_COM + 1] - (zs[Z_PB + 1] + xc.y);
        gb[r0 + 2] = zs[Z_COM + 2] - (zs[Z_PB + 2] + xc.z);
      }
      r0 = grow(T, HB_KF_MOM_KIN, k, 0);
      if (r0 >= 0) {
        gb[r0] = zs[Z_H + 3] - hang.x / mass_p;
        gb[r0 + 1] = zs[Z_H + 4] - hang.y / mass_p;
        gb[r0 + 2] = zs[Z_H + 5] - hang.z / mass_p;
      }
      r0 = grow(T, HB_KF_FEET_DIST, k, 0);
      if (r0 >= 0) gb[r0] = feet_y;
    }
  }
  // base-quaternion error e = qd^-1 (x) q - (0,0,0,1) = A q - e4 (quaternion.py:64-70); columns of A
  double Aq[4][4];
  {
    const double dx = -pre_bq[0], dy = -pre_bq[1], dz = -pre_bq[2], dw = pre_bq[3];
    // (dw, dv) (x) (bw, bv): v = dw bv + bw dv + dv x bv ; w = dw bw - dv.bv ; column a: b = e_a
    // b = e_x
    Aq[0][0] = dw; Aq[1][0] = dz; Aq[2][0] = -dy; Aq[3][0] = -dx;
    Aq[0][1] = -dz; Aq[1][1] = dw; Aq[2][1] = dx; Aq[3][1] = -dy;
    Aq[0][2] = dy; Aq[1][2] = -dx; Aq[2][2] = dw; Aq[3][2] = -dz;
    Aq[0][3] = dx; Aq[1][3] = dy; Aq[2][3] = dz; Aq[3][3] = dw;
  }
  double eq[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) eq[i] = Aq[i][0] * q0 + Aq[i][1] * q1 + Aq[i][2] * q2 + Aq[i][3] * q3 - (i == 3 ? 1.0 : 0.0);
  const double frame_cost = (phi - 3.0) * (phi - 3.0);
  const bool want_terms = (mask & HB_EVAL_COST_TERMS_BIT) != 0;
  if (mask & (HB_EVAL_F | HB_EVAL_GRAD_F | HB_EVAL_COST_TERMS_BIT)) {
    // quaternion-velocity cost (all knots) and, for k >= 1, base quaternion / joint / frame costs
    double c_bqv = 0.0, c_bq = 0.0, c_joint = 0.0, c_frame = 0.0;
    if (lane < 4) {
      const double e = qdv[lane] - pre_bqv;
      c_bqv = T.w_bqv * e * e;
      gbuf[3 + lane] += 2.0 * T.w_bqv * e;
      if (k1) {
        c_bq = T.w_bq * eq[lane] * eq[lane];
        double gq = 0.0;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          double t = 0.0;
#pragma unroll
          for (int i = 0; i < 4; ++i) t += Aq[i][a] * eq[i];
          if (a == lane) gq = t;
        }
        gbuf[7 + lane] += 2.0 * T.w_bq * gq;
      }
    }
    if (lane < HB_N_JOINTS && k1) {
      const double sd = zs[Z_SD + lane], e = zs[Z_S + lane] - pre_jr;
      if (T.joint_cost_kind == 0) {
        // kinodynamic planner.py:506-520: sumsqr of the broadcast n x n matrix (SURVEY.md A.11)
        const double t = sd + C.wj[lane] * e;
        c_joint = T.w_joint * ((HB_N_JOINTS - 1) * sd * sd + t * t);
        gbuf[11 + lane] += T.w_joint * (2.0 * (HB_N_JOINTS - 1) * sd + 2.0 * t);
        gbuf[34 + lane] += T.w_joint * 2.0 * C.wj[lane] * t;
      } else {
        // pose finder planner.py:584-588: e^T diag(w) e
        c_joint = T.w_joint * (e * C.wj[lane]) * e;
        gbuf[34 + lane] += T.w_joint * 2.0 * C.wj[lane] * e;
      }
    }
    if (lane == 31 && k1) c_frame = T.w_frame * frame_cost;
    if (want_terms) {
      // solution report (hb_eval_cost_terms): one value per named cost expression of this knot
      double* ct = fpart + (b * N + k) * HB_COST_TERMS;
      const double t_frame = warp_sum(c_frame), t_bq = warp_sum(c_bq), t_bqv = warp_sum(c_bqv), t_j = warp_sum(c_joint);
      if (lane == 0) {
        ct[HB_CT_FRAME_QUAT] = t_frame;
        ct[HB_CT_BASE_QUAT] = t_bq;
        ct[HB_CT_BASE_QUAT_VEL] = t_bqv;
        ct[HB_CT_JOINTS] = t_j;
      }
    } else {
      double cost = (c_bqv + c_bq) + c_joint + c_frame;
      cost = warp_sum(cost);
      if (lane == 0 && (mask & HB_EVAL_F)) fpart[(b * N + k) * 2 + 1] = cost;
    }
  }
  __syncwarp();

  HB_PHASE(0, 3);  // g rows, costs
  const bool want_jac = (mask & HB_EVAL_JAC_G) != 0, want_grad = (mask & HB_EVAL_GRAD_F) != 0;
  double* slot = sm + L.slot;
  // ------------------------------------------------------------------ adjoint sweep, fp64: Jacobian rows
  // (Jacobian-only kernel.  The Hessian kernel gets the same values from forward tangents that its
  // direction lanes need anyway -- see "forward-mode Jacobian" below.)
  if ((want_jac || want_grad) && !WITH_HESS) {
    Seeds<double> S;
    S.wc = S.hb = S.footF[0] = S.footF[1] = S.footN[0] = S.footN[1] = S.chestN = v3<double>(0.0, 0.0, 0.0);
    if (lane < 24) {
      const int pt = lane / 3, a = lane % 3;
      const D3 frc = v3<double>(a == 0 ? -1.0 : 0.0, a == 1 ? -1.0 : 0.0, a == 2 ? -1.0 : 0.0);
      const D3 trq = cross(ld3(sm + L.arms + 3 * pt), frc);
      if (pt < 4) {
        S.footF[0] = frc;
        S.footN[0] = trq;
      } else {
        S.footF[1] = frc;
        S.footN[1] = trq;
      }
    } else if (lane < 27) {
      const int a = lane - 24;
      S.wc = v3<double>(a == 0 ? -1.0 / M : 0.0, a == 1 ? -1.0 / M : 0.0, a == 2 ? -1.0 / M : 0.0);
    } else if (lane < 30) {
      const int a = lane - 27;
      const double sc = -1.0 / mass_p;
      S.hb = v3<double>(a == 0 ? sc : 0.0, a == 1 ? sc : 0.0, a == 2 ? sc : 0.0);
    } else if (lane == 30) {
      S.footF[0] = fdu;
      S.footN[0] = cross(fdal, fdu);
      S.footF[1] = -fdu;
      S.footN[1] = cross(fdu, fdDelta) - cross(fdar, fdu);
    } else {
      S.chestN = mG;
    }
    JacEmit em;
    const int2 jkm = *reinterpret_cast<const int2*>(&T.knot_maps[k].jk_base);  // {base, table offset}
    em.map = C.jk_map + jkm.y;
    em.jac = jac + b * T.nnz_j + jkm.x;
    em.gbuf = gbuf;
    em.lane = lane;
    em.gscale = k1 ? 2.0 * T.w_frame * (phi - 3.0) : 0.0;
    em.write = want_jac;
    em.init_bases();
    D3 n0, w0, v0;
    kin_backward(T, sb, zs, S, xc, xcd, slot, em, n0, w0, v0);
    // base chain rule
    D3 gq[4], uq[4], wq[4];
    const double qraw[4] = {q0, q1, q2, q3};
    quat_maps(qraw, qdv, gq, uq, wq);
    double dq[4], dqd[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      dq[a] = dot(n0, gq[a]) + dot(w0, uq[a]);
      dqd[a] = dot(w0, wq[a]);
    }
    if (lane == 31) {
#pragma unroll
      for (int a = 0; a < 4; ++a) gbuf[7 + a] += em.gscale * dq[a];
    } else if (want_jac) {
      if (lane < 27) {
        const int bq = em.base_q();
#pragma unroll
        for (int a = 0; a < 4; ++a) em.put(bq + a, dq[a]);
      } else if (lane < 30) {
        const int bm = 4 + 648 + 81 + (lane - 27) * 57;
        em.put(bm + 0, v0.x);
        em.put(bm + 1, v0.y);
        em.put(bm + 2, v0.z);
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          em.put(bm + 3 + a, dqd[a]);
          em.put(bm + 7 + a, dq[a]);
        }
      }
      if (lane < 4) em.put(lane, 2.0 * qraw[lane]);  // unit quaternion row
    }
    __syncwarp();
    if (want_grad) {
      // gbuf order vb3 qd4 q4 sd23 s23 -> x offsets
      double* gf = grad_f + b * T.n_x + (long)k * T.x_stride;
      for (int i = lane; i < 57; i += 32) {
        int off;
        if (i < 3) off = Z_VB + i;
        else if (i < 7) off = Z_QD + i - 3;
        else if (i < 11) off = Z_Q + i - 7;
        else if (i < 34) off = Z_SD + i - 11;
        else off = Z_S + i - 34;
        if (C.zmap[off] >= 0) gf[C.zmap[off]] = gbuf[i];
      }
      if (lane < 3 && C.zmap[Z_PB + lane] >= 0) gf[C.zmap[Z_PB + lane]] = 0.0;
    }
  }
  if (!WITH_HESS) return;
  if (!with_l && !(want_jac || want_grad)) return;
  // ------------------------------------------------------------------ adjoint sweep, dual: Hessian columns
  {
    const int dirj = lane < 27 ? lane : -1;
    Dir dir;
    dir.mask = 0u;
    dir.alpha = dir.pi = dir.wpi = dir.vpi = dir.u = v3<double>(0.0, 0.0, 0.0);
    // quaternion maps, once per warp: lane a < 4 builds g_a, u_a, w_a into the point block of z, which the
    // kinematics no longer reads (the g rows are done).  The root chain rule reads them there.
    double* qdat = zs;       // [4][6]: g_a, u_a
    double* qw = zs + 48;    // [4][3]: w_a  (zs + 24: the body masses of the sweep)
    double* qK = zs + 60;    // [4][4]: K[a][b], then [4][4]: Kd[a][b] (root chain rule)
    double* qt = zs + 92;    // [4][6]: tangents of the root totals n0, w0 along q_a (closed form, below)
    static_assert(92 + 24 <= Z_VB && HB_N_JOINTS + 1 <= 24, "quaternion tables overlap z or the masses");
    if (lane < 4) {
      D3 g, u, w;
      const double qraw[4] = {q0, q1, q2, q3};
      quat_map<double>(qraw, qdv, lane, g, u, w);
      st3(qdat + 6 * lane, g);
      st3(qdat + 6 * lane + 3, u);
      st3(qw + 3 * lane, w);
    }
    __syncwarp();
    D3 wq_lane = v3<double>(0.0, 0.0, 0.0);  // d omega_0 / d qd_a for the velocity-direction lanes 3..6
    if (lane >= 3 && lane < 7) wq_lane = ld3(qw + 3 * (lane - 3));
    if (lane < 4) {
      dir.alpha = ld3(qdat + 6 * lane);
      dir.u = ld3(qdat + 6 * lane + 3);
      dir.mask = 0xffffffffu;
      dir.wpi = ld3(sb + SB_W);
      dir.vpi = ld3(sb + SB_V);
    } else if (lane < 27) {
      const int l = lane - 4 + 1;
      dir.mask = C.sub_mask[l];
      const double* bl = sb + l * SB_STRIDE;
      dir.alpha = ld3(bl + SB_AX);
      dir.pi = ld3(bl + SB_O);
      dir.wpi = ld3(bl + SB_W);
      dir.vpi = ld3(bl + SB_V);
    }
    // ---- composite (sub-tree) moments, lane = body, accumulated leaf-to-root in the still unused stage:
    //   M, P = sum m c, Pd = sum m c_dot, H = sum (m c x c_dot + I w), J = sum (I + m (|c|^2 1 - c c^T))
    // A direction rotates one sub-tree rigidly about its pivot, so the tangents of the total P, P_dot
    // and angular momentum along it are closed-form in that sub-tree's moments (composite-rigid-body
    // argument): no lane loops over the bodies for them (that loop was 0.29 ms of 1.81 ms).
    enum { CM_M = 0, CM_P = 1, CM_PD = 4, CM_H = 7, CM_J = 10, CM_STRIDE = 17 };
    double* comp = sm + L.stage;
    if (lane < nb) {
      const double* bl = sb + lane * SB_STRIDE;
      const double m = my_mass;
      const D3 c = ld3(bl + SB_O) + ld3(bl + SB_D);
      const D3 cd = ld3(bl + SB_V) + cross(ld3(bl + SB_W), ld3(bl + SB_D));
      const double* I = bl + SB_I;
      double* cm = comp + lane * CM_STRIDE;
      cm[CM_M] = m;
      st3(cm + CM_P, scale(m, c));
      st3(cm + CM_PD, scale(m, cd));
      st3(cm + CM_H, cross(scale(m, c), cd) + ld3(bl + SB_L));
      cm[CM_J + 0] = I[0] + m * (c.y * c.y + c.z * c.z);
      cm[CM_J + 1] = I[1] - m * c.x * c.y;
      cm[CM_J + 2] = I[2] - m * c.x * c.z;
      cm[CM_J + 3] = I[3] + m * (c.x * c.x + c.z * c.z);
      cm[CM_J + 4] = I[4] - m * c.y * c.z;
      cm[CM_J + 5] = I[5] + m * (c.x * c.x + c.y * c.y);
    }
    __syncwarp();
    {
      // sub-tree sums D[body][i] = sum_l S[body][l] CM[l][i] with the 0/1 mask S[body][l] = (sub_mask[body] >> l) & 1,
      // on the fp64 tensor cores: 24 bodies x 16 components x 24 bodies is exactly 3 x 2 row/column tiles of
      // 6 m8n8k4 steps, no padding.  (The FMA version broadcast-loaded all 384 moments on every lane; the
      // leaf-to-root read-modify-write version before it took 12 % of the kernel.)
      constexpr int NBODY = HB_N_JOINTS + 1;
      static_assert(NBODY % 8 == 0, "the composite-moment product tiles the bodies by 8");
      double acc[NBODY / 8][2][2];
#pragma unroll
      for (int mt = 0; mt < NBODY / 8; ++mt) {
        // fragment rows: body 8 mt + lane / 4 (a: mask row; c, d: output row)
        const unsigned rmask = __shfl_sync(0xffffffffu, my_submask, 8 * mt + (lane >> 2));
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
#pragma unroll
        for (int kt = 0; kt < NBODY / 4; ++kt) {
          const int l = 4 * kt + (lane & 3);
          const double a = ((rmask >> l) & 1u) ? 1.0 : 0.0;
#pragma unroll
          for (int nt = 0; nt < 2; ++nt)
            dmma_m8n8k4(acc[mt][nt][0], acc[mt][nt][1], a, comp[l * CM_STRIDE + 8 * nt + (lane >> 2)]);
        }
      }
      __syncwarp();  // every tile has read the moments before they are overwritten
#pragma unroll
      for (int mt = 0; mt < NBODY / 8; ++mt) {
        double* cm = comp + (8 * mt + (lane >> 2)) * CM_STRIDE + 2 * (lane & 3);
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          cm[8 * nt] = acc[mt][nt][0];
          cm[8 * nt + 1] = acc[mt][nt][1];
        }
      }
      __syncwarp();
    }
    HB_PHASE(0, 4);  // composite moments
    // tangents of P, P_dot, h (about the base origin) along this lane's (q, s) direction
    D3 tP, tPd, th;
    {
      const double* cm = comp + (lane >= 4 && lane < 27 ? lane - 3 : 0) * CM_STRIDE;
      const double Ms = cm[CM_M];
      const D3 P = ld3(cm + CM_P), Pds = ld3(cm + CM_PD), Hs = ld3(cm + CM_H);
      const D3 a = dir.alpha, beta = cross(dir.alpha, dir.wpi);
      const D3 Pr = P - scale(Ms, dir.pi);
      tP = cross(a, Pr);
      tPd = cross(a, Pds - scale(Ms, dir.vpi)) - cross(beta, Pr) + cross(dir.u, P);
      th = cross(a, Hs) - cross(cross(a, dir.pi), Pds) - cross(P, cross(a, dir.vpi)) - symmul(cm + CM_J, beta) +
           cross(P, cross(beta, dir.pi)) + symmul(cm + CM_J, dir.u);
    }
    // velocity directions (lanes 0..29 = vb, qd, sd): w_l += in_l A, v_l += in_l A x (o_l - pivot) + B;
    // momentum is linear in the velocities, so its column is again closed-form in the moments
    D3 vel_dh = v3<double>(0.0, 0.0, 0.0);
    D3 vel_pv = vel_dh;  // d Pdot / d (velocity variable of this lane), for the cross terms of the Hessian
    if (lane < 30) {
      D3 A = v3<double>(0.0, 0.0, 0.0), B = A, piv = A;
      int lv = 0;
      if (lane < 3) B = v3<double>(lane == 0 ? 1.0 : 0.0, lane == 1 ? 1.0 : 0.0, lane == 2 ? 1.0 : 0.0);
      else if (lane < 7) A = wq_lane;
      else {
        lv = lane - 6;
        A = ld3(sb + lv * SB_STRIDE + SB_AX);
        piv = ld3(sb + lv * SB_STRIDE + SB_O);
      }
      const double* cm = comp + lv * CM_STRIDE;
      const double Ms = cm[CM_M];
      const D3 P = ld3(cm + CM_P);
      const D3 pv = cross(A, P - scale(Ms, piv)) + scale(Ms, B);
      const D3 hv = symmul(cm + CM_J, A) - cross(P, cross(A, piv)) + cross(P, B);
      vel_dh = scale(-1.0 / mass_p, hv - scale(1.0 / M, cross(Pm, pv)));
      vel_pv = pv;
    }
    // ---- quaternion columns of the Hessian in closed form: the packed sweep walks the joint directions only.
    // q_a turns the whole tree about the base origin (alpha = g_a) and adds u_a to omega_0.  Every kinematic row is
    // either rotation invariant (feet distance) or a world-fixed multiplier mu dotted with a vector X that turns with
    // the tree (contact points, CoM, angular momentum about the CoM), so the root totals are
    //   w0 = I_c hb,  n0 = sum_X X x mu - omega_0 x w0 + kappa m(G)      (I_c: locked inertia about the CoM)
    // and their tangents along q_a follow from root quantities (T = sum_X X mu^T over the points and the CoM):
    //   tw0 = alpha x w0 - I_c (alpha x hb)
    //   tn0 = (T - tr(T)) alpha + dhang x hb - u_a x w0 - omega_0 x tw0 + kappa' m(G) (alpha.m(G)) + kappa (G - phi) alpha
    // (dhang: tangent of the angular momentum about the CoM, kappa' = 2 sigma w_frame).  Parked in z for the root
    // chain rule, which turns them into rows vb, qd, q of the q columns; tests/test_quat_hessian_closed_form_cpu.py
    // checks these forms against the oracle's Hessian.
    if (with_l) {
      double* Tm = qK;  // [3][3], dead before the curvature tables are built
      if (lane < 9) {
        const int i = lane / 3, j = lane % 3;
        double t = -(i == 0 ? xc.x : (i == 1 ? xc.y : xc.z)) * lamk[24 + j];
#pragma unroll
        for (int pt = 0; pt < 8; ++pt)
          t -= (sb[T.foot_body[pt >> 2] * SB_STRIDE + SB_O + i] + sm[L.arms + 3 * pt + i]) * lamk[3 * pt + j];
        Tm[lane] = t;
      }
      __syncwarp();
      if (lane < 4) {
        const D3 a = dir.alpha, om = ld3(sb + SB_W), hbv = scale(-1.0 / mass_p, ld3(lamk + 27));
        const double* J0 = comp + CM_J;  // composite moments of the root: the whole tree
        const D3 ah = cross(a, hbv);
        const D3 w0 = symmul(J0, hbv) - scale(1.0 / M, cross(Pm, cross(hbv, Pm)));  // I_c x = J0 x - P x (x x P) / M
        const D3 tw0 = cross(a, w0) - (symmul(J0, ah) - scale(1.0 / M, cross(Pm, cross(ah, Pm))));
        const D3 dhang = th - scale(1.0 / M, cross(tP, Pd) + cross(Pm, tPd));
        const double trT = Tm[0] + Tm[4] + Tm[8];
        const double cf = k1 ? 2.0 * sg * T.w_frame : 0.0, kap = cf * (phi - 3.0);
        D3 tn0 = v3<double>(Tm[0] * a.x + Tm[1] * a.y + Tm[2] * a.z, Tm[3] * a.x + Tm[4] * a.y + Tm[5] * a.z,
                            Tm[6] * a.x + Tm[7] * a.y + Tm[8] * a.z) - scale(trT, a);
        tn0 = tn0 + cross(dhang, hbv) - cross(dir.u, w0) - cross(om, tw0);
        tn0 = tn0 + scale(cf * dot(a, mG), mG) + scale(kap, matvec(G, a) - scale(phi, a));
        st3(qt + 6 * lane, tn0);
        st3(qt + 6 * lane + 3, tw0);
      }
    }
    __syncwarp();  // the stage is reused for the Jacobian columns below
    const double inL = ((dir.mask >> T.foot_body[0]) & 1u) ? 1.0 : 0.0;
    const double inR = ((dir.mask >> T.foot_body[1]) & 1u) ? 1.0 : 0.0;
    const double inC = ((dir.mask >> T.chest_body) & 1u) ? 1.0 : 0.0;
    // tangents of the feet distance u.(pL - pR) and of trace(G) along this direction
    double ty_lane, tphi_lane;
    {
      const D3 a = dir.alpha;
      const D3 tL = scale(inL, cross(a, (ld3(sb + T.foot_body[0] * SB_STRIDE + SB_O) - dir.pi) + fdal));
      const D3 tR = scale(inR, cross(a, (ld3(sb + T.foot_body[1] * SB_STRIDE + SB_O) - dir.pi) + fdar));
      ty_lane = dot(scale(inR, cross(a, fdu)), fdDelta) + dot(fdu, tL - tR);
      const D3 ac = scale(inC, a);
      tphi_lane = cross(ac, v3<double>(G[0], G[3], G[6])).x + cross(ac, v3<double>(G[1], G[4], G[7])).y +
                  cross(ac, v3<double>(G[2], G[5], G[8])).z;
    }
    HB_PHASE(0, 5);  // direction tangents of P, Pdot, h, feet distance, trace
    // ---------------------------------------------------------------- forward-mode Jacobian
    // The direction lanes already hold the tangent of every link state along q_a / s_j, so column j of
    // the kinematic rows is a few products here; the velocity columns of the momentum rows (the map is
    // linear in the velocities) take one more pass over the bodies.  This replaces the row-per-lane
    // fp64 adjoint sweep of the Jacobian-only kernel (2.87 -> see DESIGN.md).
    if (want_jac || want_grad) {
      double* stg = sm + L.stage;
      const int bm = 4 + 648 + 81;  // momentum rows inside JK (kino_layout.py::_enumerate_jk)
      if (want_jac) {
        if (lane < 27) {
#pragma unroll
          for (int pt = 0; pt < 8; ++pt) {
            const int f = pt >> 2;
            const double in = f == 0 ? inL : inR;
            const D3 r = (ld3(sb + T.foot_body[f] * SB_STRIDE + SB_O) - dir.pi) + ld3(sm + L.arms + 3 * pt);
            const D3 t = scale(-in, cross(dir.alpha, r));
            stg[4 + (3 * pt) * 27 + lane] = t.x;
            stg[4 + (3 * pt + 1) * 27 + lane] = t.y;
            stg[4 + (3 * pt + 2) * 27 + lane] = t.z;
          }
          const D3 tc = scale(-1.0 / M, tP);
          stg[4 + 648 + lane] = tc.x;
          stg[4 + 648 + 27 + lane] = tc.y;
          stg[4 + 648 + 54 + lane] = tc.z;
          const D3 dh = scale(-1.0 / mass_p, th - scale(1.0 / M, cross(tP, Pd) + cross(Pm, tPd)));
          const int cq = lane < 4 ? 7 + lane : 34 + lane - 4;
          stg[bm + cq] = dh.x;
          stg[bm + 57 + cq] = dh.y;
          stg[bm + 114 + cq] = dh.z;
          if (lane < 4) stg[lane] = 2.0 * zs[Z_Q + lane];  // unit quaternion row
          else stg[bm + 171 + lane - 4] = ty_lane;          // feet distance row
        }
        if (lane < 30) {
          const int cv = lane < 7 ? lane : lane + 4;  // velocity columns: vb 0..2, qd 3..6, sd 11..33
          stg[bm + cv] = vel_dh.x;
          stg[bm + 57 + cv] = vel_dh.y;
          stg[bm + 114 + cv] = vel_dh.z;
        }
      }
      // frame-orientation cost: d/dz w (phi - 3)^2 = 2 w (phi - 3) dphi/dz
      if (want_grad && lane < 27 && k1)
        gbuf[lane < 4 ? 7 + lane : 34 + lane - 4] += 2.0 * T.w_frame * (phi - 3.0) * tphi_lane;
      HB_PHASE(0, 6);  // Jacobian columns staged
      __syncwarp();
      if (want_jac) {
        const int4 jkm = *reinterpret_cast<const int4*>(&T.knot_maps[k].jk_base);  // {base, offset, count, -}
        double* jb = jac + b * T.nnz_j + jkm.x;
        // destination-sorted list: entry << 16 | slot (measured 1.145 ms against 1.162 ms in entry order)
        const unsigned* lst = C.jk_list + jkm.y;
        const int n = jkm.z;
        // KIN_SCAT list loads in flight before the dependent stores: <= 927 entries in two trips
        for (int eb = lane; eb < n; eb += 32 * KIN_SCAT) {
          unsigned w[KIN_SCAT];
#pragma unroll
          for (int u = 0; u < KIN_SCAT; ++u) w[u] = (eb + 32 * u) < n ? lst[eb + 32 * u] : 0xffffffffu;
#pragma unroll
          for (int u = 0; u < KIN_SCAT; ++u)
            if (w[u] != 0xffffffffu) jb[w[u] & 0xffffu] = stg[w[u] >> 16];
        }
      }
      if (want_grad) {
        // gbuf order vb3 qd4 q4 sd23 s23 -> x offsets
        double* gf = grad_f + b * T.n_x + (long)k * T.x_stride;
        for (int i = lane; i < 57; i += 32) {
          int off;
          if (i < 3) off = Z_VB + i;
          else if (i < 7) off = Z_QD + i - 3;
          else if (i < 11) off = Z_Q + i - 7;
          else if (i < 34) off = Z_SD + i - 11;
          else off = Z_S + i - 34;
          if (C.zmap[off] >= 0) gf[C.zmap[off]] = gbuf[i];
        }
        if (lane < 3 && C.zmap[Z_PB + lane] >= 0) gf[C.zmap[Z_PB + lane]] = 0.0;
      }
      __syncwarp();  // the Hessian columns reuse the stage
    }
    HB_PHASE(0, 7);  // Jacobian scatter, grad_f
    if (!with_l) return;  // Jacobian / gradient only: done
    Seeds<Dual> S;
    S.footF[0] = S.footF[1] = S.footN[0] = S.footN[1] = vzero<Dual>();
    {
      // multipliers from lamk (loaded at the top of the kernel; rows that do not exist hold 0)
      S.wc = scale(-1.0 / M, ld3(lamk + 24));
      S.hb = scale(-1.0 / mass_p, ld3(lamk + 27));
      // stage I^w hbar (same for every direction)
      if (lane < nb) st3(sb + lane * SB_STRIDE + SB_IH, symmul(sb + lane * SB_STRIDE + SB_I, S.hb));
      __syncwarp();
    }
#pragma unroll
    for (int pt = 0; pt < 8; ++pt) {
      const int f = pt >> 2;
      const D3 frc = v3<double>(-lamk[3 * pt], -lamk[3 * pt + 1], -lamk[3 * pt + 2]);
      const D3 a = ld3(sm + L.arms + 3 * pt);
      const double in = f == 0 ? inL : inR;
      const V3<Dual> aD = lift<Dual>(a, scale(in, cross(dir.alpha, a)));
      S.footF[f] = S.footF[f] + lift<Dual>(frc, v3<double>(0.0, 0.0, 0.0));
      S.footN[f] = S.footN[f] + cross(aD, frc);
    }
    {
      const double kd = lamk[30];
      const St<Dual> sL = load_state(sb, T.foot_body[0], dir, Dual());
      const St<Dual> sR = load_state(sb, T.foot_body[1], dir, Dual());
      const V3<Dual> uD = lift<Dual>(fdu, scale(inR, cross(dir.alpha, fdu)));
      const V3<Dual> alD = lift<Dual>(fdal, scale(inL, cross(dir.alpha, fdal)));
      const V3<Dual> arD = lift<Dual>(fdar, scale(inR, cross(dir.alpha, fdar)));
      const V3<Dual> dD = (sL.o + alD) - (sR.o + arD);
      const V3<Dual> ku = scale(kd, uD);
      S.footF[0] = S.footF[0] + ku;
      S.footN[0] = S.footN[0] + cross(alD, ku);
      S.footF[1] = S.footF[1] - ku;
      S.footN[1] = S.footN[1] + scale(kd, cross(uD, dD)) - cross(arD, ku);
    }
    {
      // kappa = 2 sigma w (phi - 3) with its tangent; m(G) with its tangent (columns of G rotate with alpha)
      const D3 a = scale(inC, dir.alpha);
      double tG[9];
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const D3 col = v3<double>(G[j], G[3 + j], G[6 + j]);
        const D3 t = cross(a, col);
        tG[j] = t.x;
        tG[3 + j] = t.y;
        tG[6 + j] = t.z;
      }
      const double tphi = tG[0] + tG[4] + tG[8];
      const double cw = k1 ? 2.0 * sg * T.w_frame : 0.0;
      const Dual kappa = mkdual(cw * (phi - 3.0), cw * tphi);
      const V3<Dual> mGD = lift<Dual>(mG, v3<double>(tG[5] - tG[7], tG[6] - tG[2], tG[1] - tG[3]));
      S.chestN = scale(kappa, mGD);
    }
    HessEmit em;
    em.map = C.hk_map + T.knot_maps[k].hk_off;
    em.hess = hess + b * T.nnz_h + T.knot_maps[k].hk_base;
    em.stage = sm + L.stage;
    em.dirj = dirj;
    em.add_sd = em.add_s = 0.0;
    if (lane >= 4 && lane < 27 && k1) {
      const double wjl = C.wj[lane - 4];
      em.add_sd = T.joint_cost_kind == 0 ? sg * T.w_joint * 2.0 * wjl : 0.0;
      em.add_s = T.joint_cost_kind == 0 ? sg * T.w_joint * 2.0 * wjl * wjl : sg * T.w_joint * 2.0 * wjl;
    }
    V3<Dual> n0, w0, v0;
    const double lu_pre = lamk[31];  // read now: the slots of the packed sweep alias gbuf + lamk + slot
    const D3 lam_al = cross(ld3(lamk + 27), dir.alpha);  // quaternion lanes: velocity rows of their column (below)
    {
      SeedsP SP;
      SeedsT ST;
      SP.wc = S.wc;
      SP.hb = S.hb;
#pragma unroll
      for (int f = 0; f < 2; ++f) {
        SP.footF[f] = primal_of(S.footF[f]);
        SP.footN[f] = primal_of(S.footN[f]);
        ST.footF[f] = tangent_of(S.footF[f]);
        ST.footN[f] = tangent_of(S.footN[f]);
      }
      SP.chestN = primal_of(S.chestN);
      ST.chestN = tangent_of(S.chestN);
      __syncwarp();
      HB_PHASE(0, 8);  // seeds
      primal_adjoint_pass(T, sb, zs, SP, xc, xcd, my_depth, my_rank, my_parent, my_mass);
      HB_PHASE(0, 9);  // primal adjoint pass
      D3 tn0, tw0, tv0;
      {
        // Hessian of -hb.(P x Pdot)/M (see kin_tangent_sweep_packed) for every (direction, row), which also
        // initialises the stage; rows: vb3 qd4 sd23 (velocity lane = row) q4 s23 (direction lane = row - 30)
        double* stg = sm + L.stage;
        double* pslot = sm + L.gbuf;  // gbuf + lamk + slot: 474 contiguous doubles, all dead by now
        // tangents of P (rows q, s) and of Pdot (all rows) parked in the slot area for the cross terms (odd row
        // stride: the (q, s) block below reads a different row on every lane); the masses next to the quaternion
        // maps in the part of z the kinematics no longer reads
        constexpr int XT = 7;
        double* xt = pslot;           // [57][XT]: dP_r (velocity rows: zero, the place holds vel_dh), dPdot_r
        double* massv = zs + 24;      // [nb]
        if (lane < 27) {
          st3(xt + (30 + lane) * XT, tP);
          st3(xt + (30 + lane) * XT + 3, tPd);
        }
        if (lane < 30) {
          st3(xt + lane * XT, vel_dh);
          st3(xt + lane * XT + 3, vel_pv);
        }
        if (lane < nb) massv[lane] = my_mass;
        __syncwarp();
        if (lane < 27) {
          const D3 hbv = S.hb;
          const D3 a1 = cross(tPd, hbv), a2 = cross(hbv, tP);  // hb.(dP_r x dPdot_d) = dP_r.a1, hb.(dP_d x dPdot_r) = dPdot_r.a2
          double* col = stg + lane * 57;
          const double sM = -1.0 / M;
          // velocity rows (vb, qd, sd: 0..29) have dP_r = 0: half the loads and products.  A quaternion column takes
          // the whole entry there instead: the momentum row is linear in the velocities with a coefficient that turns
          // with the tree, so d/dq_a (lam_m . vel_dh_r) = vel_dh_r . (lam_m x g_a) (rows qd get the curvature of the
          // maps on top: they are replaced in the root chain rule)
          const bool qc = lane < 4;
          const D3 cr = qc ? lam_al : a2;
          const double sc = qc ? 1.0 : sM;
          const double* xr0 = xt + (qc ? 0 : 3);
#pragma unroll 5
          for (int r = 0; r < 30; ++r) col[r] = sc * dot(ld3(xr0 + XT * r), cr);
          // (q, s) x (q, s) block: hb.(dP_r x dPdot_d + dP_d x dPdot_r) is symmetric in (r, d).  Lane d takes the
          // pairs {d, d + j mod 27}, j = 0..13 -- every unordered pair exactly once, 14 per lane -- and stores the
          // value in both columns, so the stage holds every entry whichever of a mirrored pair the scatter reads.
#pragma unroll 2
          for (int j = 0; j < 14; ++j) {
            const int e = lane + j < 27 ? lane + j : lane + j - 27;
            const double* xe = xt + XT * (30 + e);
            const double v = sM * (dot(ld3(xe), a1) + dot(ld3(xe + 3), a2));
            col[30 + e] = v;
            stg[e * 57 + 30 + lane] = v;
          }
          if (lane >= 4) {  // joint regularisation on (sd_j, s_j), (s_j, s_j)
            col[7 + lane - 4] += em.add_sd;
            col[34 + lane - 4] += em.add_s;
          }
        }
        __syncwarp();
        HB_PHASE(0, 10);  // cross terms
        em.acc = true;
        kin_tangent_sweep_packed(T, sb, zs, massv, ST, S.hb, pslot, stg);
        HB_PHASE(0, 11);  // packed tangent sweep
        if (lane < 4) {  // closed form; v0 = 0 because hang does not depend on the base linear velocity
          tn0 = ld3(qt + 6 * lane);
          tw0 = ld3(qt + 6 * lane + 3);
          tv0 = v3<double>(0.0, 0.0, 0.0);
        } else {
          const double* rs = pslot + (lane < 27 ? T.root_slot[lane] : 0) * 12;
          tn0 = ld3(rs);
          tw0 = ld3(rs + 6);
          tv0 = ld3(rs + 9);
        }
        // the quaternion columns' rows vb, qd, q are complete (cross term included): stored, not added
        em.acc = lane >= 4;
      }
      n0 = lift<Dual>(ld3(sb + SB_ACC), tn0);
      w0 = lift<Dual>(ld3(sb + SB_ACC + 6), tw0);
      v0 = lift<Dual>(ld3(sb + SB_ACC + 9), tv0);
    }
    // Root chain rule dq_a = n0.g_a + w0.u_a, dqd_a = w0.w_a along direction d: the tangents of the root totals
    // against the maps, plus (quaternion directions d < 4 only) the curvature of the maps against the primal
    // totals, K[a][d] = n0.dg_a/dq_d + w0.du_a/dq_d and Kd[a][d] = w0.dw_a/dq_d.  K and Kd are the same on
    // every lane: lane 4 a + b builds entry (a, b) in dual arithmetic, the other lanes need none.
    if (lane < 16) {
      const int a = lane >> 2, bq = lane & 3;
      Dual qD[4];
      double qdv2[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        qD[i] = mkdual(zs[Z_Q + i], i == bq ? 1.0 : 0.0);
        qdv2[i] = zs[Z_QD + i];
      }
      V3<Dual> g, u, w;
      quat_map<Dual>(qD, qdv2, a, g, u, w);
      const D3 pn0 = primal_of(n0), pw0 = primal_of(w0);
      qK[lane] = dot(pn0, tangent_of(g)) + dot(pw0, tangent_of(u));
      qK[16 + lane] = dot(pw0, tangent_of(w));
    }
    __syncwarp();
    if (dirj >= 0) {
      const D3 tn0 = tangent_of(n0), tw0 = tangent_of(w0);
      em.put(0, v0.x.d);
      em.put(1, v0.y.d);
      em.put(2, v0.z.d);
      const double lu = lu_pre;
      // Hessian of w_bq |qd^-1 (x) q - 1|^2 is 2 w_bq A^T A = 2 w_bq |qd|^2 I (left-multiplication matrix)
      const double nqd = rbq[0] * rbq[0] + rbq[1] * rbq[1] + rbq[2] * rbq[2] +
                         rbq[3] * rbq[3];  // re-read (L1/L2 hit by now) rather than kept live across the sweep
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const bool qdir = lane < 4;
        const double dq = dot(tn0, ld3(qdat + 6 * a)) + dot(tw0, ld3(qdat + 6 * a + 3)) + (qdir ? qK[4 * a + lane] : 0.0);
        const double dqd = dot(tw0, ld3(qw + 3 * a)) + (qdir ? qK[16 + 4 * a + lane] : 0.0);
        const double extra = (a == lane && k1) ? 2.0 * sg * T.w_bq * nqd + 2.0 * lu : 0.0;
        em.put(3 + a, dqd);
        em.put(30 + a, dq + extra);
        // row s_j of column q_a by symmetry, on top of the cross term already staged there
        if (lane >= 4) em.stage[a * 57 + 34 + lane - 4] += dq;
      }
    }
    HB_PHASE(0, 12);  // root chain rule
    __syncwarp();
    if (em.stage) {
      // scatter the staged columns (27 directions x 57 rows) with coalesced map reads, in entry order: the staged
      // columns are read conflict-free in entry order, in destination order not (a destination-sorted list measured
      // 1.161 ms against 1.145 ms)
      const double* st = sm + L.stage;
      for (int eb = lane; eb < HSTAGE; eb += 32 * KIN_SCAT) {  // entry order: 1539 entries in three trips
        int sl[KIN_SCAT];
#pragma unroll
        for (int u = 0; u < KIN_SCAT; ++u) sl[u] = (eb + 32 * u) < HSTAGE ? em.map[eb + 32 * u] : -1;
#pragma unroll
        for (int u = 0; u < KIN_SCAT; ++u)
          if (sl[u] >= 0) em.hess[sl[u]] = st[eb + 32 * u];
      }
    }
    // velocity-diagonal entries (HK2): quaternion-velocity cost, joint regularisation
    if (lane < 27) {
      const int2 hk2m = *reinterpret_cast<const int2*>(&T.knot_maps[k].hk2_base);
      const int slot2 = C.hk2_map[hk2m.y + lane];
      if (slot2 >= 0)
        (hess + b * T.nnz_h + hk2m.x)[slot2] = lane < 4 ? 2.0 * sg * T.w_bqv : sg * T.w_joint * 2.0 * HB_N_JOINTS;
    }
    HB_PHASE(0, 13);  // Hessian scatter
  }
}

template __global__ void kino_kin_kernel<true>(const __grid_constant__ KinTopo, const KinoConst*, unsigned, const double*,
                                               const double*, long, const double*, const double*, double*, double*,
                                               double*, double*, double*, long);
template __global__ void kino_kin_kernel<false>(const __grid_constant__ KinTopo, const KinoConst*, unsigned,
                                                const double*, const double*, long, const double*, const double*,
                                                double*, double*, double*, double*, double*, long);

}  // namespace hb
