// kino_const.cuh -- device-resident constant block of one kinodynamic problem handle.
#pragma once
#include "../../include/hippopt_b200.h"
#include "hb_math.cuh"
#include "sweep_schedule.h"  // KT_* task descriptor bits, host-side scheduler

namespace hb {

// Developer instrumentation (tools/phase_profile.py builds a separate library with -DHB_PHASE_CLOCK; the shipped
// library compiles these macros away): cycles per phase of the two evaluation kernels, summed over the warps.
#ifdef HB_PHASE_CLOCK
__device__ unsigned long long hb_phase_acc[2][32];
#define HB_PHASE_INIT long long _pc = clock64();
#define HB_PHASE(kern, i)                                                                     \
  do {                                                                                        \
    __syncwarp();                                                                             \
    const long long _t = clock64();                                                           \
    if ((threadIdx.x & 31) == 0) atomicAdd(&hb_phase_acc[kern][i], (unsigned long long)(_t - _pc)); \
    _pc = _t;                                                                                 \
  } while (0)
#else
#define HB_PHASE_INIT
#define HB_PHASE(kern, i)
#endif

// internal evaluation bit (hb_eval_cost_terms): `fpart` then points to the [batch][N][HB_COST_TERMS] output
enum { HB_EVAL_COST_TERMS_BIT = 32 };

struct BodyC {
  double E[9];    // parent <- joint frame rotation
  double EA[9];   // E [a]x
  double EA2[9];  // E [a]x^2
  double r[3];    // joint origin in the parent frame
  double axis[3];
  double mass;
  double com[3];
  double inertia[6];  // about the CoM, body frame, (xx, xy, xz, yy, yz, zz)
  int parent;
  int depth;
  int slot;   // >= 0: this body owns a shared-memory branch accumulator
  int carry;  // 1: the contribution of body index+1 continues into this body (parent[index+1] == index)
  int sib_rank;  // index of this body among the children of its parent (level-wise primal adjoint pass)
};

// Scatter maps are stored RELATIVE to the first entry of their knot: the columns of one knot are contiguous in
// both compressed-column patterns, and the positions inside that range are the same for every interior knot, so
// a horizon needs two or three distinct tables (first / interior / last knot) instead of one per knot.  Every
// interior warp then reads the SAME few kilobytes (L1-resident) where the per-knot tables were an L2 round trip
// in front of every batch of scattered stores.  `*_off`: element offset of the knot's table inside the map array;
// `*_base`: what to add to its entries.
// Besides the entry-indexed tables (`*_map`: local entry -> slot) the Jacobian classes and the contact Hessian have a
// DESTINATION-SORTED list (`*_list`, `*_cnt` valid words at the same offset): word = local entry << 16 | slot for the
// staged outputs, and {slot, value descriptor} (contact_jac_desc.h) for the contact kernel's Jacobian.  Walking a list in
// order makes consecutive lanes store to consecutive addresses wherever the pattern has runs (whole point blocks of
// columns).  The kinematics Hessian is scattered in entry order and has no list.
struct alignas(16) KnotMaps {
  int jc_base, jc_off, jc_cnt, hc_base, hc_off, hc_cnt, pad0, pad1;         // contact kernel (two 16-byte loads)
  // kinematics kernel (16- and 8-byte loads); hk_cnt is an unused slot that keeps hk2_base 8-byte aligned
  int jk_base, jk_off, jk_cnt, hk_base, hk_off, hk_cnt, hk2_base, hk2_off;
};

struct KinoConst {
  int N, n_x, n_p, m, nnz_j, nnz_h, n_jc, n_jk, n_hc, terrain, has_final, has_per, h_init;
  int po_desc0, po_mass, po_init, po_final, po_dt, po_gravity, po_kt, po_kbs, po_eps, po_mu, po_max_u, po_max_fd,
      po_max_L, po_min_com_h, po_min_feet_d, po_max_feet_h, po_max_s, po_min_s, po_max_sd, po_min_sd, po_refs0,
      po_terrain;
  int yaw[3];
  // problem kind: 0 = kinodynamic OCP, 1 = static pose finder (single knot, no velocities).  The
  // kinematics kernel always works on a "virtual knot" in the kinodynamic 189-variable layout;
  // zmap[i] is the offset of virtual variable i inside the knot block of x, or -1 (absent: value 0).
  int kind, x_stride, cost_k0, joint_cost_kind;
  int po_fq, po_bq, po_bqv, po_jr, ref_stride;  // reference parameters of the kinematics costs
  short zmap[192];
  int nb, foot_body[2], chest_body, max_depth, n_slots, max_sib;
  alignas(16) int fam[HB_KF_COUNT][4];  // {first row, rows per knot, first knot, last knot}; read as one int4
  unsigned sub_mask[HB_MAX_BODIES];  // bit l: body l is in the subtree rooted at this body
  double w_swing, w_u, w_fd, w_centroid, w_comvel[3], w_frame, w_bq, w_bqv, w_joint, w_ratio, w_yaw;
  double wj[HB_N_JOINTS];
  double total_mass;
  double foot_R[2][9], foot_t[2][3], chest_R[9];
  BodyC body[HB_MAX_BODIES];
  const int* jc_map;
  const int* jk_map;
  const short* hc_index;
  const int* hc_map;
  const int* hk_map;
  const int* hk2_map;
  const KnotMaps* knot_maps;
  const int2* jc_list;
  const unsigned* jk_list;
  const unsigned* hc_list;
};

// Warp-uniform part of KinoConst.  It is passed BY VALUE as a __grid_constant__ kernel parameter:
// reads whose index is the same for every lane (tree topology inside the sweeps, row families with a
// compile-time id) become constant-bank operands instead of global loads -- in the ncu capture of the
// previous version those loads were ~40 % of the long-scoreboard stalls of the kinematics kernel.
// Lane-indexed data (joint frames, inertias, per-point families) stays in KinoConst / global memory,
// where a divergent index costs one coalesced load rather than a serialised constant fetch.
struct KinTopo {
  double mass[HB_MAX_BODIES];
  unsigned sub_mask[HB_MAX_BODIES];
  signed char parent[HB_MAX_BODIES], slot[HB_MAX_BODIES], carry[HB_MAX_BODIES];
  // (depth, sibling rank) pairs that hold at least one body, deepest first (level-wise adjoint pass)
  signed char step_depth[2 * HB_MAX_BODIES], step_rank[2 * HB_MAX_BODIES];
  int n_steps;
  int fam[HB_KF_COUNT][4];
  int nb, foot_body[2], chest_body, max_depth, n_slots, max_sib;
  // scalars of the kinematics kernel (offsets into x / p / g and weights): read from the constant bank, so
  // that the first global load of a warp is its data, not the address of its data
  int N, n_x, m, nnz_j, nnz_h, n_jk, x_stride, cost_k0, joint_cost_kind, zmap_identity;
  int po_desc0, po_mass, po_fq, po_bq, po_bqv, po_jr, ref_stride;
  double w_frame, w_bq, w_bqv, w_joint, total_mass;
  // ... and of the contact kernel
  int n_jc, n_hc, has_final, has_per, h_init;
  int po_dt, po_gravity, po_kt, po_kbs, po_eps, po_mu, po_refs0, po_terrain;
  int yaw[3];
  double w_swing, w_u, w_fd, w_centroid, w_comvel[3], w_ratio, w_yaw;
  const int* jc_map;
  const short* hc_index;
  const int* hc_map;
  const KnotMaps* knot_maps;
  const int2* jc_list;
  const unsigned* hc_list;
  // planar terrain: local Hessian entry of the 29 per-point terms of contact point i (kino_contact.cu), 32 shorts per point
  const short* hc_pt;
  // local Hessian entries of the least-squares cost rows (kino_contact.cu), 8 shorts per lane; same allocation as hc_pt
  const short* hc_ls;
  // packed tangent sweep (kino_kin.cu): sched[round * 32 + lane] = task descriptor (see KT_* below)
  const int* sched;
  signed char root_slot[32];  // slot that holds the root totals of direction d after the sweep
  int n_rounds, n_pslots;
  unsigned round_seed_mask;  // bit r: some task of round r sits on a foot / chest body (seed tangents needed)
  unsigned round_heavy_mask;  // bit r: round r holds "in" tasks (sub-tree of the direction); else pure propagation
};

// global g index of local row r of family `fam` at knot k, or -1 when the row does not exist
template <class Tab>
__device__ __forceinline__ int grow(const Tab& C, int fam, int k, int r) {
  const int base = C.fam[fam][0];
  if (base < 0 || k < C.fam[fam][2] || k > C.fam[fam][3]) return -1;
  return base + (k - C.fam[fam][2]) * C.fam[fam][1] + r;
}
// global table (lane-indexed families): one 16-byte load for {base, rows, k0, k1}
__device__ __forceinline__ int grow(const KinoConst& C, int fam, int k, int r) {
  const int4 f = __ldg(reinterpret_cast<const int4*>(C.fam[fam]));
  if (f.x < 0 || k < f.z || k > f.w) return -1;
  return f.x + (k - f.z) * f.y + r;
}

// reference sub-offsets (variables.py:13-116, SURVEY.md Appendix B.2)
enum {
  R_RATIO_L = 0, R_YAW_L = 4, R_RATIO_R = 5, R_YAW_R = 9, R_SWING = 10, R_CW = 11, R_CC = 14, R_COMV = 17,
  R_FQ = 20, R_BQ = 24, R_BQV = 28, R_JR = 32, R_COUNT = 55
};
// offsets inside one knot of x (SURVEY.md Appendix B.1)
enum {
  Z_V = 0, Z_FD = 3, Z_P = 6, Z_F = 9, Z_U = 12, Z_VB = 120, Z_QD = 123, Z_PB = 127, Z_Q = 130, Z_SD = 134,
  Z_S = 157, Z_COM = 180, Z_H = 183, NZ = 189
};

}  // namespace hb
