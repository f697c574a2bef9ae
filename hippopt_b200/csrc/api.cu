// api.cu -- C ABI (include/hippopt_b200.h): handle management, launches, fp64 probe.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "kino_const.cuh"
#include "contact_jac_desc.h"
// single translation unit: the kernels are included by hippopt_b200.cu before this file


static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                      \
  do {                                                                                      \
    cudaError_t e__ = (expr);                                                               \
    if (e__ != cudaSuccess) return fail(HB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
  } while (0)

enum { KIND_KINO = 1, KIND_TOY = 2 };

// a handle's tables and scratch live on the device that was current at creation: calls from another current
// device would launch on the wrong GPU with foreign pointers
#define CHECK_DEVICE(h, what)                                                                          \
  do {                                                                                                 \
    int cur__ = -1;                                                                                    \
    cudaGetDevice(&cur__);                                                                             \
    if ((h)->device >= 0 && cur__ != (h)->device)                                                      \
      return fail(HB_ERR_INVALID, std::string(what) + ": the handle belongs to CUDA device " +         \
                                      std::to_string((h)->device) + ", the current device is " +       \
                                      std::to_string(cur__) + " (cudaSetDevice before the call)");      \
  } while (0)

struct hb_problem_s {
  int kind = 0;
  int launches = 0;
  int device = -1;  // CUDA device the handle's tables live on (advisor finding, round 1): checked at every call
  // kinodynamic
  hb::KinoConst host{};
  hb::KinoConst* dev = nullptr;
  hb::KinTopo topo{};  // warp-uniform tables, passed by value to the kinematics kernel
  int *d_jc = nullptr, *d_jk = nullptr, *d_hc = nullptr, *d_hk = nullptr, *d_hk2 = nullptr, *d_sched = nullptr;
  short* d_hci = nullptr;
  short* d_hc_pt = nullptr;
  hb::KnotMaps* d_knot_maps = nullptr;
  int2* d_jc_list = nullptr;
  unsigned *d_jk_list = nullptr, *d_hc_list = nullptr;
  // per-knot cost partial sums, one scratch buffer per stream so that evaluations enqueued on
  // different streams (HostPipeline) do not share scratch
  std::map<cudaStream_t, std::pair<double*, int64_t>> fpart;
  bool jac_adjoint = false;  // hb_set_option(HB_OPT_JAC_ADJOINT)
  // optional per-kernel timing (CUDA events on the launching stream)
  bool prof = false;
  std::vector<cudaEvent_t> prof_ev;  // 4 events per hb_eval: start, after contact, after kin, after reduce
  // toy
  hb::ToyProblem* toy = nullptr;
  // host-buffer pipeline (hb_eval_host): device staging slabs, one per internal stream
  enum { HOST_STREAMS = 3, HOST_CHUNK = 128 };
  cudaStream_t hst[HOST_STREAMS] = {nullptr, nullptr, nullptr};
  double* hslab[HOST_STREAMS] = {nullptr, nullptr, nullptr};
  int64_t hslab_chunk = 0;  // instances one slab holds
  // single-chunk hb_eval_host calls that repeat with the same mask and the same (pinned) host buffers -- what a CPU-side
  // IPOPT does at every iterate -- are captured once as a CUDA graph and replayed: one launch instead of 2-3 copies,
  // 2-3 kernels and the fork / join events of the small-batch overlap
  struct HostGraph {
    uint32_t mask = 0;
    const void* ptr[8] = {};
    int64_t batch = 0;
    int seen = 0;
    bool unusable = false;
    cudaGraphExec_t exec = nullptr;
    int launches = 0;
    int64_t h2d = 0, d2h = 0;
  };
  std::vector<HostGraph> hgraphs;
  void drop_host_graphs() {
    for (auto& g : hgraphs)
      if (g.exec) cudaGraphExecDestroy(g.exec);
    hgraphs.clear();
  }
  double* d_p = nullptr;    // parameters of the current solve
  int64_t p_cap = 0, p_stride = -1, p_batch = 0;
  int64_t h2d_bytes = 0, d2h_bytes = 0;
  // small batches (a CPU-side IPOPT evaluates ONE instance): the contact kernel runs on an auxiliary stream next to
  // the kinematics kernel -- a handful of warps leave the GPU empty, so the two kernels' single-warp latencies
  // (33 us and 47 us) overlap instead of adding up
  cudaStream_t aux = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // host copies of what the handle was created from (hb_save) and the tables a non-Python caller needs: CCS
  // patterns of jac_g / hess_l and the affine description of lbg / ubg (hb_kino_attach_tables)
  std::vector<int32_t> c_icfg, c_jc, c_jk, c_hc, c_hk, c_hk2, lb_idx, ub_idx;
  std::vector<int16_t> c_hci;
  std::vector<double> c_dcfg, lb_val, ub_val;
  std::vector<int64_t> jac_colind, jac_row, hess_colind, hess_row;
};


// cudaFuncSetAttribute is per device: a process that drives several GPUs must opt every one of them in to the
// large dynamic shared-memory carve-out (advisor finding, round 1).  Guarded by a mutex: cheap, and hb_eval may be
// called from several host threads.
#include <mutex>
static int device_sms[64] = {0};
static cudaError_t ensure_kernel_attributes(int dev) {
  static std::mutex mu;
  static bool done[64] = {false};
  std::lock_guard<std::mutex> lock(mu);
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  if (done[dev]) return cudaSuccess;
  const int big = 200 * 1024;
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(hb::kino_contact_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::kino_contact_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::kino_contact_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::kino_kin_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::kino_kin_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::pose_contact_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::pose_contact_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::pose_contact_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)) != cudaSuccess) return e;
  const int lu_big = 210 * 1024;
  if ((e = cudaFuncSetAttribute(hb::lu_factor_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lu_big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::lu_factor_kernel<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lu_big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::lu_factor_kernel<3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lu_big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::lu_factor_kernel<1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lu_big)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::lu_factor_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lu_big)) != cudaSuccess) return e;
  const int lu_staged = 232448 - 1024 - 2560;
  if ((e = cudaFuncSetAttribute(hb::lu_solve_staged_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, lu_staged)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(hb::lu_solve_staged_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, lu_staged)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&device_sms[dev], cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  done[dev] = true;
  return cudaSuccess;
}

__global__ void reduce_f_kernel(const double* __restrict__ fpart, double* __restrict__ f, int n_terms, long batch) {
  const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const double* fp = fpart + b * n_terms;
  double acc = 0.0;
  for (int i = 0; i < n_terms; ++i) acc += fp[i];
  f[b] = acc;
}

// contact kernel of a terrain (hb_kino_create accepts 0, 1 and 2)
static decltype(&hb::kino_contact_kernel<0>) kino_contact_kernel_for(int terrain) {
  return terrain == 0 ? hb::kino_contact_kernel<0> : terrain == 2 ? hb::kino_contact_kernel<2> : hb::kino_contact_kernel<1>;
}
static decltype(&hb::pose_contact_kernel<0>) pose_contact_kernel_for(int terrain) {
  return terrain == 0 ? hb::pose_contact_kernel<0> : terrain == 2 ? hb::pose_contact_kernel<2> : hb::pose_contact_kernel<1>;
}

// ---------------------------------------------------------------------------------------------
// Schedule of the packed tangent sweep: sweep_schedule.h (host-only, also reachable through
// hb_debug_sweep_schedule for the CPU tests)
static hb::SweepTopo sweep_topo_of(const hb::KinoConst& C) {
  hb::SweepTopo T;
  T.nb = C.nb;
  for (int l = 0; l < 32; ++l) {
    T.parent[l] = l < C.nb ? C.body[l].parent : -1;
    T.sub_mask[l] = C.sub_mask[l];
  }
  T.foot_body[0] = C.foot_body[0];
  T.foot_body[1] = C.foot_body[1];
  T.chest_body = C.chest_body;
  T.n_base = 0;  // the kernel fills the four quaternion columns in closed form (kino_kin.cu)
  return T;
}

extern "C" int hb_debug_sweep_schedule_n_base(int32_t nb, const int32_t* parent, int32_t foot_l, int32_t foot_r,
                                              int32_t chest, int32_t typed, int32_t n_base, int32_t* tasks,
                                              int32_t* info) {
  if (!parent || !tasks || !info || nb < 2 || nb > 28 || n_base < 0 || n_base > 4)
    return fail(HB_ERR_INVALID, "hb_debug_sweep_schedule: bad argument");
  hb::SweepTopo T;
  T.nb = nb;
  T.n_base = n_base;
  for (int l = 0; l < 32; ++l) {
    T.parent[l] = l < nb ? parent[l] : -1;
    T.sub_mask[l] = 0u;
  }
  for (int l = 0; l < nb; ++l)
    for (int b = l; b >= 0; b = T.parent[b]) T.sub_mask[b] |= 1u << l;
  T.foot_body[0] = foot_l;
  T.foot_body[1] = foot_r;
  T.chest_body = chest;
  const hb::SweepSchedule s = hb::build_sweep_schedule(T, typed != 0, typed >= 2 ? 0 : 1);
  if (s.n_rounds <= 0) return fail(HB_ERR_UNSUPPORTED, "hb_debug_sweep_schedule: no schedule");
  for (size_t i = 0; i < s.tasks.size() && i < 32 * 32; ++i) tasks[i] = s.tasks[i];
  info[0] = s.n_rounds;
  info[1] = s.n_slots;
  info[2] = s.n_tasks;
  info[3] = s.n_heavy_tasks;
  info[4] = (int32_t)s.heavy_mask;
  info[5] = (int32_t)s.seed_mask;
  for (int d = 0; d < 27 && d < 4 + nb - 1; ++d) info[6 + d] = s.root_slot[d];
  return HB_OK;
}

extern "C" int hb_debug_sweep_schedule(int32_t nb, const int32_t* parent, int32_t foot_l, int32_t foot_r, int32_t chest,
                                       int32_t typed, int32_t* tasks, int32_t* info) {
  return hb_debug_sweep_schedule_n_base(nb, parent, foot_l, foot_r, chest, typed, 4, tasks, info);
}

template <class T>
static cudaError_t upload(T** dst, const T* src, size_t n) {
  cudaError_t e = cudaMalloc(dst, n * sizeof(T) + 16);
  if (e != cudaSuccess) return e;
  return cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice);
}

extern "C" int hb_kino_create(const int32_t* icfg, const double* dcfg, const int32_t* jc_map, const int32_t* jk_map,
                              const int16_t* hc_index, const int32_t* hc_map, const int32_t* hk_map,
                              const int32_t* hk2_map, hb_handle* out) {
  if (!icfg || !dcfg || !jc_map || !jk_map || !hc_index || !hc_map || !hk_map || !hk2_map || !out)
    return fail(HB_ERR_INVALID, "hb_kino_create: null argument");
  hb_problem_s* h = new hb_problem_s();
  h->kind = KIND_KINO;
  cudaGetDevice(&h->device);
  hb::KinoConst& C = h->host;
  C.N = icfg[HB_KI_HORIZON];
  C.n_x = icfg[HB_KI_N_X];
  C.n_p = icfg[HB_KI_N_P];
  C.m = icfg[HB_KI_M];
  C.nnz_j = icfg[HB_KI_NNZ_J];
  C.nnz_h = icfg[HB_KI_NNZ_H];
  C.n_jc = icfg[HB_KI_N_JC];
  C.n_jk = icfg[HB_KI_N_JK];
  C.n_hc = icfg[HB_KI_N_HC];
  C.terrain = icfg[HB_KI_TERRAIN];
  C.has_final = icfg[HB_KI_HAS_FINAL];
  C.has_per = icfg[HB_KI_HAS_PERIODICITY];
  C.h_init = icfg[HB_KI_H_INIT];
  C.po_desc0 = icfg[HB_KI_PO_DESC0];
  C.po_mass = icfg[HB_KI_PO_MASS];
  C.po_init = icfg[HB_KI_PO_INIT];
  C.po_final = icfg[HB_KI_PO_FINAL];
  C.po_dt = icfg[HB_KI_PO_DT];
  C.po_gravity = icfg[HB_KI_PO_GRAVITY];
  C.po_kt = icfg[HB_KI_PO_KT];
  C.po_kbs = icfg[HB_KI_PO_KBS];
  C.po_eps = icfg[HB_KI_PO_EPS];
  C.po_mu = icfg[HB_KI_PO_MU];
  C.po_max_u = icfg[HB_KI_PO_MAX_U];
  C.po_max_fd = icfg[HB_KI_PO_MAX_FD];
  C.po_max_L = icfg[HB_KI_PO_MAX_L];
  C.po_min_com_h = icfg[HB_KI_PO_MIN_COM_H];
  C.po_min_feet_d = icfg[HB_KI_PO_MIN_FEET_D];
  C.po_max_feet_h = icfg[HB_KI_PO_MAX_FEET_H];
  C.po_max_s = icfg[HB_KI_PO_MAX_S];
  C.po_min_s = icfg[HB_KI_PO_MIN_S];
  C.po_max_sd = icfg[HB_KI_PO_MAX_SD];
  C.po_min_sd = icfg[HB_KI_PO_MIN_SD];
  C.po_refs0 = icfg[HB_KI_PO_REFS0];
  C.po_terrain = icfg[HB_KI_PO_TERRAIN];
  C.yaw[0] = icfg[HB_KI_YAW_BR];
  C.yaw[1] = icfg[HB_KI_YAW_TR];
  C.yaw[2] = icfg[HB_KI_YAW_TL];
  C.nb = icfg[HB_KI_N_BODIES];
  C.foot_body[0] = icfg[HB_KI_FOOT_BODY_L];
  C.foot_body[1] = icfg[HB_KI_FOOT_BODY_R];
  C.chest_body = icfg[HB_KI_CHEST_BODY];
  C.kind = icfg[HB_KI_KIND];
  C.x_stride = icfg[HB_KI_X_STRIDE];
  C.cost_k0 = icfg[HB_KI_COST_K0];
  C.joint_cost_kind = icfg[HB_KI_JOINT_COST_KIND];
  C.po_fq = icfg[HB_KI_PO_FQ];
  C.po_bq = icfg[HB_KI_PO_BQ];
  C.po_bqv = icfg[HB_KI_PO_BQV];
  C.po_jr = icfg[HB_KI_PO_JR];
  C.ref_stride = icfg[HB_KI_REF_STRIDE];
  for (int i = 0; i < 192; ++i) C.zmap[i] = i < 189 ? (short)icfg[HB_KI_ZMAP0 + i] : (short)-1;
  if (C.kind != 0 && C.kind != 1) {
    delete h;
    return fail(HB_ERR_INVALID, "hb_kino_create: kind must be 0 (kinodynamic) or 1 (pose finder)");
  }
  if (C.kind == 1 && C.N != 1) {
    delete h;
    return fail(HB_ERR_UNSUPPORTED, "hb_kino_create: the pose finder is a single-knot problem");
  }
  if (C.terrain != 0 && C.terrain != 1 && C.terrain != 2) {
    delete h;
    return fail(HB_ERR_UNSUPPORTED,
                "hb_kino_create: terrain must be 0 (planar), 1 (two smooth steps) or 2 (general smooth steps)");
  }
  if (C.terrain == 2 && (C.n_p - C.po_terrain < 10 || (C.n_p - C.po_terrain) % 10 != 0)) {
    delete h;
    return fail(HB_ERR_INVALID, "hb_kino_create: terrain 2 needs n_p - po_terrain to be a positive multiple of 10 "
                                "(one (l, w, height, ox, oy, oz, yaw, n_x, n_y, n_z) record per step)");
  }
  if (C.nb < 2 || C.nb > HB_MAX_BODIES || C.nb - 1 != HB_N_JOINTS) {
    delete h;
    return fail(HB_ERR_INVALID, "hb_kino_create: the kernels are laid out for 23 joints / <= 32 bodies");
  }
  for (int f = 0; f < HB_KF_COUNT; ++f)
    for (int i = 0; i < 4; ++i) C.fam[f][i] = icfg[HB_KI_FAM0 + 4 * f + i];
  C.w_swing = dcfg[HB_KD_W_SWING];
  C.w_u = dcfg[HB_KD_W_U];
  C.w_fd = dcfg[HB_KD_W_FD];
  C.w_centroid = dcfg[HB_KD_W_CENTROID];
  for (int i = 0; i < 3; ++i) C.w_comvel[i] = dcfg[HB_KD_W_COMVEL0 + i];
  C.w_frame = dcfg[HB_KD_W_FRAME];
  C.w_bq = dcfg[HB_KD_W_BQ];
  C.w_bqv = dcfg[HB_KD_W_BQV];
  C.w_joint = dcfg[HB_KD_W_JOINT];
  C.w_ratio = dcfg[HB_KD_W_RATIO];
  C.w_yaw = dcfg[HB_KD_W_YAW];
  for (int i = 0; i < HB_N_JOINTS; ++i) C.wj[i] = dcfg[HB_KD_WJ0 + i];
  C.total_mass = dcfg[HB_KD_TOTAL_MASS];
  for (int f = 0; f < 2; ++f) {
    for (int i = 0; i < 9; ++i) C.foot_R[f][i] = dcfg[HB_KD_FOOT_R0 + 9 * f + i];
    for (int i = 0; i < 3; ++i) C.foot_t[f][i] = dcfg[HB_KD_FOOT_T0 + 3 * f + i];
  }
  for (int i = 0; i < 9; ++i) C.chest_R[i] = dcfg[HB_KD_CHEST_R0 + i];
  C.max_depth = 0;
  C.n_slots = 0;
  for (int l = 0; l < C.nb; ++l) {
    hb::BodyC& B = C.body[l];
    const double* d = dcfg + HB_KD_BODY0 + HB_KD_BODY_STRIDE * l;
    for (int i = 0; i < 9; ++i) B.E[i] = d[i];
    for (int i = 0; i < 3; ++i) B.r[i] = d[9 + i];
    for (int i = 0; i < 3; ++i) B.axis[i] = d[12 + i];
    B.mass = d[15];
    for (int i = 0; i < 3; ++i) B.com[i] = d[16 + i];
    const double* I = d + 19;
    B.inertia[0] = I[0];
    B.inertia[1] = I[1];
    B.inertia[2] = I[2];
    B.inertia[3] = I[4];
    B.inertia[4] = I[5];
    B.inertia[5] = I[8];
    const double a[3] = {B.axis[0], B.axis[1], B.axis[2]};
    const double A[9] = {0, -a[2], a[1], a[2], 0, -a[0], -a[1], a[0], 0};
    double A2[9];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) A2[3 * i + j] = A[3 * i] * A[j] + A[3 * i + 1] * A[3 + j] + A[3 * i + 2] * A[6 + j];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        B.EA[3 * i + j] = B.E[3 * i] * A[j] + B.E[3 * i + 1] * A[3 + j] + B.E[3 * i + 2] * A[6 + j];
        B.EA2[3 * i + j] = B.E[3 * i] * A2[j] + B.E[3 * i + 1] * A2[3 + j] + B.E[3 * i + 2] * A2[6 + j];
      }
    B.parent = l == 0 ? -1 : icfg[HB_KI_PARENT0 + l];
    if (l > 0 && (B.parent < 0 || B.parent >= l)) {
      delete h;
      return fail(HB_ERR_INVALID, "hb_kino_create: bodies must be ordered parent-before-child");
    }
    B.depth = l == 0 ? 0 : C.body[B.parent].depth + 1;
    if (B.depth > C.max_depth) C.max_depth = B.depth;
    B.slot = -1;
    B.carry = 0;
  }
  C.max_sib = 1;
  {
    int n_children[HB_MAX_BODIES] = {0};
    C.body[0].sib_rank = 0;
    for (int l = 1; l < C.nb; ++l) {
      const int p = C.body[l].parent;
      C.body[l].sib_rank = n_children[p]++;
      if (n_children[p] > C.max_sib) C.max_sib = n_children[p];
    }
  }
  for (int l = 1; l < C.nb; ++l) {
    const int p = C.body[l].parent;
    if (p == l - 1) C.body[p].carry = 1;
    else if (p != 0 && C.body[p].slot < 0) C.body[p].slot = C.n_slots++;
  }
  for (int j = 0; j < HB_MAX_BODIES; ++j) C.sub_mask[j] = 0u;
  for (int l = 0; l < C.nb; ++l) {
    int bdy = l;
    while (bdy >= 0) {
      C.sub_mask[bdy] |= (1u << l);
      bdy = C.body[bdy].parent;
    }
  }
  {
    hb::KinTopo& T = h->topo;
    static_cast<hb::KinScalars&>(T) = C;
    for (int l = 0; l < HB_MAX_BODIES; ++l) {
      const bool in = l < C.nb;
      T.mass[l] = in ? C.body[l].mass : 0.0;
      T.parent[l] = (signed char)(in ? C.body[l].parent : -1);
      T.slot[l] = (signed char)(in ? C.body[l].slot : -1);
      T.carry[l] = (signed char)(in ? C.body[l].carry : 0);
    }
    T.n_steps = 0;
    for (int dep = C.max_depth; dep >= 1; --dep)
      for (int r = 0; r < C.max_sib; ++r) {
        bool any = false;
        for (int l = 1; l < C.nb; ++l) any = any || (C.body[l].depth == dep && C.body[l].sib_rank == r);
        if (any) {
          T.step_depth[T.n_steps] = (signed char)dep;
          T.step_rank[T.n_steps] = (signed char)r;
          T.n_steps++;
        }
      }
    T.zmap_identity = 1;
    for (int i = 0; i < 189; ++i) T.zmap_identity = T.zmap_identity && C.zmap[i] == i;
  }
  const size_t N = C.N;
  h->c_icfg.assign(icfg, icfg + HB_KI_COUNT);
  h->c_dcfg.assign(dcfg, dcfg + HB_KD_COUNT);
  h->c_jc.assign(jc_map, jc_map + N * C.n_jc);
  h->c_jk.assign(jk_map, jk_map + N * C.n_jk);
  h->c_hci.assign(hc_index, hc_index + 129 * 129);
  h->c_hc.assign(hc_map, hc_map + N * C.n_hc);
  h->c_hk.assign(hk_map, hk_map + N * 27 * 57);
  h->c_hk2.assign(hk2_map, hk2_map + N * 27);
  cudaError_t e = cudaSuccess;
  {
    // knot-relative tables (KnotMaps in kino_const.cuh): identical rows are stored once, each with its
    // destination-sorted list
    std::vector<hb::KnotMaps> km(N);
    bool too_wide = false;
    auto relative = [&](const int32_t* map, size_t n, int hb::KnotMaps::*base, int hb::KnotMaps::*off,
                        int hb::KnotMaps::*cnt, int** dst_rel, void** dst_list, bool with_desc) {
      std::vector<int32_t> rel, list, counts, row(n);
      const size_t words = with_desc ? 2 : 1;
      for (size_t k = 0; k < N; ++k) {
        int32_t lo = INT32_MAX;
        for (size_t i = 0; i < n; ++i)
          if (map[k * n + i] >= 0 && map[k * n + i] < lo) lo = map[k * n + i];
        if (lo == INT32_MAX) lo = 0;
        for (size_t i = 0; i < n; ++i) row[i] = map[k * n + i] >= 0 ? map[k * n + i] - lo : -1;
        size_t c = 0;
        for (; c * n < rel.size(); ++c)
          if (std::equal(row.begin(), row.end(), rel.begin() + c * n)) break;
        if (c * n == rel.size()) {
          rel.insert(rel.end(), row.begin(), row.end());
          std::vector<std::pair<int32_t, int32_t>> order;  // (slot, entry)
          for (size_t i = 0; i < n; ++i) {
            if (row[i] < 0) continue;
            if (with_desc && hb::contact_jac_descriptor((int)i, C.terrain) == hb::JC_SKIP) continue;
            order.emplace_back(row[i], (int32_t)i);
          }
          std::sort(order.begin(), order.end());
          counts.push_back((int32_t)order.size());
          for (size_t i = 0; i < n; ++i) {
            if (i >= order.size()) {
              for (size_t w = 0; w < words; ++w) list.push_back(-1);
            } else if (with_desc) {
              list.push_back(order[i].first);
              list.push_back(hb::contact_jac_descriptor(order[i].second, C.terrain));
            } else {
              too_wide = too_wide || order[i].first >= 65536 || order[i].second >= 65536;
              list.push_back((int32_t)(((uint32_t)order[i].second << 16) | (uint32_t)order[i].first));
            }
          }
        }
        km[k].*base = lo;
        km[k].*off = (int)(c * n);
        if (cnt) km[k].*cnt = counts[c];
      }
      cudaError_t err = upload(dst_rel, rel.data(), rel.size());
      if (err == cudaSuccess && dst_list) err = upload(reinterpret_cast<int32_t**>(dst_list), list.data(), list.size());
      return err;
    };
    using KM = hb::KnotMaps;
    if (e == cudaSuccess) e = relative(jc_map, C.n_jc, &KM::jc_base, &KM::jc_off, &KM::jc_cnt, &h->d_jc, (void**)&h->d_jc_list, C.kind == 0);
    if (e == cudaSuccess) e = relative(jk_map, C.n_jk, &KM::jk_base, &KM::jk_off, &KM::jk_cnt, &h->d_jk, (void**)&h->d_jk_list, false);
    if (e == cudaSuccess) e = relative(hc_map, C.n_hc, &KM::hc_base, &KM::hc_off, &KM::hc_cnt, &h->d_hc, (void**)&h->d_hc_list, false);
    if (e == cudaSuccess) e = relative(hk_map, 27 * 57, &KM::hk_base, &KM::hk_off, nullptr, &h->d_hk, nullptr, false);
    if (e == cudaSuccess) e = relative(hk2_map, 27, &KM::hk2_base, &KM::hk2_off, nullptr, &h->d_hk2, nullptr, false);
    if (e == cudaSuccess) e = upload(&h->d_knot_maps, km.data(), km.size());
    if (too_wide) {
      hb_destroy(h);
      return fail(HB_ERR_UNSUPPORTED, "hb_kino_create: a knot's columns hold more than 65535 non-zeros (packed scatter lists)");
    }
  }
  if (e == cudaSuccess) e = upload(&h->d_hci, hc_index, (size_t)129 * 129);
  if (e == cudaSuccess) {
    // per-point Hessian terms of the planar contact kernel, in the order kino_contact.cu lists them: 11 complementarity /
    // friction / swing terms, 6 control regularisations, 12 momentum cross terms -> 29 local entries per point, padded to 32
    // followed by the 7 local entries per lane of the least-squares cost rows, padded to 8, in the kernel's slot order
    std::vector<int16_t> pt(8 * 32 + 32 * 8, -1);
    enum { V = 0, FD = 3, P = 6, F = 9, U = 12, COM = 120, NV = 129 };
    for (int i = 0; i < 8; ++i) {
      const int o = 15 * i;
      int n = 0;
      auto term = [&](int vi, int vj) { pt[32 * i + n++] = hc_index[vi * NV + vj]; };
      term(o + P + 2, o + P + 2);
      term(o + P + 2, o + U);
      term(o + P + 2, o + U + 1);
      term(o + P + 2, o + F + 2);
      term(o + V + 2, o + F + 2);
      term(o + FD + 2, o + P + 2);
      term(o + V, o + V);
      term(o + V + 1, o + V + 1);
      term(o + F, o + F);
      term(o + F + 1, o + F + 1);
      term(o + F + 2, o + F + 2);
      for (int c = 0; c < 3; ++c) {
        term(o + U + c, o + U + c);
        term(o + FD + c, o + FD + c);
      }
      for (int a = 0; a < 3; ++a)
        for (int bb = 0; bb < 3; ++bb) {
          if (a == bb) continue;
          term(o + P + a, o + F + bb);
          term(COM + a, o + F + bb);
        }
    }
    int16_t* ls = pt.data() + 8 * 32;
    for (int lane = 0; lane < 32; ++lane) {
      auto entry = [&](int pi, int ci, int pj, int cj) { return hc_index[(15 * pi + ci) * NV + 15 * pj + cj]; };
      for (int u = 0; u < 4; ++u) {  // p_c of points (a, (a + d) mod 8), t = 36 c + 8 d + a
        const int t = lane + 32 * u, c = t / 36, q = t % 36, a = q & 7;
        if (t < 108) ls[8 * lane + u] = entry(a, P + c, (a + (q >> 3)) & 7, P + c);
      }
      {  // (p_x, p_y) of points (4 foot + i, 4 foot + j), lane = 16 foot + 4 i + j, where one yaw row holds both points
        const int foot = lane >> 4, i = (lane >> 2) & 3, j = lane & 3;
        bool on_row = false;
        for (int s = 0; s < 2; ++s) {
          const bool hi = i == C.yaw[s] || i == C.yaw[s + 1], hj = j == C.yaw[s] || j == C.yaw[s + 1];
          on_row = on_row || (hi && hj);
        }
        if (on_row) ls[8 * lane + 4] = entry(4 * foot + i, P, 4 * foot + j, P + 1);
      }
      for (int u = 5; u < 7; ++u) {  // f_c of points (a, (a + d) mod 4) of one foot, t = 10 (3 foot + c) + 4 d + a
        const int t = lane + 32 * (u - 5), foot = t / 30, c = (t / 10) % 3, q = t % 10, a = q & 3;
        if (t < 60) ls[8 * lane + u] = entry(4 * foot + a, F + c, 4 * foot + ((a + (q >> 2)) & 3), F + c);
      }
    }
    e = upload(&h->d_hc_pt, pt.data(), pt.size());
  }
  C.jc_map = h->d_jc;
  C.jk_map = h->d_jk;
  C.hc_index = h->d_hci;
  C.hc_map = h->d_hc;
  C.hk_map = h->d_hk;
  C.hk2_map = h->d_hk2;
  C.knot_maps = h->d_knot_maps;
  C.jc_list = h->d_jc_list;
  C.jk_list = h->d_jk_list;
  C.hc_list = h->d_hc_list;
  h->topo.knot_maps = h->d_knot_maps;
  h->topo.jc_list = h->d_jc_list;
  h->topo.hc_list = h->d_hc_list;
  h->topo.jc_map = h->d_jc;
  h->topo.hc_index = h->d_hci;
  h->topo.hc_pt = h->d_hc_pt;
  h->topo.hc_ls = h->d_hc_pt ? h->d_hc_pt + 8 * 32 : nullptr;
  h->topo.hc_map = h->d_hc;
  {
    // 4 warps per CTA; the kinematics kernels keep one branch accumulator per body whose children do not
    // directly follow it in the joint list (n_slots): an interleaved joint order does not fit
    const size_t kin_smem = (size_t)hb::kin_smem_layout(C.nb, C.n_slots, true).total * sizeof(double) * (hb::KIN_H_THREADS / 32);
    if (kin_smem > 200 * 1024) {
      hb_destroy(h);
      return fail(HB_ERR_UNSUPPORTED,
                  "hb_kino_create: this joint order needs " + std::to_string(C.n_slots) +
                      " branch accumulators (" + std::to_string(kin_smem / 1024) +
                      " KB of shared memory per CTA > 200 KB): list the joints of a limb consecutively");
    }
    hb::SweepSchedule sch = hb::build_sweep_schedule(sweep_topo_of(C), true);
    if (sch.n_rounds <= 0 || sch.n_rounds > 32) sch = hb::build_sweep_schedule(sweep_topo_of(C), false);
    if (sch.n_rounds <= 0 || sch.n_rounds > 32 || sch.n_slots > 62 || sch.n_slots * 12 > 58 + 32 + C.n_slots * 32 * 12) {
      hb_destroy(h);
      return fail(HB_ERR_UNSUPPORTED, "hb_kino_create: no sweep schedule for this tree within the kernel's limits");
    }
    if (e == cudaSuccess) e = upload(&h->d_sched, sch.tasks.data(), sch.tasks.size());
    h->topo.sched = h->d_sched;
    h->topo.n_rounds = sch.n_rounds;
    h->topo.n_pslots = sch.n_slots;
    h->topo.round_seed_mask = sch.seed_mask;
    h->topo.round_heavy_mask = sch.heavy_mask;
    for (int d = 0; d < 32; ++d) h->topo.root_slot[d] = (signed char)sch.root_slot[d];
  }
  if (e == cudaSuccess) e = upload(&h->dev, &C, 1);
  if (e != cudaSuccess) {
    hb_destroy(h);
    return fail(HB_ERR_CUDA, std::string("hb_kino_create: ") + cudaGetErrorString(e));
  }
  *out = h;
  return HB_OK;
}

extern "C" int hb_toy_create(int32_t horizon, int32_t integrator, double dt, hb_handle* out) {
  if (!out || horizon < 2 || (integrator != 0 && integrator != 1)) return fail(HB_ERR_INVALID, "hb_toy_create: bad argument");
  hb_problem_s* h = new hb_problem_s();
  h->kind = KIND_TOY;
  cudaGetDevice(&h->device);
  h->toy = hb::toy_create(horizon, integrator, dt);
  if (!h->toy) {
    delete h;
    return fail(HB_ERR_CUDA, "hb_toy_create: device allocation failed");
  }
  *out = h;
  return HB_OK;
}

extern "C" int hb_destroy(hb_handle h) {
  if (!h) return HB_OK;
  cudaFree(h->d_jc);
  cudaFree(h->d_jk);
  cudaFree(h->d_hci);
  cudaFree(h->d_hc_pt);
  cudaFree(h->d_hc);
  cudaFree(h->d_hk);
  cudaFree(h->d_hk2);
  cudaFree(h->d_knot_maps);
  h->drop_host_graphs();
  cudaFree(h->d_jc_list);
  cudaFree(h->d_jk_list);
  cudaFree(h->d_hc_list);
  cudaFree(h->d_sched);
  cudaFree(h->dev);
  for (auto& kv : h->fpart) cudaFree(kv.second.first);
  for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
  for (int i = 0; i < hb_problem_s::HOST_STREAMS; ++i) {
    cudaFree(h->hslab[i]);
    if (h->hst[i]) cudaStreamDestroy(h->hst[i]);
  }
  cudaFree(h->d_p);
  if (h->aux) cudaStreamDestroy(h->aux);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->toy) hb::toy_destroy(h->toy);
  delete h;
  return HB_OK;
}

extern "C" int hb_dims(hb_handle h, int64_t* n_x, int64_t* n_p, int64_t* m, int64_t* nnz_j, int64_t* nnz_h) {
  if (!h) return fail(HB_ERR_INVALID, "hb_dims: null handle");
  if (h->kind == KIND_TOY) {
    hb::toy_dims(h->toy, n_x, n_p, m, nnz_j, nnz_h);
    return HB_OK;
  }
  if (n_x) *n_x = h->host.n_x;
  if (n_p) *n_p = h->host.n_p;
  if (m) *m = h->host.m;
  if (nnz_j) *nnz_j = h->host.nnz_j;
  if (nnz_h) *nnz_h = h->host.nnz_h;
  return HB_OK;
}

extern "C" int hb_pattern_jac(hb_handle h, int64_t* colind, int64_t* row) {
  if (!h || !colind || !row) return fail(HB_ERR_INVALID, "hb_pattern_jac: null argument");
  if (h->kind != KIND_TOY) {
    if (h->jac_row.empty())
      return fail(HB_ERR_UNSUPPORTED, "hb_pattern_jac: no pattern attached to this handle (hb_kino_attach_tables)");
    std::copy(h->jac_colind.begin(), h->jac_colind.end(), colind);
    std::copy(h->jac_row.begin(), h->jac_row.end(), row);
    return HB_OK;
  }
  hb::toy_pattern_jac(h->toy, colind, row);
  return HB_OK;
}

extern "C" int hb_pattern_hess(hb_handle h, int64_t* colind, int64_t* row) {
  if (!h || !colind || !row) return fail(HB_ERR_INVALID, "hb_pattern_hess: null argument");
  if (h->kind != KIND_TOY) {
    if (h->hess_row.empty())
      return fail(HB_ERR_UNSUPPORTED, "hb_pattern_hess: no pattern attached to this handle (hb_kino_attach_tables)");
    std::copy(h->hess_colind.begin(), h->hess_colind.end(), colind);
    std::copy(h->hess_row.begin(), h->hess_row.end(), row);
    return HB_OK;
  }
  hb::toy_pattern_hess(h->toy, colind, row);
  return HB_OK;
}

extern "C" int hb_eval(hb_handle h, uint32_t mask, const double* x, const double* p, int64_t p_stride,
                       const double* lam_g, const double* sigma, double* f, double* grad_f, double* g,
                       double* jac_vals, double* hess_vals, int64_t batch, void* stream) {
  if (!h) return fail(HB_ERR_INVALID, "hb_eval: null handle");
  if (batch <= 0) return fail(HB_ERR_INVALID, "hb_eval: batch must be positive");
  if (!x || !p) return fail(HB_ERR_INVALID, "hb_eval: x and p are required");
  if ((mask & HB_EVAL_F) && !f) return fail(HB_ERR_INVALID, "hb_eval: f requested but NULL");
  if ((mask & HB_EVAL_GRAD_F) && !grad_f) return fail(HB_ERR_INVALID, "hb_eval: grad_f requested but NULL");
  if ((mask & HB_EVAL_G) && !g) return fail(HB_ERR_INVALID, "hb_eval: g requested but NULL");
  if ((mask & HB_EVAL_JAC_G) && !jac_vals) return fail(HB_ERR_INVALID, "hb_eval: jac_vals requested but NULL");
  if ((mask & HB_EVAL_HESS_L) && (!hess_vals || !lam_g || !sigma))
    return fail(HB_ERR_INVALID, "hb_eval: hess_vals, lam_g and sigma are required for HB_EVAL_HESS_L");
  if (!(mask & 31u)) return fail(HB_ERR_INVALID, "hb_eval: empty mask");
  CHECK_DEVICE(h, "hb_eval");
  cudaStream_t st = (cudaStream_t)stream;
  h->launches = 0;
  if (h->kind == KIND_TOY) {
    const int rc = hb::toy_eval(h->toy, mask, x, p, p_stride, lam_g, sigma, f, grad_f, g, jac_vals, hess_vals, batch, st);
    if (rc < 0) return fail(HB_ERR_CUDA, "hb_eval(toy): launch failed");
    h->launches = rc;
    return HB_OK;
  }
  const hb::KinoConst& C = h->host;
  if (p_stride != 0 && p_stride != C.n_p) return fail(HB_ERR_INVALID, "hb_eval: p_stride must be 0 or n_p");
  double* d_fpart = nullptr;
  if (mask & HB_EVAL_F) {
    const int64_t need = batch * C.N * 2;
    auto& slot = h->fpart[st];
    if (need > slot.second) {
      cudaFree(slot.first);
      slot.first = nullptr;
      slot.second = 0;
      CUDA_TRY(cudaMalloc(&slot.first, need * sizeof(double)));
      slot.second = need;
    }
    d_fpart = slot.first;
  }
  const int warps_per_block = 4;
  const long total_warps = (long)batch * C.N;
  const unsigned grid = (unsigned)((total_warps + warps_per_block - 1) / warps_per_block);
  // The "Hessian" variant of the kinematics kernel also serves Jacobian / gradient requests: its forward-mode
  // Jacobian (closed-form tangents, no sweep: 0.42 ms) beats the row-per-lane adjoint sweep of the lean
  // variant (0.62 ms), which is left with f and g.  hb_set_option(HB_OPT_JAC_ADJOINT) selects the adjoint sweep:
  // an independent algorithm for the same numbers (tests).
  const bool with_hess = (mask & HB_EVAL_HESS_L) != 0 ||
                         (!h->jac_adjoint && (mask & (HB_EVAL_JAC_G | HB_EVAL_GRAD_F)) != 0);
  auto mark = [&]() -> int {
    if (!h->prof) return HB_OK;
    cudaEvent_t e;
    CUDA_TRY(cudaEventCreate(&e));
    h->prof_ev.push_back(e);
    CUDA_TRY(cudaEventRecord(e, st));
    return HB_OK;
  };
  if (mark() != HB_OK) return HB_ERR_CUDA;
  // fewer warps than one kernel's residency on the whole GPU (8 per SM for the kinematics kernel): run the contact
  // kernel beside the kinematics kernel.  Not while profiling (the per-kernel events assume one stream).
  int dev_now = 0;
  CUDA_TRY(cudaGetDevice(&dev_now));
  CUDA_TRY(ensure_kernel_attributes(dev_now));
  const bool overlap = !h->prof && C.kind == 0 && total_warps <= 8L * device_sms[dev_now];
  cudaStream_t st_contact = st;
  if (overlap) {
    if (!h->aux) {
      CUDA_TRY(cudaStreamCreateWithFlags(&h->aux, cudaStreamNonBlocking));
      CUDA_TRY(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventRecord(h->ev_fork, st));         // inputs on `st` are complete before the fork
    CUDA_TRY(cudaStreamWaitEvent(h->aux, h->ev_fork, 0));
    st_contact = h->aux;
  }
  {
    const size_t smem = (size_t)(C.kind == 1 ? hb::pose_contact_smem_layout(C.n_hc) : hb::kino_contact_smem_layout(C.n_hc)).total *
                        sizeof(double) * warps_per_block;
    // the shared block holds the kernel's n_hc Hessian accumulators (191 planar, 255 on the smooth steps)
    if (C.kind == 1) {
      const auto kernel = pose_contact_kernel_for(C.terrain);
      kernel<<<grid, 32 * warps_per_block, smem, st>>>(h->dev, mask, x, p, (long)p_stride, lam_g, sigma, d_fpart, grad_f, g,
                                                       jac_vals, hess_vals, (long)batch);
    } else {
      const auto kernel = kino_contact_kernel_for(C.terrain);
      kernel<<<grid, 32 * warps_per_block, smem, st_contact>>>(h->topo, h->dev, mask, x, p, (long)p_stride, lam_g, sigma,
                                                               d_fpart, grad_f, g, jac_vals, hess_vals, (long)batch);
    }
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    if (overlap) CUDA_TRY(cudaEventRecord(h->ev_join, h->aux));
  }
  if (mark() != HB_OK) return HB_ERR_CUDA;
  {
    // the Hessian variant has its own CTA shape (KIN_H_THREADS, kino_kin.cu): occupancy tuning
    const int kin_warps = with_hess ? hb::KIN_H_THREADS / 32 : warps_per_block;
    const unsigned kin_grid = (unsigned)((total_warps + kin_warps - 1) / kin_warps);
    const size_t smem = (size_t)hb::kin_smem_layout(C.nb, C.n_slots, with_hess).total * sizeof(double) * kin_warps;
    if (with_hess)
      hb::kino_kin_kernel<true><<<kin_grid, 32 * kin_warps, smem, st>>>(h->topo, h->dev, mask, x, p, (long)p_stride,
                                                                         lam_g, sigma, d_fpart, grad_f, g, jac_vals,
                                                                         hess_vals, (long)batch);
    else
      hb::kino_kin_kernel<false><<<grid, 32 * warps_per_block, smem, st>>>(h->topo, h->dev, mask, x, p, (long)p_stride,
                                                                          lam_g, sigma, d_fpart, grad_f, g, jac_vals,
                                                                          hess_vals, (long)batch);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  // join: everything after this call on `st` (the f reduction, the caller's copies) sees both kernels' outputs
  if (overlap) CUDA_TRY(cudaStreamWaitEvent(st, h->ev_join, 0));
  if (mark() != HB_OK) return HB_ERR_CUDA;
  if (mask & HB_EVAL_F) {
    reduce_f_kernel<<<(unsigned)((batch + 127) / 128), 128, 0, st>>>(d_fpart, f, 2 * C.N, (long)batch);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
  }
  if (mark() != HB_OK) return HB_ERR_CUDA;
  return HB_OK;
}

// ---------------------------------------------------------------------------------------------
// host-buffer pipeline
extern "C" int hb_host_set_parameters(hb_handle h, const double* p, int64_t p_stride, int64_t batch) {
  if (!h || !p) return fail(HB_ERR_INVALID, "hb_host_set_parameters: null argument");
  int64_t n_p = 0;
  hb_dims(h, nullptr, &n_p, nullptr, nullptr, nullptr);
  if (p_stride != 0 && p_stride != n_p) return fail(HB_ERR_INVALID, "hb_host_set_parameters: p_stride must be 0 or n_p");
  if (p_stride != 0 && batch <= 0) return fail(HB_ERR_INVALID, "hb_host_set_parameters: batch must be positive");
  const int64_t need = p_stride == 0 ? n_p : n_p * batch;
  if (need > h->p_cap || p_stride != h->p_stride) h->drop_host_graphs();  // the graphs hold d_p and the stride
  if (need > h->p_cap) {
    cudaFree(h->d_p);
    h->d_p = nullptr;
    h->p_cap = 0;
    CUDA_TRY(cudaMalloc(&h->d_p, (size_t)need * sizeof(double)));
    h->p_cap = need;
  }
  CUDA_TRY(cudaMemcpy(h->d_p, p, (size_t)need * sizeof(double), cudaMemcpyHostToDevice));
  h->p_stride = p_stride;
  h->p_batch = p_stride == 0 ? 0 : batch;
  return HB_OK;
}

extern "C" int hb_eval_host(hb_handle h, uint32_t mask, const double* x, const double* lam_g, const double* sigma,
                            double* f, double* grad_f, double* g, double* jac_vals, double* hess_vals,
                            int64_t batch) {
  if (!h) return fail(HB_ERR_INVALID, "hb_eval_host: null handle");
  if (batch <= 0) return fail(HB_ERR_INVALID, "hb_eval_host: batch must be positive");
  if (!x) return fail(HB_ERR_INVALID, "hb_eval_host: x is required");
  if (h->p_stride < 0) return fail(HB_ERR_INVALID, "hb_eval_host: call hb_host_set_parameters first");
  if (h->p_stride != 0 && batch > h->p_batch)
    return fail(HB_ERR_INVALID, "hb_eval_host: batch exceeds the batch the parameters were set for");
  if ((mask & HB_EVAL_F) && !f) return fail(HB_ERR_INVALID, "hb_eval_host: f requested but NULL");
  if ((mask & HB_EVAL_GRAD_F) && !grad_f) return fail(HB_ERR_INVALID, "hb_eval_host: grad_f requested but NULL");
  if ((mask & HB_EVAL_G) && !g) return fail(HB_ERR_INVALID, "hb_eval_host: g requested but NULL");
  if ((mask & HB_EVAL_JAC_G) && !jac_vals) return fail(HB_ERR_INVALID, "hb_eval_host: jac_vals requested but NULL");
  const bool need_l = (mask & HB_EVAL_HESS_L) != 0;
  if (need_l && (!hess_vals || !lam_g || !sigma))
    return fail(HB_ERR_INVALID, "hb_eval_host: hess_vals, lam_g and sigma are required for HB_EVAL_HESS_L");
  if (!(mask & 31u)) return fail(HB_ERR_INVALID, "hb_eval_host: empty mask");
  int64_t n_x = 0, n_p = 0, m = 0, nnz_j = 0, nnz_h = 0;
  hb_dims(h, &n_x, &n_p, &m, &nnz_j, &nnz_h);
  const int S = hb_problem_s::HOST_STREAMS;
  const int64_t chunk = batch < hb_problem_s::HOST_CHUNK ? batch : (int64_t)hb_problem_s::HOST_CHUNK;
  // slab of one stream: x | lam | sigma | f | grad_f | g | jac | hess, each for `chunk` instances
  const int64_t per_inst = n_x + m + 1 + 1 + n_x + m + nnz_j + nnz_h;
  if (chunk > h->hslab_chunk) {
    h->drop_host_graphs();
    for (int i = 0; i < S; ++i) {
      cudaFree(h->hslab[i]);
      h->hslab[i] = nullptr;
    }
    h->hslab_chunk = 0;
    for (int i = 0; i < S; ++i) {
      if (!h->hst[i]) CUDA_TRY(cudaStreamCreateWithFlags(&h->hst[i], cudaStreamNonBlocking));
      CUDA_TRY(cudaMalloc(&h->hslab[i], (size_t)(per_inst * chunk) * sizeof(double)));
    }
    h->hslab_chunk = chunk;
  }
  const int64_t cap = h->hslab_chunk;
  int launches = 0;
  int64_t h2d = 0, d2h = 0;
  const int64_t n_chunks = (batch + chunk - 1) / chunk;
  auto enqueue = [&]() -> int {
    launches = 0;
    h2d = d2h = 0;
    for (int64_t ci = 0; ci < n_chunks; ++ci) {
      const int64_t lo = ci * chunk, n = (lo + chunk <= batch ? chunk : batch - lo);
      const int si = (int)(ci % S);
      cudaStream_t st = h->hst[si];
      double* d_x = h->hslab[si];
      double* d_lam = d_x + cap * n_x;
      double* d_sig = d_lam + cap * m;
      double* d_f = d_sig + cap;
      double* d_gf = d_f + cap;
      double* d_g = d_gf + cap * n_x;
      double* d_j = d_g + cap * m;
      double* d_h = d_j + cap * nnz_j;
      auto up = [&](double* dst, const double* src, int64_t count) {
        h2d += count * 8;
        return cudaMemcpyAsync(dst, src, (size_t)count * 8, cudaMemcpyHostToDevice, st);
      };
      auto down = [&](double* dst, const double* src, int64_t count) {
        d2h += count * 8;
        return cudaMemcpyAsync(dst, src, (size_t)count * 8, cudaMemcpyDeviceToHost, st);
      };
      // copies whose source and destination ranges are adjacent on BOTH sides are merged into one transfer: a caller
      // that keeps x | lam_g | sigma and f | grad_f | g | jac | hess in one pinned block each (HostPipeline does) pays
      // one copy per direction instead of up to eight -- at one instance per call the fixed cost of a copy (~8 us)
      // is what the call consists of
      struct Span {
        double* dst;
        const double* src;
        int64_t count;
      };
      auto run = [&](std::vector<Span>& v, bool to_device) -> cudaError_t {
        size_t i = 0;
        while (i < v.size()) {
          Span cur = v[i++];
          while (i < v.size() && v[i].dst == cur.dst + cur.count && v[i].src == cur.src + cur.count) cur.count += v[i++].count;
          const cudaError_t e = to_device ? up(cur.dst, cur.src, cur.count) : down(cur.dst, cur.src, cur.count);
          if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
      };
      std::vector<Span> in = {{d_x, x + lo * n_x, n * n_x}};
      if (need_l) {
        in.push_back({d_lam, lam_g + lo * m, n * m});
        in.push_back({d_sig, sigma + lo, n});
      }
      CUDA_TRY(run(in, true));
      const double* pc = h->p_stride == 0 ? h->d_p : h->d_p + lo * n_p;
      const int rc = hb_eval(h, mask, d_x, pc, h->p_stride, need_l ? d_lam : nullptr, need_l ? d_sig : nullptr, d_f, d_gf,
                             d_g, d_j, d_h, n, st);
      if (rc != HB_OK) return rc;
      launches += h->launches;
      std::vector<Span> out;
      if (mask & HB_EVAL_F) out.push_back({f + lo, d_f, n});
      if (mask & HB_EVAL_GRAD_F) out.push_back({grad_f + lo * n_x, d_gf, n * n_x});
      if (mask & HB_EVAL_G) out.push_back({g + lo * m, d_g, n * m});
      if (mask & HB_EVAL_JAC_G) out.push_back({jac_vals + lo * nnz_j, d_j, n * nnz_j});
      if (need_l) out.push_back({hess_vals + lo * nnz_h, d_h, n * nnz_h});
      CUDA_TRY(run(out, false));
    }
    return HB_OK;
  };
  // ---- graph replay of repeating single-chunk calls
  hb_problem_s::HostGraph* hg = nullptr;
  if (n_chunks == 1 && !h->prof) {
    const void* key[8] = {x, lam_g, sigma, f, grad_f, g, jac_vals, hess_vals};
    for (auto& e : h->hgraphs)
      if (e.mask == mask && e.batch == batch && std::equal(key, key + 8, e.ptr)) hg = &e;
    if (!hg && h->hgraphs.size() < 8) {
      h->hgraphs.emplace_back();
      hg = &h->hgraphs.back();
      hg->mask = mask;
      hg->batch = batch;
      std::copy(key, key + 8, hg->ptr);
      for (const void* q : key) {  // pageable buffers make a copy synchronous: not for a graph
        if (!q) continue;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, q) != cudaSuccess || at.type != cudaMemoryTypeHost) hg->unusable = true;
      }
      cudaGetLastError();
    }
    if (hg && hg->unusable) hg = nullptr;
  }
  if (hg && hg->exec) {
    CUDA_TRY(cudaGraphLaunch(hg->exec, h->hst[0]));
    CUDA_TRY(cudaStreamSynchronize(h->hst[0]));
    h->launches = hg->launches;
    h->h2d_bytes = hg->h2d;
    h->d2h_bytes = hg->d2h;
    return HB_OK;
  }
  if (hg && hg->seen++ >= 1) {  // second call with this key: everything it needs exists by now, capture it
    cudaGraph_t graph = nullptr;
    bool ok = cudaStreamBeginCapture(h->hst[0], cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (ok) {
      const int rc = enqueue();
      const cudaError_t ee = cudaStreamEndCapture(h->hst[0], &graph);  // always: the stream must leave capture mode
      ok = rc == HB_OK && ee == cudaSuccess && graph != nullptr;
    }
    if (ok) ok = cudaGraphInstantiate(&hg->exec, graph, 0) == cudaSuccess;
    if (graph) cudaGraphDestroy(graph);
    if (ok) {
      hg->launches = launches;
      hg->h2d = h2d;
      hg->d2h = d2h;
      CUDA_TRY(cudaGraphLaunch(hg->exec, h->hst[0]));
      CUDA_TRY(cudaStreamSynchronize(h->hst[0]));
      h->launches = launches;
      h->h2d_bytes = h2d;
      h->d2h_bytes = d2h;
      return HB_OK;
    }
    cudaGetLastError();  // not capturable on this driver / configuration: run as before, and do not try again
    hg->exec = nullptr;
    hg->unusable = true;
  }
  {
    const int rc = enqueue();
    if (rc != HB_OK) return rc;
  }
  for (int i = 0; i < S; ++i) CUDA_TRY(cudaStreamSynchronize(h->hst[i]));
  h->launches = launches;
  h->h2d_bytes = h2d;
  h->d2h_bytes = d2h;
  return HB_OK;
}

extern "C" int hb_host_last_traffic(hb_handle h, int64_t* h2d_bytes, int64_t* d2h_bytes) {
  if (!h) return fail(HB_ERR_INVALID, "hb_host_last_traffic: null handle");
  if (h2d_bytes) *h2d_bytes = h->h2d_bytes;
  if (d2h_bytes) *d2h_bytes = h->d2h_bytes;
  return HB_OK;
}

extern "C" int hb_host_alloc(void** ptr, int64_t bytes) {
  if (!ptr || bytes <= 0) return fail(HB_ERR_INVALID, "hb_host_alloc: bad argument");
  CUDA_TRY(cudaHostAlloc(ptr, (size_t)bytes, cudaHostAllocDefault));
  return HB_OK;
}

extern "C" int hb_host_free(void* ptr) {
  if (ptr) CUDA_TRY(cudaFreeHost(ptr));
  return HB_OK;
}

// ---------------------------------------------------------------------------------------------
// batched LU of the KKT stage blocks (lu.cu)

// The kernel variant both launch paths use for (n, batch, nrhs) on a device with `sms` SMs:
//   rpt, mb   lu_factor_kernel<RPT, MB>: panel rows per thread (n <= RPT * LU_THREADS) and CTAs per SM the register
//             allocation is tuned for -- the 128-register MB = 2 build when the batch exceeds one CTA per SM and two
//             CTAs fit an SM's shared memory
//   ct        lu_solve_staged_kernel<CT>: 8-column tiles of right-hand sides per CTA, 4 or 3
//   chunks    column chunks (CTAs) per matrix of the solve
struct LuPlan {
  int rpt, mb, ct, chunks;
};
static LuPlan lu_plan(int64_t n, int64_t batch, int64_t nrhs, int sms) {
  LuPlan p{};
  const size_t smem = hb::lu_factor_smem((int)n);
  const bool two = batch > sms && 2 * (smem + 2048) <= 227 * 1024;
  p.rpt = n <= hb::LU_THREADS ? 1 : n <= 2 * hb::LU_THREADS ? 2 : 3;
  p.mb = two && p.rpt < 3 ? 2 : 1;
  // staged substitution (lu.cu): 32 or 24 right-hand sides per CTA while two CTAs fit an SM, else on one CTA per SM
  // (lu_staged_smem(768, 3) = 196 112 B fits one)
  const size_t two_per_sm = (233472 / 2) - 1024 - 2560, one_per_sm = 232448 - 1024 - 2560;  // minus the static arrays
  if (hb::lu_staged_smem((int)n, 4) <= two_per_sm) p.ct = 4;
  else if (hb::lu_staged_smem((int)n, 3) <= two_per_sm) p.ct = 3;
  else if (hb::lu_staged_smem((int)n, 4) <= one_per_sm) p.ct = 4;
  else p.ct = 3;
  p.chunks = (int)((nrhs + 8 * p.ct - 1) / (8 * p.ct));
  return p;
}

extern "C" int hb_debug_lu_plan(int64_t n, int64_t batch, int64_t nrhs, int32_t sms, int32_t* out) {
  if (!out || n <= 0 || n > 768 || batch <= 0 || nrhs <= 0 || sms <= 0)
    return fail(HB_ERR_INVALID, "hb_debug_lu_plan: need 0 < n <= 768, batch > 0, nrhs > 0, sms > 0, out");
  const LuPlan p = lu_plan(n, batch, nrhs, sms);
  out[0] = p.rpt;
  out[1] = p.mb;
  out[2] = p.ct;
  out[3] = p.chunks;
  return HB_OK;
}

namespace hb {
// one thread per point: the production surface and frame jets, unchanged, written out for the tests
template <int TERRAIN>
__global__ void debug_terrain_kernel(const double* __restrict__ tp, int n_steps, const double* __restrict__ pts, long n,
                                     double* __restrict__ out) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double* t = tp + 10 * (TERRAIN == 1 ? 1 : n_steps) * i;
  const double x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
  double* o = out + HB_SMOOTH_TERRAIN_OUT * i;
  const BJ<4> T = terrain_surface<TERRAIN>(t, n_steps, x, y);
  for (int k = 0; k < BJ<4>::SIZE; ++k) o[k] = T.c[k];
  TFrame F;
  terrain_frame<TERRAIN>(t, n_steps, x, y, z, F);
  const TJ* f[18] = {&F.h, &F.gx, &F.gy, &F.n[0], &F.n[1], &F.n[2], &F.xh[0], &F.xh[1], &F.xh[2],
                     &F.yh[0], &F.yh[1], &F.yh[2], &F.Dn[0][0], &F.Dn[0][1], &F.Dn[1][0], &F.Dn[1][1],
                     &F.Dn[2][0], &F.Dn[2][1]};
  for (int a = 0; a < 18; ++a)
    for (int k = 0; k < 10; ++k) o[BJ<4>::SIZE + 10 * a + k] = f[a]->c[k];
}
static_assert(BJ<4>::SIZE + 18 * 10 == HB_SMOOTH_TERRAIN_OUT, "hb_debug_smooth_terrain output layout");
}  // namespace hb

extern "C" int hb_debug_smooth_terrain(const double* tp, const double* pts, int64_t n, double* out, void* stream) {
  if (!tp || !pts || !out || n <= 0) return fail(HB_ERR_INVALID, "hb_debug_smooth_terrain: null argument or n <= 0");
  hb::debug_terrain_kernel<1><<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(tp, 0, pts, (long)n, out);
  CUDA_TRY(cudaGetLastError());
  return HB_OK;
}

extern "C" int hb_debug_tilted_terrain(const double* tp, int32_t n_steps, const double* pts, int64_t n, double* out,
                                       void* stream) {
  if (!tp || !pts || !out || n <= 0 || n_steps <= 0)
    return fail(HB_ERR_INVALID, "hb_debug_tilted_terrain: null argument, n <= 0 or n_steps <= 0");
  hb::debug_terrain_kernel<2><<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(tp, n_steps, pts, (long)n,
                                                                                            out);
  CUDA_TRY(cudaGetLastError());
  return HB_OK;
}

extern "C" int hb_lu_factor_batched(double* A, int32_t* piv, int32_t* info, int64_t n, int64_t batch, void* stream) {
  if (!A || !piv || !info) return fail(HB_ERR_INVALID, "hb_lu_factor_batched: null argument");
  if (n <= 0 || n > 768 || batch <= 0) return fail(HB_ERR_INVALID, "hb_lu_factor_batched: need 0 < n <= 768, batch > 0");
  const size_t smem = hb::lu_factor_smem((int)n);
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(ensure_kernel_attributes(dev));
  const LuPlan p = lu_plan(n, batch, 1, device_sms[dev]);  // (the solve fields are not used here)
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)batch;
  if (p.rpt == 1 && p.mb == 2) hb::lu_factor_kernel<1, 2><<<grid, hb::LU_THREADS, smem, st>>>(A, piv, info, (int)n);
  else if (p.rpt == 1) hb::lu_factor_kernel<1, 1><<<grid, hb::LU_THREADS, smem, st>>>(A, piv, info, (int)n);
  else if (p.rpt == 2 && p.mb == 2) hb::lu_factor_kernel<2, 2><<<grid, hb::LU_THREADS, smem, st>>>(A, piv, info, (int)n);
  else if (p.rpt == 2) hb::lu_factor_kernel<2, 1><<<grid, hb::LU_THREADS, smem, st>>>(A, piv, info, (int)n);
  else hb::lu_factor_kernel<3, 1><<<grid, hb::LU_THREADS, smem, st>>>(A, piv, info, (int)n);
  CUDA_TRY(cudaGetLastError());
  return HB_OK;
}

extern "C" int hb_lu_solve_batched(const double* LU, const int32_t* piv, double* Bm, int64_t n, int64_t nrhs,
                                   int64_t batch, void* stream) {
  if (!LU || !piv || !Bm) return fail(HB_ERR_INVALID, "hb_lu_solve_batched: null argument");
  if (n <= 0 || n > 768 || batch <= 0 || nrhs <= 0)
    return fail(HB_ERR_INVALID, "hb_lu_solve_batched: need 0 < n <= 768, batch > 0, nrhs > 0");
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(ensure_kernel_attributes(dev));
  const LuPlan p = lu_plan(n, batch, nrhs, device_sms[dev]);
  const size_t smem = hb::lu_staged_smem((int)n, p.ct);
  const int n_chunks = p.chunks;
  const unsigned grid = (unsigned)(batch * n_chunks);
  if (p.ct == 4) hb::lu_solve_staged_kernel<4><<<grid, hb::LU_THREADS, smem, (cudaStream_t)stream>>>(LU, piv, Bm, (int)n, (int)nrhs, n_chunks);
  else hb::lu_solve_staged_kernel<3><<<grid, hb::LU_THREADS, smem, (cudaStream_t)stream>>>(LU, piv, Bm, (int)n, (int)nrhs, n_chunks);
  CUDA_TRY(cudaGetLastError());
  return HB_OK;
}

extern "C" int hb_ccs_group_mul(const double* vals, const int32_t* ptr, const int32_t* entry, const int32_t* idx,
                                const double* w, const double* x, double* y, int64_t n_out, int64_t n_in, int64_t nnz,
                                int64_t batch, void* stream) {
  if (!vals || !ptr || !entry || !idx || !x || !y) return fail(HB_ERR_INVALID, "hb_ccs_group_mul: null argument");
  if (n_out <= 0 || n_in <= 0 || nnz < 0 || batch <= 0) return fail(HB_ERR_INVALID, "hb_ccs_group_mul: bad sizes");
  const long total = (long)batch * n_out;
  hb::ccs_group_mul_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      vals, ptr, entry, idx, w, x, y, (int)n_out, (int)n_in, (long)nnz, (long)batch);
  CUDA_TRY(cudaGetLastError());
  return HB_OK;
}

extern "C" int hb_kkt_assemble_stage(const int32_t* hdr, const int32_t* tab, const double* hess_vals, int64_t nnz_h,
                                     const double* jac_vals, int64_t nnz_j, const double* sigma_I, int64_t m_I,
                                     const double* delta, double delta_c, const double* RX, int64_t n_x, const double* RE,
                                     int64_t m_E, const double* prev_sol, double* D, double* rhs, int64_t batch,
                                     void* stream) {
  if (!hdr || !tab || !hess_vals || !jac_vals || !delta || !RX || !RE || !D || !rhs)
    return fail(HB_ERR_INVALID, "hb_kkt_assemble_stage: null argument");
  hb::KktStage S;
  S.nb = hdr[hb::KS_NB];
  S.nx = hdr[hb::KS_NX];
  S.nv = hdr[hb::KS_NV];
  S.ne = hdr[hb::KS_NE];
  S.R = hdr[hb::KS_R];
  S.n_cpl = hdr[hb::KS_NCPL];
  S.n_cpl_next = hdr[hb::KS_NCPL_NEXT];
  S.n_direct = hdr[hb::KS_NDIRECT];
  S.n_targets = hdr[hb::KS_NTARGETS];
  S.n_an = hdr[hb::KS_NAN];
  S.nb_prev = hdr[hb::KS_NB_PREV];
  const int n_contrib = hdr[hb::KS_NCONTRIB], n_a = hdr[hb::KS_NA];
  if (batch <= 0 || S.nb <= 0 || S.nx <= 0 || S.nx > S.nb || S.nv < 0 || S.nv > S.nx || S.ne < 0 || S.nx + S.ne > S.nb ||
      S.R <= 0 || S.n_cpl < 0 || S.n_cpl_next < 0 || S.n_direct < 0 || S.n_targets < 0 || n_contrib < 0 || n_a < 0 ||
      S.n_an < 0 || (S.n_cpl > 0 && S.nb_prev <= 0))
    return fail(HB_ERR_INVALID, "hb_kkt_assemble_stage: inconsistent stage header");
  if (S.n_targets > 0 && (!sigma_I || m_I <= 0)) return fail(HB_ERR_INVALID, "hb_kkt_assemble_stage: sigma_I missing");
  if (S.n_cpl > 0 && !prev_sol) return fail(HB_ERR_INVALID, "hb_kkt_assemble_stage: the previous stage's solution is missing");
  const int32_t* t = tab;  // tables in header order
  S.direct_val = t, t += S.n_direct;
  S.direct_pos = t, t += S.n_direct;
  S.tgt_pos = t, t += S.n_targets;
  S.tgt_ptr = t, t += S.n_targets + 1;
  S.tgt_sig = t, t += n_contrib;
  S.tgt_e1 = t, t += n_contrib;
  S.tgt_e2 = t, t += n_contrib;
  S.var = t, t += S.nv;
  S.eq = t, t += S.ne;
  S.cpl = t, t += S.n_cpl;
  S.a_ptr = t, t += S.n_cpl + 1;
  S.a_val = t, t += n_a;
  S.a_col = t, t += n_a;
  S.an_val = t, t += S.n_an;
  S.an_row = t, t += S.n_an;
  S.an_col = t;
  hb::kkt_assemble_kernel<<<(unsigned)batch, 512, 0, (cudaStream_t)stream>>>(S, hess_vals, (long)nnz_h, jac_vals, (long)nnz_j,
                                                                           sigma_I, (long)m_I, delta, delta_c, RX, (long)n_x,
                                                                           RE, (long)m_E, prev_sol, D, rhs);
  CUDA_TRY(cudaGetLastError());
  return HB_OK;
}

extern "C" int hb_interpolate_humanoid_states(int64_t batch, int64_t n_points, int64_t n_joints, const double* initial,
                                              const double* final_, const int32_t* schedule,
                                              const double* phases_left, int64_t n_phases_left, int64_t stride_left,
                                              const double* phases_right, int64_t n_phases_right,
                                              int64_t stride_right, double* states, double* x, int64_t x_stride,
                                              int64_t knot0, void* stream) {
  if (!initial || !final_ || !schedule || !phases_left || !phases_right)
    return fail(HB_ERR_INVALID, "hb_interpolate_humanoid_states: null argument");
  if (!states && !x) return fail(HB_ERR_INVALID, "hb_interpolate_humanoid_states: no output requested");
  if (batch <= 0 || n_points <= 0 || n_points > (1 << 20) || n_joints < 0 || n_phases_left <= 0 || n_phases_right <= 0)
    return fail(HB_ERR_INVALID, "hb_interpolate_humanoid_states: need batch > 0, 0 < n_points <= 2^20, phases > 0");
  if (x && (n_joints != 23 || knot0 < 0 || x_stride < (knot0 + n_points) * hb::IZ_N))
    return fail(HB_ERR_INVALID,
                "hb_interpolate_humanoid_states: the guess layout has 23 joints and 189 variables per knot; "
                "x_stride must cover knots knot0 .. knot0 + n_points - 1");
  const long total = (long)batch * n_points, per_cta = hb::IW_ITEMS * hb::IW_WARPS;
  const size_t smem = (size_t)per_cta * (82 + n_joints) * sizeof(double);
  if (smem > 48 * 1024) return fail(HB_ERR_INVALID, "hb_interpolate_humanoid_states: too many joints (n_joints <= 430)");
  hb::interp_states_kernel<<<(unsigned)((total + per_cta - 1) / per_cta), 32 * hb::IW_WARPS, smem, (cudaStream_t)stream>>>(
      total, (int)n_points, (int)n_joints, initial, final_, schedule, phases_left, (long)stride_left, phases_right,
      (long)stride_right, states, x, (long)x_stride, (int)knot0);
  CUDA_TRY(cudaGetLastError());
  return HB_OK;
}

extern "C" int hb_profile_enable(hb_handle h, int enable) {
  if (!h) return fail(HB_ERR_INVALID, "hb_profile_enable: null handle");
  for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
  h->prof_ev.clear();
  h->prof = enable != 0;
  return HB_OK;
}

extern "C" int hb_profile_read(hb_handle h, double* ms, int64_t* n_evals) {
  if (!h || !ms || !n_evals) return fail(HB_ERR_INVALID, "hb_profile_read: null argument");
  ms[0] = ms[1] = ms[2] = 0.0;
  const size_t n = h->prof_ev.size() / 4;
  if (n) CUDA_TRY(cudaEventSynchronize(h->prof_ev[4 * n - 1]));
  for (size_t i = 0; i < n; ++i)
    for (int j = 0; j < 3; ++j) {
      float t = 0.f;
      CUDA_TRY(cudaEventElapsedTime(&t, h->prof_ev[4 * i + j], h->prof_ev[4 * i + j + 1]));
      ms[j] += t;
    }
  *n_evals = (int64_t)n;
  return HB_OK;
}

extern "C" int hb_last_launch_count(hb_handle h) { return h ? h->launches : 0; }

extern "C" int hb_set_option(hb_handle h, int32_t option, int32_t value) {
  if (!h) return fail(HB_ERR_INVALID, "hb_set_option: null handle");
  if (option == HB_OPT_JAC_ADJOINT) {
    h->jac_adjoint = value != 0;
    return HB_OK;
  }
  return fail(HB_ERR_INVALID, "hb_set_option: unknown option");
}

extern "C" const char* hb_last_error(void) { return g_err.c_str(); }

// ---------------------------------------------------------------------------------------------
// fp64 FMA throughput probe: 8 independent FMA chains per thread, enough CTAs to fill the chip.
__global__ void __launch_bounds__(256) fp64_probe_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-3, a1 = a0 + 1.0, a2 = a0 + 2.0, a3 = a0 + 3.0, a4 = a0 + 4.0, a5 = a0 + 5.0,
         a6 = a0 + 6.0, a7 = a0 + 7.0;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c);
    a1 = fma(a1, m, c);
    a2 = fma(a2, m, c);
    a3 = fma(a3, m, c);
    a4 = fma(a4, m, c);
    a5 = fma(a5, m, c);
    a6 = fma(a6, m, c);
    a7 = fma(a7, m, c);
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

extern "C" int hb_probe_fp64_tflops(double* tflops, void* stream) {
  if (!tflops) return fail(HB_ERR_INVALID, "hb_probe_fp64_tflops: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0, sms = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int blocks = sms * 8, threads = 256, iters = 1 << 14;
  double* buf = nullptr;
  CUDA_TRY(cudaMalloc(&buf, (size_t)blocks * threads * sizeof(double)));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CUDA_TRY(cudaEventRecord(e0, st));
    fp64_probe_kernel<<<blocks, threads, 0, st>>>(buf, iters);
    CUDA_TRY(cudaEventRecord(e1, st));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
    const double tf = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(buf);
  *tflops = best;
  return HB_OK;
}

// ---------------------------------------------------------------------------------------------
// tables for callers without the Python layout compiler, and (de)serialisation of a handle
extern "C" int hb_kino_attach_tables(hb_handle h, const int64_t* jac_colind, const int64_t* jac_row,
                                     const int64_t* hess_colind, const int64_t* hess_row, const int32_t* lb_idx,
                                     const double* lb_val, const int32_t* ub_idx, const double* ub_val) {
  if (!h || h->kind != KIND_KINO) return fail(HB_ERR_INVALID, "hb_kino_attach_tables: kinodynamic / pose-finder handle required");
  if (!jac_colind || !jac_row || !hess_colind || !hess_row || !lb_idx || !lb_val || !ub_idx || !ub_val)
    return fail(HB_ERR_INVALID, "hb_kino_attach_tables: null argument");
  const hb::KinoConst& C = h->host;
  if (jac_colind[C.n_x] != C.nnz_j || hess_colind[C.n_x] != C.nnz_h)
    return fail(HB_ERR_INVALID, "hb_kino_attach_tables: colind does not end at nnz");
  for (int r = 0; r < C.m; ++r)
    if (lb_idx[r] >= C.n_p || ub_idx[r] >= C.n_p) return fail(HB_ERR_INVALID, "hb_kino_attach_tables: parameter index out of range");
  h->jac_colind.assign(jac_colind, jac_colind + C.n_x + 1);
  h->jac_row.assign(jac_row, jac_row + C.nnz_j);
  h->hess_colind.assign(hess_colind, hess_colind + C.n_x + 1);
  h->hess_row.assign(hess_row, hess_row + C.nnz_h);
  h->lb_idx.assign(lb_idx, lb_idx + C.m);
  h->lb_val.assign(lb_val, lb_val + C.m);
  h->ub_idx.assign(ub_idx, ub_idx + C.m);
  h->ub_val.assign(ub_val, ub_val + C.m);
  return HB_OK;
}

extern "C" int hb_bounds(hb_handle h, const double* p, double* lbg, double* ubg) {
  if (!h || !p || !lbg || !ubg) return fail(HB_ERR_INVALID, "hb_bounds: null argument");
  if (h->kind != KIND_KINO || h->lb_idx.empty())
    return fail(HB_ERR_UNSUPPORTED, "hb_bounds: no bound table attached to this handle (hb_kino_attach_tables)");
  for (int r = 0; r < h->host.m; ++r) {
    lbg[r] = h->lb_idx[r] >= 0 ? h->lb_val[r] * p[h->lb_idx[r]] : h->lb_val[r];
    ubg[r] = h->ub_idx[r] >= 0 ? h->ub_val[r] * p[h->ub_idx[r]] : h->ub_val[r];
  }
  return HB_OK;
}

namespace {
const uint64_t HB_BLOB_MAGIC = 0x3130424f4c424248ull;  // "HBBLOB01"
template <class T>
bool put_vec(FILE* f, const std::vector<T>& v) {
  const uint64_t n = v.size();
  return fwrite(&n, sizeof(n), 1, f) == 1 && (n == 0 || fwrite(v.data(), sizeof(T), n, f) == n);
}
template <class T>
bool get_vec(FILE* f, std::vector<T>& v) {
  uint64_t n = 0;
  if (fread(&n, sizeof(n), 1, f) != 1 || n > (1ull << 31)) return false;
  v.resize(n);
  return n == 0 || fread(v.data(), sizeof(T), n, f) == n;
}
}  // namespace

extern "C" int hb_save(hb_handle h, const char* path) {
  if (!h || !path) return fail(HB_ERR_INVALID, "hb_save: null argument");
  if (h->kind != KIND_KINO) return fail(HB_ERR_UNSUPPORTED, "hb_save: kinodynamic / pose-finder handles (the toy OCP has hb_toy_create)");
  FILE* f = fopen(path, "wb");
  if (!f) return fail(HB_ERR_INVALID, std::string("hb_save: cannot open ") + path);
  bool ok = fwrite(&HB_BLOB_MAGIC, sizeof(HB_BLOB_MAGIC), 1, f) == 1;
  ok = ok && put_vec(f, h->c_icfg) && put_vec(f, h->c_dcfg) && put_vec(f, h->c_jc) && put_vec(f, h->c_jk) &&
       put_vec(f, h->c_hci) && put_vec(f, h->c_hc) && put_vec(f, h->c_hk) && put_vec(f, h->c_hk2) &&
       put_vec(f, h->jac_colind) && put_vec(f, h->jac_row) && put_vec(f, h->hess_colind) && put_vec(f, h->hess_row) &&
       put_vec(f, h->lb_idx) && put_vec(f, h->lb_val) && put_vec(f, h->ub_idx) && put_vec(f, h->ub_val);
  ok = (fclose(f) == 0) && ok;
  return ok ? HB_OK : fail(HB_ERR_INVALID, std::string("hb_save: write failed: ") + path);
}

extern "C" int hb_load(const char* path, hb_handle* out) {
  if (!path || !out) return fail(HB_ERR_INVALID, "hb_load: null argument");
  FILE* f = fopen(path, "rb");
  if (!f) return fail(HB_ERR_INVALID, std::string("hb_load: cannot open ") + path);
  uint64_t magic = 0;
  std::vector<int32_t> icfg, jc, jk, hc, hk, hk2, lbi, ubi;
  std::vector<int16_t> hci;
  std::vector<double> dcfg, lbv, ubv;
  std::vector<int64_t> jcol, jrow, hcol, hrow;
  bool ok = fread(&magic, sizeof(magic), 1, f) == 1 && magic == HB_BLOB_MAGIC;
  ok = ok && get_vec(f, icfg) && get_vec(f, dcfg) && get_vec(f, jc) && get_vec(f, jk) && get_vec(f, hci) && get_vec(f, hc) &&
       get_vec(f, hk) && get_vec(f, hk2) && get_vec(f, jcol) && get_vec(f, jrow) && get_vec(f, hcol) && get_vec(f, hrow) &&
       get_vec(f, lbi) && get_vec(f, lbv) && get_vec(f, ubi) && get_vec(f, ubv);
  fclose(f);
  if (!ok || icfg.size() != HB_KI_COUNT || dcfg.size() != HB_KD_COUNT || hci.size() != 129 * 129)
    return fail(HB_ERR_INVALID, std::string("hb_load: not a hippopt_b200 problem file of this library version: ") + path);
  const size_t N = (size_t)icfg[HB_KI_HORIZON];
  if (jc.size() != N * (size_t)icfg[HB_KI_N_JC] || jk.size() != N * (size_t)icfg[HB_KI_N_JK] ||
      hc.size() != N * (size_t)icfg[HB_KI_N_HC] || hk.size() != N * 27 * 57 || hk2.size() != N * 27)
    return fail(HB_ERR_INVALID, std::string("hb_load: inconsistent table sizes in ") + path);
  const int rc = hb_kino_create(icfg.data(), dcfg.data(), jc.data(), jk.data(), hci.data(), hc.data(), hk.data(), hk2.data(), out);
  if (rc != HB_OK) return rc;
  if (!jrow.empty()) {
    const int rc2 = hb_kino_attach_tables(*out, jcol.data(), jrow.data(), hcol.data(), hrow.data(), lbi.data(), lbv.data(),
                                          ubi.data(), ubv.data());
    if (rc2 != HB_OK) {
      hb_destroy(*out);
      *out = nullptr;
      return rc2;
    }
  }
  return HB_OK;
}

// ---------------------------------------------------------------------------------------------
// per-expression cost values (solution report)
extern "C" int hb_eval_cost_terms(hb_handle h, const double* x, const double* p, int64_t p_stride, double* terms,
                                  int64_t batch, void* stream) {
  if (!h || !x || !p || !terms) return fail(HB_ERR_INVALID, "hb_eval_cost_terms: null argument");
  if (batch <= 0) return fail(HB_ERR_INVALID, "hb_eval_cost_terms: batch must be positive");
  if (h->kind != KIND_KINO || h->host.kind != 0)
    return fail(HB_ERR_UNSUPPORTED, "hb_eval_cost_terms: kinodynamic OCP handles only");
  const hb::KinoConst& C = h->host;
  if (p_stride != 0 && p_stride != C.n_p) return fail(HB_ERR_INVALID, "hb_eval_cost_terms: p_stride must be 0 or n_p");
  CHECK_DEVICE(h, "hb_eval_cost_terms");
  cudaStream_t st = (cudaStream_t)stream;
  const int wpb = 4;
  const long total_warps = (long)batch * C.N;
  const unsigned grid = (unsigned)((total_warps + wpb - 1) / wpb);
  const unsigned mask = hb::HB_EVAL_COST_TERMS_BIT;
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(ensure_kernel_attributes(dev));
  const size_t smem_c = (size_t)hb::kino_contact_smem_layout(C.n_hc).total * sizeof(double) * wpb;
  const auto contact_kernel = kino_contact_kernel_for(C.terrain);
  contact_kernel<<<grid, 32 * wpb, smem_c, st>>>(h->topo, h->dev, mask, x, p, (long)p_stride, nullptr, nullptr, terms, nullptr,
                                                 nullptr, nullptr, nullptr, (long)batch);
  CUDA_TRY(cudaGetLastError());
  const size_t smem_k = (size_t)hb::kin_smem_layout(C.nb, C.n_slots, false).total * sizeof(double) * wpb;
  hb::kino_kin_kernel<false><<<grid, 32 * wpb, smem_k, st>>>(h->topo, h->dev, mask, x, p, (long)p_stride, nullptr, nullptr,
                                                            terms, nullptr, nullptr, nullptr, nullptr, (long)batch);
  CUDA_TRY(cudaGetLastError());
  h->launches = 2;
  return HB_OK;
}

#ifdef HB_PHASE_CLOCK
// developer build only (tools/phase_profile.py): read and reset the per-phase cycle sums
extern "C" int hb_debug_phase_read(unsigned long long* out64) {
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpyFromSymbol(out64, hb::hb_phase_acc, sizeof(unsigned long long) * 64));
  static unsigned long long zero[64] = {0};
  CUDA_TRY(cudaMemcpyToSymbol(hb::hb_phase_acc, zero, sizeof(zero)));
  return HB_OK;
}
#endif

// ---------------------------------------------------------------------------------------------
// CasADi's external-function (codegen) ABI for the five nlpsol oracle functions (SURVEY.md 8(b)):
//   cs.external("hb_nlp_jac_g", "libhippopt_b200.so") loads F, F_n_in, F_n_out, F_sparsity_in / _out, F_work,
//   F_name_in / _out, F_incref / _decref, F_alloc_mem / _init_mem / _free_mem / _checkout / _release by name [ext].
// External functions carry no handle, so a problem is BOUND to them per process (hb_external_bind); they then share
// one host pipeline and an x-keyed cache -- f, grad_f, g and jac_g at the same x cost ONE evaluation, hess_l a second
// one -- the compiled counterpart of hippopt_b200/plugin.py's OracleCache, without the Python callback in between.
typedef long long int casadi_int;
namespace {
struct ExternalBinding {
  hb_handle h = nullptr;
  int64_t n_x = 0, n_p = 0, m = 0, nnz_j = 0, nnz_h = 0;
  double *x = nullptr, *p = nullptr, *lam = nullptr, *sigma = nullptr;      // pinned staging of the inputs
  double *f = nullptr, *grad = nullptr, *g = nullptr, *jac = nullptr, *hess = nullptr;  // pinned results
  bool have_first = false, have_p = false;
  long evals_first = 0, evals_hess = 0;
  std::vector<casadi_int> sp_x, sp_p, sp_one, sp_g, sp_jac, sp_hess;
  std::mutex mu;
} g_ext;

std::vector<casadi_int> dense_sp(casadi_int n) {
  std::vector<casadi_int> s = {n, 1, 0, n};
  for (casadi_int i = 0; i < n; ++i) s.push_back(i);
  return s;
}
std::vector<casadi_int> ccs_sp(casadi_int nrow, casadi_int ncol, const std::vector<int64_t>& colind, const std::vector<int64_t>& row) {
  std::vector<casadi_int> s = {nrow, ncol};
  s.insert(s.end(), colind.begin(), colind.end());
  s.insert(s.end(), row.begin(), row.end());
  return s;
}
// two pinned blocks in hb_eval_host's slab order -- x | lam_g | sigma and f | grad_f | g | jac | hess -- so that an
// evaluation is one copy in each direction; p has its own buffer (uploaded only when it changes)
void ext_free() {
  if (g_ext.x) cudaFreeHost(g_ext.x);
  if (g_ext.f) cudaFreeHost(g_ext.f);
  if (g_ext.p) cudaFreeHost(g_ext.p);
  g_ext.x = g_ext.lam = g_ext.sigma = g_ext.f = g_ext.grad = g_ext.g = g_ext.jac = g_ext.hess = g_ext.p = nullptr;
}
// copies x / p into the staging buffers; returns true when x changed (the first-order cache is then stale)
int ext_inputs(const double** arg) {
  const size_t bx = sizeof(double) * g_ext.n_x, bp = sizeof(double) * g_ext.n_p;
  bool changed = !g_ext.have_first;
  if (arg[0]) {
    if (memcmp(g_ext.x, arg[0], bx) != 0) {
      memcpy(g_ext.x, arg[0], bx);
      changed = true;
    }
  } else {
    for (int64_t i = 0; i < g_ext.n_x; ++i)
      if (g_ext.x[i] != 0.0) changed = true;
    memset(g_ext.x, 0, bx);
  }
  bool p_changed = !g_ext.have_p;
  if (arg[1]) {
    if (memcmp(g_ext.p, arg[1], bp) != 0) {
      memcpy(g_ext.p, arg[1], bp);
      p_changed = true;
    }
  } else {
    memset(g_ext.p, 0, bp);
  }
  if (p_changed) {
    if (hb_host_set_parameters(g_ext.h, g_ext.p, 0, 1) != HB_OK) return -1;
    g_ext.have_p = true;
    changed = true;
  }
  return changed ? 1 : 0;
}
int ext_first_order(const double** arg) {
  if (!g_ext.h) return fail(HB_ERR_INVALID, "hb_nlp_*: no problem bound (hb_external_bind)");
  const int ch = ext_inputs(arg);
  if (ch < 0) return 1;
  if (ch) {
    if (hb_eval_host(g_ext.h, HB_EVAL_F | HB_EVAL_GRAD_F | HB_EVAL_G | HB_EVAL_JAC_G, g_ext.x, nullptr, nullptr, g_ext.f,
                     g_ext.grad, g_ext.g, g_ext.jac, nullptr, 1) != HB_OK)
      return 1;
    g_ext.have_first = true;
    ++g_ext.evals_first;
  }
  return 0;
}
}  // namespace

extern "C" int hb_external_bind(hb_handle h) {
  std::lock_guard<std::mutex> lock(g_ext.mu);
  ext_free();
  g_ext.h = nullptr;
  g_ext.have_first = g_ext.have_p = false;
  g_ext.evals_first = g_ext.evals_hess = 0;
  if (!h) return HB_OK;  // unbind
  if (h->kind == KIND_KINO && h->jac_row.empty())
    return fail(HB_ERR_INVALID, "hb_external_bind: attach the patterns first (hb_kino_attach_tables / hb_load)");
  hb_dims(h, &g_ext.n_x, &g_ext.n_p, &g_ext.m, &g_ext.nnz_j, &g_ext.nnz_h);
  std::vector<int64_t> jc(g_ext.n_x + 1), jr(g_ext.nnz_j), hc(g_ext.n_x + 1), hr(g_ext.nnz_h);
  if (hb_pattern_jac(h, jc.data(), jr.data()) != HB_OK || hb_pattern_hess(h, hc.data(), hr.data()) != HB_OK) return HB_ERR_INVALID;
  g_ext.sp_x = dense_sp(g_ext.n_x);
  g_ext.sp_p = dense_sp(g_ext.n_p);
  g_ext.sp_one = dense_sp(1);
  g_ext.sp_g = dense_sp(g_ext.m);
  g_ext.sp_jac = ccs_sp(g_ext.m, g_ext.n_x, jc, jr);
  g_ext.sp_hess = ccs_sp(g_ext.n_x, g_ext.n_x, hc, hr);
  const size_t n_in = (size_t)(g_ext.n_x + g_ext.m + 1), n_out = (size_t)(1 + g_ext.n_x + g_ext.m + g_ext.nnz_j + g_ext.nnz_h);
  CUDA_TRY(cudaHostAlloc((void**)&g_ext.x, sizeof(double) * n_in, cudaHostAllocDefault));
  CUDA_TRY(cudaHostAlloc((void**)&g_ext.f, sizeof(double) * n_out, cudaHostAllocDefault));
  CUDA_TRY(cudaHostAlloc((void**)&g_ext.p, sizeof(double) * (size_t)(g_ext.n_p > 0 ? g_ext.n_p : 1), cudaHostAllocDefault));
  memset(g_ext.x, 0, sizeof(double) * n_in);
  memset(g_ext.f, 0, sizeof(double) * n_out);
  memset(g_ext.p, 0, sizeof(double) * (size_t)(g_ext.n_p > 0 ? g_ext.n_p : 1));
  g_ext.lam = g_ext.x + g_ext.n_x;
  g_ext.sigma = g_ext.lam + g_ext.m;
  g_ext.grad = g_ext.f + 1;
  g_ext.g = g_ext.grad + g_ext.n_x;
  g_ext.jac = g_ext.g + g_ext.m;
  g_ext.hess = g_ext.jac + g_ext.nnz_j;
  g_ext.h = h;
  return HB_OK;
}

extern "C" int hb_external_stats(int64_t* first_order_evaluations, int64_t* hessian_evaluations) {
  if (first_order_evaluations) *first_order_evaluations = g_ext.evals_first;
  if (hessian_evaluations) *hessian_evaluations = g_ext.evals_hess;
  return HB_OK;
}

#define HB_EXT_COMMON(F, NIN, NOUT)                                                                         \
  extern "C" casadi_int F##_n_in(void) { return NIN; }                                                     \
  extern "C" casadi_int F##_n_out(void) { return NOUT; }                                                   \
  extern "C" int F##_work(casadi_int* sz_arg, casadi_int* sz_res, casadi_int* sz_iw, casadi_int* sz_w) {   \
    if (sz_arg) *sz_arg = NIN;                                                                             \
    if (sz_res) *sz_res = NOUT;                                                                            \
    if (sz_iw) *sz_iw = 0;                                                                                 \
    if (sz_w) *sz_w = 0;                                                                                   \
    return 0;                                                                                              \
  }                                                                                                        \
  extern "C" void F##_incref(void) {}                                                                      \
  extern "C" void F##_decref(void) {}                                                                      \
  extern "C" int F##_alloc_mem(void) { return 0; }                                                         \
  extern "C" int F##_init_mem(int) { return 0; }                                                           \
  extern "C" void F##_free_mem(int) {}                                                                     \
  extern "C" int F##_checkout(void) { return 0; }                                                          \
  extern "C" void F##_release(int) {}

static const char* ext_in_name(casadi_int i) {
  static const char* n[] = {"x", "p", "lam_f", "lam_g"};
  return i >= 0 && i < 4 ? n[i] : nullptr;
}

// ---- nlp_f: (x, p) -> f
HB_EXT_COMMON(hb_nlp_f, 2, 1)
extern "C" const char* hb_nlp_f_name_in(casadi_int i) { return i < 2 ? ext_in_name(i) : nullptr; }
extern "C" const char* hb_nlp_f_name_out(casadi_int i) { return i == 0 ? "f" : nullptr; }
extern "C" const casadi_int* hb_nlp_f_sparsity_in(casadi_int i) { return i == 0 ? g_ext.sp_x.data() : (i == 1 ? g_ext.sp_p.data() : nullptr); }
extern "C" const casadi_int* hb_nlp_f_sparsity_out(casadi_int i) { return i == 0 ? g_ext.sp_one.data() : nullptr; }
extern "C" int hb_nlp_f(const double** arg, double** res, casadi_int*, double*, int) {
  std::lock_guard<std::mutex> lock(g_ext.mu);
  if (ext_first_order(arg)) return 1;
  if (res[0]) res[0][0] = g_ext.f[0];
  return 0;
}
// ---- nlp_g: (x, p) -> g
HB_EXT_COMMON(hb_nlp_g, 2, 1)
extern "C" const char* hb_nlp_g_name_in(casadi_int i) { return i < 2 ? ext_in_name(i) : nullptr; }
extern "C" const char* hb_nlp_g_name_out(casadi_int i) { return i == 0 ? "g" : nullptr; }
extern "C" const casadi_int* hb_nlp_g_sparsity_in(casadi_int i) { return hb_nlp_f_sparsity_in(i); }
extern "C" const casadi_int* hb_nlp_g_sparsity_out(casadi_int i) { return i == 0 ? g_ext.sp_g.data() : nullptr; }
extern "C" int hb_nlp_g(const double** arg, double** res, casadi_int*, double*, int) {
  std::lock_guard<std::mutex> lock(g_ext.mu);
  if (ext_first_order(arg)) return 1;
  if (res[0]) memcpy(res[0], g_ext.g, sizeof(double) * g_ext.m);
  return 0;
}
// ---- nlp_grad_f: (x, p) -> (f, grad_f)
HB_EXT_COMMON(hb_nlp_grad_f, 2, 2)
extern "C" const char* hb_nlp_grad_f_name_in(casadi_int i) { return i < 2 ? ext_in_name(i) : nullptr; }
extern "C" const char* hb_nlp_grad_f_name_out(casadi_int i) { return i == 0 ? "f" : (i == 1 ? "grad_f_x" : nullptr); }
extern "C" const casadi_int* hb_nlp_grad_f_sparsity_in(casadi_int i) { return hb_nlp_f_sparsity_in(i); }
extern "C" const casadi_int* hb_nlp_grad_f_sparsity_out(casadi_int i) { return i == 0 ? g_ext.sp_one.data() : (i == 1 ? g_ext.sp_x.data() : nullptr); }
extern "C" int hb_nlp_grad_f(const double** arg, double** res, casadi_int*, double*, int) {
  std::lock_guard<std::mutex> lock(g_ext.mu);
  if (ext_first_order(arg)) return 1;
  if (res[0]) res[0][0] = g_ext.f[0];
  if (res[1]) memcpy(res[1], g_ext.grad, sizeof(double) * g_ext.n_x);
  return 0;
}
// ---- nlp_jac_g: (x, p) -> (g, jac_g)
HB_EXT_COMMON(hb_nlp_jac_g, 2, 2)
extern "C" const char* hb_nlp_jac_g_name_in(casadi_int i) { return i < 2 ? ext_in_name(i) : nullptr; }
extern "C" const char* hb_nlp_jac_g_name_out(casadi_int i) { return i == 0 ? "g" : (i == 1 ? "jac_g_x" : nullptr); }
extern "C" const casadi_int* hb_nlp_jac_g_sparsity_in(casadi_int i) { return hb_nlp_f_sparsity_in(i); }
extern "C" const casadi_int* hb_nlp_jac_g_sparsity_out(casadi_int i) { return i == 0 ? g_ext.sp_g.data() : (i == 1 ? g_ext.sp_jac.data() : nullptr); }
extern "C" int hb_nlp_jac_g(const double** arg, double** res, casadi_int*, double*, int) {
  std::lock_guard<std::mutex> lock(g_ext.mu);
  if (ext_first_order(arg)) return 1;
  if (res[0]) memcpy(res[0], g_ext.g, sizeof(double) * g_ext.m);
  if (res[1]) memcpy(res[1], g_ext.jac, sizeof(double) * g_ext.nnz_j);
  return 0;
}
// ---- nlp_hess_l: (x, p, lam_f, lam_g) -> triu(hess_l)
HB_EXT_COMMON(hb_nlp_hess_l, 4, 1)
extern "C" const char* hb_nlp_hess_l_name_in(casadi_int i) { return ext_in_name(i); }
extern "C" const char* hb_nlp_hess_l_name_out(casadi_int i) { return i == 0 ? "triu_hess_gamma_x_x" : nullptr; }
extern "C" const casadi_int* hb_nlp_hess_l_sparsity_in(casadi_int i) {
  return i < 2 ? hb_nlp_f_sparsity_in(i) : (i == 2 ? g_ext.sp_one.data() : (i == 3 ? g_ext.sp_g.data() : nullptr));
}
extern "C" const casadi_int* hb_nlp_hess_l_sparsity_out(casadi_int i) { return i == 0 ? g_ext.sp_hess.data() : nullptr; }
extern "C" int hb_nlp_hess_l(const double** arg, double** res, casadi_int*, double*, int) {
  std::lock_guard<std::mutex> lock(g_ext.mu);
  if (!g_ext.h) return fail(HB_ERR_INVALID, "hb_nlp_hess_l: no problem bound (hb_external_bind)");
  const int ch = ext_inputs(arg);
  if (ch < 0) return 1;
  if (ch) g_ext.have_first = false;  // x moved without a first-order call in between: that cache is stale
  g_ext.sigma[0] = arg[2] ? arg[2][0] : 0.0;
  if (arg[3]) memcpy(g_ext.lam, arg[3], sizeof(double) * g_ext.m);
  else memset(g_ext.lam, 0, sizeof(double) * g_ext.m);
  if (hb_eval_host(g_ext.h, HB_EVAL_HESS_L, g_ext.x, g_ext.lam, g_ext.sigma, nullptr, nullptr, nullptr, nullptr, g_ext.hess, 1) != HB_OK)
    return 1;
  ++g_ext.evals_hess;
  if (res[0]) memcpy(res[0], g_ext.hess, sizeof(double) * g_ext.nnz_h);
  return 0;
}
