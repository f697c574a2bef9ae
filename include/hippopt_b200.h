/* hippopt_b200.h -- C ABI of the B200-native NLP evaluator for hippopt's multiple-shooting OCPs.
 *
 * What this boundary replaces.  hippopt has no FFI of its own: the numerical hot path is the set of
 * NLP oracle functions CasADi builds and IPOPT calls at every iteration of ``opti.solve()``
 *   /root/reference/src/hippopt/base/opti_solver.py:479   (single blocking call into CasADi)
 *   [ext] nlpsol oracle functions nlp_f, nlp_grad_f, nlp_g, nlp_jac_g, nlp_hess_l
 * for the problem that
 *   /root/reference/src/hippopt/turnkey_planners/humanoid_kinodynamic/planner.py:27-176
 * assembles.  A CasADi ``Callback`` / ``external`` shim (INTEGRATION.md) forwards exactly those five
 * evaluations to hb_eval(); the sparsity queries replace ``Function.sparsity_out`` of nlp_jac_g /
 * nlp_hess_l (compressed-column, Hessian upper triangle).
 *
 * Conventions
 *   - plain C types only; every pointer marked "device" is a CUDA device pointer owned by the caller
 *     (fp64, contiguous, instance-major: x[b*n_x + i]); the library never allocates or frees caller
 *     buffers and keeps no reference to them after the call returns (work is enqueued on `stream`).
 *   - return 0 on success, non-zero error code otherwise (CasADi external-function convention);
 *     hb_last_error() gives a message.  NaN/Inf in outputs are passed through, not trapped.
 *   - the layout tables (row offsets, scatter maps) are computed by the host-side layout compiler
 *     (hippopt_b200/kino_layout.py) and copied into the handle at creation.
 */
#ifndef HIPPOPT_B200_H
#define HIPPOPT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hb_problem_s* hb_handle;

/* evaluation mask bits for hb_eval (any combination) */
enum {
  HB_EVAL_F = 1,      /* nlp_f       : f[b]                         */
  HB_EVAL_GRAD_F = 2, /* nlp_grad_f  : grad_f[b*n_x + i]            */
  HB_EVAL_G = 4,      /* nlp_g       : g[b*m + r]                   */
  HB_EVAL_JAC_G = 8,  /* nlp_jac_g   : jac_vals[b*nnz_j + slot]     */
  HB_EVAL_HESS_L = 16 /* nlp_hess_l  : hess_vals[b*nnz_h + slot]    */
};

enum { HB_OK = 0, HB_ERR_INVALID = 1, HB_ERR_CUDA = 2, HB_ERR_UNSUPPORTED = 3 };

#define HB_MAX_BODIES 32
#define HB_N_JOINTS 23
#define HB_N_POINTS 8

/* ---- integer configuration table of the kinodynamic problem (indices into icfg[]) ---- */
enum {
  HB_KI_HORIZON = 0,
  HB_KI_N_X,
  HB_KI_N_P,
  HB_KI_M,
  HB_KI_NNZ_J,
  HB_KI_NNZ_H,
  HB_KI_N_JC,
  HB_KI_N_JK,
  HB_KI_N_HC,
  HB_KI_TERRAIN,          /* 0 planar (planar_terrain.py), 1 sum of two smooth steps (the stairs), 2 sum of K general
                             smooth steps (the ramp); all for either kind.  1: the steps' ten parameters
                             (l, w, height, ox, oy) x 2 at HB_KI_PO_TERRAIN in p.  2: K records
                             (l, w, height, ox, oy, oz, yaw, n_x, n_y, n_z) from HB_KI_PO_TERRAIN to the end of p;
                             K = (n_p - HB_KI_PO_TERRAIN) / 10, which must be a whole number >= 1 (else HB_ERR_INVALID) */
  HB_KI_HAS_FINAL,
  HB_KI_HAS_PERIODICITY,
  HB_KI_H_INIT,           /* x offset of initial_state.centroidal_momentum */
  /* parameter offsets inside p (SURVEY.md Appendix B.2) */
  HB_KI_PO_DESC0,
  HB_KI_PO_MASS,
  HB_KI_PO_INIT,
  HB_KI_PO_FINAL,
  HB_KI_PO_DT,
  HB_KI_PO_GRAVITY,
  HB_KI_PO_KT,
  HB_KI_PO_KBS,
  HB_KI_PO_EPS,
  HB_KI_PO_MU,
  HB_KI_PO_MAX_U,
  HB_KI_PO_MAX_FD,
  HB_KI_PO_MAX_L,
  HB_KI_PO_MIN_COM_H,
  HB_KI_PO_MIN_FEET_D,
  HB_KI_PO_MAX_FEET_H,
  HB_KI_PO_MAX_S,
  HB_KI_PO_MIN_S,
  HB_KI_PO_MAX_SD,
  HB_KI_PO_MIN_SD,
  HB_KI_PO_REFS0,
  HB_KI_PO_TERRAIN,
  /* yaw task corner indices inside a foot (planner.py:780-828) */
  HB_KI_YAW_BR,
  HB_KI_YAW_TR,
  HB_KI_YAW_TL,
  /* model topology */
  HB_KI_N_BODIES,
  HB_KI_FOOT_BODY_L,
  HB_KI_FOOT_BODY_R,
  HB_KI_CHEST_BODY,
  /* problem kind and the "virtual knot" mapping used by the kinematics kernel */
  HB_KI_KIND,             /* 0 kinodynamic OCP (planner.py:27-176), 1 pose finder (humanoid_pose_finder/planner.py:303-413) */
  HB_KI_X_STRIDE,         /* doubles between consecutive knots in x (189, or 0 for a single knot) */
  HB_KI_COST_K0,          /* first knot on which apply_to_first_elements=False expressions exist (1, or 0) */
  HB_KI_JOINT_COST_KIND,  /* 0: planner.py:506-520 (kinodynamic), 1: e^T diag(w) e (pose finder :584-588) */
  HB_KI_PO_FQ,            /* parameter offsets of the cost references at knot 0 ... */
  HB_KI_PO_BQ,
  HB_KI_PO_BQV,
  HB_KI_PO_JR,
  HB_KI_REF_STRIDE,       /* ... and their stride per knot */
  HB_KI_ZMAP0,            /* 189 entries: virtual knot variable -> offset inside the knot block of x, or -1 */
  HB_KI_PARENT0 = HB_KI_ZMAP0 + 189,               /* HB_MAX_BODIES entries */
  HB_KI_FAM0 = HB_KI_PARENT0 + HB_MAX_BODIES,      /* HB_KF_COUNT x 4 entries: base, rows, k0, k1 */
  HB_KI_COUNT_BASE = HB_KI_FAM0
};

/* constraint families in the reference's subject_to order (planner.py:124-176); the first
 * HB_KF_PT_COUNT ids repeat per contact point: family id = point * HB_KF_PT_COUNT + local id */
enum {
  HB_KF_PT_F_IC = 0,
  HB_KF_PT_F_DYN,
  HB_KF_PT_P_IC,
  HB_KF_PT_P_DYN,
  HB_KF_PT_PLANAR,
  HB_KF_PT_DCC,
  HB_KF_PT_HEIGHT,
  HB_KF_PT_NORMAL,
  HB_KF_PT_FRICTION,
  HB_KF_PT_U_BOUNDS,
  HB_KF_PT_FD_BOUNDS,
  HB_KF_PT_FK,
  HB_KF_PT_COUNT
};
enum {
  HB_KF_PB_IC = HB_KF_PT_COUNT * HB_N_POINTS,
  HB_KF_PB_DYN,
  HB_KF_Q_IC,
  HB_KF_Q_DYN,
  HB_KF_S_IC,
  HB_KF_S_DYN,
  HB_KF_COM_IC,
  HB_KF_COM_DYN,
  HB_KF_H_IC,
  HB_KF_H_DYN,
  HB_KF_UNIT_QUAT,
  HB_KF_COM_KIN,
  HB_KF_MOM_KIN,
  HB_KF_L_BOUNDS,
  HB_KF_COM_HEIGHT,
  HB_KF_FEET_DIST,
  HB_KF_S_BOUNDS,
  HB_KF_SD_BOUNDS,
  HB_KF_FINAL,
  HB_KF_FEET_RELH,
  HB_KF_PERIODICITY,
  HB_KF_COUNT
};
#define HB_KI_COUNT (HB_KI_COUNT_BASE + 4 * HB_KF_COUNT)

/* ---- double configuration table (indices into dcfg[]) ---- */
enum {
  HB_KD_W_SWING = 0,     /* swing_foot_height_cost_multiplier                      */
  HB_KD_W_U,             /* contact_velocity_control_cost_multiplier               */
  HB_KD_W_FD,            /* contact_force_control_cost_multiplier                  */
  HB_KD_W_CENTROID,      /* contacts_centroid_cost_multiplier                      */
  HB_KD_W_COMVEL0,       /* 3: com_linear_velocity multiplier * weights            */
  HB_KD_W_FRAME = HB_KD_W_COMVEL0 + 3,
  HB_KD_W_BQ,
  HB_KD_W_BQV,
  HB_KD_W_JOINT,
  HB_KD_W_RATIO,
  HB_KD_W_YAW,
  HB_KD_WJ0,             /* 23: joint_regularization_cost_weights                  */
  HB_KD_TOTAL_MASS = HB_KD_WJ0 + HB_N_JOINTS,
  HB_KD_FOOT_R0,         /* 2 x 9 : sole frame rotation in its body                */
  HB_KD_FOOT_T0 = HB_KD_FOOT_R0 + 18, /* 2 x 3                                     */
  HB_KD_CHEST_R0 = HB_KD_FOOT_T0 + 6, /* 9                                         */
  HB_KD_BODY0 = HB_KD_CHEST_R0 + 9    /* per body 31 doubles: E(9) r(3) axis(3) mass(1) com(3) inertia(9) pad(3) */
};
#define HB_KD_BODY_STRIDE 31
#define HB_KD_COUNT (HB_KD_BODY0 + HB_KD_BODY_STRIDE * HB_MAX_BODIES)

/* Create an evaluator for the humanoid kinodynamic OCP.  All arrays are HOST pointers and are copied.
 *   icfg[HB_KI_COUNT], dcfg[HB_KD_COUNT]          configuration tables (enums above)
 *   jc_map[N*n_jc], jk_map[N*n_jk]                local Jacobian entry -> CCS slot (-1: absent)
 *   hc_index[129*129]                             contact-block variable pair -> local Hessian entry
 *   hc_map[N*n_hc], hk_map[N*27*57], hk2_map[N*27] local Hessian entry -> CCS slot (-1: absent)
 * replaces: graph construction in planner.py:27-176 + nlpsol init [ext]. */
int hb_kino_create(const int32_t* icfg, const double* dcfg, const int32_t* jc_map, const int32_t* jk_map,
                   const int16_t* hc_index, const int32_t* hc_map, const int32_t* hk_map,
                   const int32_t* hk2_map, hb_handle* out);

/* Create an evaluator for the mass-falling toy OCP of /root/reference/test/test_multiple_shooting.py:
 * 210-353 (3 masses, ForwardEuler or ImplicitTrapezoid defects, horizon N).  integrator: 0 Euler, 1 trapezoid. */
int hb_toy_create(int32_t horizon, int32_t integrator, double dt, hb_handle* out);

int hb_destroy(hb_handle h);

/* problem dimensions: n_x, n_p, m, nnz(jac_g), nnz(hess_l upper) */
int hb_dims(hb_handle h, int64_t* n_x, int64_t* n_p, int64_t* m, int64_t* nnz_j, int64_t* nnz_h);

/* Sparsity of jac_g (m x n_x) and hess_l (n_x x n_x, upper triangle) in compressed-column form,
 * written to HOST arrays colind[n_x+1], row[nnz].  replaces: Function.sparsity_out() of nlp_jac_g / nlp_hess_l [ext].
 * The toy OCP's layout lives in the library; kinodynamic / pose-finder handles answer once their tables are
 * attached (hb_kino_attach_tables: done by hippopt_b200.evaluator at creation, or restored by hb_load). */
int hb_pattern_jac(hb_handle h, int64_t* colind, int64_t* row);
int hb_pattern_hess(hb_handle h, int64_t* colind, int64_t* row);

/* Tables a caller without the Python layout compiler needs, copied into the handle (HOST pointers):
 *   CCS patterns of jac_g / hess_l, and lbg / ubg as an affine function of ONE parameter per row:
 *   lbg[r] = lb_idx[r] >= 0 ? lb_val[r] * p[lb_idx[r]] : lb_val[r]   (same for ubg; +-inf as IEEE infinities)
 * replaces: opti.lbg / opti.ubg evaluated at the parameter values (opti_solver.py:616-619). */
int hb_kino_attach_tables(hb_handle h, const int64_t* jac_colind, const int64_t* jac_row, const int64_t* hess_colind,
                          const int64_t* hess_row, const int32_t* lb_idx, const double* lb_val, const int32_t* ub_idx,
                          const double* ub_val);
/* lbg[m], ubg[m] (HOST) for one parameter vector p[n_p] (HOST) */
int hb_bounds(hb_handle h, const double* p, double* lbg, double* ubg);

/* Serialise a kinodynamic / pose-finder handle (configuration tables, scatter maps, attached tables) to a file and
 * create a handle from such a file: a C / C++ / Go caller links the library, calls hb_load on a file written once by
 * the Python layout compiler for its (robot, settings, horizon), and never needs Python at run time. */
int hb_save(hb_handle h, const char* path);
int hb_load(const char* path, hb_handle* out);

/* Evaluate the requested NLP functions for `batch` independent instances.
 *   x      device [batch*n_x]          decision vectors
 *   p      device [batch*n_p] or [n_p] parameters (p_stride = n_p, or 0 to share one vector)
 *   lam_g  device [batch*m]            constraint multipliers (HB_EVAL_HESS_L only)
 *   sigma  device [batch]              objective factor       (HB_EVAL_HESS_L only)
 *   outputs may be NULL when their bit is not in `mask`.
 *   stream: cudaStream_t (NULL = default stream).
 * replaces: nlp_f / nlp_grad_f / nlp_g / nlp_jac_g / nlp_hess_l calls inside opti_solver.py:479. */
int hb_eval(hb_handle h, uint32_t mask, const double* x, const double* p, int64_t p_stride,
            const double* lam_g, const double* sigma, double* f, double* grad_f, double* g,
            double* jac_vals, double* hess_vals, int64_t batch, void* stream);

/* Per-expression cost values of the kinodynamic OCP, for the solution report (not an IPOPT callback).
 * replaces: opti_solution.value(self._cost_expressions[name]) for every named cost, opti_solver.py:526-529
 * (names: `name=` arguments of planner.py:215-895 + the "[k]" suffix of multiple_shooting_solver.py:810;
 * hippopt_b200/naming.py maps the slots below to those names).
 *   terms  device [batch][horizon][HB_COST_TERMS]: the value (multiplier included) of cost expression `slot` at
 *          knot k, 0 where the expression does not exist (apply_to_first_elements = False at k = 0).
 * The sum over slots and knots is f (up to the order of the additions). */
enum {
  HB_CT_SWING0 = 0,       /* 8: <point>.p_swing_height_regularization        planner.py:855-875 */
  HB_CT_UV0 = 8,          /* 8: <point>.u_v_regularization                   planner.py:877-884 */
  HB_CT_FDOT0 = 16,       /* 8: <point>.f_dot_regularization                 planner.py:886-893 */
  HB_CT_FRATIO0 = 24,     /* 8: <point>.f_regularization (force ratio)       planner.py:756-771 */
  HB_CT_COM_VELOCITY = 32,/* com_velocity_error                              planner.py:432-447 */
  HB_CT_CENTROID,         /* contacts_centroid_cost                          planner.py:248-264 */
  HB_CT_YAW_LEFT,         /* left_yaw_regularization                         planner.py:780-853 */
  HB_CT_YAW_RIGHT,        /* right_yaw_regularization                                           */
  HB_CT_FRAME_QUAT,       /* frame_quaternion_error                          planner.py:449-477 */
  HB_CT_BASE_QUAT,        /* base_quaternion_error                           planner.py:479-491 */
  HB_CT_BASE_QUAT_VEL,    /* base_quaternion_velocity_error                  planner.py:493-503 */
  HB_CT_JOINTS,           /* joint_positions_error                           planner.py:505-520 */
  HB_COST_TERMS
};
int hb_eval_cost_terms(hb_handle h, const double* x, const double* p, int64_t p_stride, double* terms,
                       int64_t batch, void* stream);

/* Host-buffer form of hb_eval: the call a CPU-side solver (IPOPT inside opti_solver.py:479) makes.
 * Every pointer is a HOST pointer (pinned memory from hb_host_alloc gives full copy/compute overlap;
 * pageable memory works, more slowly).  The batch is cut into chunks pipelined over internal CUDA
 * streams: H2D of x / lam_g / sigma, the kernels, D2H of the requested outputs.  Blocking: all outputs
 * are complete in host memory when the call returns.  Device staging buffers belong to the handle.
 *
 * Parameters do not change between the iterations of one solve (opti.set_value before opti.solve,
 * opti_solver.py:296-344), so they are uploaded once with hb_host_set_parameters:
 *   p host [batch*n_p] (p_stride = n_p) or [n_p] (p_stride = 0, shared by every instance).
 * hb_eval_host fails with HB_ERR_INVALID if no parameters were set or `batch` exceeds the batch they
 * were set for (p_stride = n_p).
 *
 * A call that fits one chunk (batch <= 128) and repeats with the same mask and the same PINNED host pointers -- one
 * instance per call, every iterate, is what a CPU-side IPOPT does -- is captured as a CUDA graph on its second
 * occurrence and replayed from then on (copies, kernels and their events as one launch; up to 8 such call shapes per
 * handle).  The host buffers of such a call must stay allocated (and pinned) for as long as they are passed with that
 * handle; new parameters of another size drop the graphs. */
int hb_host_set_parameters(hb_handle h, const double* p, int64_t p_stride, int64_t batch);
int hb_eval_host(hb_handle h, uint32_t mask, const double* x, const double* lam_g, const double* sigma,
                 double* f, double* grad_f, double* g, double* jac_vals, double* hess_vals, int64_t batch);
/* bytes copied host->device and device->host by the last hb_eval_host */
int hb_host_last_traffic(hb_handle h, int64_t* h2d_bytes, int64_t* d2h_bytes);
/* page-locked host memory for callers that do not link the CUDA runtime themselves */
int hb_host_alloc(void** ptr, int64_t bytes);
int hb_host_free(void* ptr);

/* number of kernel launches the last hb_eval / hb_eval_host enqueued (for bench.py's gpu_launches claim) */
int hb_last_launch_count(hb_handle h);

/* Evaluator options.  HB_OPT_JAC_ADJOINT (default 0): when jac_g / grad_f are requested WITHOUT hess_l,
 * compute the kinematic rows with the row-per-lane adjoint sweep instead of the forward-mode columns -- an
 * independent algorithm for the same numbers (agreement to rounding is part of the GPU tests), 0.2 ms
 * slower per 30 720 knot-evals. */
enum { HB_OPT_JAC_ADJOINT = 1 };
int hb_set_option(hb_handle h, int32_t option, int32_t value);

/* Per-kernel device timing of the kinodynamic evaluator.  While enabled, every hb_eval records CUDA
 * events on its stream around the contact kernel, the kinematics kernel and the f reduction.
 * hb_profile_read sums the elapsed milliseconds {contact, kinematics, reduce} over the hb_eval calls
 * made since hb_profile_enable(h, 1) and returns their number. */
int hb_profile_enable(hb_handle h, int enable);
int hb_profile_read(hb_handle h, double* ms3, int64_t* n_evals);

/* Batched dense LU with partial pivoting for the stage blocks of the KKT sweep (hippopt_b200/kkt.py;
 * SURVEY.md 8(f) row f2).  replaces: the numeric factorisation / solve IPOPT delegates to its sparse
 * linear solver once per iteration (MUMPS [ext] below opti_solver.py:479), restricted to the dense
 * per-knot blocks the stage ordering leaves.
 *   A     device [batch][n*n]   column-major, leading dimension n; overwritten by L (unit, below) and U
 *   piv   device [batch][n]     piv[j] = row (>= j) interchanged with row j.  Interchanges are applied to
 *                               the panel and the trailing columns only (16-column panels); the factors are
 *                               meant for hb_lu_solve_batched, not for LAPACK's getrs
 *   info  device [batch]        0, or 1 + index of the first exactly-zero / NaN pivot column
 *   Bm    device [batch][n*nrhs] row-major right-hand sides (entry (i, c) at i*nrhs + c), overwritten by X
 * n <= 768 (panel and right-hand sides live in shared memory).  One CTA per matrix (and per 24 or 32
 * right-hand sides). */
int hb_lu_factor_batched(double* A, int32_t* piv, int32_t* info, int64_t n, int64_t batch, void* stream);
int hb_lu_solve_batched(const double* LU, const int32_t* piv, double* Bm, int64_t n, int64_t nrhs, int64_t batch,
                        void* stream);
/* Host-only: the kernel variants hb_lu_factor_batched / hb_lu_solve_batched launch for (n, batch, nrhs) on a device
 * with `sms` SMs (the same function picks them), for tests that must know which variant a case runs.
 *   out[4]  RPT (panel rows per thread), MB (CTAs per SM of the factor kernel's register budget), ct (8-column tiles of
 *           right-hand sides per CTA of the solve: 3 or 4), column chunks per matrix */
int hb_debug_lu_plan(int64_t n, int64_t batch, int64_t nrhs, int32_t sms, int32_t* out);

/* One stage of the block-tridiagonal KKT sweep (hippopt_b200/kkt.py::StageKKT) assembled in one launch from the CCS
 * value arrays: the dense symmetric stage block D (batch x nb x nb) = hess_l block + J_I^T Sigma J_I + shifts, with the
 * stage's equality rows in both triangles and the coupling term A_k S_{k-1}^{-1} A_k^T subtracted, and the right-hand
 * sides rhs (batch x nb x (R + n_cpl_next), row-major) = [b_k - A_k w_{k-1} | A_{k+1}^T; 0].  hb_lu_factor_batched(D) and
 * hb_lu_solve_batched(D, rhs) follow; the solution is `prev_sol` of the next stage.
 *   hdr   HOST   int32[13]: nb, nx (variable slots), nv (live variables), ne (equality rows), R, n_cpl, n_cpl_next,
 *                n_direct, n_targets, n_contrib, n_a, n_an, nb_prev (block size of stage k - 1: stages may differ)
 *   tab   device int32 tables in this order: direct_val[n_direct] (>= 0: hess_vals index, < 0: ~index into jac_vals),
 *                direct_pos[n_direct]; tgt_pos[n_targets], tgt_ptr[n_targets + 1], tgt_sig / tgt_e1 / tgt_e2[n_contrib]
 *                (D[tgt_pos] += sum sigma_I[sig] jac[e1] jac[e2]); var[nv], eq[ne] (rows of RX / RE); cpl[n_cpl] (block
 *                rows of the coupling equations); a_ptr[n_cpl + 1], a_val / a_col[n_a] (A_k by row: jac_vals index,
 *                variable slot of stage k - 1); an_val / an_row / an_col[n_an] (A_{k+1}: rhs[an_col][R + an_row])
 *   RX    device [batch][n_x][R], RE device [batch][m_E][R]; prev_sol device [batch][nb_prev][R + n_cpl] or NULL
 * One CTA per instance; fixed summation order (bit-reproducible).
 * replaces: the assembly of the KKT matrix inside IPOPT / MUMPS [ext] for the stage ordering of kkt.py. */
int hb_kkt_assemble_stage(const int32_t* hdr, const int32_t* tab, const double* hess_vals, int64_t nnz_h,
                          const double* jac_vals, int64_t nnz_j, const double* sigma_I, int64_t m_I, const double* delta,
                          double delta_c, const double* RX, int64_t n_x, const double* RE, int64_t m_E,
                          const double* prev_sol, double* D, double* rhs, int64_t batch, void* stream);

/* Deterministic sparse products with the CCS value arrays the evaluation kernels write, for solvers that keep their
 * iterates on the device (hippopt_b200.ipsolver): y[b][o] = sum_{q in [ptr[o], ptr[o+1])} w[q] vals[b][entry[q]] x[b][idx[q]]
 * (w may be NULL = 1).  With (ptr, entry, idx) grouped by row this is jac_g x, by column jac_g^T lam, by row over the
 * mirrored upper triangle hess_l x.  One thread per output element, fixed summation order (no atomics).
 * replaces: the sparse products inside IPOPT's residual and step computations [ext]. */
int hb_ccs_group_mul(const double* vals, const int32_t* ptr, const int32_t* entry, const int32_t* idx, const double* w,
                     const double* x, double* y, int64_t n_out, int64_t n_in, int64_t nnz, int64_t batch, void* stream);

/* Initial guesses / reference trajectories on the device (SURVEY.md 8(f) row f3).
 * replaces: humanoid_state_interpolator (robot_planning/utilities/interpolators.py:396-448) with its callees
 * linear_interpolator (:24-50), quaternion_slerp (:53-77), transform_interpolator (:80-103),
 * feet_contact_points_interpolator (:312-337) and the per-point arithmetic of foot_contact_state_interpolator
 * (:171-229), for `batch` instances at once.  The phase bookkeeping of foot_contact_state_interpolator
 * (:106-169, :231-309) depends on times only; the caller passes its result as `schedule`
 * (hippopt_b200/interpolators.py foot_contact_schedule builds it and raises the reference's ValueErrors).
 *   initial, final   device [batch][82 + n_joints]  state blocks: 8 x (p[3], f[3], position_in_foot_frame[3]),
 *                                                   base position[3], quaternion xyzw[4], joints, com[3]
 *                                                   (points 0-3 left foot, 4-7 right; descriptors read from initial)
 *   schedule         device [2][n_points][5] int32  per foot (left, right) and point: kind (0 stance of phase a,
 *                                                   1 swing from a.transform to a.mid_swing_transform, 2 swing from
 *                                                   a.mid_swing_transform to b.transform), a, b, sample j of n
 *                                                   (np.linspace(0, 1, n)[j]); a, b are NOT range-checked on the device
 *   phases_*         device [n_phases][17] doubles per instance, instances `stride_*` doubles apart (0: shared):
 *                                                   transform position[3], quaternion[4], mid-swing position[3],
 *                                                   quaternion[4], force[3]
 *   states           device [batch][n_points][82 + n_joints] or NULL
 *   x                device [batch][x_stride] or NULL: the same values written into the kinodynamic NLP's decision
 *                    vector at knots knot0 .. knot0 + n_points - 1 (p, f of the points, base, joints, com; other
 *                    entries untouched; n_joints must be 23) */
int hb_interpolate_humanoid_states(int64_t batch, int64_t n_points, int64_t n_joints, const double* initial,
                                   const double* final_, const int32_t* schedule, const double* phases_left,
                                   int64_t n_phases_left, int64_t stride_left, const double* phases_right,
                                   int64_t n_phases_right, int64_t stride_right, double* states, double* x,
                                   int64_t x_stride, int64_t knot0, void* stream);

/* CasADi external-function (codegen) ABI [ext] for the five nlpsol oracle functions, exported under the names
 *   hb_nlp_f (x, p -> f), hb_nlp_g (x, p -> g), hb_nlp_grad_f (x, p -> f, grad_f), hb_nlp_jac_g (x, p -> g, jac_g),
 *   hb_nlp_hess_l (x, p, lam_f, lam_g -> triu hess_l)
 * each with F(const double** arg, double** res, casadi_int* iw, double* w, int mem), F_n_in, F_n_out, F_sparsity_in,
 * F_sparsity_out (compact CCS vectors), F_work, F_name_in, F_name_out, F_incref, F_decref, F_alloc_mem, F_init_mem,
 * F_free_mem, F_checkout, F_release, so that `casadi.external("hb_nlp_jac_g", "libhippopt_b200.so")` loads them.
 * replaces: the generated-C oracle functions of `nlpsol` (SURVEY.md 8(b)); the alternative to the Python Callback shim.
 * External functions carry no handle: hb_external_bind(h) binds ONE problem per process (NULL unbinds); they share a host
 * pipeline and an x-keyed cache (f, grad_f, g, jac_g at one x = one evaluation).  hb_external_stats counts them. */
int hb_external_bind(hb_handle h);
int hb_external_stats(int64_t* first_order_evaluations, int64_t* hessian_evaluations);
typedef long long int hb_casadi_int; /* CasADi's casadi_int */
int hb_nlp_f(const double** arg, double** res, hb_casadi_int* iw, double* w, int mem);
hb_casadi_int hb_nlp_f_n_in(void);
hb_casadi_int hb_nlp_f_n_out(void);
const hb_casadi_int* hb_nlp_f_sparsity_in(hb_casadi_int i);
const hb_casadi_int* hb_nlp_f_sparsity_out(hb_casadi_int i);
int hb_nlp_f_work(hb_casadi_int* sz_arg, hb_casadi_int* sz_res, hb_casadi_int* sz_iw, hb_casadi_int* sz_w);
const char* hb_nlp_f_name_in(hb_casadi_int i);
const char* hb_nlp_f_name_out(hb_casadi_int i);
void hb_nlp_f_incref(void);
void hb_nlp_f_decref(void);
int hb_nlp_f_alloc_mem(void);
int hb_nlp_f_init_mem(int mem);
void hb_nlp_f_free_mem(int mem);
int hb_nlp_f_checkout(void);
void hb_nlp_f_release(int mem);
int hb_nlp_g(const double** arg, double** res, hb_casadi_int* iw, double* w, int mem);
hb_casadi_int hb_nlp_g_n_in(void);
hb_casadi_int hb_nlp_g_n_out(void);
const hb_casadi_int* hb_nlp_g_sparsity_in(hb_casadi_int i);
const hb_casadi_int* hb_nlp_g_sparsity_out(hb_casadi_int i);
int hb_nlp_g_work(hb_casadi_int* sz_arg, hb_casadi_int* sz_res, hb_casadi_int* sz_iw, hb_casadi_int* sz_w);
const char* hb_nlp_g_name_in(hb_casadi_int i);
const char* hb_nlp_g_name_out(hb_casadi_int i);
void hb_nlp_g_incref(void);
void hb_nlp_g_decref(void);
int hb_nlp_g_alloc_mem(void);
int hb_nlp_g_init_mem(int mem);
void hb_nlp_g_free_mem(int mem);
int hb_nlp_g_checkout(void);
void hb_nlp_g_release(int mem);
int hb_nlp_grad_f(const double** arg, double** res, hb_casadi_int* iw, double* w, int mem);
hb_casadi_int hb_nlp_grad_f_n_in(void);
hb_casadi_int hb_nlp_grad_f_n_out(void);
const hb_casadi_int* hb_nlp_grad_f_sparsity_in(hb_casadi_int i);
const hb_casadi_int* hb_nlp_grad_f_sparsity_out(hb_casadi_int i);
int hb_nlp_grad_f_work(hb_casadi_int* sz_arg, hb_casadi_int* sz_res, hb_casadi_int* sz_iw, hb_casadi_int* sz_w);
const char* hb_nlp_grad_f_name_in(hb_casadi_int i);
const char* hb_nlp_grad_f_name_out(hb_casadi_int i);
void hb_nlp_grad_f_incref(void);
void hb_nlp_grad_f_decref(void);
int hb_nlp_grad_f_alloc_mem(void);
int hb_nlp_grad_f_init_mem(int mem);
void hb_nlp_grad_f_free_mem(int mem);
int hb_nlp_grad_f_checkout(void);
void hb_nlp_grad_f_release(int mem);
int hb_nlp_jac_g(const double** arg, double** res, hb_casadi_int* iw, double* w, int mem);
hb_casadi_int hb_nlp_jac_g_n_in(void);
hb_casadi_int hb_nlp_jac_g_n_out(void);
const hb_casadi_int* hb_nlp_jac_g_sparsity_in(hb_casadi_int i);
const hb_casadi_int* hb_nlp_jac_g_sparsity_out(hb_casadi_int i);
int hb_nlp_jac_g_work(hb_casadi_int* sz_arg, hb_casadi_int* sz_res, hb_casadi_int* sz_iw, hb_casadi_int* sz_w);
const char* hb_nlp_jac_g_name_in(hb_casadi_int i);
const char* hb_nlp_jac_g_name_out(hb_casadi_int i);
void hb_nlp_jac_g_incref(void);
void hb_nlp_jac_g_decref(void);
int hb_nlp_jac_g_alloc_mem(void);
int hb_nlp_jac_g_init_mem(int mem);
void hb_nlp_jac_g_free_mem(int mem);
int hb_nlp_jac_g_checkout(void);
void hb_nlp_jac_g_release(int mem);
int hb_nlp_hess_l(const double** arg, double** res, hb_casadi_int* iw, double* w, int mem);
hb_casadi_int hb_nlp_hess_l_n_in(void);
hb_casadi_int hb_nlp_hess_l_n_out(void);
const hb_casadi_int* hb_nlp_hess_l_sparsity_in(hb_casadi_int i);
const hb_casadi_int* hb_nlp_hess_l_sparsity_out(hb_casadi_int i);
int hb_nlp_hess_l_work(hb_casadi_int* sz_arg, hb_casadi_int* sz_res, hb_casadi_int* sz_iw, hb_casadi_int* sz_w);
const char* hb_nlp_hess_l_name_in(hb_casadi_int i);
const char* hb_nlp_hess_l_name_out(hb_casadi_int i);
void hb_nlp_hess_l_incref(void);
void hb_nlp_hess_l_decref(void);
int hb_nlp_hess_l_alloc_mem(void);
int hb_nlp_hess_l_init_mem(int mem);
void hb_nlp_hess_l_free_mem(int mem);
int hb_nlp_hess_l_checkout(void);
void hb_nlp_hess_l_release(int mem);

/* Host-only: the (direction, body) task table of the kinematics kernel's packed tangent sweep for a tree
 * (hippopt_b200/csrc/sweep_schedule.h), for the CPU tests of the scheduler.  parent[nb]; typed: homogeneous rounds.
 *   tasks[32*32]  descriptor of (round, lane), 0 = idle
 *   info[40]      n_rounds, n_slots, n_tasks, n_heavy_tasks, heavy_mask, seed_mask, root_slot[27] */
int hb_debug_sweep_schedule(int32_t nb, const int32_t* parent, int32_t foot_l, int32_t foot_r, int32_t chest,
                            int32_t typed, int32_t* tasks, int32_t* info);
/* The same with n_base (0..4) of the four base quaternion directions in the sweep; hb_debug_sweep_schedule keeps all
 * four.  The kinematics kernel runs the schedule with none (its quaternion columns are closed-form). */
int hb_debug_sweep_schedule_n_base(int32_t nb, const int32_t* parent, int32_t foot_l, int32_t foot_r, int32_t chest,
                                   int32_t typed, int32_t n_base, int32_t* tasks, int32_t* info);

/* The smooth-step terrain jets of the contact kernel (hippopt_b200/csrc/kino_smooth.cuh), evaluated by the production
 * smooth_steps_surface and terrain_frame<1> at n points, for tests that compare them with a symbolic reference.
 *   tp   device [n][10]   terrain parameters of each point, (l, w, height, ox, oy) x 2
 *   pts  device [n][3]    (x, y, z)
 *   out  device [n][HB_SMOOTH_TERRAIN_OUT]  the 15 normalised coefficients of the order-4 surface jet T(x, y), then the
 *        TFrame fields in declaration order, 10 trivariate coefficients each: h, gx, gy, n[3], xh[3], yh[3], Dn[3][2] */
#define HB_SMOOTH_TERRAIN_OUT 195
int hb_debug_smooth_terrain(const double* tp, const double* pts, int64_t n, double* out, void* stream);

/* The same for kernel terrain 2 (tilted_steps_surface, K = n_steps general steps) with the same output layout.
 *   tp   device [n][10 n_steps]  terrain parameters of each point, (l, w, height, ox, oy, oz, yaw, n_x, n_y, n_z) per step */
int hb_debug_tilted_terrain(const double* tp, int32_t n_steps, const double* pts, int64_t n, double* out, void* stream);

const char* hb_last_error(void);

/* fp64 FMA throughput probe (TFLOP/s) used as roofline denominator when none is published */
int hb_probe_fp64_tflops(double* tflops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HIPPOPT_B200_H */
