/*
 * tsidb.h — C ABI of the B200-native batched TSID tick (libtsidb.so).
 *
 * This is the drop-in boundary for the per-tick hot path of
 * UW-RoboSoccer/tsid_control.  In the reference that path crosses the
 * boost.python binding of the `tsid` C++ library four times per tick
 * (ref:main.py:119-127):
 *
 *     HQPData = formulation.computeProblemData(t, q, v)      ref:main.py:119
 *     sol     = solver.solve(HQPData)                        ref:main.py:121
 *     tau     = formulation.getActuatorForces(sol)           ref:main.py:126
 *     dv      = formulation.getAccelerations(sol)            ref:main.py:127
 *     f       = formulation.getContactForce(name, sol)       ref:ctrl/WalkController.py:263,273
 *
 * for ONE robot.  Here one call does the same for n_envs independent robots.
 * Plain pointers and sizes only; no torch types.  All floating point is IEEE
 * fp64.  Per-env solver outcome is reported in status[] with the TSID
 * HQP_STATUS enum values so `status != 0` keeps the meaning it has at
 * ref:main.py:122.
 *
 * Ownership: the caller owns every buffer; the library owns the model/conf
 * constants and its workspace.  One handle per device; a handle is not
 * re-entrant: it has ONE set of workspaces, work counters and side streams, so
 * all calls on one handle must be ordered with each other on one CUDA stream
 * (two ticks enqueued on different streams, or a tsidb_compute_host issued while
 * an earlier asynchronous tsidb_compute is still running, race on them); use one
 * handle per stream.  Device entry points are asynchronous on `cuda_stream`.
 * There is no CPU fallback: every entry point fails (<0) without a CUDA device.
 *
 * Streams: a tick is enqueued on `cuda_stream`; internally the three contact-class
 * kernel chains (double support / single support / flight) are forked onto side
 * streams of the handle with events and joined back before the call returns, so the
 * caller sees ordinary stream order (also inside CUDA-graph capture).
 *
 * Environment knobs (diagnostics and tuning, not needed in normal use):
 *   TSIDB_CLASS_STREAMS=0   read by tsidb_create: keep every kernel of a tick on the caller's stream
 *   TSIDB_SMALL_N=n         read by tsidb_create: ticks of at most n envs (default 1024) run as ONE launch, one warp per env
 *                           through all three stages (no class sort, no per-class launches); 0 = always the batched pipeline
 *   TSIDB_SMALL_LOCAL_N=n   read by tsidb_create: such ticks of at most n envs (default 2 per SM) keep the hand-off images
 *                           between the stages in shared memory; 0 = always through global memory (tsidb_debug_terms needs it)
 *   TSIDB_SCHED_HINT=0      read by tsidb_create: no longest-first order inside the contact classes (tsidb_set_sched_hint)
 *   TSIDB_HOST_CHUNKS=k     read by tsidb_compute_host: k equal chunks instead of the tapered 1/8,3/8,3/8,1/8 split
 *   TSIDB_HOST_TAPER=d      read by tsidb_compute_host: first/last chunk = 1/d of the batch
 *   TSIDB_HOST_SPLIT=a,b,.. read by tsidb_compute_host: chunk sizes in 64ths of the batch (sum 64), e.g. 8,16,24,16
 *   TSIDB_HOST_TRACE=1      read by tsidb_compute_host: event time stamps per chunk on stderr
 */
#ifndef TSIDB_H_
#define TSIDB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSIDB_MAX_BODIES 24 /* floating base + revolute joints             */
#define TSIDB_MAX_NA 23     /* actuated joints                             */
#define TSIDB_MAX_NV 29
#define TSIDB_NFORCE 12     /* Contact6d: 4 corner forces, sole frame      */

/* TSID HQP_STATUS_* [UPSTREAM tsid solvers/fwd.hpp]; ref:main.py:122 tests != 0 */
enum {
  TSIDB_STATUS_UNKNOWN = -1,
  TSIDB_STATUS_OPTIMAL = 0,
  TSIDB_STATUS_INFEASIBLE = 1,
  TSIDB_STATUS_UNBOUNDED = 2,
  TSIDB_STATUS_MAX_ITER_REACHED = 3,
  TSIDB_STATUS_ERROR = 4
};

/* contact_mask bits (replaces formulation.addRigidContact/removeRigidContact,
 * ref:ctrl/WalkController.py:83-85,124-126, ref:legacy/biped.py:174,183,191-197,205-211) */
enum { TSIDB_CONTACT_LF = 1, TSIDB_CONTACT_RF = 2 };
enum { TSIDB_LAYOUT_ROWS = 0, TSIDB_LAYOUT_SOA = 1 };

/*
 * Compiled robot model — what tsid.RobotWrapper(urdf, [root], FreeFlyer)
 * holds after ref:ctrl/WalkController.py:13-19.  Produced by
 * tsid_control_b200/model_compiler.py.  Body 0 is the free-flyer; bodies
 * 1..na are JointModelRZ in Pinocchio order.  Matrices are row-major.
 */
typedef struct tsidb_model {
  int32_t nb;                               /* bodies = na + 1                       */
  int32_t parent[TSIDB_MAX_BODIES];         /* parent body, -1 for body 0            */
  double jR[TSIDB_MAX_BODIES][9];           /* joint placement in the parent body    */
  double jp[TSIDB_MAX_BODIES][3];
  double mass[TSIDB_MAX_BODIES];
  double com[TSIDB_MAX_BODIES][3];          /* lever, body frame                     */
  double inertia[TSIDB_MAX_BODIES][9];      /* about the CoM, body frame             */
  int32_t foot_body[2];                     /* [0]=LF, [1]=RF: parent body of sole   */
  double fR[2][9];                          /* sole frame placement in that body     */
  double fp[2][3];
  double gravity[3];                        /* (0,0,-9.81)                           */
} tsidb_model;

/*
 * Controller constants — the values ref:ctrl/conf.py:21-72 /
 * ref:legacy/op3_conf.py:4-50 feed into the tsid task objects at
 * ref:ctrl/WalkController.py:55-187 / ref:legacy/biped.py:31-151.
 */
typedef struct tsidb_conf {
  /* Contact6d (ref:ctrl/WalkController.py:55-70) */
  double contact_points[3][4];              /* corners in the sole frame             */
  double contact_normal[3];
  double mu, fmin, fmax;
  double kp_contact[6], kd_contact[6];
  double w_force_reg;                       /* conf.w_forceRef                        */
  double force_reg_weights[6];              /* [UPSTREAM Contact6d] 1,1,1e-3,2,2,2   */
  /* TaskSE3Equality feet (ref:ctrl/WalkController.py:90-104,131-144) */
  double w_foot, kp_foot[6], kd_foot[6];
  /* TaskComEquality (ref:ctrl/WalkController.py:147-152) */
  double w_com, kp_com[3], kd_com[3];
  /* TaskJointPosture (ref:ctrl/WalkController.py:159-165) */
  double w_posture, kp_posture[TSIDB_MAX_NA], kd_posture[TSIDB_MAX_NA];
  /* legacy TaskAMEquality (ref:legacy/biped.py:82-87); w_am <= 0 disables */
  double w_am, kp_am[3];
  /* TaskActuationBounds (ref:ctrl/WalkController.py:168-176); enabled iff w_torque_bounds > 0 */
  int32_t use_torque_bounds;
  double tau_min[TSIDB_MAX_NA], tau_max[TSIDB_MAX_NA];
  /* TaskJointBounds (ref:ctrl/WalkController.py:178-184); enabled iff w_joint_bounds > 0 */
  int32_t use_joint_bounds;
  double v_min[TSIDB_MAX_NA], v_max[TSIDB_MAX_NA];
  double joint_bounds_dt;                   /* [UPSTREAM TaskJointBounds] 2*conf.dt  */
  /* SolverHQuadProgFast (ref:ctrl/WalkController.py:186-187) */
  double hessian_reg;                       /* [UPSTREAM] 1e-8                       */
  int32_t max_iter;                         /* [UPSTREAM] 1000                       */
  int32_t pad_;
} tsidb_conf;

typedef struct tsidb_handle tsidb_handle;

/* Array layouts.  Every per-env array (state, references, outputs) of one call uses
 * the same `layout` argument:
 *   TSIDB_LAYOUT_ROWS (0)  [N][dof] row-major — the PyTorch-natural [N, dof] tensor
 *   TSIDB_LAYOUT_SOA  (1)  [dof][N]           — struct of arrays
 * so neither needs a transposing copy.
 *
 * Per-env task references, one struct of device (or host) pointers.  A NULL
 * pointer selects the reference the controller was constructed with
 * (tsidb_set_default_refs), broadcast to every env.                          */
typedef struct tsidb_refs {
  const double* com;        /* [9]  pos, vel, acc            TaskComEquality.setReference  ref:ctrl/WalkController.py:152 */
  const double* foot_lf;    /* [24] SE3 pos (p, R col-major) 12, vel 6, acc 6   task_LF.setReference ref:ctrl/WalkController.py:196 */
  const double* foot_rf;    /* [24]                                             task_RF.setReference ref:ctrl/WalkController.py:197 */
  const double* contact_lf; /* [12] SE3 (p, R col-major)     contactLF.setReference ref:ctrl/WalkController.py:81 */
  const double* contact_rf; /* [12]                          contactRF.setReference ref:ctrl/WalkController.py:122 */
  const double* posture;    /* [na]                          postureTask.setReference ref:ctrl/WalkController.py:165 */
} tsidb_refs;

/* Optional per-env diagnostics/outputs (any pointer may be NULL). */
typedef struct tsidb_aux_out {
  double* com;        /* [9]  com, vcom, acom_drift   robot.com(data) ref:main.py:135          */
  double* foot_lf;    /* [12] sole placement (p, R col-major)  robot.framePosition ref:main.py:139 */
  double* foot_rf;    /* [12]                                                     ref:main.py:141 */
  double* wrench;     /* [12] T*f per foot (LF 6, RF 6), the f_lf/f_rf of ref:ctrl/WalkController.py:263,273 */
  /* sol.lambda [UPSTREAM HQPOutput]: Lagrange multipliers of the inequality rows in the working set, in working-set
   * order, and the row each one belongs to (tsidb_ci_row numbering, -1 = unused slot); zero / -1 when status != 0.
   * The multipliers of the always-active equalities are not formed: the equalities are eliminated, not added one
   * by one (the reference itself never reads sol.lambda). */
  double* lambda;      /* [32] always row-major [N][32] */
  int32_t* lambda_row; /* [32] always row-major [N][32] */
} tsidb_aux_out;

/* ---- lifecycle ------------------------------------------------------------------ */
/* replaces WalkController.__init__ / Biped.__init__ up to solver.resize
 * (ref:ctrl/WalkController.py:12-187, ref:legacy/biped.py:7-151) */
int tsidb_create(const tsidb_model* model, const tsidb_conf* conf, int max_envs, int device,
                 tsidb_handle** out);
void tsidb_destroy(tsidb_handle* h);
const char* tsidb_last_error(void);
/* model sizes: na, nv, nq, and the reference's one-sided inequality count 2*nIn
 * (for mapping active_set bits to CI rows) */
int tsidb_sizes(const tsidb_handle* h, int* na, int* nv, int* nq);

/* default references broadcast when a tsidb_refs pointer is NULL (host pointers,
 * same element order as tsidb_refs, contiguous) */
int tsidb_set_default_refs(tsidb_handle* h, const double* com9, const double* foot_lf24,
                           const double* foot_rf24, const double* contact_lf12,
                           const double* contact_rf12, const double* posture_na);

/* ---- the tick ------------------------------------------------------------------- */
/*
 * computeProblemData + solve + getActuatorForces/getAccelerations/getContactForce
 * for n_envs robots (ref:main.py:119-127).  All pointers are DEVICE pointers.
 *   q [nq], v [nv]            state, in the layout selected by `layout`
 *   contact_mask [n_envs]     TSIDB_CONTACT_* bits
 *   tau [na], ddq [nv]        outputs, same layout
 *   f [24]                    LF corner forces 0..11, RF 12..23, 0 for a foot not in contact
 *   status, iters [n_envs]    HQP status / eiquadprog iteration count
 *   active_set [3][n_envs]    (may be NULL) bit r of the 192-bit word = one-sided
 *                             canonical inequality row r is in the final working set;
 *                             row numbering in tsidb_ci_row()
 */
int tsidb_compute(tsidb_handle* h, int n_envs, int layout,
                  const double* q, const double* v, const uint8_t* contact_mask,
                  const tsidb_refs* refs, double* tau, double* ddq, double* f,
                  int32_t* status, int32_t* iters, uint64_t* active_set,
                  const tsidb_aux_out* aux, void* cuda_stream);

/* Same tick with HOST buffers ([N][dof] row-major, contiguous): pinned staging,
 * H2D, kernels, D2H inside the call; returns after the results are in host memory.
 * This is the call the reference-side binding makes (INTEGRATION.md).
 * ddq and f may be NULL: a caller that only drives the actuators (ref:main.py:126)
 * then gets tau, status and iters back and the accelerations and contact forces
 * stay on the device (168 instead of 592 bytes per env over PCIe).              */
int tsidb_compute_host(tsidb_handle* h, int n_envs, const double* q, const double* v,
                       const uint8_t* contact_mask, const tsidb_refs* refs_host,
                       double* tau, double* ddq, double* f, int32_t* status, int32_t* iters,
                       uint64_t* active_set);

/* The same host-buffer tick when the references and the contact phases already live on the DEVICE — the gait state
 * of tsidb_gait_state(), advanced there by tsidb_gait_step(), or any [N][dof] device arrays of the caller — so that
 * only q and v (424 B per robot/v1 env instead of 1 233 B) cross PCIe on the way in.  This is the deployment the
 * reference intends around update_tasks (ref:ctrl/WalkController.py:189-206): the simulator hands over the state,
 * the walking references are generated next to the solver.  contact_mask_dev and the arrays of refs_dev are device
 * pointers (null = all feet in contact / handle defaults); q, v and the outputs are host pointers as above. */
int tsidb_compute_host_devrefs(tsidb_handle* h, int n_envs, const double* q, const double* v,
                               const uint8_t* contact_mask_dev, const tsidb_refs* refs_dev,
                               double* tau, double* ddq, double* f, int32_t* status, int32_t* iters,
                               uint64_t* active_set);

/* Diagnostics for parity tests: the dynamics terms the last tick handed from the dynamics kernel to the solver stages
 * for ONE env — M [nv][nv], nle [nv], the sole Jacobians JF [2][6][nv] (LOCAL frame, LF then RF), the dv block of the
 * Hessian H [nv][nv] (lower triangle significant) and the dv part of the gradient g [nv] — what
 * RobotWrapper::computeAllTerms / the solver's H, g build produce inside ref:main.py:119,121.  Host pointers;
 * synchronous.  Valid when the last tick ran without a contact mask or with at most TSIDB_SMALL_N envs (no class sort:
 * slot == env) on a handle created with TSIDB_SMALL_LOCAL_N=0 (the images of the smallest ticks otherwise stay in shared
 * memory); n_contacts = contacts of that env in that tick.  A tsidb_problem_data call also fills these images (slot ==
 * env, every env of that call): after it this function reads that call's terms. */
int tsidb_debug_terms(tsidb_handle* h, int env, int n_contacts, double* M, double* nle, double* JF, double* H, double* g);

/* ---- the assembled QP without the solve ---------------------------------------------------------------------------
 * formulation.computeProblemData (ref:main.py:119) for n_envs robots: exactly the problem SolverHQuadProgFast hands to
 * eiquadprog for each env,
 *     min 1/2 x^T H x + g^T x   s.t.   CE x + ce0 = 0,   CI x + ci0 >= 0,
 * in compact variables x = [dv; f of the feet in contact, LF first] (n = nv + 12 nc; the force-block order of the tick).
 *   equality rows:   base dynamics (6; ce0 = h_u), then the contact-motion rows of the feet in contact, LF first;
 *   inequality rows: the blocks [LF force (in contact), RF force (in contact), actuation (use_torque_bounds), joint bounds
 *                    (use_joint_bounds)], each stacked [lower rows (A, -lb); upper rows (-A, ub)] as SolverHQuadProgFast
 *                    stacks a two-sided constraint.
 * Every array is per env, row-major, DEVICE memory, zero outside the env's (n, neq, nin); any pointer may be NULL (that
 * part is not written).  H, CE and CI must be 16-byte aligned.  The maxima come from tsidb_problem_sizes:
 * n_max = nv + 24, neq_max = 18, nin_max = 2 (34 + na use_torque_bounds + nv use_joint_bounds) (robot/v1: 50 / 18 / 160). */
typedef struct tsidb_problem_out {
  double* H;      /* [N][n_max][n_max]   full symmetric Hessian, regulariser included */
  double* g;      /* [N][n_max]                                                         */
  double* CE;     /* [N][neq_max][n_max]                                                */
  double* ce0;    /* [N][neq_max]                                                       */
  double* CI;     /* [N][nin_max][n_max]  one-sided rows                                */
  double* ci0;    /* [N][nin_max]                                                       */
  int32_t* sizes; /* [N][3]  n, neq, nin of this env                                    */
  /* The struct grew at its end with the actuation map, tau = TA x + ta0 (getActuatorForces: TA = [M_a | -J_c,a^T],
   * ta0 = h_a); a caller that zero-initialises the struct keeps the six parts above and nothing more. */
  double* TA;     /* [N][na][n_max]      16-byte aligned like H, CE and CI                */
  double* ta0;    /* [N][na]                                                            */
} tsidb_problem_out;

int tsidb_problem_sizes(const tsidb_handle* h, int* n_max, int* neq_max, int* nin_max);
/* q, v, contact_mask and refs as in tsidb_compute (`layout` applies to them only; the outputs are always row-major per
 * env); a NULL mask means double support, NULL refs the handle's defaults.  Asynchronous on cuda_stream.  The call keeps
 * no state that a later tick reads (it leaves the scheduling hint's forecast alone), but it uses the handle's image
 * workspaces, so it is ordered with the other calls on the handle like any of them, and tsidb_debug_terms reads its
 * images afterwards. */
int tsidb_problem_data(tsidb_handle* h, int n_envs, int layout, const double* q, const double* v,
                       const uint8_t* contact_mask, const tsidb_refs* refs, const tsidb_problem_out* out, void* cuda_stream);

/* ---- solving a caller-supplied QP ---------------------------------------------------------------------------------
 * tsidb_qp_solve runs eiquadprog-fast (the solver SolverHQuadProgFast calls, with the handle's conf.max_iter) on n_envs
 * problems in the layout tsidb_problem_data writes, possibly modified or enlarged by the caller: qp->H, g, CE, ce0, CI,
 * ci0 and sizes are read (DEVICE memory, per env row-major with the strides n_max, neq_max, nin_max, which may exceed
 * tsidb_problem_sizes).  Nothing outside an env's own (n, neq, nin) = qp->sizes[e] is read, so padding may hold anything.
 * Required: H, g, sizes, out->x, out->status; CE and ce0 when neq_max > 0; CI and ci0 when nin_max > 0; TA and ta0 when
 * out->tau is given.  n_max <= TSIDB_QP_MAX_N, neq_max <= n_max, nin_max <= TSIDB_QP_MAX_NIN.  Any other output pointer
 * may be NULL.  An env whose sizes violate 1 <= n <= n_max, 0 <= neq <= min(n, neq_max), 0 <= nin <= nin_max gets
 * TSIDB_STATUS_ERROR and zero outputs; the rest of the batch is solved.  Statuses as the tick maps eiquadprog's result
 * (H not positive definite or an unbounded step: INFEASIBLE; max_iter: MAX_ITER_REACHED; a redundant equality row:
 * ERROR); x, the working set and the multipliers are written for OPTIMAL and MAX_ITER_REACHED, zeros (active: -1)
 * otherwise.  At the optimum H x + g = CI^T lambda + CE^T lambda_eq over the working set.
 * The call uses none of the handle's workspaces or forecast (only its launch counter), so it may be enqueued on any
 * stream, also while a tick of the same handle runs on another one.  Asynchronous on cuda_stream, no host round trip. */
#define TSIDB_QP_MAX_N 64
#define TSIDB_QP_MAX_NIN 512
typedef struct tsidb_qp_out {
  double* x;          /* [N][n_max]    primal solution, in the caller's variable order                              */
  int32_t* status;    /* [N]           TSIDB_STATUS_*                                                               */
  int32_t* iters;     /* [N]           eiquadprog iteration count                                                   */
  int32_t* active;    /* [N][n_max]    CI rows of the final working set in working-set order, -1 padded             */
  double* lambda;     /* [N][n_max]    their multipliers, same order                                                */
  double* lambda_eq;  /* [N][neq_max]  multipliers of the equality rows                                             */
  double* tau;        /* [N][na]       TA x + ta0                                                                   */
} tsidb_qp_out;

int tsidb_qp_solve(tsidb_handle* h, int n_envs, int n_max, int neq_max, int nin_max, const tsidb_problem_out* qp,
                   const tsidb_qp_out* out, void* cuda_stream);

/* ---- differentiating the QP solve ---------------------------------------------------------------------------------
 * tsidb_qp_grad is the adjoint (reverse-mode derivative) of tsidb_qp_solve: given the problem qp that was solved (same
 * strides and required arrays as the solve; TA also when grad_in->tau is given), the solve's result sol (x, status,
 * active, lambda and, when neq_max > 0, lambda_eq are read) and the gradients of a loss with respect to the solve's
 * outputs, grad_in (x, lambda, lambda_eq, tau: dL/d of each, same layout; a NULL part counts as zero; status, iters and
 * active must be NULL), it writes dL/d of the problem's parts into grad_out (H, g, CE, ce0, CI, ci0, TA, ta0: NULL = not
 * written; sizes must be NULL), every byte of each requested part with zeros in the padding.  All DEVICE memory.
 * The derivative is the one of the KKT system of the final working set W (rows CE and CI_W, multipliers lambda_eq and
 * lambda): at a degenerate point (a row of W with a zero multiplier, or an inactive row with zero slack) it is the
 * one-sided derivative that keeps W.  With G = [CE; CI_W], nu = [lambda_eq; lambda_W] and (p, q) the solution of
 * H p + G' q = dL/dx + TA' dL/dtau, G p = -[dL/dlambda_eq; dL/dlambda_W]:  dg = -p, dG = nu p' - q x', d[ce0; ci0_W] = -q,
 * dTA = dL/dtau x', dta0 = dL/dtau; rows of CI outside W get zero.  The solve reads only the lower triangle of H, so
 * dL/dH is lower triangular: dH = tril(P + P', -1) + diag(P) with P = -p x'; a caller with a symmetric H by
 * construction gets the same total as with the symmetric convention.
 * An env is differentiated (status[e] = TSIDB_STATUS_OPTIMAL) when sol->status[e] is OPTIMAL, its sizes fit the strides,
 * its working set is valid (entries in [0, nin), no duplicate, -1 padding after the last entry, neq + |W| <= n), H is
 * positive definite and the rows of W are independent; otherwise status[e] = TSIDB_STATUS_ERROR and its gradients are
 * zero.  Nothing outside an env's (n, neq, nin) and working set is read.  No workspace of the handle is used, so the call
 * may run on any stream.  Asynchronous on cuda_stream, no host round trip. */
int tsidb_qp_grad(tsidb_handle* h, int n_envs, int n_max, int neq_max, int nin_max, const tsidb_problem_out* qp,
                  const tsidb_qp_out* sol, const tsidb_qp_out* grad_in, const tsidb_problem_out* grad_out, int32_t* status,
                  void* cuda_stream);

/* ---- differentiating through the task references ------------------------------------------------------------------
 * tsidb_refs_grad is the adjoint of the map references -> (g, ce0) of tsidb_problem_data: given dg = dL/dg [N][n_max] and
 * dce0 = dL/dce0 [N][neq_max] (row-major DEVICE arrays with the caller's strides, n_max >= and neq_max >= the values of
 * tsidb_problem_sizes, e.g. what tsidb_qp_grad returns; NULL counts as zero), it writes dL/d of each reference array the
 * caller asks for in `out` (NULL = not written).  Only g and the contact-motion rows of ce0 depend on the references, and
 * only columns 0..nv of dg and rows 6..6+6nc of dce0 are read, so padding and appended variables or rows may hold
 * anything.  q, v, contact_mask, refs and `layout` as in tsidb_problem_data; `layout` also applies to the outputs.  The
 * gradient is taken with respect to the raw doubles of each array (the 9 column-major entries of an SE3 reference's
 * rotation, not a tangent vector), for a NULL reference array with respect to the default that was used; every requested
 * byte is written, and the contact reference of a foot that is not in contact gets exact zeros.  The SE3 logarithm is
 * differentiated branch by branch as the tick computes it (INTEGRATION.md, "Differentiating through the references").
 * No workspace of the handle is used, so the call may run on any stream.  Asynchronous on cuda_stream. */
typedef struct tsidb_refs_out { /* dL/d of each tsidb_refs array, same shapes; NULL = not written */
  double *com, *foot_lf, *foot_rf, *contact_lf, *contact_rf, *posture;
} tsidb_refs_out;
int tsidb_refs_grad(tsidb_handle* h, int n_envs, int layout, const double* q, const double* v, const uint8_t* contact_mask,
                    const tsidb_refs* refs, int n_max, int neq_max, const double* dg, const double* dce0,
                    const tsidb_refs_out* out, void* cuda_stream);

/* ---- differentiating with respect to the state ----------------------------------------------------------------------
 * tsidb_state_grad is the adjoint of all of tsidb_problem_data (H, g, CE, ce0, CI, ci0, TA, ta0) with respect to q and
 * v: given `grad` = dL/d of each part (DEVICE arrays in the layout tsidb_qp_grad writes, with the caller's strides n_max,
 * neq_max, nin_max >= the values of tsidb_problem_sizes; grad NULL or a NULL part counts as zero), it writes dL/dq [N][nq]
 * and dL/dv [N][nv] (NULL = not written, not both), in the call's `layout` like q and v.  q, v, contact_mask and refs as
 * in tsidb_problem_data.  grad->H is the gradient with respect to every entry of the full H the export writes, so the
 * lower-triangular gradient of tsidb_qp_grad composes unchanged.  Only the entries inside an env's own (n, neq, nin)
 * that depend on the state are read (INTEGRATION.md, "Differentiating with respect to the state", lists them); padding,
 * appended variables and rows and the constant blocks may hold anything.  The gradient is with respect to the raw doubles
 * of q (the free-flyer quaternion's 4 components through the tick's unnormalised quat -> R formula).  A joint-bound entry
 * of ci0 that the export clips to +-1e10 has zero derivative.  No workspace of the handle is used, so the call may run
 * on any stream.  Asynchronous on cuda_stream. */
int tsidb_state_grad(tsidb_handle* h, int n_envs, int layout, const double* q, const double* v, const uint8_t* contact_mask,
                     const tsidb_refs* refs, int n_max, int neq_max, int nin_max, const tsidb_problem_out* grad, double* dq,
                     double* dv, void* cuda_stream);

/* controller.integrate_dv(q, v, dv, dt) (ref:ctrl/WalkController.py:291-295,
 * ref:legacy/biped.py:236-240): v_mean = v + dt/2*dv; v += dt*dv;
 * q = pin.integrate(q, dt*v_mean).  In place on device arrays.                   */
int tsidb_integrate(tsidb_handle* h, int n_envs, int layout, double* q, double* v,
                    const double* dv, double dt, void* cuda_stream);

/* robot.framePosition / robot.com without a solve (ref:ctrl/WalkController.py:73,79,120,151):
 * used at construction and at contact switches.                                   */
int tsidb_kinematics(tsidb_handle* h, int n_envs, int layout, const double* q,
                     const double* v, const tsidb_aux_out* aux, void* cuda_stream);

/* ---- gait phase machine and closed-loop rollout on the device --------------------------------
 * What the reference intends around update_tasks (ref:ctrl/WalkController.py:189-206; the call is commented out
 * at ref:main.py:117) and never finishes (ref:ctrl/Walk_Planner.py:14-32 does not run): per-env gait phase,
 * contact switching with the legacy semantics (ref:legacy/biped.py:168-212), swing-foot references with the
 * FootTrajectory shape (ref:ctrl/Foot_Trajectory.py:8-19), CoM reference by LIPM Euler steps
 * (ref:ctrl/LIPM.py:44-47).  State and references live in library-owned device arrays; see
 * tsid_control_b200/csrc/tsidb_gait.cuh for the exact rules and tests/gait_ref.py for their numpy restatement. */
typedef struct tsidb_gait_conf {
  double dt;             /* conf.dt            ref:ctrl/conf.py:21 */
  double step_duration;  /* conf.step_duration ref:ctrl/conf.py:27 (duration of one swing) */
  double step_length;    /* conf.step_length   ref:ctrl/conf.py:26 */
  double step_height;    /* conf.step_height   ref:ctrl/conf.py:24 */
  double com_height;     /* LIPM h0            ref:ctrl/LIPM.py:6,15 */
} tsidb_gait_conf;

/* (re)start the gait of n_envs envs from the default references: phase0 [N] in [0,1) and vcmd [N][2] are DEVICE
 * pointers (NULL = 0).  Asynchronous on cuda_stream except for one small synchronising upload. */
int tsidb_gait_reset(tsidb_handle* h, int n_envs, const tsidb_gait_conf* conf, const double* phase0,
                     const double* vcmd, void* cuda_stream);
/* device pointers of the gait's references / contact mask / phase / failure counters (any out pointer may be NULL);
 * valid until tsidb_destroy.  refs_out->posture is NULL (the default posture reference applies). */
int tsidb_gait_state(tsidb_handle* h, tsidb_refs* refs_out, const uint8_t** mask_out, const double** phase_out,
                     const int32_t** fails_out);
/* advance the phase machine by one tick given the sole placements the tick measured (tsidb_aux_out.foot_*,
 * [N][12] row-major device arrays) and its status (may be NULL). */
int tsidb_gait_step(tsidb_handle* h, int n_envs, const double* foot_lf_now, const double* foot_rf_now,
                    const int32_t* status, void* cuda_stream);
/* n_steps x { tick with the gait's references and mask -> integrate_dv -> gait step } with no host round trip:
 * the batched, closed-loop form of ref:main.py:110-128.  q, v ([N][nq], [N][nv], DEVICE, row-major) are
 * advanced in place; tau/ddq/f/status/iters hold the last step's outputs.  use_graph != 0 captures the step in
 * a CUDA graph and replays it (launch-bound small batches).  Returns after the last step has been enqueued
 * (use_graph: after it has finished). */
int tsidb_rollout(tsidb_handle* h, int n_envs, int n_steps, double* q, double* v, double* tau, double* ddq,
                  double* f, int32_t* status, int32_t* iters, int use_graph, void* cuda_stream);

/* per-env diagnostics from a tick's auxiliary outputs (all [N][k] row-major DEVICE arrays; any output may be NULL):
 *   cop [3]            controller.get_cop(sol)              ref:ctrl/WalkController.py:255-289
 *   capture_point [3]  Biped.compute_capture_point(com, dcom, w)  ref:legacy/biped.py:224-227 (omega = w)
 *   support [4]        Biped.compute_support_polygon()      ref:legacy/biped.py:229-234 (lf.xy, rf.xy)      */
int tsidb_diagnostics(tsidb_handle* h, int n_envs, const tsidb_aux_out* aux, const uint8_t* contact_mask,
                      double omega, double* cop, double* capture_point, double* support, void* cuda_stream);

/* canonical one-sided inequality row numbering used by active_set:
 *   block 0: LF force rows (17), block 1: RF force rows (17),
 *   block 2: actuation rows (na), block 3: joint-bound rows (nv)
 *   row = 2*offset(block) + side*rows(block) + i   (side 0 = lower, 1 = upper),
 *   i.e. each two-sided block is stacked [lower rows; upper rows] exactly as
 *   [UPSTREAM SolverHQuadProgFast] stacks CI.  Returns -1 when out of range.      */
int tsidb_ci_row(const tsidb_handle* h, int block, int side, int i);

/* measured FP64 DFMA throughput of this device (TFLOP/s), the roofline
 * denominator for the solver kernels (BASELINE.md §2 asks for it).               */
int tsidb_fp64_peak(int device, double* tflops_out);

/* counters: kernel launches issued by this handle since creation */
int64_t tsidb_launch_count(const tsidb_handle* h);

/* Instrumentation for bench.py (the reference has no counterpart; its only timer is the unused
 * start_time of ref:main.py:54,113).  With timing on, every tick records CUDA events between its
 * kernels on the launching stream; tsidb_last_tick_ms waits for the last tick and returns the
 * durations of {class sort, dynamics+assembly, equality elimination, null-space basis,
 * active set+decode} in milliseconds.  A timed tick runs stage by stage on the launching stream
 * (the contact-class chains are not forked onto side streams), so the five durations add up to
 * slightly more than an untimed tick takes.                                                      */
int tsidb_set_timing(tsidb_handle* h, int on);
int tsidb_last_tick_ms(tsidb_handle* h, float* ms5);

/* Scheduling hint (no counterpart in the reference; never changes a result).  The class sort of a tick orders the envs
 * of a contact class by their active-set iteration count in the handle's PREVIOUS tick, most iterations first, so the
 * longest solves start first and the per-class kernels end with a shorter tail.  In closed loop the counts change slowly
 * from tick to tick (consecutive ticks of a replayed rollout: +2.8 % ticks/s); for a batch that is ticked again unchanged
 * the forecast is exact (+5 %).  On by default (TSIDB_SCHED_HINT=0 at tsidb_create turns it off); off, every env of a class shares one bucket. */
int tsidb_set_sched_hint(tsidb_handle* h, int on);

/* ---- the reference's planners on the device (SURVEY.md §8f-1), one thread per env ---------------------------
 * tsidb_foot_trajectory: FootTrajectory(t = [t0, t1], start, target, step_height, rise_ratio) of
 * ref:ctrl/Foot_Trajectory.py:6-43 evaluated at t[e] for every env: start4/target4 [N][4] = (x, y, z, yaw),
 * out16 [N][16] = value, 1st, 2nd and 3rd derivative of (x, y, z, yaw).  (The reference's get_velocity /
 * get_acceleration return the 2nd and 3rd derivative, :35,:43.)  All arrays are device pointers. */
int tsidb_foot_trajectory(tsidb_handle* h, int n_envs, double t0, double t1, const double* start4, const double* target4,
                          double step_height, double rise_ratio, const double* t, double* out16, void* cuda_stream);
/* tsidb_gait_set_plan: hand a footstep plan (the output of tsidb_footstep_plan, device pointers; copied) to the gait
 * phase machine: from then on the swing foot of every gait step goes to the env's next footstep of that side along
 * FootTrajectory([0, step_duration], start, target, step_height, rise_ratio) — x, y and yaw linear in time, z the 3-
 * or 4-knot spline — with the first and second derivatives as the velocity / acceleration reference of the foot
 * task; an exhausted plan sets the foot down where it is.  steps == NULL returns to straight steps along x.  Needs
 * tsidb_gait_reset first (n_envs <= its n_envs). */
int tsidb_gait_set_plan(tsidb_handle* h, int n_envs, const double* steps, const int32_t* n_steps, int max_steps,
                        double rise_ratio, void* cuda_stream);
/* tsidb_footstep_plan: FootstepPlanner(step_width, step_length).plan(path, init_supports) of
 * ref:ctrl/Footstep_Planner.py:92-125 per env: path [N][max_pts][2] with n_pts[e] valid points (null: max_pts for
 * every env), init8 [N][2][4] the two initial supports (x, y, yaw, side 0 = left / 1 = right), steps
 * [N][max_steps][4] = (x, y, yaw, side), n_steps[e] = footsteps written (initial supports included; -1: max_steps
 * too small).  Device pointers. */
int tsidb_footstep_plan(tsidb_handle* h, int n_envs, const double* path, const int32_t* n_pts, int max_pts, const double* init8,
                        double step_length, double step_width, double* steps, int32_t* n_steps, int max_steps, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* TSIDB_H_ */
