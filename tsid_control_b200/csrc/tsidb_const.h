/* tsidb_const.h — per-handle constant block (lives in __constant__ memory on the device)
 * and the shared-memory layout of one env's workspace.  Shared by tsidb.cu (host side fills
 * it) and tsidb_kernels.cuh (device side reads it).                                      */
#ifndef TSIDB_CONST_H_
#define TSIDB_CONST_H_
#include <stdint.h>

#define TSIDB_NVX 26   /* largest nv this build keeps in shared memory (robot/v1)          */
#define TSIDB_NX 50    /* nv + 24                                                          */
#define TSIDB_MRED 32  /* n - nEq = na + 6*nc <= 32: one lane per reduced coordinate       */
#define TSIDB_WARPS_PER_BLOCK 16   /* dynamics kernel: warps per CTA (they share the staged model constants) */
#define TSIDB_D_CTAS_PER_SM 1     /* dynamics kernel: resident CTAs per SM (16 warps)                       */
#define TSIDB_E_WARPS 8            /* elimination kernel, double support: one-warp CTAs resident per SM */
#define TSIDB_E_WARPS_LIGHT 12     /* elimination kernel, single support and flight */
/* warps per CTA of the per-class kernels (the resident warps per SM above are split into CTAs of this width; a
 * narrow CTA returns its shared memory and registers as soon as its warps run out of work) */
#define TSIDB_E_CTA_WARPS 1
#define TSIDB_A_CTA_WARPS_DS 4
#define TSIDB_A_CTA_WARPS_SS 4
#define TSIDB_A_CTA_WARPS(NC) ((NC) == 2 ? TSIDB_A_CTA_WARPS_DS : TSIDB_A_CTA_WARPS_SS)
/* CTA-wide phase lock-step (all warps of a CTA run the same phase at the same time, so one instruction-cache
 * line serves all of them).  It paid off for the fused 215 KB kernel of the first generation; with one kernel
 * per stage the code fits the instruction cache and free-running warps hide each other's latencies better
 * (measured: elimination 1.82 -> 1.63 ms, dynamics 1.24 -> 1.17 ms), so both are off. */
#define TSIDB_LOCK_D 0
#define TSIDB_LOCK_E 0
#define TSIDB_MAX_SLOTS 6

struct DevConst {
  int32_t nb, na, nv, nq;
  int32_t maxdepth;
  int32_t parent[24];
  int32_t depth[24];
  int32_t sibrank[24];      /* rank among the children of the same parent              */
  int32_t maxsib[8];        /* per depth: largest sibling count                        */
  int32_t foot_body[2];
  uint32_t foot_support[2]; /* bit b set: body b is on the chain root -> foot          */
  int32_t use_tb, use_jb, use_am, max_iter;
  int32_t nin_ref_fixed;    /* reference one-sided rows that do not depend on contacts  */
  int32_t pad0;
  double jR[24][9], jp[24][3], mass[24], com[24][3], inertia[24][9];
  double fR[2][9], fp[2][3];
  double gravity[3];
  /* Contact6d */
  double T[6][12];          /* force generator                                          */
  double fric[4][3];        /* pyramid rows of one corner                               */
  double nrm[3];
  double fmin, fmax;
  double kp_contact[6], kd_contact[6], kp_foot[6], kd_foot[6], kp_com[3], kd_com[3];
  double kp_post[23], kd_post[23], kp_am[3];
  double w_foot, w_com, w_post, w_am, w_freg, hreg;
  double tau_min[23], tau_max[23], v_min[23], v_max[23], jb_dt;
  /* force block of the Hessian, identical for every env and foot:
   * H_f = w_freg (W T)^T (W T) + hreg I = Lf Lf^T                                      */
  double Lf[12][12];        /* lower Cholesky factor                                    */
  double Lfinv[12][12];     /* its inverse (lower)                                      */
  double Hf_trace, Lfinv_trace;
  /* default references (tsidb_set_default_refs) */
  double ref_com[9], ref_foot[2][24], ref_contact[2][12], ref_posture[23];
};

/* shared-memory layout of one env in the dynamics kernel (doubles) */
#define SM_LDM 27
#define SM_LDB 19
#define SM_oM 0                         /* region 0, reused in time: subtree-sum scratch of K1 (609) -> M 26 x 27 -> dv
                                           block of the Hessian 26 x 27                                        702 */
#define SM_oH SM_oM
#define SM_oGv (SM_oM + 702)            /* gradient (follows H: one bulk store)    50 */
#define SM_oJF (SM_oGv + 50)            /* JF       2 x 6 x 26                    312 */
#define SM_oJcom (SM_oJF + 312)         /* Jcom     3 x 26                         78 */
#define SM_oAg (SM_oJcom + 78)          /* Ag_ang   3 x 26                         78 */
#define SM_oNle (SM_oAg + 78)           /* nle      26                             26 */
#define SM_oBv (SM_oNle + 26)           /* task vectors                            64 */
#define SM_oFr (SM_oBv + 64)            /* frames and CoM                          64 */
#define SM_oQV (SM_oFr + 64)            /* q (32) and v (32)                       64 */
#define SM_oRef (SM_oQV + 64)           /* this env's references, staged by asynchronous copies at the start of the env:
                                           com 9 (+1), foot LF 24, foot RF 24, contact LF 12, contact RF 12, posture 24   106 */
#define RF_COM 0
#define RF_FOOT 10   /* + 24 f */
#define RF_CONTACT 58 /* + 12 f */
#define RF_POST 82
#define SM_oQVn (SM_oRef + 106)         /* q (32) and v (32) of the warp's NEXT env, prefetched by asynchronous copies
                                           while the current env is computed         64 */
#ifndef TSIDB_SMALL_PROFILE
#define TSIDB_SMALL_PROFILE 0   /* 1: the single-launch kernel leaves clock stamps of its stages (tools/small_profile.py) */
#endif
#define SM_PER_ENV (SM_oQVn + 64)       /*                                       1608 */
/* task vectors inside oBv */
#define BV_MOT 0   /* 2 x 6 contact motion rhs, by foot */
#define BV_FOOT 12 /* 2 x 6 foot task rhs               */
#define BV_COM 24  /* 3 */
#define BV_AM 27   /* 3 */
#define BV_POST 30 /* na */
/* frames inside oFr */
#define FR_OMF 0   /* 2 x 12: p(3), R row-major (9) */
#define FR_VF 24   /* 2 x 6 */
#define FR_AF 36   /* 2 x 6 */
#define FR_COM 48  /* com 3, vcom 3, acom 3 */
#define FR_L 57    /* angular momentum about the CoM 3, its drift 3 */
/* shared-memory layout of one env in the elimination kernel.  [0, SE_IMAGE) is the assembly image written by
 * the dynamics kernel (one bulk copy); the Hessian block is factored in place. */
#define SE_oH 0                     /* H -> L  26 x 27                         702 */
#define SE_oG (SE_oH + 702)         /* gradient / Q^T w_unc / w_hat             50 */
#define SE_oMu (SE_oG + 50)         /* base rows of M, 6 x 27                  162 */
#define SE_oJF (SE_oMu + 162)       /* JF 2 x 6 x 26                           312 */
#define SE_oNle (SE_oJF + 312)      /* base nle                                  8 */
#define SE_oBm (SE_oNle + 8)        /* contact-motion rhs 2 x 6                 12 */
#define SE_oSc (SE_oBm + 12)        /* contact mask, pad                         2 */
#define SE_IMAGE (SE_oSc + 2)       /* doubles handed over per env            1248 */

/* constants of the QP export (tsidb_problem_data), a section of the handle's global table (TBL_oPROB) filled on the
 * host by tsidb_fill_problem_table: every env shares them and the export reads them with lane-dependent indices */
#define PT_oHF 0                    /* force block of the Hessian w_freg (W T)^T (W T) + hreg I   12 x 12 */
#define PT_oB (PT_oHF + 144)        /* Contact6d inequality rows (pyramid 16, normal 1)           17 x 12 */
#define PT_oT (PT_oB + 204)         /* force generator T                                           6 x 12 */
#define PT_oTMIN (PT_oT + 72)       /* tau_min, tau_max, v_min, v_max                          4 x 24    */
#define PT_oTMAX (PT_oTMIN + 24)
#define PT_oVMIN (PT_oTMAX + 24)
#define PT_oVMAX (PT_oVMIN + 24)
#define PT_SIZE (PT_oVMAX + 24)     /*                                                          516       */

/* output arrays of the QP export (tsidb_problem_out of include/tsidb.h); a null pointer: that part is not written */
struct ProblemOut {
  double *H, *g, *CE, *ce0, *CI, *ci0;
  int32_t* sizes;
  double *TA, *ta0; /* actuation map tau = TA x + ta0 */
};

/* arguments of the generic QP solve (tsidb_qp_solve): caller-supplied problems in the layout of tsidb_problem_out, the
 * caller's strides, and the outputs of tsidb_qp_out (include/tsidb.h) */
struct QpArgs {
  int32_t n_envs, n_max, neq_max, nin_max, na, max_iter;
  const double *H, *g, *CE, *ce0, *CI, *ci0, *TA, *ta0;
  const int32_t* sizes;
  double* x;
  int32_t *status, *iters, *active;
  double *lambda, *lambda_eq, *tau;
};

/* arguments of the adjoint of the QP solve (tsidb_qp_grad): the solved problem and its solution (read), the incoming
 * gradients (NULL = zero) and the requested gradients of the problem's parts (NULL = not written), same layouts */
struct QpGradArgs {
  int32_t n_envs, n_max, neq_max, nin_max, na;
  const double *H, *CE, *CI, *TA;
  const int32_t* sizes;
  const double *x, *lambda, *lambda_eq;
  const int32_t *sol_status, *active;
  const double *gx, *glambda, *glambda_eq, *gtau;
  double *dH, *dg, *dCE, *dce0, *dCI, *dci0, *dTA, *dta0;
  int32_t* status;
};

/* arguments of the adjoint of the reference terms (tsidb_refs_grad): dL/dg [N][n_max] and dL/dce0 [N][neq_max] (NULL =
 * zero) and dL/d of the tsidb_refs arrays com, foot_lf, foot_rf, contact_lf, contact_rf, posture (NULL = not written) */
struct RefsGradArgs {
  int32_t n_max, neq_max;
  const double *dg, *dce0;
  double* out[6];
};

/* arguments of the adjoint of the export in q and v (tsidb_state_grad): dL/d of the parts of tsidb_problem_out with the
 * caller's strides (NULL = zero) and dL/dq [N][nq], dL/dv [N][nv] in the call's layout (NULL = not written) */
struct StateGradArgs {
  int32_t n_max, neq_max, nin_max, pad_;
  const double *H, *g, *CE, *ce0, *CI, *ci0, *TA, *ta0;
  double *dq, *dv;
};

struct TickArgs {
  int32_t n_envs, layout, pad_;
  const double* q;
  const double* v;
  const uint8_t* mask;
  const double* r_com;
  const double* r_foot[2];
  const double* r_contact[2];
  const double* r_posture;
  double* tau;
  double* ddq;
  double* f;
  int32_t* status;
  int32_t* iters;
  uint64_t* active;   /* [3][n_envs] */
  double* o_com;      /* aux outputs, may be null */
  double* o_foot[2];
  double* o_wrench;
  double* o_lambda;       /* [N][32] multipliers of the working set, may be null */
  int32_t* o_lambda_row;  /* [N][32] their rows (tsidb_ci_row numbering), may be null */
  int32_t* counter;   /* dynamic work counter of the active-set kernel */
  double* ws;         /* hand-off images of the active-set kernel, SA_IMAGE doubles per slot */
  double* ws3;        /* assembly images dynamics -> elimination kernel, SE_IMAGE doubles per slot */
  const int32_t* perm; /* slot -> env (class sort), null = identity */
  int32_t kin_only;   /* stop after the kinematics (tsidb_kinematics) */
  int32_t slot;       /* constant-memory slot of the handle */
  int32_t* pred;      /* [n_envs] iteration counts of the previous tick on this handle (scheduling hint), may be null */
  const double* tables; /* the lane-indexed constants in the order the kernels stage them in shared memory (TBL_*), made
                         * once per handle by tsidb_tables_kernel: coalesced loads instead of lane-divergent constant reads */
};

#endif
