/* emu_qp_grad.cpp — runs the adjoint of the generic QP solve of the CUDA kernel header (qp_grad_env) on the host, one
 * emulated warp per env with its shared memory poisoned with NaN: what tsidb_qp_grad computes, without a GPU (test
 * infrastructure, tests/emu_qp_grad.py). */
#include "emu_cuda.h"

#include "../../tsid_control_b200/csrc/tsidb_host_const.h"
static DevConst g_const[TSIDB_MAX_SLOTS];
#include "../../tsid_control_b200/csrc/tsidb_kernels.cuh"

namespace emu { Warp W; }

static const QpGradArgs* g_a;
static double* g_sm;
static int g_env;

static void lane_entry(int lane) {
  qp_grad_env(*g_a, g_sm, g_env, lane);
  emu::W.done[lane] = true;
  swapcontext(&emu::W.ctx[lane], &emu::W.sched);
}

static int run_warp(int env) {
  const size_t STK = 1 << 18;
  emu::Warp& W = emu::W;
  W.arrived = 0;
  for (int l = 0; l < 32; l++) {
    W.done[l] = false;
    getcontext(&W.ctx[l]);
    W.ctx[l].uc_stack.ss_sp = W.stacks + l * STK;
    W.ctx[l].uc_stack.ss_size = STK;
    W.ctx[l].uc_link = &W.sched;
    makecontext(&W.ctx[l], (void (*)())lane_entry, 1, l);
  }
  for (;;) {
    bool all = true;
    for (int l = 0; l < 32; l++) {
      if (W.done[l]) continue;
      all = false;
      W.cur = l;
      swapcontext(&W.sched, &W.ctx[l]);
    }
    if (all) break;
  }
  if (W.arrived != 0) { fprintf(stderr, "emu: env %d: %d lanes left waiting at a collective\n", env, W.arrived); return -3; }
  return 0;
}

/* tsidb_qp_grad on the host, after the stride checks of the host side */
extern "C" int emu_qp_grad(int n_envs, int n_max, int neq_max, int nin_max, int na, const tsidb_problem_out* qp,
                           const tsidb_qp_out* sol, const tsidb_qp_out* gin, const tsidb_problem_out* gout, int32_t* status) {
  const size_t STK = 1 << 18;
  emu::Warp& W = emu::W;
  if (!W.stacks) W.stacks = (char*)malloc(32 * STK);
  if (n_max < 1 || n_max > TSIDB_QP_MAX_N || neq_max < 0 || neq_max > n_max || nin_max < 0 || nin_max > TSIDB_QP_MAX_NIN)
    return -1;
  QpGradArgs a;
  a.n_envs = n_envs; a.n_max = n_max; a.neq_max = neq_max; a.nin_max = nin_max; a.na = na;
  a.H = qp->H; a.CE = qp->CE; a.CI = qp->CI; a.TA = qp->TA; a.sizes = qp->sizes;
  a.x = sol->x; a.lambda = sol->lambda; a.lambda_eq = sol->lambda_eq; a.sol_status = sol->status; a.active = sol->active;
  a.gx = gin->x; a.glambda = gin->lambda; a.glambda_eq = gin->lambda_eq; a.gtau = gin->tau;
  a.dH = gout->H; a.dg = gout->g; a.dCE = gout->CE; a.dce0 = gout->ce0; a.dCI = gout->CI; a.dci0 = gout->ci0;
  a.dTA = gout->TA; a.dta0 = gout->ta0;
  a.status = status;
  const int smn = qg_layout(n_max, nin_max).per_env;
  g_sm = (double*)malloc(smn * sizeof(double));
  g_a = &a;
  int rc = 0;
  for (int env = 0; env < n_envs && rc == 0; env++) {
    for (int k = 0; k < smn; k++) g_sm[k] = NAN;
    g_env = env;
    rc = run_warp(env);
  }
  free(g_sm);
  return rc;
}
