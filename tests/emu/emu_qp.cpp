/* emu_qp.cpp — runs the generic QP solve of the CUDA kernel header (qp_env) on the host, one emulated warp per env with
 * its shared memory poisoned with NaN: what tsidb_qp_solve computes, without a GPU (test infrastructure, tests/emu_qp.py). */
#include "emu_cuda.h"

#include "../../tsid_control_b200/csrc/tsidb_host_const.h"
static DevConst g_const[TSIDB_MAX_SLOTS];
#include "../../tsid_control_b200/csrc/tsidb_kernels.cuh"

namespace emu { Warp W; }

static const QpArgs* g_q;
static double* g_sm;
static int g_env;

static void lane_entry(int lane) {
  qp_env(*g_q, g_sm, g_env, lane);
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

/* tsidb_qp_solve on the host, after the host-side argument checks the tests exercise on the GPU */
extern "C" int emu_qp_solve(int n_envs, int n_max, int neq_max, int nin_max, int na, int max_iter, const tsidb_problem_out* qp,
                            const tsidb_qp_out* out) {
  const size_t STK = 1 << 18;
  emu::Warp& W = emu::W;
  if (!W.stacks) W.stacks = (char*)malloc(32 * STK);
  if (n_max < 1 || n_max > TSIDB_QP_MAX_N || neq_max < 0 || neq_max > n_max || nin_max < 0 || nin_max > TSIDB_QP_MAX_NIN)
    return -1;
  QpArgs q;
  q.n_envs = n_envs; q.n_max = n_max; q.neq_max = neq_max; q.nin_max = nin_max; q.na = na; q.max_iter = max_iter;
  q.H = qp->H; q.g = qp->g; q.CE = qp->CE; q.ce0 = qp->ce0; q.CI = qp->CI; q.ci0 = qp->ci0; q.TA = qp->TA; q.ta0 = qp->ta0;
  q.sizes = qp->sizes;
  q.x = out->x; q.status = out->status; q.iters = out->iters; q.active = out->active;
  q.lambda = out->lambda; q.lambda_eq = out->lambda_eq; q.tau = out->tau;
  const int smn = qp_layout(n_max, nin_max).per_env;
  g_sm = (double*)malloc(smn * sizeof(double));
  g_q = &q;
  int rc = 0;
  for (int env = 0; env < n_envs && rc == 0; env++) {
    for (int k = 0; k < smn; k++) g_sm[k] = NAN;
    g_env = env;
    rc = run_warp(env);
  }
  free(g_sm);
  return rc;
}
