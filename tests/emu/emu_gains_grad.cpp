/* emu_gains_grad.cpp — runs the adjoint of the export in the gains and weights of the CUDA kernel header (gains_grad_env:
 * staging, K1, gains_adjoint_env) on the host, one emulated warp per env: what tsidb_gains_grad computes, without a GPU
 * (test infrastructure, tests/emu_gains_grad.py). */
#include "emu_cuda.h"

#include <string>

#include "../../tsid_control_b200/csrc/tsidb_host_const.h"
static DevConst g_const[TSIDB_MAX_SLOTS];
#include "../../tsid_control_b200/csrc/tsidb_kernels.cuh"

namespace emu { Warp W; }

static double g_mdl[MDL_SIZE]; /* the CTA-shared copy the kernel keeps in shared memory */
static const TickArgs* g_args;
static const GainsGradArgs* g_r;
static double* g_sm;
static double g_frg[144]; /* the force regularisation's Gram matrix the library keeps in its global table */
static int g_env;

static void lane_entry(int lane) {
  const DevConst& C = g_const[0];
  if (C.nv == 26) gains_grad_env<26>(C, g_mdl, g_sm, *g_args, *g_r, g_env, lane);
  else gains_grad_env<24>(C, g_mdl, g_sm, *g_args, *g_r, g_env, lane);
  emu::W.done[lane] = true;
  swapcontext(&emu::W.ctx[lane], &emu::W.sched);
}

static int run_warp(int env) {
  const size_t STK = 1 << 20;
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
  long spins = 0;
  for (;;) {
    bool all = true;
    for (int l = 0; l < 32; l++) {
      if (W.done[l]) continue;
      all = false;
      W.cur = l;
      swapcontext(&W.sched, &W.ctx[l]);
    }
    if (all) break;
    if (++spins > 3000000L) { fprintf(stderr, "emu: env %d: lanes diverged at a collective (deadlock)\n", env); return -2; }
  }
  if (W.arrived != 0) { fprintf(stderr, "emu: env %d: %d lanes left waiting at a collective\n", env, W.arrived); return -3; }
  return 0;
}

/* model and conf constants; defaults = the default references (com 9, foot 2 x 24, contact 2 x 12, posture na) */
extern "C" int emu_gains_grad_fill_const(const tsidb_model* m, const tsidb_conf* c, const double* defaults) {
  std::string err;
  if (!tsidb_fill_devconst(m, c, &g_const[0], &err)) { fprintf(stderr, "emu: %s\n", err.c_str()); return -1; }
  DevConst& C = g_const[0];
  memcpy(C.ref_com, defaults, 9 * sizeof(double));
  memcpy(C.ref_foot[0], defaults + 9, 24 * sizeof(double));
  memcpy(C.ref_foot[1], defaults + 33, 24 * sizeof(double));
  memcpy(C.ref_contact[0], defaults + 57, 12 * sizeof(double));
  memcpy(C.ref_contact[1], defaults + 69, 12 * sizeof(double));
  memcpy(C.ref_posture, defaults + 81, C.na * sizeof(double));
  tsidb_force_gram(c, C.T, reinterpret_cast<double(*)[12]>(g_frg));
  return 0;
}

/* tsidb_gains_grad on the host, shared memory poisoned with NaN before every env (a read of anything the kernel did not
 * write shows up in the output) */
extern "C" int emu_gains_grad(const TickArgs* a_in, const GainsGradArgs* r) {
  const size_t STK = 1 << 20;
  emu::Warp& W = emu::W;
  if (!W.stacks) W.stacks = (char*)malloc(32 * STK);
  TickArgs a = *a_in;
  stage_model(g_const[0], g_mdl, 0, 1);
  g_sm = (double*)malloc(SM_PER_ENV * sizeof(double));
  g_args = &a;
  GainsGradArgs rr = *r;
  rr.frg = g_frg;
  g_r = &rr;
  int rc = 0;
  for (int env = 0; env < a.n_envs && rc == 0; env++) {
    for (int k = 0; k < SM_PER_ENV; k++) g_sm[k] = NAN;
    g_env = env;
    rc = run_warp(env);
  }
  free(g_sm);
  return rc;
}
