/* emu_state_grad.cpp — runs the adjoint of the QP export in q and v of the CUDA kernel header (state_grad_env: staging,
 * K1, K2, state_adjoint_env, the tangent K1 passes) on the host, one emulated warp per env: what tsidb_state_grad
 * computes, without a GPU (test infrastructure, tests/emu_state_grad.py). */
#include "emu_cuda.h"

#include <string>

#include "../../tsid_control_b200/csrc/tsidb_host_const.h"
static DevConst g_const[TSIDB_MAX_SLOTS];
#include "../../tsid_control_b200/csrc/tsidb_kernels.cuh"

namespace emu { Warp W; }

static double g_mdl[MDL_SIZE]; /* the CTA-shared copy the kernel keeps in shared memory */
static const TickArgs* g_args;
static const StateGradArgs* g_r;
static double* g_sm;
static int g_env;

static void lane_entry(int lane) {
  const DevConst& C = g_const[0];
  double* cb = g_sm + 2 * K1_DUAL_SIZE;
  if (C.nv == 26) state_grad_env<26>(C, g_mdl, g_sm, cb, *g_args, *g_r, g_env, lane);
  else state_grad_env<24>(C, g_mdl, g_sm, cb, *g_args, *g_r, g_env, lane);
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
extern "C" int emu_state_grad_fill_const(const tsidb_model* m, const tsidb_conf* c, const double* defaults) {
  std::string err;
  if (!tsidb_fill_devconst(m, c, &g_const[0], &err)) { fprintf(stderr, "emu: %s\n", err.c_str()); return -1; }
  DevConst& C = g_const[0];
  memcpy(C.ref_com, defaults, 9 * sizeof(double));
  memcpy(C.ref_foot[0], defaults + 9, 24 * sizeof(double));
  memcpy(C.ref_foot[1], defaults + 33, 24 * sizeof(double));
  memcpy(C.ref_contact[0], defaults + 57, 12 * sizeof(double));
  memcpy(C.ref_contact[1], defaults + 69, 12 * sizeof(double));
  memcpy(C.ref_posture, defaults + 81, C.na * sizeof(double));
  return 0;
}

/* tsidb_state_grad on the host, shared memory poisoned with NaN before every env (a read of anything the kernel did not
 * write shows up in the output) */
extern "C" int emu_state_grad(const TickArgs* a_in, const StateGradArgs* r) {
  const size_t STK = 1 << 20;
  emu::Warp& W = emu::W;
  if (!W.stacks) W.stacks = (char*)malloc(32 * STK);
  TickArgs a = *a_in;
  stage_model(g_const[0], g_mdl, 0, 1);
  const int per_env = 2 * K1_DUAL_SIZE + SM_oRef; /* tangent workspace and cotangents, as one warp of the kernel */
  g_sm = (double*)aligned_alloc(16, per_env * sizeof(double));
  g_args = &a;
  g_r = r;
  int rc = 0;
  for (int env = 0; env < a.n_envs && rc == 0; env++) {
    for (int k = 0; k < per_env; k++) g_sm[k] = NAN;
    g_env = env;
    rc = run_warp(env);
  }
  free(g_sm);
  return rc;
}
