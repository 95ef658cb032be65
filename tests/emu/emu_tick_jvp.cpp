/* emu_tick_jvp.cpp — runs the forward derivative of export + solve of the CUDA kernel header (tick_jvp_env: staging, K1,
 * K2, the KKT factors, per direction the tangent K1, the right-hand sides and the solve) on the host, one emulated warp
 * per env: what tsidb_tick_jvp computes, without a GPU (test infrastructure, tests/emu_tick_jvp.py). */
#include "emu_cuda.h"

#include <string>

#include "../../tsid_control_b200/csrc/tsidb_host_const.h"
static DevConst g_const[TSIDB_MAX_SLOTS];
#include "../../tsid_control_b200/csrc/tsidb_kernels.cuh"

namespace emu { Warp W; }

static double g_mdl[MDL_SIZE]; /* the CTA-shared copy the kernel keeps in shared memory */
static const TickArgs* g_args;
static const JvpArgs* g_j;
static double* g_sm;
static int g_env;

static void lane_entry(int lane) {
  const DevConst& C = g_const[0];
  Dual* ds = reinterpret_cast<Dual*>(g_sm);
  double* sm = g_sm + JV_DUALS;
  double* qs = sm + JV_SIZE;
  if (C.nv == 26) tick_jvp_env<26>(C, g_mdl, ds, sm, qs, *g_args, *g_j, g_env, lane);
  else tick_jvp_env<24>(C, g_mdl, ds, sm, qs, *g_args, *g_j, g_env, lane);
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
extern "C" int emu_tick_jvp_fill_const(const tsidb_model* m, const tsidb_conf* c, const double* defaults) {
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

/* tsidb_tick_jvp on the host, after the stride checks of the host side; shared memory poisoned with NaN before every
 * env (a read of anything the kernel did not write shows up in the output) */
extern "C" int emu_tick_jvp(const TickArgs* a_in, const JvpArgs* j) {
  const size_t STK = 1 << 20;
  emu::Warp& W = emu::W;
  if (!W.stacks) W.stacks = (char*)malloc(32 * STK);
  if (j->n_max > TSIDB_QP_MAX_N || j->neq_max > j->n_max || j->nin_max > TSIDB_QP_MAX_NIN || j->n_dirs < 1) return -1;
  TickArgs a = *a_in;
  stage_model(g_const[0], g_mdl, 0, 1);
  const int per_env = TSIDB_J_PER_WARP(j->n_max, j->nin_max); /* one warp of the kernel */
  g_sm = (double*)aligned_alloc(16, per_env * sizeof(double));
  g_args = &a;
  g_j = j;
  int rc = 0;
  for (int env = 0; env < a.n_envs && rc == 0; env++) {
    for (int k = 0; k < per_env; k++) g_sm[k] = NAN;
    g_env = env;
    rc = run_warp(env);
  }
  free(g_sm);
  return rc;
}
