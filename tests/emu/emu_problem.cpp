/* emu_problem.cpp — runs the QP export of the CUDA kernel header (dynamics_env, then problem_env) on the host, one
 * emulated warp per env: what tsidb_problem_data computes, without a GPU (test infrastructure, tests/emu_problem.py). */
#include "emu_cuda.h"

#include <string>

#include "../../tsid_control_b200/csrc/tsidb_host_const.h"
static DevConst g_const[TSIDB_MAX_SLOTS];
#include "../../tsid_control_b200/csrc/tsidb_kernels.cuh"

namespace emu { Warp W; }

static double g_mdl[MDL_SIZE];   /* the CTA-shared copies the kernels keep in shared memory */
static double g_pt[PT_SIZE];     /* the QP export's section of the handle's table */
static const TickArgs* g_args;
static const ProblemOut* g_out;
static double* g_sm;
static int g_env, g_stage;

static void lane_entry(int lane) {
  const DevConst& C = g_const[0];
  if (g_stage == 0) {
    if (C.nv == 26) dynamics_env<26>(C, g_mdl, g_sm, *g_args, g_env, g_env, lane);
    else dynamics_env<24>(C, g_mdl, g_sm, *g_args, g_env, g_env, lane);
  } else {
    if (C.nv == 26) problem_env<26>(C, g_pt, g_sm, *g_args, *g_out, g_env, lane);
    else problem_env<24>(C, g_pt, g_sm, *g_args, *g_out, g_env, lane);
  }
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

extern "C" int emu_problem_fill_const(const tsidb_model* m, const tsidb_conf* c) {
  std::string err;
  if (!tsidb_fill_devconst(m, c, &g_const[0], &err)) { fprintf(stderr, "emu: %s\n", err.c_str()); return -1; }
  tsidb_fill_problem_table(c, &g_const[0], g_pt);
  return 0;
}

/* tsidb_problem_data on the host: per env the dynamics stage, then the QP export, with shared memory poisoned with NaN
 * before each stage (a read of anything the stage did not write shows up in the output) */
extern "C" int emu_problem(const TickArgs* a_in, const ProblemOut* out) {
  const size_t STK = 1 << 20;
  emu::Warp& W = emu::W;
  if (!W.stacks) W.stacks = (char*)malloc(32 * STK);
  TickArgs a = *a_in;
  stage_model(g_const[0], g_mdl, 0, 1);
  const int smn = SM_PER_ENV > PB<TSIDB_NVX>::per_env ? SM_PER_ENV : PB<TSIDB_NVX>::per_env;
  g_sm = (double*)calloc(smn, sizeof(double));
  a.ws = (double*)calloc((size_t)a.n_envs * SA_IMAGE, sizeof(double));
  a.ws3 = (double*)calloc((size_t)a.n_envs * SE_IMAGE, sizeof(double));
  a.perm = nullptr;
  g_args = &a;
  g_out = out;
  int rc = 0;
  for (int env = 0; env < a.n_envs && rc == 0; env++) {
    for (int stage = 0; stage < 2 && rc == 0; stage++) {
      for (int k = 0; k < smn; k++) g_sm[k] = NAN;
      g_env = env;
      g_stage = stage;
      rc = run_warp(env);
    }
  }
  free(g_sm);
  free(a.ws);
  free(a.ws3);
  return rc;
}
