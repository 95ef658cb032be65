/* tsidb.cu — host side of libtsidb.so: the C ABI of include/tsidb.h over the sm_100a kernels
 * of tsidb_kernels.cuh.  No torch types, no CPU fallback: every entry point needs a CUDA device. */
#include <cuda_runtime.h>
#include <vector>
#include <nvtx3/nvToolsExt.h> /* header-only: ranges cost nothing unless a profiler is attached */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>

#include "../../include/tsidb.h"
#include "tsidb_host_const.h"
#include "tsidb_kernels.cuh"
#include "tsidb_gait.cuh"

static thread_local std::string g_err;
static std::mutex g_slot_mu;
static bool g_slot_used[8][TSIDB_MAX_SLOTS]; /* per device */

#define CK(call)                                                                             \
  do {                                                                                       \
    cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess) {                                                                 \
      g_err = std::string(#call) + ": " + cudaGetErrorString(e_);                            \
      return -2;                                                                             \
    }                                                                                        \
  } while (0)

#define TSIDB_HOST_STREAMS 3   /* tsidb_compute_host: chunks rotate over these streams (copy/compute overlap) */
#define TSIDB_MAX_CHUNKS 8     /* independent work counters / workspace windows */
#define TSIDB_NCOUNTER 48      /* ints per chunk: 16 work counters and class sizes, then the bins of the class sort */

struct tsidb_handle {
  int device, slot, max_envs, sm_count;
  DevConst dc;
  int32_t* counter;      /* device, TSIDB_NCOUNTER per chunk ([16..16+TSIDB_NKEY): sizes of the (class, bucket) bins of the class sort): work counters of the active-set ([0],[4],[5]), elimination ([8..10]) and basis ([12..14]) kernels, [1..3] class sizes */
  double* ws;            /* device: solver images, SA_IMAGE doubles per slot */
  double* ws3;           /* device: assembly images, SE_IMAGE doubles per slot */
  int32_t* perm;         /* device: slot -> env */
  int32_t* cls_pos;      /* device: per-env (class, position) */
  int64_t launches;
  int timing;            /* tsidb_set_timing: record events between the tick's kernels */
  cudaEvent_t ev[6];     /* start, after class sort, dynamics, elimination, J2, active set */
  /* staging for tsidb_compute_host */
  double *h_in, *h_out;  /* pinned */
  double *d_in, *d_out;  /* device */
  uint8_t *h_mask, *d_mask;
  int32_t *h_int, *d_int;    /* status, iters */
  uint64_t *h_act, *d_act;
  cudaStream_t stream[TSIDB_HOST_STREAMS];
  /* the three contact-class chains E -> G -> A of a tick are independent: double support stays on the tick's own
   * stream, single support and flight run on side streams (per chunk in flight), forked and joined with events */
  cudaStream_t side[TSIDB_MAX_CHUNKS][2];
  cudaEvent_t ev_fork[TSIDB_MAX_CHUNKS], ev_join[TSIDB_MAX_CHUNKS][2];
  int class_streams;     /* 0: every kernel on the tick's stream (also whenever per-kernel timing is on) */
  /* gait phase machine (tsidb_gait_*): state and references, allocated at the first tsidb_gait_reset */
  GaitConf gconf;
  GaitState gait;
  double* g_foot_now[2];   /* sole placements measured by the last tick of a rollout, [N][12] */
  double* g_defaults;      /* device copy of the default references: com 9, feet 2x24, contacts 2x12 */
  int gait_ready;
  int gait_n;              /* envs initialised by the last tsidb_gait_reset */
  double* tables;          /* TickArgs::tables */
  int32_t* pred;           /* [max_envs] iteration counts of the previous tick (longest-first order of the class sort) */
  int sched_hint;          /* TSIDB_SCHED_HINT (default 1): use them */
  int small_n;             /* ticks of at most this many envs run as ONE launch (tsidb_tick_small_kernel); TSIDB_SMALL_N */
  int small_local_n;       /* ... and of at most this many with the hand-off images in shared memory; TSIDB_SMALL_LOCAL_N */
};

/* ------------------------------------------------------------------ small kernels */
/* integrate_dv (ref:ctrl/WalkController.py:291-295): one thread per env.
 * v_mean = v + dt/2 dv; v += dt dv; q = pin.integrate(q, dt v_mean)  [pinocchio SE3 (+) exp6,
 * quaternion sign continuity + first-order normalisation; revolute joints add] */
__global__ void tsidb_integrate_kernel(int n_envs, int layout, int na, double* q, double* v, const double* dv, double dt) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n_envs) return;
  const int nv = na + 6, nq = na + 7;
  auto qi = [&](int d) -> size_t { return layout ? ((size_t)d * n_envs + env) : ((size_t)env * nq + d); };
  auto vi = [&](int d) -> size_t { return layout ? ((size_t)d * n_envs + env) : ((size_t)env * nv + d); };
  double vm[6];
  for (int i = 0; i < nv; i++) {
    const double vo = v[vi(i)], a = dv[vi(i)];
    const double m = dt * (vo + 0.5 * dt * a);
    v[vi(i)] = vo + dt * a;
    if (i < 6) vm[i] = m;
    else q[qi(i + 1)] += m;
  }
  const double* lv = vm;
  const double* w = vm + 3;
  const double t2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
  const double t = sqrt(t2);
  const double prec3 = 1.220703125e-4;
  double st, ct;
  sincos(t, &st, &ct);
  const double a_wxv = (t > prec3) ? (1.0 - ct) / t2 : 0.5 - t2 / 24.0;
  const double a_v = (t > prec3) ? st / t : 1.0 - t2 / 6.0;
  const double a_w = (t > prec3) ? (1.0 - a_v) / t2 : 1.0 / 6.0 - t2 / 120.0;
  const double dg = (t > prec3) ? ct : 1.0 - t2 / 2.0;
  double wxv[3];
  cross3(w, lv, wxv);
  const double wdv = dot3(w, lv);
  double p1[3], R1[9];
  for (int k = 0; k < 3; k++) p1[k] = a_v * lv[k] + (a_w * wdv) * w[k] + a_wxv * wxv[k];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) R1[3 * i + j] = a_wxv * w[i] * w[j];
  R1[1] -= a_v * w[2]; R1[2] += a_v * w[1];
  R1[3] += a_v * w[2]; R1[5] -= a_v * w[0];
  R1[6] -= a_v * w[1]; R1[7] += a_v * w[0];
  R1[0] += dg; R1[4] += dg; R1[8] += dg;
  /* current base rotation */
  const double x = q[qi(3)], y = q[qi(4)], z = q[qi(5)], ww = q[qi(6)];
  double R0[9];
  {
    double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    double twx = tx * ww, twy = ty * ww, twz = tz * ww, txx = tx * x, txy = ty * x, txz = tz * x;
    double tyy = ty * y, tyz = tz * y, tzz = tz * z;
    R0[0] = 1 - (tyy + tzz); R0[1] = txy - twz; R0[2] = txz + twy;
    R0[3] = txy + twz; R0[4] = 1 - (txx + tzz); R0[5] = tyz - twx;
    R0[6] = txz - twy; R0[7] = tyz + twx; R0[8] = 1 - (txx + tyy);
  }
  double dp[3];
  mv3(R0, p1, dp);
  for (int k = 0; k < 3; k++) q[qi(k)] += dp[k];
  /* quaternion of R1 (Eigen's conversion) */
  double q1[4];
  double tr = R1[0] + R1[4] + R1[8];
  if (tr > 0) {
    double s = sqrt(tr + 1.0);
    q1[3] = 0.5 * s;
    s = 0.5 / s;
    q1[0] = (R1[7] - R1[5]) * s; q1[1] = (R1[2] - R1[6]) * s; q1[2] = (R1[3] - R1[1]) * s;
  } else {
    int i = 0;
    if (R1[4] > R1[0]) i = 1;
    if (R1[8] > R1[4 * i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    double s = sqrt(R1[4 * i] - R1[4 * j] - R1[4 * k] + 1.0);
    q1[i] = 0.5 * s;
    s = 0.5 / s;
    q1[3] = (R1[3 * k + j] - R1[3 * j + k]) * s;
    q1[j] = (R1[3 * j + i] + R1[3 * i + j]) * s;
    q1[k] = (R1[3 * k + i] + R1[3 * i + k]) * s;
  }
  double r[4] = {ww * q1[0] + x * q1[3] + y * q1[2] - z * q1[1], ww * q1[1] + y * q1[3] + z * q1[0] - x * q1[2],
                 ww * q1[2] + z * q1[3] + x * q1[1] - y * q1[0], ww * q1[3] - x * q1[0] - y * q1[1] - z * q1[2]};
  const double dotp = r[0] * x + r[1] * y + r[2] * z + r[3] * ww;
  if (dotp < 0) for (int k = 0; k < 4; k++) r[k] = -r[k];
  const double N2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2] + r[3] * r[3];
  const double al = (3.0 - N2) / 2.0;
  for (int k = 0; k < 4; k++) q[qi(3 + k)] = r[k] * al;
}

/* FP64 throughput probe: 8 independent DFMA chains per thread */
__global__ void tsidb_dfma_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x * 1e-3, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; i++) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

/* ------------------------------------------------------------------ C ABI */
extern "C" const char* tsidb_last_error(void) { return g_err.c_str(); }

static int upload_const(tsidb_handle* h) {
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyToSymbol(g_const, &h->dc, sizeof(DevConst), (size_t)h->slot * sizeof(DevConst), cudaMemcpyHostToDevice));
  /* the lane-indexed constants once more, as a global table in staging order (TickArgs::tables) */
  tsidb_tables_kernel<<<1, 128>>>(h->slot, h->tables);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  return 0;
}

/* everything of tsidb_create that can fail after the handle exists; on any failure the caller destroys the handle
 * (tsidb_destroy tolerates members that were never created), which also returns the constant-memory slot */
static int create_impl(tsidb_handle* h, const tsidb_conf* conf, const cudaDeviceProp& prop, int max_envs, int device) {
  h->sm_count = prop.multiProcessorCount;
  const size_t smem = ((size_t)TSIDB_WARPS_PER_BLOCK * SM_PER_ENV + MDL_SIZE) * sizeof(double);
  /* Every CTA of the elimination, basis and active-set kernels is one warp; WARPS of them are to be resident per SM
   * (1 KB of shared memory is reserved per CTA on top of its own), so every kernel asks for the largest
   * shared-memory carve-out. */
  const size_t per_sm = (size_t)prop.sharedMemPerMultiprocessor, rsv = (size_t)prop.reservedSharedMemPerBlock;
#define TSIDB_ATTR(KERNEL, BYTES, RESIDENT, WHAT, CARVEOUT)                                                                       \
  do {                                                                                                                   \
    if ((size_t)(RESIDENT) * ((size_t)(BYTES) + rsv) > per_sm) {                                                         \
      g_err = std::string("tsidb_create: an SM does not hold the planned number of resident CTAs of the ") + WHAT;       \
      return -2;                                                                                                         \
    }                                                                                                                    \
    CK((cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BYTES))));                       \
    CK((cudaFuncSetAttribute(KERNEL, cudaFuncAttributePreferredSharedMemoryCarveout, (int)(CARVEOUT))));                  \
  } while (0)
#define TSIDB_AS_SMEM(NV, NC) ((size_t)TSIDB_A_CTA_WARPS(NC) * a_layout(NV, NC).per_env * sizeof(double))
#define TSIDB_AS_ATTR(NV, NC, W) TSIDB_ATTR((tsidb_activeset_kernel<NV, NC, W>), TSIDB_AS_SMEM(NV, NC), (W) / TSIDB_A_CTA_WARPS(NC), "active-set kernel", cudaSharedmemCarveoutMaxShared)
  TSIDB_AS_ATTR(26, 2, TSIDB_AS_WARPS_DS); TSIDB_AS_ATTR(26, 1, TSIDB_AS_WARPS_SS); TSIDB_AS_ATTR(26, 0, TSIDB_AS_WARPS_FL);
  TSIDB_AS_ATTR(24, 2, TSIDB_AS_WARPS_DS); TSIDB_AS_ATTR(24, 1, TSIDB_AS_WARPS_SS); TSIDB_AS_ATTR(24, 0, TSIDB_AS_WARPS_FL);
#undef TSIDB_AS_ATTR
  /* the dynamics kernel runs alone at the head of the tick and has global loads and a few spills: it asks only for
   * the carve-out it needs (the next configuration up), which leaves it a larger L1 */
  int d_carve = (int)((100 * TSIDB_D_CTAS_PER_SM * (smem + rsv) + per_sm - 1) / per_sm);
  if (const char* e = getenv("TSIDB_D_CARVEOUT")) { const int v = atoi(e); if (v >= d_carve && v <= 100) d_carve = v; } /* tuning knob */
  TSIDB_ATTR(tsidb_dynamics_kernel<26>, smem, TSIDB_D_CTAS_PER_SM, "dynamics kernel", d_carve);
  TSIDB_ATTR(tsidb_dynamics_kernel<24>, smem, TSIDB_D_CTAS_PER_SM, "dynamics kernel", d_carve);
  TSIDB_ATTR(tsidb_refs_grad_kernel<26>, TSIDB_R_SMEM, 1, "references gradient kernel", cudaSharedmemCarveoutMaxShared);
  TSIDB_ATTR(tsidb_refs_grad_kernel<24>, TSIDB_R_SMEM, 1, "references gradient kernel", cudaSharedmemCarveoutMaxShared);
  TSIDB_ATTR(tsidb_state_grad_kernel<26>, TSIDB_S_SMEM, 1, "state gradient kernel", cudaSharedmemCarveoutMaxShared);
  TSIDB_ATTR(tsidb_state_grad_kernel<24>, TSIDB_S_SMEM, 1, "state gradient kernel", cudaSharedmemCarveoutMaxShared);
  CK((cudaFuncSetAttribute(tsidb_tick_small_kernel<26, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(TSIDB_SMALL_SMEM_DOUBLES(26) * sizeof(double)))));
  CK((cudaFuncSetAttribute(tsidb_tick_small_kernel<24, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(TSIDB_SMALL_SMEM_DOUBLES(24) * sizeof(double)))));
  CK((cudaFuncSetAttribute(tsidb_tick_small_kernel<26, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(TSIDB_SMALL_LOCAL_SMEM_DOUBLES(26) * sizeof(double)))));
  CK((cudaFuncSetAttribute(tsidb_tick_small_kernel<24, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(TSIDB_SMALL_LOCAL_SMEM_DOUBLES(24) * sizeof(double)))));
  h->small_n = 1024;
  if (const char* e = getenv("TSIDB_SMALL_N")) h->small_n = atoi(e);
  /* up to this many envs the single launch keeps the hand-off images in shared memory (3 envs per SM fit); the images of
   * such a tick never reach global memory, so tsidb_debug_terms needs TSIDB_SMALL_LOCAL_N=0 */
  h->small_local_n = 2 * prop.multiProcessorCount;
  if (const char* e = getenv("TSIDB_SMALL_LOCAL_N")) h->small_local_n = atoi(e);
#define TSIDB_E_SMEM(NV, NC) (((size_t)TSIDB_E_CTA_WARPS * e_per_env(NV, NC) + 144) * sizeof(double))
#define TSIDB_E_ATTR(NV, NC, W) TSIDB_ATTR((tsidb_eliminate_kernel<NV, NC, W>), TSIDB_E_SMEM(NV, NC), (W) / TSIDB_E_CTA_WARPS, "elimination kernel", cudaSharedmemCarveoutMaxShared)
  TSIDB_E_ATTR(26, 2, TSIDB_E_WARPS); TSIDB_E_ATTR(26, 1, TSIDB_E_WARPS_LIGHT); TSIDB_E_ATTR(26, 0, TSIDB_E_WARPS_LIGHT);
  TSIDB_E_ATTR(24, 2, TSIDB_E_WARPS); TSIDB_E_ATTR(24, 1, TSIDB_E_WARPS_LIGHT); TSIDB_E_ATTR(24, 0, TSIDB_E_WARPS_LIGHT);
#undef TSIDB_E_ATTR
  TSIDB_ATTR(tsidb_problem_kernel<26>, TSIDB_P_SMEM(26), TSIDB_P_CTAS_PER_SM, "QP export kernel", cudaSharedmemCarveoutMaxShared);
  TSIDB_ATTR(tsidb_problem_kernel<24>, TSIDB_P_SMEM(24), TSIDB_P_CTAS_PER_SM, "QP export kernel", cudaSharedmemCarveoutMaxShared);
  TSIDB_ATTR(tsidb_qp_kernel, qp_layout(TSIDB_QP_MAX_N, TSIDB_QP_MAX_NIN).per_env * sizeof(double), 1, "generic QP kernel",
             cudaSharedmemCarveoutMaxShared);
  TSIDB_ATTR(tsidb_qp_grad_kernel, qg_layout(TSIDB_QP_MAX_N, TSIDB_QP_MAX_NIN).per_env * sizeof(double), 1,
             "QP gradient kernel", cudaSharedmemCarveoutMaxShared);
#undef TSIDB_ATTR
  CK(cudaMalloc(&h->counter, TSIDB_NCOUNTER * TSIDB_MAX_CHUNKS * sizeof(int32_t)));
  CK(cudaMalloc(&h->pred, (size_t)max_envs * sizeof(int32_t)));
  CK(cudaMemset(h->pred, 0, (size_t)max_envs * sizeof(int32_t)));
  h->sched_hint = 1;
  if (const char* e = getenv("TSIDB_SCHED_HINT")) h->sched_hint = atoi(e);
  CK(cudaMalloc(&h->ws, (size_t)max_envs * SA_IMAGE * sizeof(double)));
  CK(cudaMalloc(&h->ws3, (size_t)max_envs * SE_IMAGE * sizeof(double)));
  CK(cudaMalloc(&h->perm, (size_t)max_envs * sizeof(int32_t)));
  CK(cudaMalloc(&h->cls_pos, (size_t)max_envs * sizeof(int32_t)));
  CK(cudaMalloc(&h->tables, TBL_SIZE * sizeof(double)));
  if (upload_const(h) != 0) return -2;
  {
    double pt[PT_SIZE];
    tsidb_fill_problem_table(conf, &h->dc, pt);
    CK(cudaMemcpy(h->tables + TBL_oPROB, pt, sizeof pt, cudaMemcpyHostToDevice));
  }
  /* host-call staging: inputs q(nq) v(nv) refs(9+24+24+12+12+na); outputs tau(na) ddq(nv) f(24) */
  const int na = h->dc.na, nv = h->dc.nv, nq = h->dc.nq;
  const size_t in_per = nq + nv + 9 + 24 + 24 + 12 + 12 + na, out_per = na + nv + 24;
  CK(cudaMallocHost(&h->h_in, in_per * max_envs * sizeof(double)));
  CK(cudaMallocHost(&h->h_out, out_per * max_envs * sizeof(double)));
  CK(cudaMalloc(&h->d_in, in_per * max_envs * sizeof(double)));
  CK(cudaMalloc(&h->d_out, out_per * max_envs * sizeof(double)));
  CK(cudaMallocHost(&h->h_mask, max_envs));
  CK(cudaMalloc(&h->d_mask, max_envs));
  CK(cudaMallocHost(&h->h_int, 2 * sizeof(int32_t) * max_envs));
  CK(cudaMalloc(&h->d_int, 2 * sizeof(int32_t) * max_envs));
  CK(cudaMallocHost(&h->h_act, 3 * sizeof(uint64_t) * max_envs));
  CK(cudaMalloc(&h->d_act, 3 * sizeof(uint64_t) * max_envs));
  for (int i = 0; i < TSIDB_HOST_STREAMS; i++) CK(cudaStreamCreateWithFlags(&h->stream[i], cudaStreamNonBlocking));
  for (int c = 0; c < TSIDB_MAX_CHUNKS; c++) {
    CK(cudaEventCreateWithFlags(&h->ev_fork[c], cudaEventDisableTiming));
    for (int i = 0; i < 2; i++) {
      CK(cudaStreamCreateWithFlags(&h->side[c][i], cudaStreamNonBlocking));
      CK(cudaEventCreateWithFlags(&h->ev_join[c][i], cudaEventDisableTiming));
    }
  }
  h->class_streams = 1;
  if (const char* e = getenv("TSIDB_CLASS_STREAMS")) h->class_streams = atoi(e) != 0; /* tuning knob */
  return 0;
}

extern "C" void tsidb_destroy(tsidb_handle* h);

extern "C" int tsidb_create(const tsidb_model* model, const tsidb_conf* conf, int max_envs, int device, tsidb_handle** out) {
  if (!model || !conf || !out || max_envs <= 0) { g_err = "tsidb_create: bad argument"; return -1; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    g_err = "tsidb_create: no CUDA device (there is no CPU fallback for the TSID tick)";
    return -3;
  }
  if (device < 0 || device >= ndev || device >= 8) { g_err = "tsidb_create: bad device index"; return -1; }
  /* everything that can be checked without owning anything comes first */
  DevConst dc;
  std::string err;
  if (!tsidb_fill_devconst(model, conf, &dc, &err)) { g_err = "tsidb_create: " + err; return -1; }
  if (dc.nv != 26 && dc.nv != 24) {
    g_err = "tsidb_create: this build instantiates the tick kernels for nv = 26 (robot/v1) and nv = 24 (robot/v0)";
    return -1;
  }
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if ((size_t)prop.sharedMemPerBlockOptin < ((size_t)TSIDB_WARPS_PER_BLOCK * SM_PER_ENV + MDL_SIZE) * sizeof(double)) {
    g_err = "tsidb_create: device offers less opt-in shared memory per block than the kernel needs";
    return -2;
  }
  tsidb_handle* h = new tsidb_handle();
  memset((void*)h, 0, sizeof *h);
  h->dc = dc;
  h->device = device;
  h->max_envs = max_envs;
  h->slot = -1;
  {
    std::lock_guard<std::mutex> lk(g_slot_mu);
    for (int s = 0; s < TSIDB_MAX_SLOTS; s++)
      if (!g_slot_used[device][s]) { g_slot_used[device][s] = true; h->slot = s; break; }
  }
  if (h->slot < 0) { g_err = "tsidb_create: all constant-memory slots of this device are in use"; delete h; return -1; }
  const int rc = create_impl(h, conf, prop, max_envs, device);
  if (rc != 0) {
    const std::string keep = g_err; /* tsidb_destroy must not hide the cause */
    tsidb_destroy(h);               /* frees whatever was allocated so far and returns the slot */
    cudaGetLastError();
    g_err = keep;
    return rc;
  }
  *out = h;
  return 0;
}

extern "C" void tsidb_destroy(tsidb_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaFree(h->counter); cudaFree(h->ws); cudaFree(h->ws3); cudaFree(h->perm); cudaFree(h->cls_pos); cudaFree(h->tables); cudaFree(h->pred);
  cudaFreeHost(h->h_in); cudaFreeHost(h->h_out); cudaFree(h->d_in); cudaFree(h->d_out);
  cudaFreeHost(h->h_mask); cudaFree(h->d_mask);
  cudaFreeHost(h->h_int); cudaFree(h->d_int);
  cudaFreeHost(h->h_act); cudaFree(h->d_act);
  for (int i = 0; i < TSIDB_HOST_STREAMS; i++)
    if (h->stream[i]) cudaStreamDestroy(h->stream[i]);
  for (int c = 0; c < TSIDB_MAX_CHUNKS; c++) {
    if (h->ev_fork[c]) cudaEventDestroy(h->ev_fork[c]);
    for (int i = 0; i < 2; i++) {
      if (h->side[c][i]) cudaStreamDestroy(h->side[c][i]);
      if (h->ev_join[c][i]) cudaEventDestroy(h->ev_join[c][i]);
    }
  }
  for (int i = 0; i < 6; i++)
    if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  if (h->gait_ready) {
    cudaFree(h->gait.phi); cudaFree(h->gait.mask); cudaFree(h->gait.vcmd); cudaFree(h->gait.lipm); cudaFree(h->gait.origin);
    cudaFree(h->gait.com); cudaFree(h->gait.foot[0]); cudaFree(h->gait.foot[1]); cudaFree(h->gait.contact[0]);
    cudaFree(h->gait.contact[1]); cudaFree(h->gait.fails); cudaFree(h->g_foot_now[0]); cudaFree(h->g_foot_now[1]);
    cudaFree(h->g_defaults);
    cudaFree(h->gait.step_idx); cudaFree(h->gait.swing); cudaFree((void*)h->gait.steps); cudaFree((void*)h->gait.n_steps);
  }
  {
    std::lock_guard<std::mutex> lk(g_slot_mu);
    if (h->slot >= 0) g_slot_used[h->device][h->slot] = false;
  }
  delete h;
}

extern "C" int tsidb_sizes(const tsidb_handle* h, int* na, int* nv, int* nq) {
  if (!h) { g_err = "tsidb_sizes: null handle"; return -1; }
  if (na) *na = h->dc.na;
  if (nv) *nv = h->dc.nv;
  if (nq) *nq = h->dc.nq;
  return 0;
}

extern "C" int tsidb_set_default_refs(tsidb_handle* h, const double* com9, const double* foot_lf24, const double* foot_rf24,
                                      const double* contact_lf12, const double* contact_rf12, const double* posture_na) {
  if (!h) { g_err = "tsidb_set_default_refs: null handle"; return -1; }
  if (com9) memcpy(h->dc.ref_com, com9, 9 * sizeof(double));
  if (foot_lf24) memcpy(h->dc.ref_foot[0], foot_lf24, 24 * sizeof(double));
  if (foot_rf24) memcpy(h->dc.ref_foot[1], foot_rf24, 24 * sizeof(double));
  if (contact_lf12) memcpy(h->dc.ref_contact[0], contact_lf12, 12 * sizeof(double));
  if (contact_rf12) memcpy(h->dc.ref_contact[1], contact_rf12, 12 * sizeof(double));
  if (posture_na) memcpy(h->dc.ref_posture, posture_na, h->dc.na * sizeof(double));
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize()); /* constants may be in use by a running tick */
  return upload_const(h);
}

/* the dynamics kernel over a.n_envs envs on a persistent grid (kernel D of the tick; also the first stage of the QP export) */
static int launch_dynamics(tsidb_handle* h, const TickArgs& a, cudaStream_t st) {
  const int warps = TSIDB_WARPS_PER_BLOCK;
  int blocks = (a.n_envs + warps - 1) / warps;
  if (blocks > TSIDB_D_CTAS_PER_SM * h->sm_count) blocks = TSIDB_D_CTAS_PER_SM * h->sm_count; /* persistent */
  const size_t smem = ((size_t)warps * SM_PER_ENV + MDL_SIZE) * sizeof(double);
  if (h->dc.nv == 26) tsidb_dynamics_kernel<26><<<blocks, 32 * warps, smem, st>>>(a);
  else tsidb_dynamics_kernel<24><<<blocks, 32 * warps, smem, st>>>(a);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

/* One tick over a.n_envs envs on stream st.  `base` / `chunk` select a window of the workspaces and a work
 * counter of its own, so that chunks of one host call can be in flight on different streams. */
static int launch_tick(tsidb_handle* h, TickArgs& a, cudaStream_t st, int base = 0, int chunk = 0) {
  CK(cudaSetDevice(h->device));
  if (base + a.n_envs > h->max_envs) { g_err = "n_envs exceeds the handle's max_envs (workspace size)"; return -1; }
  int32_t* counter = h->counter + TSIDB_NCOUNTER * chunk; /* [0],[4],[5]: active-set work counters per class, [1..3]: class sizes, [8..10]: elimination, [12..14]: basis work counters */
  int32_t* perm = h->perm + base;
  int32_t* cls_pos = h->cls_pos + base;
  a.counter = counter;
  a.slot = h->slot;
  a.tables = h->tables;
  a.pred = h->pred + base;
  a.ws = h->ws + (size_t)base * SA_IMAGE;
  a.ws3 = h->ws3 + (size_t)base * SE_IMAGE;
  a.perm = nullptr;
  const int n = a.n_envs;
  const bool timed = h->timing && !a.kin_only && chunk == 0 && base == 0;
  if (timed) CK(cudaEventRecord(h->ev[0], st));
  struct NvtxRange { explicit NvtxRange(const char* n) { nvtxRangePushA(n); } ~NvtxRange() { nvtxRangePop(); } };
  NvtxRange r_tick("tsidb:tick");
  if (!a.kin_only && !timed && n <= h->small_n) {
    /* small batch: one launch, one warp per env through all three stages (tsidb_tick_small_kernel) */
    NvtxRange r("tsidb:tick_small");
    if (n <= h->small_local_n) {
      if (h->dc.nv == 26) tsidb_tick_small_kernel<26, true><<<n, 32, TSIDB_SMALL_LOCAL_SMEM_DOUBLES(26) * sizeof(double), st>>>(a);
      else tsidb_tick_small_kernel<24, true><<<n, 32, TSIDB_SMALL_LOCAL_SMEM_DOUBLES(24) * sizeof(double), st>>>(a);
    } else {
      if (h->dc.nv == 26) tsidb_tick_small_kernel<26, false><<<n, 32, TSIDB_SMALL_SMEM_DOUBLES(26) * sizeof(double), st>>>(a);
      else tsidb_tick_small_kernel<24, false><<<n, 32, TSIDB_SMALL_SMEM_DOUBLES(24) * sizeof(double), st>>>(a);
    }
    CK(cudaGetLastError());
    h->launches += 1;
    return 0;
  }
  if (!a.kin_only) {
    NvtxRange r("tsidb:class_sort");
    CK(cudaMemsetAsync(counter, 0, TSIDB_NCOUNTER * sizeof(int32_t), st));
    if (a.mask) {
      /* class sort (double support, single support, flight) -> slot order */
      const int th = 256;
      tsidb_classify_kernel<<<(n + th - 1) / th, th, 0, st>>>(n, a.mask, h->sched_hint ? a.pred : nullptr, cls_pos, counter + 1, counter + 16);
      tsidb_permute_kernel<<<(n + th - 1) / th, th, 0, st>>>(n, cls_pos, counter + 16, perm);
      a.perm = perm;
      h->launches += 2;
    }
  }
  if (timed) CK(cudaEventRecord(h->ev[1], st));
  {
    NvtxRange r("tsidb:dynamics");
    if (const int rc = launch_dynamics(h, a, st)) return rc;
  }
  if (timed) CK(cudaEventRecord(h->ev[2], st));
  if (!a.kin_only) {
    /* One launch per kernel and contact class (NC = 2 double support, 1 single support, 0 flight): every size is a
     * compile-time constant and the lighter classes fit more warps per SM.  The class sizes are only known on the
     * device, so every class gets a full persistent grid and the CTAs of an empty class return at once.  Without
     * a mask all envs are double support.  The chains E -> G -> A of the classes do not depend on each other: with
     * class streams on, single support and flight run on side streams, so that the SMs a kernel's last CTAs leave
     * idle are picked up by the next ready kernel of another class.  Per-kernel timing keeps everything on one
     * stream, stage by stage. */
    /* grids: as many CTAs as an SM holds of the kernel, times the SMs (never more warps than envs) */
    const int sms = h->sm_count;
    auto grid = [&](int resident_warps, int cta_warps) {
      const long g = (long)(resident_warps / cta_warps) * sms, need = (n + cta_warps - 1) / cta_warps;
      return (int)(g < need ? g : need);
    };
    const int nv26 = h->dc.nv == 26;
#define TSIDB_E_LAUNCH(NV, NC, W, S) \
  tsidb_eliminate_kernel<NV, NC, W><<<grid(W, TSIDB_E_CTA_WARPS), 32 * TSIDB_E_CTA_WARPS, TSIDB_E_SMEM(NV, NC), S>>>(a)
#define TSIDB_AS_LAUNCH(NV, NC, W, S) \
  tsidb_activeset_kernel<NV, NC, W><<<grid(W, TSIDB_A_CTA_WARPS(NC)), 32 * TSIDB_A_CTA_WARPS(NC), TSIDB_AS_SMEM(NV, NC), S>>>(a)
    auto launch_e = [&](int nc, cudaStream_t s) {
      if (nv26) { if (nc == 2) TSIDB_E_LAUNCH(26, 2, TSIDB_E_WARPS, s); else if (nc == 1) TSIDB_E_LAUNCH(26, 1, TSIDB_E_WARPS_LIGHT, s); else TSIDB_E_LAUNCH(26, 0, TSIDB_E_WARPS_LIGHT, s); }
      else { if (nc == 2) TSIDB_E_LAUNCH(24, 2, TSIDB_E_WARPS, s); else if (nc == 1) TSIDB_E_LAUNCH(24, 1, TSIDB_E_WARPS_LIGHT, s); else TSIDB_E_LAUNCH(24, 0, TSIDB_E_WARPS_LIGHT, s); }
    };
    auto launch_a = [&](int nc, cudaStream_t s) {
      if (nv26) { if (nc == 2) TSIDB_AS_LAUNCH(26, 2, TSIDB_AS_WARPS_DS, s); else if (nc == 1) TSIDB_AS_LAUNCH(26, 1, TSIDB_AS_WARPS_SS, s); else TSIDB_AS_LAUNCH(26, 0, TSIDB_AS_WARPS_FL, s); }
      else { if (nc == 2) TSIDB_AS_LAUNCH(24, 2, TSIDB_AS_WARPS_DS, s); else if (nc == 1) TSIDB_AS_LAUNCH(24, 1, TSIDB_AS_WARPS_SS, s); else TSIDB_AS_LAUNCH(24, 0, TSIDB_AS_WARPS_FL, s); }
    };
    const int ncls = a.perm ? 3 : 1;
    NvtxRange r("tsidb:eliminate+basis+activeset");
    if (h->class_streams && !timed && ncls == 3) {
      CK(cudaEventRecord(h->ev_fork[chunk], st));
      for (int c = 0; c < 3; c++) {
        const int nc = 2 - c;
        cudaStream_t s = c == 0 ? st : h->side[chunk][c - 1];
        if (c > 0) CK(cudaStreamWaitEvent(s, h->ev_fork[chunk], 0));
        launch_e(nc, s); launch_a(nc, s);
        CK(cudaGetLastError());
        if (c > 0) {
          CK(cudaEventRecord(h->ev_join[chunk][c - 1], s));
          CK(cudaStreamWaitEvent(st, h->ev_join[chunk][c - 1], 0));
        }
      }
    } else {
      for (int c = 0; c < ncls; c++) launch_e(2 - c, st);
      CK(cudaGetLastError());
      if (timed) CK(cudaEventRecord(h->ev[3], st));
      if (timed) CK(cudaEventRecord(h->ev[4], st)); /* the basis is built inside the elimination kernel: stage 4 is empty */
      for (int c = 0; c < ncls; c++) launch_a(2 - c, st);
      CK(cudaGetLastError());
    }
    h->launches += 2 * ncls;
#undef TSIDB_E_LAUNCH
#undef TSIDB_AS_LAUNCH
  } else if (timed) {
    CK(cudaEventRecord(h->ev[3], st));
    CK(cudaEventRecord(h->ev[4], st));
  }
  if (timed) CK(cudaEventRecord(h->ev[5], st));
  return 0;
}

extern "C" int tsidb_compute(tsidb_handle* h, int n_envs, int layout, const double* q, const double* v,
                             const uint8_t* contact_mask, const tsidb_refs* refs, double* tau, double* ddq, double* f,
                             int32_t* status, int32_t* iters, uint64_t* active_set, const tsidb_aux_out* aux,
                             void* cuda_stream) {
  if (!h || !q || !v || !tau || !ddq || !f || !status || !iters) { g_err = "tsidb_compute: null argument"; return -1; }
  if (n_envs <= 0) { g_err = "tsidb_compute: n_envs must be positive"; return -1; }
  if (layout != 0 && layout != 1) { g_err = "tsidb_compute: layout must be 0 ([N][dof]) or 1 ([dof][N])"; return -1; }
  TickArgs a;
  memset(&a, 0, sizeof a);
  a.n_envs = n_envs; a.layout = layout;
  a.q = q; a.v = v; a.mask = contact_mask;
  if (refs) {
    a.r_com = refs->com; a.r_foot[0] = refs->foot_lf; a.r_foot[1] = refs->foot_rf;
    a.r_contact[0] = refs->contact_lf; a.r_contact[1] = refs->contact_rf; a.r_posture = refs->posture;
  }
  a.tau = tau; a.ddq = ddq; a.f = f; a.status = status; a.iters = iters; a.active = active_set;
  if (aux) { a.o_com = aux->com; a.o_foot[0] = aux->foot_lf; a.o_foot[1] = aux->foot_rf; a.o_wrench = aux->wrench; a.o_lambda = aux->lambda; a.o_lambda_row = aux->lambda_row; }
  return launch_tick(h, a, (cudaStream_t)cuda_stream);
}

extern "C" int tsidb_kinematics(tsidb_handle* h, int n_envs, int layout, const double* q, const double* v,
                                const tsidb_aux_out* aux, void* cuda_stream) {
  if (!h || !q || !aux) { g_err = "tsidb_kinematics: null argument"; return -1; }
  if (n_envs <= 0 || (layout != 0 && layout != 1)) { g_err = "tsidb_kinematics: bad n_envs/layout"; return -1; }
  TickArgs a;
  memset(&a, 0, sizeof a);
  a.n_envs = n_envs; a.layout = layout; a.q = q; a.v = v; a.kin_only = 1;
  a.o_com = aux->com; a.o_foot[0] = aux->foot_lf; a.o_foot[1] = aux->foot_rf;
  return launch_tick(h, a, (cudaStream_t)cuda_stream);
}

static bool is_pinned(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}

/* The host-buffer tick.  The batch is cut into up to 4 chunks that rotate over 3 streams, so the H2D copy of
 * chunk k+1 and the D2H copy of chunk k-1 run under the kernels of chunk k.  A caller buffer that is pinned
 * (cudaHostAlloc / cudaHostRegister / torch pin_memory) is the DMA source or target itself; a pageable one
 * goes through the handle's pinned staging, chunk by chunk. */
static int compute_host_impl(tsidb_handle* h, int n_envs, const double* q, const double* v, const uint8_t* contact_mask,
                             const tsidb_refs* refs, bool dev_refs, double* tau, double* ddq, double* f, int32_t* status,
                             int32_t* iters, uint64_t* active_set);

extern "C" int tsidb_compute_host(tsidb_handle* h, int n_envs, const double* q, const double* v, const uint8_t* contact_mask,
                                  const tsidb_refs* refs, double* tau, double* ddq, double* f, int32_t* status,
                                  int32_t* iters, uint64_t* active_set) {
  return compute_host_impl(h, n_envs, q, v, contact_mask, refs, false, tau, ddq, f, status, iters, active_set);
}

extern "C" int tsidb_compute_host_devrefs(tsidb_handle* h, int n_envs, const double* q, const double* v,
                                          const uint8_t* contact_mask_dev, const tsidb_refs* refs_dev, double* tau, double* ddq,
                                          double* f, int32_t* status, int32_t* iters, uint64_t* active_set) {
  return compute_host_impl(h, n_envs, q, v, contact_mask_dev, refs_dev, true, tau, ddq, f, status, iters, active_set);
}

/* dev_refs: the contact mask and the reference arrays are device pointers and are used in place (chunk by chunk);
 * otherwise they are host arrays and travel with q and v */
static int compute_host_impl(tsidb_handle* h, int n_envs, const double* q, const double* v, const uint8_t* contact_mask,
                             const tsidb_refs* refs, bool dev_refs, double* tau, double* ddq, double* f, int32_t* status,
                             int32_t* iters, uint64_t* active_set) {
  /* ddq and f are optional: a caller that only drives the actuators (ref:main.py:126) passes NULL and the accelerations
   * and contact forces stay on the device (592 -> 168 bytes per env back over PCIe) */
  if (!h || !q || !v || !tau || !status || !iters) { g_err = "tsidb_compute_host: null argument"; return -1; }
  if (n_envs <= 0 || n_envs > h->max_envs) { g_err = "tsidb_compute_host: n_envs exceeds the handle's max_envs"; return -1; }
  CK(cudaSetDevice(h->device));
  const int na = h->dc.na, nv = h->dc.nv, nq = h->dc.nq;
  const size_t N = (size_t)n_envs;
  /* device / staging layout: [q | v | com | foot_lf | foot_rf | contact_lf | contact_rf | posture], each [N][nd] */
  struct Seg { const double* src; int nd; bool pinned; } segs[8] = {
      {q, nq, false}, {v, nv, false}, {refs ? refs->com : nullptr, 9, false}, {refs ? refs->foot_lf : nullptr, 24, false},
      {refs ? refs->foot_rf : nullptr, 24, false}, {refs ? refs->contact_lf : nullptr, 12, false},
      {refs ? refs->contact_rf : nullptr, 12, false}, {refs ? refs->posture : nullptr, na, false}};
  size_t off[9];
  off[0] = 0;
  const int n_host_segs = dev_refs ? 2 : 8; /* q and v always come from the host */
  for (int s = 0; s < 8; s++) {
    off[s + 1] = off[s] + ((segs[s].src && s < n_host_segs) ? N * segs[s].nd : 0);
    if (segs[s].src && s < n_host_segs) segs[s].pinned = is_pinned(segs[s].src);
  }
  const bool mask_pinned = !dev_refs && contact_mask && is_pinned(contact_mask);
  const bool out_pinned[3] = {is_pinned(tau), ddq && is_pinned(ddq), f && is_pinned(f)};
  const bool st_pinned = is_pinned(status), it_pinned = is_pinned(iters);
  const bool act_pinned = active_set && is_pinned(active_set);
  double* d_tau = h->d_out;
  double* d_ddq = h->d_out + N * na;
  double* d_f = h->d_out + N * (na + nv);
  double* s_tau = h->h_out;
  double* s_ddq = h->h_out + N * na;
  double* s_f = h->h_out + N * (na + nv);

  /* chunk boundaries: the first chunk's H2D copy and the last chunk's D2H copy cannot overlap with kernels, so for
   * large batches those two chunks are small (1/8 of the batch each) and the middle ones large (3/8 each) */
  int nch = n_envs >= 16384 ? 4 : (n_envs >= 2048 ? 2 : 1);
  bool tapered = nch == 4;
  if (const char* e = getenv("TSIDB_HOST_CHUNKS")) { /* tuning knob: equal chunks */
    const int v = atoi(e);
    if (v >= 1 && v <= TSIDB_MAX_CHUNKS) { nch = v; tapered = false; }
  }
  size_t bound[TSIDB_MAX_CHUNKS + 1];
  bound[0] = 0;
  int split64[TSIDB_MAX_CHUNKS], nsplit = 0;
  if (const char* e = getenv("TSIDB_HOST_SPLIT")) { /* tuning knob: chunk sizes in 64ths of the batch, e.g. "8,20,28,8" */
    int sum = 0;
    for (const char* p = e; *p && nsplit < TSIDB_MAX_CHUNKS;) {
      const int v = atoi(p);
      if (v <= 0) { nsplit = 0; break; }
      split64[nsplit++] = v; sum += v;
      while (*p && *p != ',') p++;
      if (*p == ',') p++;
    }
    if (sum != 64) nsplit = 0;
  }
  if (nsplit >= 2 && n_envs >= 16384) {
    nch = nsplit; tapered = false;
    size_t acc = 0;
    for (int c = 0; c < nch; c++) { acc += split64[c]; bound[c + 1] = (c + 1 == nch) ? N : ((N * acc / 64 + 7) & ~(size_t)7); }
  } else if (tapered) {
    int den = 8;
    if (const char* e = getenv("TSIDB_HOST_TAPER")) { const int v = atoi(e); if (v >= 3 && v <= 64) den = v; } /* tuning knob */
    const size_t e8 = (N / den + 7) & ~(size_t)7;
    bound[1] = e8; bound[2] = (N / 2 + 7) & ~(size_t)7; bound[3] = N - e8; bound[4] = N;
  } else {
    const size_t cs = ((N + nch - 1) / nch + 7) & ~(size_t)7;
    nch = (int)((N + cs - 1) / cs);
    for (int c = 1; c <= nch; c++) bound[c] = (c * cs < N) ? c * cs : N;
  }
  /* TSIDB_HOST_TRACE=1: event time stamps per chunk (copies in, kernels, copies out) printed to stderr */
  const bool trace = getenv("TSIDB_HOST_TRACE") != nullptr;
  cudaEvent_t tev[TSIDB_MAX_CHUNKS][4];
  if (trace)
    for (int c = 0; c < nch; c++)
      for (int i = 0; i < 4; i++) CK(cudaEventCreate(&tev[c][i]));
  for (int c = 0; c < nch; c++) {
    cudaStream_t st = h->stream[c % TSIDB_HOST_STREAMS];
    const size_t o = bound[c];
    if (trace) CK(cudaEventRecord(tev[c][0], st));
    const int m = (int)(bound[c + 1] - bound[c]);
    for (int s = 0; s < n_host_segs; s++) {
      if (!segs[s].src) continue;
      const size_t cnt = (size_t)m * segs[s].nd, eo = off[s] + o * segs[s].nd;
      const double* src = segs[s].src + o * segs[s].nd;
      if (!segs[s].pinned) { memcpy(h->h_in + eo, src, cnt * sizeof(double)); src = h->h_in + eo; }
      CK(cudaMemcpyAsync(h->d_in + eo, src, cnt * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    if (contact_mask && !dev_refs) {
      const uint8_t* src = contact_mask + o;
      if (!mask_pinned) { memcpy(h->h_mask + o, src, m); src = h->h_mask + o; }
      CK(cudaMemcpyAsync(h->d_mask + o, src, m, cudaMemcpyHostToDevice, st));
    }
    TickArgs a;
    memset(&a, 0, sizeof a);
    a.n_envs = m; a.layout = 0;
    auto dptr = [&](int s) -> const double* {
      if (!segs[s].src) return nullptr;
      return (s < n_host_segs) ? h->d_in + off[s] + o * segs[s].nd : segs[s].src + o * segs[s].nd; /* device array: in place */
    };
    a.q = dptr(0); a.v = dptr(1); a.r_com = dptr(2); a.r_foot[0] = dptr(3); a.r_foot[1] = dptr(4);
    a.r_contact[0] = dptr(5); a.r_contact[1] = dptr(6); a.r_posture = dptr(7);
    a.mask = contact_mask ? (dev_refs ? contact_mask + o : h->d_mask + o) : nullptr;
    a.tau = d_tau + o * na; a.ddq = d_ddq + o * nv; a.f = d_f + o * 24;
    a.status = h->d_int + o; a.iters = h->d_int + N + o;
    a.active = active_set ? h->d_act + 3 * o : nullptr; /* [3][m] block of this chunk */
    if (trace) CK(cudaEventRecord(tev[c][1], st));
    int rc = launch_tick(h, a, st, (int)o, c);
    if (rc) return rc;
    if (trace) CK(cudaEventRecord(tev[c][2], st));
    CK(cudaMemcpyAsync(out_pinned[0] ? tau + o * na : s_tau + o * na, a.tau, (size_t)m * na * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (ddq) CK(cudaMemcpyAsync(out_pinned[1] ? ddq + o * nv : s_ddq + o * nv, a.ddq, (size_t)m * nv * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (f) CK(cudaMemcpyAsync(out_pinned[2] ? f + o * 24 : s_f + o * 24, a.f, (size_t)m * 24 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(st_pinned ? status + o : h->h_int + o, a.status, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(it_pinned ? iters + o : h->h_int + N + o, a.iters, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (active_set) {
      for (int w = 0; w < 3; w++) {
        uint64_t* dst = act_pinned ? active_set + (size_t)w * N + o : h->h_act + (size_t)w * N + o;
        CK(cudaMemcpyAsync(dst, h->d_act + 3 * o + (size_t)w * m, (size_t)m * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
      }
    }
    if (trace) CK(cudaEventRecord(tev[c][3], st));
  }
  for (int i = 0; i < TSIDB_HOST_STREAMS && i < nch; i++) CK(cudaStreamSynchronize(h->stream[i]));
  if (trace) {
    for (int c = 0; c < nch; c++) {
      float t[4];
      for (int i = 0; i < 4; i++) { CK(cudaEventElapsedTime(&t[i], tev[0][0], tev[c][i])); }
      fprintf(stderr, "[tsidb host trace] chunk %d (%d envs): enqueued %.3f  inputs on device %.3f  kernels done %.3f  outputs on host %.3f ms\n",
              c, (int)(bound[c + 1] - bound[c]), t[0], t[1], t[2], t[3]);
    }
    for (int c = 0; c < nch; c++)
      for (int i = 0; i < 4; i++) cudaEventDestroy(tev[c][i]);
  }
  if (!out_pinned[0]) memcpy(tau, s_tau, N * na * sizeof(double));
  if (ddq && !out_pinned[1]) memcpy(ddq, s_ddq, N * nv * sizeof(double));
  if (f && !out_pinned[2]) memcpy(f, s_f, N * 24 * sizeof(double));
  if (!st_pinned) memcpy(status, h->h_int, N * sizeof(int32_t));
  if (!it_pinned) memcpy(iters, h->h_int + N, N * sizeof(int32_t));
  if (active_set && !act_pinned) memcpy(active_set, h->h_act, 3 * N * sizeof(uint64_t));
  return 0;
}

/* The dynamics terms the last tick handed from the dynamics kernel to the solver stages, for ONE env: read back from
 * the assembly image (Hessian dv block, gradient, base rows of M, sole Jacobians, base nle) and the solve-independent part
 * of the solver image (rows 6.. of M, nle_a).  Diagnostics for the parity tests (SURVEY.md section 7 step 5: M, h, J against
 * the oracle), synchronous; valid when the last tick ran without a contact mask or as a small batch (slot == env). */
extern "C" int tsidb_debug_terms(tsidb_handle* h, int env, int n_contacts, double* M /*[nv][nv]*/, double* nle /*[nv]*/,
                                 double* JF /*[2][6][nv]*/, double* H /*[nv][nv]*/, double* g /*[nv]*/) {
  if (!h || !M || !nle || !JF || !H || !g) { g_err = "tsidb_debug_terms: null argument"; return -1; }
  if (env < 0 || env >= h->max_envs || n_contacts < 0 || n_contacts > 2) { g_err = "tsidb_debug_terms: env or contact count out of range"; return -1; }
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  const int nv = h->dc.nv, na = h->dc.na;
  std::vector<double> ea(SE_IMAGE), sa(SA_IMAGE);
  CK(cudaMemcpy(ea.data(), h->ws3 + (size_t)env * SE_IMAGE, SE_IMAGE * sizeof(double), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(sa.data(), h->ws + (size_t)env * SA_IMAGE, SA_IMAGE * sizeof(double), cudaMemcpyDeviceToHost));
  const ALayout L = a_layout(nv, n_contacts);
  for (int i = 0; i < nv; i++)
    for (int j = 0; j < nv; j++) {
      H[i * nv + j] = ea[SE_oH + i * SM_LDM + j];
      M[i * nv + j] = (i < 6) ? ea[SE_oMu + i * SM_LDM + j] : sa[L.oMa + (i - 6) * SA_LDM + j];
    }
  for (int i = 0; i < nv; i++) {
    g[i] = ea[SE_oG + i];
    nle[i] = (i < 6) ? ea[SE_oNle + i] : sa[L.oNle + i - 6];
  }
  for (int r = 0; r < 12; r++)
    for (int j = 0; j < nv; j++) JF[r * nv + j] = ea[SE_oJF + r * TSIDB_NVX + j];
  (void)na;
  return 0;
}

static void problem_maxima(const tsidb_handle* h, int* n_max, int* neq_max, int* nin_max) {
  *n_max = h->dc.nv + 24;
  *neq_max = 18;
  *nin_max = 2 * (34 + (h->dc.use_tb ? h->dc.na : 0) + (h->dc.use_jb ? h->dc.nv : 0));
}

extern "C" int tsidb_problem_sizes(const tsidb_handle* h, int* n_max, int* neq_max, int* nin_max) {
  if (!h || !n_max || !neq_max || !nin_max) { g_err = "tsidb_problem_sizes: null argument"; return -1; }
  problem_maxima(h, n_max, neq_max, nin_max);
  return 0;
}

/* computeProblemData without the solve: the dynamics kernel (no class sort, slot == env, never the single-launch path,
 * whose images stay in shared memory) leaves every env's images in the handle's workspaces, then the export kernel writes
 * the compact problem of every env.  pred, the work counters and the timing events are not touched. */
extern "C" int tsidb_problem_data(tsidb_handle* h, int n_envs, int layout, const double* q, const double* v,
                                  const uint8_t* contact_mask, const tsidb_refs* refs, const tsidb_problem_out* out,
                                  void* cuda_stream) {
  if (!h || !q || !v || !out) { g_err = "tsidb_problem_data: null argument"; return -1; }
  if (n_envs <= 0 || n_envs > h->max_envs) { g_err = "tsidb_problem_data: n_envs must be in [1, max_envs]"; return -1; }
  if (layout != 0 && layout != 1) { g_err = "tsidb_problem_data: layout must be 0 ([N][dof]) or 1 ([dof][N])"; return -1; }
  for (const double* p : {out->H, out->CE, out->CI})
    if (((uintptr_t)p & 15) != 0) { g_err = "tsidb_problem_data: H, CE and CI must be 16-byte aligned"; return -1; }
  if (((uintptr_t)out->TA & 15) != 0) { g_err = "tsidb_problem_data: TA must be 16-byte aligned"; return -1; }
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  TickArgs a;
  memset(&a, 0, sizeof a);
  a.n_envs = n_envs; a.layout = layout;
  a.q = q; a.v = v; a.mask = contact_mask;
  if (refs) {
    a.r_com = refs->com; a.r_foot[0] = refs->foot_lf; a.r_foot[1] = refs->foot_rf;
    a.r_contact[0] = refs->contact_lf; a.r_contact[1] = refs->contact_rf; a.r_posture = refs->posture;
  }
  a.slot = h->slot;
  a.tables = h->tables;
  a.ws = h->ws;
  a.ws3 = h->ws3;
  a.perm = nullptr;
  if (const int rc = launch_dynamics(h, a, st)) return rc;
  ProblemOut o;
  o.H = out->H; o.g = out->g; o.CE = out->CE; o.ce0 = out->ce0; o.CI = out->CI; o.ci0 = out->ci0; o.sizes = out->sizes;
  o.TA = out->TA; o.ta0 = out->ta0;
  long blocks = (n_envs + TSIDB_P_CTA_WARPS - 1) / TSIDB_P_CTA_WARPS;
  if (blocks > (long)TSIDB_P_CTAS_PER_SM * h->sm_count) blocks = (long)TSIDB_P_CTAS_PER_SM * h->sm_count; /* persistent */
  if (h->dc.nv == 26) tsidb_problem_kernel<26><<<(int)blocks, 32 * TSIDB_P_CTA_WARPS, TSIDB_P_SMEM(26), st>>>(a, o);
  else tsidb_problem_kernel<24><<<(int)blocks, 32 * TSIDB_P_CTA_WARPS, TSIDB_P_SMEM(24), st>>>(a, o);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

/* eiquadprog-fast on caller-supplied problems: one launch of the generic QP kernel, no workspace of the handle */
extern "C" int tsidb_qp_solve(tsidb_handle* h, int n_envs, int n_max, int neq_max, int nin_max, const tsidb_problem_out* qp,
                              const tsidb_qp_out* out, void* cuda_stream) {
  if (!h || !qp || !out) { g_err = "tsidb_qp_solve: null argument"; return -1; }
  if (n_envs <= 0) { g_err = "tsidb_qp_solve: n_envs must be positive"; return -1; }
  if (n_max < 1 || n_max > TSIDB_QP_MAX_N || neq_max < 0 || neq_max > n_max || nin_max < 0 || nin_max > TSIDB_QP_MAX_NIN) {
    g_err = "tsidb_qp_solve: strides must satisfy 1 <= n_max <= TSIDB_QP_MAX_N (64), 0 <= neq_max <= n_max, "
            "0 <= nin_max <= TSIDB_QP_MAX_NIN (512)";
    return -1;
  }
  if (!qp->H || !qp->g || !qp->sizes || !out->x || !out->status) {
    g_err = "tsidb_qp_solve: H, g, sizes, x and status are required";
    return -1;
  }
  if ((neq_max > 0 && (!qp->CE || !qp->ce0)) || (nin_max > 0 && (!qp->CI || !qp->ci0))) {
    g_err = "tsidb_qp_solve: CE and ce0 are required when neq_max > 0, CI and ci0 when nin_max > 0";
    return -1;
  }
  if (out->tau && (!qp->TA || !qp->ta0)) { g_err = "tsidb_qp_solve: tau needs TA and ta0"; return -1; }
  for (const void* p : {(const void*)qp->H, (const void*)qp->g, (const void*)qp->CE, (const void*)qp->ce0, (const void*)qp->CI,
                        (const void*)qp->ci0, (const void*)qp->TA, (const void*)qp->ta0, (const void*)out->x,
                        (const void*)out->lambda, (const void*)out->lambda_eq, (const void*)out->tau})
    if (((uintptr_t)p & 7) != 0) { g_err = "tsidb_qp_solve: fp64 arrays must be 8-byte aligned"; return -1; }
  for (const void* p : {(const void*)qp->sizes, (const void*)out->status, (const void*)out->iters, (const void*)out->active})
    if (((uintptr_t)p & 3) != 0) { g_err = "tsidb_qp_solve: int32 arrays must be 4-byte aligned"; return -1; }
  CK(cudaSetDevice(h->device));
  QpArgs q;
  q.n_envs = n_envs; q.n_max = n_max; q.neq_max = neq_max; q.nin_max = nin_max; q.na = h->dc.na; q.max_iter = h->dc.max_iter;
  q.H = qp->H; q.g = qp->g; q.CE = qp->CE; q.ce0 = qp->ce0; q.CI = qp->CI; q.ci0 = qp->ci0; q.TA = qp->TA; q.ta0 = qp->ta0;
  q.sizes = qp->sizes;
  q.x = out->x; q.status = out->status; q.iters = out->iters; q.active = out->active;
  q.lambda = out->lambda; q.lambda_eq = out->lambda_eq; q.tau = out->tau;
  const size_t smem = qp_layout(n_max, nin_max).per_env * sizeof(double);
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tsidb_qp_kernel, 32, smem));
  if (per_sm < 1) { g_err = "tsidb_qp_solve: the kernel does not fit an SM"; return -2; }
  long blocks = (long)per_sm * h->sm_count; /* persistent */
  if (blocks > n_envs) blocks = n_envs;
  tsidb_qp_kernel<<<(int)blocks, 32, smem, (cudaStream_t)cuda_stream>>>(q);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

/* adjoint of tsidb_qp_solve: one launch of the QP gradient kernel, no workspace of the handle */
extern "C" int tsidb_qp_grad(tsidb_handle* h, int n_envs, int n_max, int neq_max, int nin_max, const tsidb_problem_out* qp,
                             const tsidb_qp_out* sol, const tsidb_qp_out* grad_in, const tsidb_problem_out* grad_out,
                             int32_t* status, void* cuda_stream) {
  if (!h || !qp || !sol || !grad_in || !grad_out) { g_err = "tsidb_qp_grad: null argument"; return -1; }
  if (n_envs <= 0) { g_err = "tsidb_qp_grad: n_envs must be positive"; return -1; }
  if (n_max < 1 || n_max > TSIDB_QP_MAX_N || neq_max < 0 || neq_max > n_max || nin_max < 0 || nin_max > TSIDB_QP_MAX_NIN) {
    g_err = "tsidb_qp_grad: strides must satisfy 1 <= n_max <= TSIDB_QP_MAX_N (64), 0 <= neq_max <= n_max, "
            "0 <= nin_max <= TSIDB_QP_MAX_NIN (512)";
    return -1;
  }
  if (!qp->H || !qp->g || !qp->sizes || !sol->x || !sol->status || !sol->active || !sol->lambda || !status) {
    g_err = "tsidb_qp_grad: H, g, sizes, the solution's x, status, active and lambda, and status are required";
    return -1;
  }
  if ((neq_max > 0 && (!qp->CE || !qp->ce0 || !sol->lambda_eq)) || (nin_max > 0 && (!qp->CI || !qp->ci0))) {
    g_err = "tsidb_qp_grad: CE, ce0 and lambda_eq are required when neq_max > 0, CI and ci0 when nin_max > 0";
    return -1;
  }
  if (grad_in->tau && !qp->TA) { g_err = "tsidb_qp_grad: a tau gradient needs TA"; return -1; }
  if (grad_in->status || grad_in->iters || grad_in->active || grad_out->sizes) {
    g_err = "tsidb_qp_grad: grad_in's status, iters, active and grad_out's sizes must be NULL";
    return -1;
  }
  for (const void* p : {(const void*)qp->H, (const void*)qp->g, (const void*)qp->CE, (const void*)qp->ce0, (const void*)qp->CI,
                        (const void*)qp->ci0, (const void*)qp->TA, (const void*)qp->ta0, (const void*)sol->x,
                        (const void*)sol->lambda, (const void*)sol->lambda_eq, (const void*)grad_in->x,
                        (const void*)grad_in->lambda, (const void*)grad_in->lambda_eq, (const void*)grad_in->tau,
                        (const void*)grad_out->H, (const void*)grad_out->g, (const void*)grad_out->CE, (const void*)grad_out->ce0,
                        (const void*)grad_out->CI, (const void*)grad_out->ci0, (const void*)grad_out->TA, (const void*)grad_out->ta0})
    if (((uintptr_t)p & 7) != 0) { g_err = "tsidb_qp_grad: fp64 arrays must be 8-byte aligned"; return -1; }
  for (const void* p : {(const void*)qp->sizes, (const void*)sol->status, (const void*)sol->active, (const void*)status})
    if (((uintptr_t)p & 3) != 0) { g_err = "tsidb_qp_grad: int32 arrays must be 4-byte aligned"; return -1; }
  CK(cudaSetDevice(h->device));
  QpGradArgs a;
  a.n_envs = n_envs; a.n_max = n_max; a.neq_max = neq_max; a.nin_max = nin_max; a.na = h->dc.na;
  a.H = qp->H; a.CE = qp->CE; a.CI = qp->CI; a.TA = qp->TA; a.sizes = qp->sizes;
  a.x = sol->x; a.lambda = sol->lambda; a.lambda_eq = sol->lambda_eq; a.sol_status = sol->status; a.active = sol->active;
  a.gx = grad_in->x; a.glambda = grad_in->lambda; a.glambda_eq = grad_in->lambda_eq; a.gtau = grad_in->tau;
  a.dH = grad_out->H; a.dg = grad_out->g; a.dCE = grad_out->CE; a.dce0 = grad_out->ce0; a.dCI = grad_out->CI;
  a.dci0 = grad_out->ci0; a.dTA = grad_out->TA; a.dta0 = grad_out->ta0;
  a.status = status;
  const size_t smem = qg_layout(n_max, nin_max).per_env * sizeof(double);
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tsidb_qp_grad_kernel, 32, smem));
  if (per_sm < 1) { g_err = "tsidb_qp_grad: the kernel does not fit an SM"; return -2; }
  long blocks = (long)per_sm * h->sm_count; /* persistent */
  if (blocks > n_envs) blocks = n_envs;
  tsidb_qp_grad_kernel<<<(int)blocks, 32, smem, (cudaStream_t)cuda_stream>>>(a);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

/* adjoint of the reference terms: one launch that recomputes K1 per env, no workspace of the handle */
extern "C" int tsidb_refs_grad(tsidb_handle* h, int n_envs, int layout, const double* q, const double* v,
                               const uint8_t* contact_mask, const tsidb_refs* refs, int n_max, int neq_max, const double* dg,
                               const double* dce0, const tsidb_refs_out* out, void* cuda_stream) {
  if (!h || !q || !v || !out) { g_err = "tsidb_refs_grad: null argument"; return -1; }
  if (n_envs <= 0 || n_envs > h->max_envs) { g_err = "tsidb_refs_grad: n_envs must be in [1, max_envs]"; return -1; }
  if (layout != 0 && layout != 1) { g_err = "tsidb_refs_grad: layout must be 0 ([N][dof]) or 1 ([dof][N])"; return -1; }
  int nx, neq, nin;
  problem_maxima(h, &nx, &neq, &nin);
  if (n_max < nx || neq_max < neq) {
    g_err = "tsidb_refs_grad: n_max and neq_max must be at least tsidb_problem_sizes' n_max and neq_max";
    return -1;
  }
  for (const void* p : {(const void*)q, (const void*)v, (const void*)dg, (const void*)dce0, (const void*)out->com,
                        (const void*)out->foot_lf, (const void*)out->foot_rf, (const void*)out->contact_lf,
                        (const void*)out->contact_rf, (const void*)out->posture})
    if (((uintptr_t)p & 7) != 0) { g_err = "tsidb_refs_grad: fp64 arrays must be 8-byte aligned"; return -1; }
  CK(cudaSetDevice(h->device));
  TickArgs a;
  memset(&a, 0, sizeof a);
  a.n_envs = n_envs; a.layout = layout;
  a.q = q; a.v = v; a.mask = contact_mask;
  if (refs) {
    a.r_com = refs->com; a.r_foot[0] = refs->foot_lf; a.r_foot[1] = refs->foot_rf;
    a.r_contact[0] = refs->contact_lf; a.r_contact[1] = refs->contact_rf; a.r_posture = refs->posture;
  }
  a.slot = h->slot;
  a.tables = h->tables;
  RefsGradArgs r;
  r.n_max = n_max; r.neq_max = neq_max; r.dg = dg; r.dce0 = dce0;
  r.out[0] = out->com; r.out[1] = out->foot_lf; r.out[2] = out->foot_rf;
  r.out[3] = out->contact_lf; r.out[4] = out->contact_rf; r.out[5] = out->posture;
  int blocks = (n_envs + TSIDB_R_CTA_WARPS - 1) / TSIDB_R_CTA_WARPS;
  if (blocks > h->sm_count) blocks = h->sm_count; /* persistent */
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (h->dc.nv == 26) tsidb_refs_grad_kernel<26><<<blocks, 32 * TSIDB_R_CTA_WARPS, TSIDB_R_SMEM, st>>>(a, r);
  else tsidb_refs_grad_kernel<24><<<blocks, 32 * TSIDB_R_CTA_WARPS, TSIDB_R_SMEM, st>>>(a, r);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

/* adjoint of the export in q and v: one launch that recomputes K1 and K2 per env and runs K1 in tangent arithmetic along
 * every raw input direction, no workspace of the handle */
extern "C" int tsidb_state_grad(tsidb_handle* h, int n_envs, int layout, const double* q, const double* v,
                                const uint8_t* contact_mask, const tsidb_refs* refs, int n_max, int neq_max, int nin_max,
                                const tsidb_problem_out* grad, double* dq, double* dv, void* cuda_stream) {
  if (!h || !q || !v) { g_err = "tsidb_state_grad: null argument"; return -1; }
  if (!dq && !dv) { g_err = "tsidb_state_grad: dq and dv are both NULL"; return -1; }
  if (n_envs <= 0 || n_envs > h->max_envs) { g_err = "tsidb_state_grad: n_envs must be in [1, max_envs]"; return -1; }
  if (layout != 0 && layout != 1) { g_err = "tsidb_state_grad: layout must be 0 ([N][dof]) or 1 ([dof][N])"; return -1; }
  int nx, neq, nin;
  problem_maxima(h, &nx, &neq, &nin);
  if (n_max < nx || neq_max < neq || nin_max < nin) {
    g_err = "tsidb_state_grad: n_max, neq_max and nin_max must be at least tsidb_problem_sizes' maxima";
    return -1;
  }
  tsidb_problem_out none;
  memset(&none, 0, sizeof none);
  const tsidb_problem_out& gr = grad ? *grad : none;
  for (const void* p : {(const void*)q, (const void*)v, (const void*)gr.H, (const void*)gr.g, (const void*)gr.CE,
                        (const void*)gr.ce0, (const void*)gr.CI, (const void*)gr.ci0, (const void*)gr.TA, (const void*)gr.ta0,
                        (const void*)dq, (const void*)dv})
    if (((uintptr_t)p & 7) != 0) { g_err = "tsidb_state_grad: fp64 arrays must be 8-byte aligned"; return -1; }
  CK(cudaSetDevice(h->device));
  TickArgs a;
  memset(&a, 0, sizeof a);
  a.n_envs = n_envs; a.layout = layout;
  a.q = q; a.v = v; a.mask = contact_mask;
  if (refs) {
    a.r_com = refs->com; a.r_foot[0] = refs->foot_lf; a.r_foot[1] = refs->foot_rf;
    a.r_contact[0] = refs->contact_lf; a.r_contact[1] = refs->contact_rf; a.r_posture = refs->posture;
  }
  a.slot = h->slot;
  a.tables = h->tables;
  StateGradArgs r;
  memset(&r, 0, sizeof r);
  r.n_max = n_max; r.neq_max = neq_max; r.nin_max = nin_max;
  r.H = gr.H; r.g = gr.g; r.CE = gr.CE; r.ce0 = gr.ce0; r.CI = gr.CI; r.ci0 = gr.ci0; r.TA = gr.TA; r.ta0 = gr.ta0;
  r.dq = dq; r.dv = dv;
  int blocks = (n_envs + TSIDB_S_CTA_WARPS - 1) / TSIDB_S_CTA_WARPS;
  if (blocks > h->sm_count) blocks = h->sm_count; /* persistent */
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (h->dc.nv == 26) tsidb_state_grad_kernel<26><<<blocks, 32 * TSIDB_S_CTA_WARPS, TSIDB_S_SMEM, st>>>(a, r);
  else tsidb_state_grad_kernel<24><<<blocks, 32 * TSIDB_S_CTA_WARPS, TSIDB_S_SMEM, st>>>(a, r);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

extern "C" int tsidb_integrate(tsidb_handle* h, int n_envs, int layout, double* q, double* v, const double* dv, double dt,
                               void* cuda_stream) {
  if (!h || !q || !v || !dv) { g_err = "tsidb_integrate: null argument"; return -1; }
  if (n_envs <= 0 || (layout != 0 && layout != 1)) { g_err = "tsidb_integrate: bad n_envs/layout"; return -1; }
  CK(cudaSetDevice(h->device));
  const int threads = 128;
  tsidb_integrate_kernel<<<(n_envs + threads - 1) / threads, threads, 0, (cudaStream_t)cuda_stream>>>(
      n_envs, layout, h->dc.na, q, v, dv, dt);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

/* ------------------------------------------------------------------ gait phase machine and closed-loop rollout */
static int gait_alloc(tsidb_handle* h) {
  if (h->gait_ready) return 0;
  const size_t N = (size_t)h->max_envs;
  CK(cudaMalloc(&h->gait.phi, N * sizeof(double)));
  CK(cudaMalloc(&h->gait.mask, N));
  CK(cudaMalloc(&h->gait.vcmd, 2 * N * sizeof(double)));
  CK(cudaMalloc(&h->gait.lipm, 4 * N * sizeof(double)));
  CK(cudaMalloc(&h->gait.origin, 24 * N * sizeof(double)));
  CK(cudaMalloc(&h->gait.com, 9 * N * sizeof(double)));
  for (int f = 0; f < 2; f++) {
    CK(cudaMalloc(&h->gait.foot[f], 24 * N * sizeof(double)));
    CK(cudaMalloc(&h->gait.contact[f], 12 * N * sizeof(double)));
    CK(cudaMalloc(&h->g_foot_now[f], 12 * N * sizeof(double)));
  }
  CK(cudaMalloc(&h->gait.fails, N * sizeof(int32_t)));
  CK(cudaMalloc(&h->gait.step_idx, N * sizeof(int32_t)));
  CK(cudaMalloc(&h->gait.swing, 16 * N * sizeof(double)));
  CK(cudaMalloc(&h->g_defaults, 81 * sizeof(double)));
  h->gait_ready = 1;
  return 0;
}

extern "C" int tsidb_gait_reset(tsidb_handle* h, int n_envs, const tsidb_gait_conf* gc, const double* phase0, const double* vcmd,
                                void* cuda_stream) {
  if (!h || !gc) { g_err = "tsidb_gait_reset: null argument"; return -1; }
  if (n_envs <= 0 || n_envs > h->max_envs) { g_err = "tsidb_gait_reset: n_envs exceeds the handle's max_envs"; return -1; }
  if (!(gc->dt > 0) || !(gc->step_duration > 0) || !(gc->com_height > 0)) { g_err = "tsidb_gait_reset: dt, step_duration and com_height must be positive"; return -1; }
  CK(cudaSetDevice(h->device));
  if (gait_alloc(h)) return -2;
  h->gconf.dt = gc->dt; h->gconf.step_duration = gc->step_duration; h->gconf.step_length = gc->step_length;
  h->gconf.step_height = gc->step_height; h->gconf.w2 = 9.80665 / gc->com_height; /* ref:ctrl/LIPM.py:15 */
  h->gconf.com_z = h->dc.ref_com[2];
  if (!h->gait.steps) { h->gconf.rise_ratio = 0.5; h->gconf.max_steps = 0; }
  double d[81];
  memcpy(d, h->dc.ref_com, 9 * sizeof(double));
  memcpy(d + 9, h->dc.ref_foot[0], 24 * sizeof(double));
  memcpy(d + 33, h->dc.ref_foot[1], 24 * sizeof(double));
  memcpy(d + 57, h->dc.ref_contact[0], 12 * sizeof(double));
  memcpy(d + 69, h->dc.ref_contact[1], 12 * sizeof(double));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  CK(cudaMemcpyAsync(h->g_defaults, d, sizeof d, cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st)); /* d is a stack buffer */
  const int th = 128;
  tsidb_gait_reset_kernel<<<(n_envs + th - 1) / th, th, 0, st>>>(n_envs, h->gconf, h->gait, h->g_defaults, phase0, vcmd);
  CK(cudaGetLastError());
  h->launches += 1;
  h->gait_n = n_envs;
  return 0;
}

/* plan = output of tsidb_footstep_plan (or any [N][max_steps][4] footsteps): copied into the handle; the swing foot of
 * every later gait step goes to the env's next footstep of that side along FootTrajectory(rise_ratio) */
extern "C" int tsidb_gait_set_plan(tsidb_handle* h, int n_envs, const double* steps, const int32_t* n_steps, int max_steps,
                                   double rise_ratio, void* cuda_stream) {
  if (!h || !h->gait_ready) { g_err = "tsidb_gait_set_plan: call tsidb_gait_reset first"; return -1; }
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (!steps) { /* back to straight steps */
    CK(cudaStreamSynchronize(st));
    cudaFree((void*)h->gait.steps); cudaFree((void*)h->gait.n_steps);
    h->gait.steps = nullptr; h->gait.n_steps = nullptr; h->gconf.max_steps = 0;
    return 0;
  }
  if (!n_steps || n_envs <= 0 || n_envs > h->gait_n || max_steps < 3 || !(rise_ratio > 0.0) || !(rise_ratio < 1.0)) {
    g_err = "tsidb_gait_set_plan: bad n_envs (<= envs of the last tsidb_gait_reset) / max_steps / rise_ratio";
    return -1;
  }
  if (h->gait.steps && h->gconf.max_steps != max_steps) {
    CK(cudaStreamSynchronize(st));
    cudaFree((void*)h->gait.steps); cudaFree((void*)h->gait.n_steps);
    h->gait.steps = nullptr; h->gait.n_steps = nullptr;
  }
  if (!h->gait.steps) {
    double* sp; int32_t* np_;
    CK(cudaMalloc(&sp, (size_t)h->max_envs * max_steps * 4 * sizeof(double)));
    CK(cudaMalloc(&np_, (size_t)h->max_envs * sizeof(int32_t)));
    CK(cudaMemsetAsync(np_, 0, (size_t)h->max_envs * sizeof(int32_t), st));
    h->gait.steps = sp; h->gait.n_steps = np_;
  }
  CK(cudaMemcpyAsync((void*)h->gait.steps, steps, (size_t)n_envs * max_steps * 4 * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync((void*)h->gait.n_steps, n_steps, (size_t)n_envs * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  h->gconf.rise_ratio = rise_ratio;
  h->gconf.max_steps = max_steps;
  /* execution starts at footstep 2 (0 and 1 are the initial supports); feet already in the air start their swing */
  tsidb_gait_plan_init_kernel<<<(n_envs + 127) / 128, 128, 0, st>>>(n_envs, h->gconf, h->gait);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

extern "C" int tsidb_gait_state(tsidb_handle* h, tsidb_refs* refs_out, const uint8_t** mask_out, const double** phase_out,
                                const int32_t** fails_out) {
  if (!h || !h->gait_ready) { g_err = "tsidb_gait_state: call tsidb_gait_reset first"; return -1; }
  if (refs_out) {
    refs_out->com = h->gait.com; refs_out->foot_lf = h->gait.foot[0]; refs_out->foot_rf = h->gait.foot[1];
    refs_out->contact_lf = h->gait.contact[0]; refs_out->contact_rf = h->gait.contact[1]; refs_out->posture = nullptr;
  }
  if (mask_out) *mask_out = h->gait.mask;
  if (phase_out) *phase_out = h->gait.phi;
  if (fails_out) *fails_out = h->gait.fails;
  return 0;
}

extern "C" int tsidb_gait_step(tsidb_handle* h, int n_envs, const double* foot_lf_now, const double* foot_rf_now,
                               const int32_t* status, void* cuda_stream) {
  if (!h || !h->gait_ready) { g_err = "tsidb_gait_step: call tsidb_gait_reset first"; return -1; }
  if (!foot_lf_now || !foot_rf_now) { g_err = "tsidb_gait_step: null foot placements"; return -1; }
  if (n_envs <= 0 || n_envs > h->max_envs) { g_err = "tsidb_gait_step: bad n_envs"; return -1; }
  CK(cudaSetDevice(h->device));
  const int th = 128;
  tsidb_gait_step_kernel<<<(n_envs + th - 1) / th, th, 0, (cudaStream_t)cuda_stream>>>(n_envs, h->gconf, h->gait, foot_lf_now,
                                                                                         foot_rf_now, status);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

/* one closed-loop step on stream st: tick with the gait's references -> integrate -> phase machine */
static int rollout_step(tsidb_handle* h, int n, double* q, double* v, double* tau, double* ddq, double* f, int32_t* status,
                        int32_t* iters, cudaStream_t st) {
  TickArgs a;
  memset(&a, 0, sizeof a);
  a.n_envs = n; a.layout = 0; a.q = q; a.v = v; a.mask = h->gait.mask;
  a.r_com = h->gait.com; a.r_foot[0] = h->gait.foot[0]; a.r_foot[1] = h->gait.foot[1];
  a.r_contact[0] = h->gait.contact[0]; a.r_contact[1] = h->gait.contact[1];
  a.tau = tau; a.ddq = ddq; a.f = f; a.status = status; a.iters = iters;
  a.o_foot[0] = h->g_foot_now[0]; a.o_foot[1] = h->g_foot_now[1];
  int rc = launch_tick(h, a, st);
  if (rc) return rc;
  const int th = 128;
  tsidb_integrate_kernel<<<(n + th - 1) / th, th, 0, st>>>(n, 0, h->dc.na, q, v, ddq, h->gconf.dt);
  tsidb_gait_step_kernel<<<(n + th - 1) / th, th, 0, st>>>(n, h->gconf, h->gait, h->g_foot_now[0], h->g_foot_now[1], status);
  CK(cudaGetLastError());
  h->launches += 2;
  return 0;
}

extern "C" int tsidb_rollout(tsidb_handle* h, int n_envs, int n_steps, double* q, double* v, double* tau, double* ddq, double* f,
                             int32_t* status, int32_t* iters, int use_graph, void* cuda_stream) {
  if (!h || !q || !v || !tau || !ddq || !f || !status || !iters) { g_err = "tsidb_rollout: null argument"; return -1; }
  if (!h->gait_ready) { g_err = "tsidb_rollout: call tsidb_gait_reset first"; return -1; }
  if (n_envs <= 0 || n_envs > h->max_envs || n_steps < 0) { g_err = "tsidb_rollout: bad n_envs / n_steps"; return -1; }
  if (n_envs > h->gait_n) { g_err = "tsidb_rollout: n_envs exceeds the envs initialised by the last tsidb_gait_reset"; return -1; }
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (!use_graph || n_steps < 2) {
    for (int k = 0; k < n_steps; k++) {
      int rc = rollout_step(h, n_envs, q, v, tau, ddq, f, status, iters, st);
      if (rc) return rc;
    }
    return 0;
  }
  /* the step is the same every time (all state lives in device memory): capture it once, replay it */
  cudaStream_t cap = st;
  bool own = false;
  if (!cap) {
    /* the legacy default stream cannot be captured: replay on a stream of our own, ordered after the work the
     * caller has already queued on the default stream (and synchronised before returning, below) */
    CK(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
    own = true;
    cudaEvent_t ev;
    CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CK(cudaEventRecord(ev, st));
    CK(cudaStreamWaitEvent(cap, ev, 0));
    CK(cudaEventDestroy(ev));
  }
  const int timing = h->timing;
  h->timing = 0;
  const int64_t l0 = h->launches;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  CK(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
  int rc = rollout_step(h, n_envs, q, v, tau, ddq, f, status, iters, cap);
  cudaError_t ce = cudaStreamEndCapture(cap, &graph);
  h->timing = timing;
  if (rc || ce != cudaSuccess) {
    if (graph) cudaGraphDestroy(graph);
    if (own) cudaStreamDestroy(cap);
    if (!rc) { g_err = std::string("tsidb_rollout: stream capture failed: ") + cudaGetErrorString(ce); rc = -2; }
    return rc;
  }
  const int64_t per_step = h->launches - l0;
  ce = cudaGraphInstantiate(&exec, graph, 0);
  for (int k = 0; k < n_steps && ce == cudaSuccess; k++) ce = cudaGraphLaunch(exec, cap);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(cap); /* exec must outlive its launches */
  h->launches = l0 + per_step * n_steps;
  if (exec) cudaGraphExecDestroy(exec);
  cudaGraphDestroy(graph);
  if (own) cudaStreamDestroy(cap);
  if (ce != cudaSuccess) { g_err = std::string("tsidb_rollout: graph replay failed: ") + cudaGetErrorString(ce); return -2; }
  return 0;
}

extern "C" int tsidb_diagnostics(tsidb_handle* h, int n_envs, const tsidb_aux_out* aux, const uint8_t* contact_mask, double omega,
                                 double* cop, double* capture_point, double* support, void* cuda_stream) {
  if (!h || !aux || !aux->com || !aux->foot_lf || !aux->foot_rf || !aux->wrench) {
    g_err = "tsidb_diagnostics: needs the four auxiliary outputs of a tick (com, foot_lf, foot_rf, wrench)";
    return -1;
  }
  if (n_envs <= 0 || !(omega > 0)) { g_err = "tsidb_diagnostics: bad n_envs / omega"; return -1; }
  CK(cudaSetDevice(h->device));
  const int th = 128;
  tsidb_diagnostics_kernel<<<(n_envs + th - 1) / th, th, 0, (cudaStream_t)cuda_stream>>>(
      n_envs, aux->com, aux->foot_lf, aux->foot_rf, aux->wrench, contact_mask, omega, cop, capture_point, support);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

extern "C" int tsidb_foot_trajectory(tsidb_handle* h, int n_envs, double t0, double t1, const double* start4, const double* target4,
                                     double step_height, double rise_ratio, const double* t, double* out16, void* cuda_stream) {
  if (!h || !start4 || !target4 || !t || !out16) { g_err = "tsidb_foot_trajectory: null argument"; return -1; }
  if (n_envs <= 0 || !(t1 > t0) || !(rise_ratio > 0.0) || !(rise_ratio < 1.0)) { g_err = "tsidb_foot_trajectory: bad n_envs / knots / rise_ratio"; return -1; }
  CK(cudaSetDevice(h->device));
  const int th = 128;
  tsidb_foot_trajectory_kernel<<<(n_envs + th - 1) / th, th, 0, (cudaStream_t)cuda_stream>>>(n_envs, t0, t1, start4, target4, step_height,
                                                                                              rise_ratio, t, out16);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

extern "C" int tsidb_footstep_plan(tsidb_handle* h, int n_envs, const double* path, const int32_t* n_pts, int max_pts, const double* init8,
                                   double step_length, double step_width, double* steps, int32_t* n_steps, int max_steps, void* cuda_stream) {
  if (!h || !path || !init8 || !steps || !n_steps) { g_err = "tsidb_footstep_plan: null argument"; return -1; }
  if (n_envs <= 0 || max_pts < 2 || max_steps < 3 || !(step_length > 0.0)) { g_err = "tsidb_footstep_plan: bad sizes"; return -1; }
  CK(cudaSetDevice(h->device));
  const int th = 64;
  tsidb_footstep_plan_kernel<<<(n_envs + th - 1) / th, th, 0, (cudaStream_t)cuda_stream>>>(n_envs, path, n_pts, max_pts, init8, step_length,
                                                                                            step_width, steps, n_steps, max_steps);
  CK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

extern "C" int tsidb_ci_row(const tsidb_handle* h, int block, int side, int i) {
  if (!h || block < 0 || block > 3 || side < 0 || side > 1 || i < 0) return -1;
  const int na = h->dc.na, nv = h->dc.nv;
  const int rows[4] = {17, 17, na, nv};
  const int off[4] = {0, 17, 34, 34 + na};
  if (i >= rows[block]) return -1;
  return 2 * off[block] + side * rows[block] + i;
}

extern "C" int64_t tsidb_launch_count(const tsidb_handle* h) { return h ? h->launches : 0; }

extern "C" int tsidb_set_sched_hint(tsidb_handle* h, int on) {
  if (!h) { g_err = "tsidb_set_sched_hint: null handle"; return -1; }
  h->sched_hint = on ? 1 : 0;
  return 0;
}

extern "C" int tsidb_set_timing(tsidb_handle* h, int on) {
  if (!h) { g_err = "tsidb_set_timing: null handle"; return -1; }
  CK(cudaSetDevice(h->device));
  if (on && !h->ev[0])
    for (int i = 0; i < 6; i++) CK(cudaEventCreate(&h->ev[i]));
  h->timing = on ? 1 : 0;
  return 0;
}

extern "C" int tsidb_last_tick_ms(tsidb_handle* h, float* ms5) {
  if (!h || !ms5) { g_err = "tsidb_last_tick_ms: null argument"; return -1; }
  if (!h->timing || !h->ev[0]) { g_err = "tsidb_last_tick_ms: timing is off (tsidb_set_timing)"; return -1; }
  CK(cudaSetDevice(h->device));
  CK(cudaEventSynchronize(h->ev[5]));
  for (int i = 0; i < 5; i++) CK(cudaEventElapsedTime(&ms5[i], h->ev[i], h->ev[i + 1]));
  return 0;
}

extern "C" int tsidb_fp64_peak(int device, double* tflops_out) {
  if (!tflops_out) { g_err = "tsidb_fp64_peak: null argument"; return -1; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) { g_err = "tsidb_fp64_peak: no such CUDA device"; return -3; }
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 20000;
  double* out;
  CK(cudaMalloc(&out, sizeof(double) * blocks * threads));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  tsidb_dfma_kernel<<<blocks, threads>>>(out, 200, 1.0000001, 1e-9); /* warm-up */
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    CK(cudaEventRecord(e0));
    tsidb_dfma_kernel<<<blocks, threads>>>(out, iters, 1.0000001, 1e-9);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 8.0 * (double)iters * blocks * threads;
    const double tf = fl / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  *tflops_out = best;
  return 0;
}
