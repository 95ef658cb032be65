/* tsidb_kernels.cuh — device code of the batched TSID tick for sm_100a.
 *
 * One warp solves one robot instance ("env"); all arithmetic is fp64.  The tick is a pipeline of persistent
 * kernels, each with the thread mapping, register budget, CTA width and resident warp count that suit its stage
 * (dynamics: one 16-warp CTA per SM; elimination and basis: 8-12 one-warp CTAs per SM on a work counter; active
 * set: 4-warp CTAs); an env's state moves from stage to stage as an "image" in HBM that the consumer pulls into
 * shared memory with one bulk asynchronous copy (TMA).  DESIGN.md §4 has the table with sizes and measured times.
 *
 *   kernel D  tsidb_dynamics_kernel        (reference function each phase replaces)
 *     K1 dynamics   lane <-> body.  World-frame FK, velocities, zero-acceleration drift (pointer jumping over the
 *                   kinematic tree: log2(depth) rounds of shuffles), composite inertias and
 *                   forces accumulated up the tree, then M (CRBA), nle (RNEA), frame Jacobians, CoM/Jcom,
 *                   centroidal angular rows.
 *                   [tsid::RobotWrapper::computeAllTerms inside computeProblemData, ref:main.py:119]
 *     K2 assembly   task right-hand sides (SE3 log, PD laws), the dv block of the Hessian (the force blocks are
 *                   constant and pre-factored on the host), gradient.
 *                   [task.compute() + SolverHQuadProgFast H/g build, ref:main.py:119,121]
 *   kernels E, A  the QP: Goldfarb-Idnani dual active set with the pivot rules of eiquadprog-fast (most
 *                   violated row, lowest index on ties; min ratio drop)
 *                   [SolverHQuadProgFast::solve -> EiquadprogFast::solve_quadprog, ref:main.py:121]
 *     E  tsidb_eliminate_kernel   the 6+6nc equalities are always active, so they are eliminated once: Cholesky of
 *                   H, Householder QR of L^-1 CE^T (lane <-> column), x0 — instead of 18 Givens sweeps; then the
 *                   n x (n-nEq) null-space basis J2 = L^-T Q2 (na+6nc <= 32 columns), one thread per column,
 *                   straight from the factor in shared memory.
 *     A  tsidb_activeset_kernel   the iterations on J2 (one lane per column / per row), then
 *        decode     dv, f, tau = h_a + M_a dv - J_a^T f.   [ref:main.py:126-127]
 *   E and A are instantiated and launched per contact class (nc = 2, 1, 0): every size is a compile-time
 *   constant; the host runs the three class chains E -> A on forked streams (tsidb.cu, launch_tick).
 *   kernel P  tsidb_problem_kernel  not part of the tick: after kernel D (slot == env) it writes each env's assembled QP
 *                   (H, g, CE, ce0, CI, ci0) to the caller's arrays instead of solving it (tsidb_problem_data).
 *
 * The file also compiles for the host under tests/emu (lock-step warp emulator that poisons shared memory with
 * NaN) so that the kernel logic can be exercised without a GPU; TSIDB_EMU selects that build.
 */
#ifndef TSIDB_KERNELS_CUH_
#define TSIDB_KERNELS_CUH_

#include <cstddef>
#include "tsidb_const.h"

#ifndef TSIDB_EMU
#include <cuda_runtime.h>
#define TSIDB_DEV __device__ __forceinline__
#define TSIDB_HD __host__ __device__
#define TSIDB_DEVNI __device__ __noinline__
#define TSIDB_DEVM __device__ __forceinline__ /* member functions */
__constant__ DevConst g_const[TSIDB_MAX_SLOTS];
#else
#define TSIDB_DEVM inline
#endif

#define FULL 0xffffffffu
#define SCHED_FENCE() asm volatile("" ::: "memory")
/* Optional CTA-wide phase alignment (TSIDB_LOCK_D / TSIDB_LOCK_E in tsidb_const.h, both off): the warps of a CTA
 * work on different envs but run the same phase at the same time, so an instruction-cache line fetched by one
 * warp serves all of them.  A no-op in the single-warp host emulation. */
#ifdef TSIDB_EMU
#define PHASE_SYNC_D() ((void)0)
#define PHASE_SYNC_E() ((void)0)
#else
#define PHASE_SYNC_D() do { if (TSIDB_LOCK_D) __syncthreads(); } while (0)
#define PHASE_SYNC_E() do { if (TSIDB_LOCK_E) __syncthreads(); } while (0)
#endif
#define TS_EPS 2.220446049250313e-16
#define TS_INF 1.7976931348623157e308

/* status values of the HQP solver (include/tsidb.h) */
#define ST_OPTIMAL 0
#define ST_INFEASIBLE 1
#define ST_MAX_ITER 3
#define ST_ERROR 4

/* ---------------------------------------------------------------- small helpers */
/* Tangent (forward-mode) scalar: a value and its derivative along one input direction.  K1 and the 3-vector helpers are
 * templates on the scalar type; instantiated with double they are the code the tick runs, with Dual they carry one
 * direction of d/dq, d/dv through the same arithmetic (tsidb_state_grad, stage 2). */
struct Dual {
  double v, d;
  TSIDB_HD Dual(double x = 0.0, double t = 0.0) : v(x), d(t) {}
};
TSIDB_DEV Dual operator+(const Dual& a, const Dual& b) { return Dual(a.v + b.v, a.d + b.d); }
TSIDB_DEV Dual operator+(const Dual& a, double b) { return Dual(a.v + b, a.d); }
TSIDB_DEV Dual operator+(double a, const Dual& b) { return Dual(a + b.v, b.d); }
TSIDB_DEV Dual operator-(const Dual& a, const Dual& b) { return Dual(a.v - b.v, a.d - b.d); }
TSIDB_DEV Dual operator-(const Dual& a, double b) { return Dual(a.v - b, a.d); }
TSIDB_DEV Dual operator-(double a, const Dual& b) { return Dual(a - b.v, -b.d); }
TSIDB_DEV Dual operator-(const Dual& a) { return Dual(-a.v, -a.d); }
TSIDB_DEV Dual operator*(const Dual& a, const Dual& b) { return Dual(a.v * b.v, a.d * b.v + a.v * b.d); }
TSIDB_DEV Dual operator*(const Dual& a, double b) { return Dual(a.v * b, a.d * b); }
TSIDB_DEV Dual operator*(double a, const Dual& b) { return Dual(a * b.v, a * b.d); }
TSIDB_DEV Dual operator/(const Dual& a, const Dual& b) { const double r = a.v / b.v; return Dual(r, (a.d - r * b.d) / b.v); }
TSIDB_DEV Dual operator/(double a, const Dual& b) { const double r = a / b.v; return Dual(r, -r * b.d / b.v); }
TSIDB_DEV Dual& operator+=(Dual& a, const Dual& b) { a.v += b.v; a.d += b.d; return a; }
/* K1's reference point, one coordinate: the base position as read, rounded toward zero to whole metres; a plain double
 * also in the tangent passes.  q - c is exact and (a reference position) - c rounds at the size of the difference, never
 * at the size of c; |q - c| < 1 m bounds the lever arms at any distance, and for a base within a metre of the origin
 * (c = 0) the arithmetic is that of world-origin algebra. */
TSIDB_DEV double ref_point(double x) { return trunc(x); }
TSIDB_DEV double ref_point(const Dual& x) { return trunc(x.v); }
TSIDB_DEV void sincos(const Dual& x, Dual* s, Dual* c) {
  double sv, cv;
  sincos(x.v, &sv, &cv);
  *s = Dual(sv, cv * x.d);
  *c = Dual(cv, -sv * x.d);
}

TSIDB_DEV double shfl(double x, int src) { return __shfl_sync(FULL, x, src); }
TSIDB_DEV Dual shfl(const Dual& x, int src) { return Dual(__shfl_sync(FULL, x.v, src), __shfl_sync(FULL, x.d, src)); }
TSIDB_DEV double warp_sum(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
  return x;
}
template <class A, class B, class O>
TSIDB_DEV void cross3(const A* a, const B* b, O* o) {
  O x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  o[0] = x; o[1] = y; o[2] = z;
}
template <class A, class B>
TSIDB_DEV auto dot3(const A* a, const B* b) -> decltype(a[0] * b[0]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
/* o = R v (R row-major) */
template <class A, class B, class O>
TSIDB_DEV void mv3(const A* R, const B* v, O* o) {
  O x = R[0] * v[0] + R[1] * v[1] + R[2] * v[2];
  O y = R[3] * v[0] + R[4] * v[1] + R[5] * v[2];
  O z = R[6] * v[0] + R[7] * v[1] + R[8] * v[2];
  o[0] = x; o[1] = y; o[2] = z;
}
/* o = R^T v */
template <class A, class B, class O>
TSIDB_DEV void mtv3(const A* R, const B* v, O* o) {
  O x = R[0] * v[0] + R[3] * v[1] + R[6] * v[2];
  O y = R[1] * v[0] + R[4] * v[1] + R[7] * v[2];
  O z = R[2] * v[0] + R[5] * v[1] + R[8] * v[2];
  o[0] = x; o[1] = y; o[2] = z;
}
template <class A, class B, class O>
TSIDB_DEV void mm3(const A* A_, const B* B_, O* C) {
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) C[3 * i + j] = A_[3 * i] * B_[j] + A_[3 * i + 1] * B_[3 + j] + A_[3 * i + 2] * B_[6 + j];
}
/* element (env, dof) of a per-env array with ndof entries per env:
 * layout 0: [N][ndof] row-major (PyTorch-natural), layout 1: SoA [ndof][N] */
TSIDB_DEV size_t eidx(const TickArgs& a, int env, int dof, int ndof) {
  return a.layout ? ((size_t)dof * a.n_envs + env) : ((size_t)env * ndof + dof);
}
TSIDB_DEV double ldin(const double* p, const TickArgs& a, int env, int dof, int ndof) { return p[eidx(a, env, dof, ndof)]; }
/* the same element through a base pointer and a stride formed once per env and array */
struct EnvRow {
  const double* p;
  size_t st;
};
TSIDB_DEV double env_at(const EnvRow& r, int dof) { return r.p[(size_t)dof * r.st]; }
TSIDB_DEV EnvRow env_row(const double* p, const TickArgs& a, int env, int ndof) {
  EnvRow r;
  r.p = p + (a.layout ? (size_t)env : (size_t)env * ndof);
  r.st = a.layout ? (size_t)a.n_envs : (size_t)1;
  return r;
}

/* pinocchio log3 (2.x) + log6: M = (R row-major, p) -> [lin; ang] */
TSIDB_DEV void log6_dev(const double* R, const double* p, double* out) {
  const double PI = 3.14159265358979323846;
  double tr = R[0] + R[4] + R[8];
  double th;
  if (tr >= 3.0) th = 0.0;
  else if (tr <= -1.0) th = PI;
  else th = acos((tr - 1.0) / 2.0);
  double w[3];
  const double prec3 = 1.220703125e-4;
  /* cos(th) is the argument of the acos and sin(th) = sqrt((1 - c)(1 + c)) on [0, pi]: no sincos on the critical
   * path of the assembly (1 - c is exact near c = 1, where the product form keeps full relative accuracy) */
  const double ct = (tr >= 3.0) ? 1.0 : ((tr <= -1.0) ? -1.0 : (tr - 1.0) / 2.0);
  const double st = sqrt(fmax((1.0 - ct) * (1.0 + ct), 0.0));
  if (th >= PI - 1e-2) {
    double cphi = -(tr - 1.0) / 2.0;
    double beta = th * th / (1.0 + cphi);
    double t0 = (R[0] + cphi) * beta, t1 = (R[4] + cphi) * beta, t2 = (R[8] + cphi) * beta;
    w[0] = (R[7] > R[5] ? 1.0 : -1.0) * (t0 > 0 ? sqrt(t0) : 0.0);
    w[1] = (R[2] > R[6] ? 1.0 : -1.0) * (t1 > 0 ? sqrt(t1) : 0.0);
    w[2] = (R[3] > R[1] ? 1.0 : -1.0) * (t2 > 0 ? sqrt(t2) : 0.0);
  } else {
    double t = ((th > prec3) ? th / st : 1.0) / 2.0;
    w[0] = t * (R[7] - R[5]);
    w[1] = t * (R[2] - R[6]);
    w[2] = t * (R[3] - R[1]);
  }
  double t2 = th * th, alpha, beta;
  if (th < prec3) {
    alpha = 1.0 - t2 / 12.0 - t2 * t2 / 720.0;
    beta = 1.0 / 12.0 + t2 / 720.0;
  } else {
    alpha = th * st / (2.0 * (1.0 - ct));
    beta = 1.0 / t2 - st / (2.0 * th * (1.0 - ct));
  }
  double wxp[3];
  cross3(w, p, wxp);
  double wdp = dot3(w, p);
#pragma unroll
  for (int k = 0; k < 3; k++) {
    out[k] = alpha * p[k] - 0.5 * wxp[k] + (beta * wdp) * w[k];
    out[3 + k] = w[k];
  }
}

/* ================================================================= K1: dynamics */
/* lane <-> body.  Everything is expressed in world AXES with Plücker vectors taken at the env's own reference point c
 * (ref_point: the base position in whole metres, a plain double also in the tangent passes), which makes the per-body work
 * independent once the placements are known; only the placement/velocity chain (top-down) and the subtree sums
 * (bottom-up) walk the tree.  Taken at the world origin instead, the inertias moved there (m |c|^2) and the momenta
 * (c x P) of a robot at distance d are O(m d^2) terms whose differences are M, h and J: their rounding grew with d^2.
 * The frames and the CoM in the Fr block stay relative to c; stage_refs_wait moves the reference positions there too,
 * and dynamics_env adds c back where a world position leaves the kernel (DESIGN.md, reference point). */
/* per-body model constants staged in shared memory, one copy per CTA: a lane reads the constants of ITS body, and
 * lane-dependent addresses into __constant__ memory are served one address at a time */
#define MDL_STRIDE 27   /* jR 9, jp 3, mass 1, com 3, inertia 9, parent, depth; odd: conflict-free lane <-> body reads */
#define MDL_oJR 0
#define MDL_oJP 9
#define MDL_oMASS 12
#define MDL_oCOM 13
#define MDL_oI 16
#define MDL_oPAR 25
#define MDL_oDEP 26
#define MDL_oPOST (TSIDB_MAX_BODIES_K * MDL_STRIDE)   /* kp_post 23, kd_post 23, ref_posture 23 */
#define TSIDB_MAX_BODIES_K 24
#define MDL_SIZE (MDL_oPOST + 70)
TSIDB_DEV void stage_model(const DevConst& C, double* mdl, int tid, int nthreads) {
  for (int k = tid; k < TSIDB_MAX_BODIES_K * MDL_STRIDE; k += nthreads) {
    const int b = k / MDL_STRIDE, j = k % MDL_STRIDE;
    double v;
    if (j < 9) v = C.jR[b][j];
    else if (j < 12) v = C.jp[b][j - 9];
    else if (j < 13) v = C.mass[b];
    else if (j < 16) v = C.com[b][j - 13];
    else if (j < 25) v = C.inertia[b][j - 16];
    else if (j < 26) v = (double)C.parent[b];
    else v = (double)C.depth[b];
    mdl[k] = v;
  }
  for (int k = tid; k < 69; k += nthreads) {
    const int j = k % 23;
    mdl[MDL_oPOST + k] = (k < 23) ? C.kp_post[j] : ((k < 46) ? C.kd_post[j] : C.ref_posture[j]);
  }
}

/* the staged tables as one global array: [ model MDL_SIZE | Lf^-1 144 | LaneConst 19 x 32 ] */
#define TBL_oMDL 0
#define TBL_oLF ((MDL_SIZE + 1) & ~1)
#define TBL_oLANE (TBL_oLF + 144)   /* LaneConst of the 32 lanes, value j of lane l at [j][l]: 19 x 32 */
#define TBL_oPROB (TBL_oLANE + 19 * 32)   /* constants of the QP export (PT_*, tsidb_const.h), filled on the host */
#define TBL_oFRG (TBL_oPROB + PT_SIZE)   /* Gram matrix of the force regularisation (W T)^T (W T), 12 x 12 (tsidb_gains_grad) */
#define TBL_SIZE (TBL_oFRG + 144)
TSIDB_DEV void load_table(double* dst, const double* src, int count /* even */, int tid, int nthreads) {
  const double2* s2 = reinterpret_cast<const double2*>(src);
  double2* d2 = reinterpret_cast<double2*>(dst);
  /* four loads in flight per trip: a single warp stages a table in three round trips to L2 instead of twelve */
  for (int k0 = tid; k0 < count / 2; k0 += 4 * nthreads) {
    double2 t[4];
#pragma unroll
    for (int u = 0; u < 4; u++) { const int k = k0 + u * nthreads; if (k < count / 2) t[u] = s2[k]; }
#pragma unroll
    for (int u = 0; u < 4; u++) { const int k = k0 + u * nthreads; if (k < count / 2) d2[k] = t[u]; }
  }
}

/* Where K1 keeps a lane's 28 inertial accumulators: registers in the double instantiation (the tick's); in the tangent
 * passes, whose values and derivatives do not fit the register file next to the rest of K1, a per-lane row of shared
 * memory past the env workspace (odd stride of 29 Duals: lanes hit different banks). */
template <class T> struct K1Acc;
template <> struct K1Acc<double> {
  double r[28];
  TSIDB_DEVM K1Acc(double*, int) {}
  TSIDB_DEVM double& operator[](int k) { return r[k]; }
};
template <> struct K1Acc<Dual> {
  Dual* p;
  TSIDB_DEVM K1Acc(Dual* sm, int lane) : p(sm + SM_oRef + 29 * lane) {}
  TSIDB_DEVM Dual& operator[](int k) { return p[k]; }
};

/* lane 0's placement (the base's R0, p0) on every lane: shuffled into registers in the double instantiation; in the
 * tangent passes lane 0 leaves it in shared memory after the accumulator rows, where the other lanes read it */
#define K1_DUAL_ROOT (SM_oRef + 29 * 32) /* tangent workspace (Duals): env workspace, 32 accumulator rows, R0 and p0 */
#define K1_DUAL_SIZE (K1_DUAL_ROOT + 12)
template <class T, int N> struct K1Root;
template <int N> struct K1Root<double, N> {
  double r[N];
  TSIDB_DEVM K1Root(const double* src, double*, int) {
#pragma unroll
    for (int k = 0; k < N; k++) r[k] = shfl(src[k], 0);
  }
  TSIDB_DEVM const double* ptr() const { return r; }
  TSIDB_DEVM double operator[](int k) const { return r[k]; }
};
template <int N> struct K1Root<Dual, N> {
  const Dual* p;
  TSIDB_DEVM K1Root(const Dual* src, Dual* dst, int lane) : p(dst) {
    if (lane == 0)
      for (int k = 0; k < N; k++) dst[k] = src[k];
    __syncwarp();
  }
  TSIDB_DEVM const Dual* ptr() const { return p; }
  TSIDB_DEVM Dual operator[](int k) const { return p[k]; }
};

template <int NV, class T>
TSIDB_DEV void k1_dynamics(const DevConst& C, const double* mdl, T* sm, int lane) {
  constexpr int nb = NV - 5, nv = NV; /* bodies = floating base + NV - 6 revolute joints */
  const bool act = lane < nb;
  const int b = act ? lane : 0;
  const int par = act && lane > 0 ? (int)mdl[b * MDL_STRIDE + MDL_oPAR] : 0;
  const T* qs = sm + SM_oQV;
  const T* vs = sm + SM_oQV + 32;

  T R[9], p[3], Vl[3], Va[3], Al[3] = {0, 0, 0}, Aa[3] = {0, 0, 0};
  T Rl[9], pl[3], qd = 0.0;
  if (lane == 0) {
    /* free flyer: q = (p, quat xyzw); v = local (lin, ang) */
    T x = qs[3], y = qs[4], z = qs[5], w = qs[6];
    T tx = 2 * x, ty = 2 * y, tz = 2 * z;
    T twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x;
    T tyy = ty * y, tyz = tz * y, tzz = tz * z;
    R[0] = 1 - (tyy + tzz); R[1] = txy - twz; R[2] = txz + twy;
    R[3] = txy + twz; R[4] = 1 - (txx + tzz); R[5] = tyz - twx;
    R[6] = txz - twy; R[7] = tyz + twx; R[8] = 1 - (txx + tyy);
    /* relative to the reference point c (ref_point) */
    p[0] = qs[0] - ref_point(qs[0]); p[1] = qs[1] - ref_point(qs[1]); p[2] = qs[2] - ref_point(qs[2]);
    T vl[3] = {vs[0], vs[1], vs[2]}, wl[3] = {vs[3], vs[4], vs[5]};
    mv3(R, wl, Va);
    mv3(R, vl, Vl);
    T c[3];
    cross3(p, Va, c);
    Vl[0] += c[0]; Vl[1] += c[1]; Vl[2] += c[2];
  } else {
    T ang = act ? qs[6 + b] : T(0.0);
    qd = act ? vs[5 + b] : T(0.0);
    T sa, ca;
    sincos(ang, &sa, &ca);
    const double* jR = mdl + b * MDL_STRIDE + MDL_oJR;
#pragma unroll
    for (int r = 0; r < 3; r++) {
      double c0 = jR[3 * r], c1 = jR[3 * r + 1];
      Rl[3 * r] = c0 * ca + c1 * sa;
      Rl[3 * r + 1] = c1 * ca - c0 * sa;
      Rl[3 * r + 2] = jR[3 * r + 2];
    }
    pl[0] = mdl[b * MDL_STRIDE + MDL_oJP]; pl[1] = mdl[b * MDL_STRIDE + MDL_oJP + 1]; pl[2] = mdl[b * MDL_STRIDE + MDL_oJP + 2];
#pragma unroll
    for (int k = 0; k < 9; k++) R[k] = Rl[k];
#pragma unroll
    for (int k = 0; k < 3; k++) { p[k] = pl[k]; Vl[k] = 0; Va[k] = 0; }
  }
  /* Top-down by POINTER JUMPING instead of one tree level at a time: every body composes its transform with its
   * current ancestor's and then points to that ancestor's ancestor: after r rounds a transform spans 2^r joints, so
   * ceil(log2(depth + 1)) rounds reach the world frame (3 instead of 6 for the humanoids here); the twists and the drift accelerations are sums along the path to the
   * root in world coordinates and are accumulated the same way.  anc = -1: the quantity is already a world one. */
  int rounds = 0;
  while ((1 << rounds) <= C.maxdepth) rounds++;
  const int par0 = (act && lane > 0) ? par : -1;
  {
    int anc = par0;
    for (int rd = 0; rd < rounds; rd++) {
      const int src = anc < 0 ? 0 : anc;
      T Rp[9], pp[3];
#pragma unroll
      for (int k = 0; k < 9; k++) Rp[k] = shfl(R[k], src);
#pragma unroll
      for (int k = 0; k < 3; k++) pp[k] = shfl(p[k], src);
      const int anc2 = __shfl_sync(FULL, anc, src);
      if (anc >= 0) {
        T Rn[9], pn[3];
        mm3(Rp, R, Rn);
        mv3(Rp, p, pn);
#pragma unroll
        for (int k = 0; k < 9; k++) R[k] = Rn[k];
#pragma unroll
        for (int k = 0; k < 3; k++) p[k] = pn[k] + pp[k];
        anc = anc2;
      }
    }
  }
  /* own twist S qd of the body's joint (the base keeps its twist): V = sum over the path to the root */
  T Sql[3] = {0, 0, 0}, Sqa[3] = {0, 0, 0};
  if (lane > 0) {
    T a[3] = {R[2], R[5], R[8]}, sl[3];
    cross3(p, a, sl);
#pragma unroll
    for (int k = 0; k < 3; k++) { Sql[k] = sl[k] * qd; Sqa[k] = a[k] * qd; Vl[k] = Sql[k]; Va[k] = Sqa[k]; }
  }
  {
    int anc = par0;
    for (int rd = 0; rd < rounds; rd++) {
      const int src = anc < 0 ? 0 : anc;
      T Vlp[3], Vap[3];
#pragma unroll
      for (int k = 0; k < 3; k++) { Vlp[k] = shfl(Vl[k], src); Vap[k] = shfl(Va[k], src); }
      const int anc2 = __shfl_sync(FULL, anc, src);
      if (anc >= 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) { Vl[k] += Vlp[k]; Va[k] += Vap[k]; }
        anc = anc2;
      }
    }
  }
  /* own drift term V x (S qd) (motion cross product; zero for the base): A = sum over the path to the root */
  if (lane > 0) {
    T c1[3], c2[3], c3[3];
    cross3(Vl, Sqa, c1);
    cross3(Va, Sql, c2);
    cross3(Va, Sqa, c3);
#pragma unroll
    for (int k = 0; k < 3; k++) { Al[k] = c1[k] + c2[k]; Aa[k] = c3[k]; }
  }
  {
    int anc = par0;
    for (int rd = 0; rd < rounds; rd++) {
      const int src = anc < 0 ? 0 : anc;
      T Alp[3], Aap[3];
#pragma unroll
      for (int k = 0; k < 3; k++) { Alp[k] = shfl(Al[k], src); Aap[k] = shfl(Aa[k], src); }
      const int anc2 = __shfl_sync(FULL, anc, src);
      if (anc >= 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) { Al[k] += Alp[k]; Aa[k] += Aap[k]; }
        anc = anc2;
      }
    }
  }
  /* motion subspace of the body's joint (revolute z): S = (p x a, a) */
  T Sa_[3] = {R[2], R[5], R[8]}, Sl_[3];
  cross3(p, Sa_, Sl_);

  /* per-body inertial quantities, world axes, reference point = c (ref_point) */
  K1Acc<T> acc(sm, lane);
  {
    double m = act ? mdl[b * MDL_STRIDE + MDL_oMASS] : 0.0;
    double cl[3] = {mdl[b * MDL_STRIDE + MDL_oCOM], mdl[b * MDL_STRIDE + MDL_oCOM + 1], mdl[b * MDL_STRIDE + MDL_oCOM + 2]};
    T cw[3];
    mv3(R, cl, cw);
    cw[0] += p[0]; cw[1] += p[1]; cw[2] += p[2];
    T RI[9], Iw[9];
    mm3(R, mdl + b * MDL_STRIDE + MDL_oI, RI);
    /* Iw = RI * R^T */
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
      for (int j = 0; j < 3; j++) Iw[3 * i + j] = RI[3 * i] * R[3 * j] + RI[3 * i + 1] * R[3 * j + 1] + RI[3 * i + 2] * R[3 * j + 2];
    T h[3] = {m * cw[0], m * cw[1], m * cw[2]};
    T c2 = dot3(cw, cw);
    /* inertia about the origin: Io = Iw + m (|c|^2 I - c c^T); xx xy xz yy yz zz */
    T Io[6] = {Iw[0] + m * (c2 - cw[0] * cw[0]), Iw[1] - m * cw[0] * cw[1], Iw[2] - m * cw[0] * cw[2],
                    Iw[4] + m * (c2 - cw[1] * cw[1]), Iw[5] - m * cw[1] * cw[2], Iw[8] + m * (c2 - cw[2] * cw[2])};
    /* momentum  P = m (Vl + Va x c),  L_o = Iw Va + c x P */
    T t[3], P[3], Lo[3];
    cross3(Va, cw, t);
    P[0] = m * (Vl[0] + t[0]); P[1] = m * (Vl[1] + t[1]); P[2] = m * (Vl[2] + t[2]);
    mv3(Iw, Va, Lo);
    cross3(cw, P, t);
    Lo[0] += t[0]; Lo[1] += t[1]; Lo[2] += t[2];
    /* force at zero joint acceleration, no gravity: Y A + V x* (Y V) */
    T fl[3], fa[3], u[3];
    cross3(Aa, cw, t);
    fl[0] = m * (Al[0] + t[0]); fl[1] = m * (Al[1] + t[1]); fl[2] = m * (Al[2] + t[2]);
    mv3(Iw, Aa, fa);
    cross3(cw, fl, t);
    fa[0] += t[0]; fa[1] += t[1]; fa[2] += t[2];
    cross3(Va, P, t);
    fl[0] += t[0]; fl[1] += t[1]; fl[2] += t[2];
    cross3(Va, Lo, t);
    cross3(Vl, P, u);
    fa[0] += t[0] + u[0]; fa[1] += t[1] + u[1]; fa[2] += t[2] + u[2];
    acc[0] = m; acc[1] = h[0]; acc[2] = h[1]; acc[3] = h[2];
#pragma unroll
    for (int k = 0; k < 6; k++) acc[4 + k] = Io[k];
    /* with gravity: + Y (lin = -g): lin -= m g, ang -= c x m g = h x (-g) */
    double mg[3] = {-C.gravity[0], -C.gravity[1], -C.gravity[2]};
    cross3(h, mg, t);
    acc[10] = fl[0] + m * mg[0]; acc[11] = fl[1] + m * mg[1]; acc[12] = fl[2] + m * mg[2];
    acc[13] = fa[0] + t[0]; acc[14] = fa[1] + t[1]; acc[15] = fa[2] + t[2];
    acc[16] = P[0]; acc[17] = P[1]; acc[18] = P[2]; acc[19] = Lo[0]; acc[20] = Lo[1]; acc[21] = Lo[2];
    acc[22] = fl[0]; acc[23] = fl[1]; acc[24] = fl[2]; acc[25] = fa[0]; acc[26] = fa[1]; acc[27] = fa[2];
  }
  /* bottom-up subtree sums through shared memory (scratch in the J2 region).  Lanes <-> the 28 components:
   * a body's index is larger than its parent's (Pinocchio's depth-first order), so ONE sweep from the last
   * body to the first leaves every subtree sum in place; each lane only ever touches its own component, so
   * the sweep needs no synchronisation. */
  T* sc = sm + SM_oH;
  if (act) {
#pragma unroll
    for (int k = 0; k < 28; k++) sc[b * 29 + k] = acc[k];
  }
  __syncwarp();
  if (lane < 28) {
    for (int c = nb - 1; c >= 1; c--) sc[C.parent[c] * 29 + lane] += sc[c * 29 + lane];
  }
  __syncwarp();
  if (act) {
#pragma unroll
    for (int k = 0; k < 28; k++) acc[k] = sc[b * 29 + k];
  }
  __syncwarp();
  /* totals and the base placement, broadcast from lane 0 */
  T mt = shfl(acc[0], 0);
  T ht[3] = {shfl(acc[1], 0), shfl(acc[2], 0), shfl(acc[3], 0)};
  T comw[3] = {ht[0] / mt, ht[1] / mt, ht[2] / mt};
  const K1Root<T, 9> R0(R, sm + K1_DUAL_ROOT, lane);
  const K1Root<T, 3> p0(p, sm + K1_DUAL_ROOT + 9, lane);
  T Y0[10];
#pragma unroll
  for (int k = 0; k < 10; k++) Y0[k] = shfl(acc[k], 0);

  T* Mm = sm + SM_oM;
  T* nle = sm + SM_oNle;
  T* Jcom = sm + SM_oJcom;
  T* Ag = sm + SM_oAg;
  T* JF = sm + SM_oJF;
  T* fr = sm + SM_oFr;

  /* zero M and JF (different branches do not couple; non-support columns are zero) */
  for (int k = lane; k < nv * SM_LDM; k += 32) Mm[k] = 0.0;
  for (int k = lane; k < 2 * 6 * TSIDB_NVX; k += 32) JF[k] = 0.0;
  __syncwarp();

  /* Lane roles from here on.  Joint lanes (1..nb-1) own column 5 + b of M, Jcom, Ag, JF.  The six base columns are
   * formed by the lanes the tree leaves idle — base dof k on lane nb + k — with the base's motion subspace and the
   * composite inertia of the whole robot, through the SAME instructions as the joint columns (round 1 ran them as a
   * second, divergent pass on lanes 0..5). */
  const bool isjoint = act && lane > 0;
  const bool isbase = lane >= nb && lane < nb + 6;
  const int kb = lane - nb; /* base dof of a base lane */
  if (isbase) {
    const int k = kb % 3;
    const T rk[3] = {R0[k], R0[3 + k], R0[6 + k]};
    if (kb < 3) { Sl_[0] = rk[0]; Sl_[1] = rk[1]; Sl_[2] = rk[2]; Sa_[0] = Sa_[1] = Sa_[2] = 0.0; }
    else { cross3(p0.ptr(), rk, Sl_); Sa_[0] = rk[0]; Sa_[1] = rk[1]; Sa_[2] = rk[2]; }
  }
  /* F = Yc S for the lane's column; nle, Jcom, Ag columns; M entries along the ancestors */
  T Fl[3], Fa[3];
  {
    const T mc = isbase ? Y0[0] : acc[0];
    T hc[3], Io[6], t[3];
#pragma unroll
    for (int k = 0; k < 3; k++) hc[k] = isbase ? Y0[1 + k] : acc[1 + k];
#pragma unroll
    for (int k = 0; k < 6; k++) Io[k] = isbase ? Y0[4 + k] : acc[4 + k];
    cross3(Sa_, hc, t);
    Fl[0] = mc * Sl_[0] + t[0]; Fl[1] = mc * Sl_[1] + t[1]; Fl[2] = mc * Sl_[2] + t[2];
    Fa[0] = Io[0] * Sa_[0] + Io[1] * Sa_[1] + Io[2] * Sa_[2];
    Fa[1] = Io[1] * Sa_[0] + Io[3] * Sa_[1] + Io[4] * Sa_[2];
    Fa[2] = Io[2] * Sa_[0] + Io[4] * Sa_[1] + Io[5] * Sa_[2];
    cross3(hc, Sl_, t);
    Fa[0] += t[0]; Fa[1] += t[1]; Fa[2] += t[2];
    if (isjoint || isbase) {
      const int c = isbase ? kb : 5 + b;
      if (isjoint) nle[c] = dot3(Sl_, &acc[10]) + dot3(Sa_, &acc[13]);
      cross3(hc, Sa_, t);
#pragma unroll
      for (int r = 0; r < 3; r++) Jcom[r * TSIDB_NVX + c] = (mc * Sl_[r] - t[r]) / mt;
      cross3(comw, Fl, t);
#pragma unroll
      for (int r = 0; r < 3; r++) Ag[r * TSIDB_NVX + c] = Fa[r] - t[r];
      /* base rows: X0^T F */
      T u[3], w[3];
      mtv3(R0.ptr(), Fl, u);
      cross3(p0.ptr(), Fl, t);
      T d[3] = {Fa[0] - t[0], Fa[1] - t[1], Fa[2] - t[2]};
      mtv3(R0.ptr(), d, w);
#pragma unroll
      for (int r = 0; r < 3; r++) {
        Mm[r * SM_LDM + c] = u[r];
        Mm[(3 + r) * SM_LDM + c] = w[r];
        if (isjoint) { Mm[c * SM_LDM + r] = u[r]; Mm[c * SM_LDM + 3 + r] = w[r]; }
      }
    }
  }
  /* walk the revolute ancestors (including the body itself) */
  {
    int j = act && lane > 0 ? b : 0;
    for (int st = 0; st < C.maxdepth; st++) {
      T sjl[3], sja[3];
#pragma unroll
      for (int k = 0; k < 3; k++) { sjl[k] = shfl(Sl_[k], j); sja[k] = shfl(Sa_[k], j); }
      const int pj = __shfl_sync(FULL, par, j); /* parent of body j: lane j holds it (no lane-indexed constant read) */
      if (j > 0) {
        T val = dot3(sjl, Fl) + dot3(sja, Fa);
        Mm[(5 + j) * SM_LDM + 5 + b] = val;
        Mm[(5 + b) * SM_LDM + 5 + j] = val;
        j = pj;
      }
    }
  }
  {
    /* base nle = X0^T Fc_root; CoM quantities; centroidal angular momentum and its drift */
    T F0l[3], F0a[3], Pt[3], Lt[3], fal[3], faa[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      F0l[k] = shfl(acc[10 + k], 0); F0a[k] = shfl(acc[13 + k], 0);
      Pt[k] = shfl(acc[16 + k], 0); Lt[k] = shfl(acc[19 + k], 0);
      fal[k] = shfl(acc[22 + k], 0); faa[k] = shfl(acc[25 + k], 0);
    }
    if (lane == 0) {
      T u[3], w[3], t[3];
      mtv3(R0.ptr(), F0l, u);
      cross3(p0.ptr(), F0l, t);
      T d[3] = {F0a[0] - t[0], F0a[1] - t[1], F0a[2] - t[2]};
      mtv3(R0.ptr(), d, w);
#pragma unroll
      for (int r = 0; r < 3; r++) { nle[r] = u[r]; nle[3 + r] = w[r]; }
      cross3(comw, Pt, t);
      T t2[3];
      cross3(comw, fal, t2);
      const T imt0 = 1.0 / mt; /* one reciprocal for this lane's six divisions by the total mass */
#pragma unroll
      for (int r = 0; r < 3; r++) {
        fr[FR_COM + r] = comw[r];
        fr[FR_COM + 3 + r] = Pt[r] * imt0;
        fr[FR_COM + 6 + r] = fal[r] * imt0;
        fr[FR_L + r] = Lt[r] - t[r];
        fr[FR_L + 3 + r] = faa[r] - t2[r];
      }
    }
  }
  /* operational frames (soles): placement, LOCAL velocity, classic-acceleration drift, LOCAL Jacobian — ONE pass for both
   * feet.  A joint lies on at most one foot's chain, so the joint lanes of the two legs form their columns at the same
   * time, each with its own foot's frame; the base columns of foot 0 are formed by the base lanes nb..nb+5, those of
   * foot 1 by the six lanes behind them (lane 0, the base body's, takes the one that does not fit below lane 32); the
   * lanes of the two foot bodies form the frames' velocity terms.  (Round 1: a loop over the feet with three divergent
   * blocks each.) */
  {
    static_assert(nb + 11 <= 32, "base columns of the second foot: five idle lanes and lane 0");
    int fm = -1, col = 0; /* this lane's foot and Jacobian column */
    if (isjoint) {
      fm = ((C.foot_support[0] >> b) & 1u) ? 0 : (((C.foot_support[1] >> b) & 1u) ? 1 : -1);
      col = 5 + b;
    } else if (isbase) {
      fm = 0; col = kb;
    } else if (lane >= nb + 6 || lane == 0) {
      const int k2 = (lane == 0) ? 32 - (nb + 6) : lane - (nb + 6); /* lanes nb+6..31 take dofs 0.., lane 0 the next one */
      if (k2 < 6) {
        fm = 1; col = k2;
        const int k = k2 % 3;
        const T rk[3] = {R0[k], R0[3 + k], R0[6 + k]};
        if (k2 < 3) { Sl_[0] = rk[0]; Sl_[1] = rk[1]; Sl_[2] = rk[2]; Sa_[0] = Sa_[1] = Sa_[2] = 0.0; }
        else { cross3(p0.ptr(), rk, Sl_); Sa_[0] = rk[0]; Sa_[1] = rk[1]; Sa_[2] = rk[2]; }
      }
    }
    const int fsel = fm < 0 ? 0 : fm;
    const int fb = C.foot_body[fsel];
    T Rb[9], pb[3];
#pragma unroll
    for (int k = 0; k < 9; k++) Rb[k] = shfl(R[k], fb);
#pragma unroll
    for (int k = 0; k < 3; k++) pb[k] = shfl(p[k], fb);
    double fRm[9], fpm[3];
#pragma unroll
    for (int k = 0; k < 9; k++) fRm[k] = C.fR[fsel][k]; /* lane-indexed constant reads: two addresses per instruction */
#pragma unroll
    for (int k = 0; k < 3; k++) fpm[k] = C.fp[fsel][k];
    T Rf[9], pf[3], t[3];
    mm3(Rb, fRm, Rf);
    mv3(Rb, fpm, pf);
    pf[0] += pb[0]; pf[1] += pb[1]; pf[2] += pb[2];
    if (fm >= 0) {
      T la[3], ll[3];
      mtv3(Rf, Sa_, la);
      cross3(pf, Sa_, t);
      T d[3] = {Sl_[0] - t[0], Sl_[1] - t[1], Sl_[2] - t[2]};
      mtv3(Rf, d, ll);
#pragma unroll
      for (int r = 0; r < 3; r++) {
        JF[(fm * 6 + r) * TSIDB_NVX + col] = ll[r];
        JF[(fm * 6 + 3 + r) * TSIDB_NVX + col] = la[r];
      }
    }
    if (isjoint && lane == fb) {
      const int f = fm;
      T vl[3], va[3], al[3], aa[3];
      mtv3(Rf, Va, va);
      cross3(pf, Va, t);
      T d[3] = {Vl[0] - t[0], Vl[1] - t[1], Vl[2] - t[2]};
      mtv3(Rf, d, vl);
      mtv3(Rf, Aa, aa);
      cross3(pf, Aa, t);
      T e[3] = {Al[0] - t[0], Al[1] - t[1], Al[2] - t[2]};
      mtv3(Rf, e, al);
      cross3(va, vl, t);
#pragma unroll
      for (int r = 0; r < 3; r++) {
        fr[FR_OMF + f * 12 + r] = pf[r];
        fr[FR_VF + f * 6 + r] = vl[r]; fr[FR_VF + f * 6 + 3 + r] = va[r];
        fr[FR_AF + f * 6 + r] = al[r] + t[r]; fr[FR_AF + f * 6 + 3 + r] = aa[r];
      }
#pragma unroll
      for (int k = 0; k < 9; k++) fr[FR_OMF + f * 12 + 3 + k] = Rf[k];
    }
  }
  __syncwarp();
}

/* ================================================================= K2: assembly */
/* tsid::TaskSE3Equality::compute in the local frame: b = Kp log6(oMf^-1 Mref) + Kd (R^T vref - v) + R^T aref - drift.
 * The adjoints restate its error E = Rf^T R_ref, ep = Rf^T (p_ref - p_f) (refs_adjoint_env, state_adjoint_env) and
 * gains_adjoint_env the whole law, so that the tick's kernels stay untouched: a change here goes there too. */
TSIDB_DEV void se3_rhs(const double* fr, int f, const double* kp, const double* kd, const double* ref12,
                       const double* vref, const double* aref, double* b6) {
  const double* pf = fr + FR_OMF + f * 12;
  const double* Rf = pf + 3;
  /* Mref: p, R column-major */
  double Rr[9], dp[3], E[9], ep[3];
#pragma unroll
  for (int c = 0; c < 3; c++)
#pragma unroll
    for (int r = 0; r < 3; r++) Rr[3 * r + c] = ref12[3 + 3 * c + r];
  dp[0] = ref12[0] - pf[0]; dp[1] = ref12[1] - pf[1]; dp[2] = ref12[2] - pf[2];
  /* E = Rf^T Rr, ep = Rf^T dp */
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) E[3 * i + j] = Rf[i] * Rr[j] + Rf[3 + i] * Rr[3 + j] + Rf[6 + i] * Rr[6 + j];
  mtv3(Rf, dp, ep);
  double pe[6];
  log6_dev(E, ep, pe);
  double vl[3] = {0, 0, 0}, va[3] = {0, 0, 0}, al[3] = {0, 0, 0}, aa[3] = {0, 0, 0};
  if (vref) { mtv3(Rf, vref, vl); mtv3(Rf, vref + 3, va); }
  if (aref) { mtv3(Rf, aref, al); mtv3(Rf, aref + 3, aa); }
  const double* vF = fr + FR_VF + f * 6;
  const double* aF = fr + FR_AF + f * 6;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    b6[k] = (kp[k] * pe[k] + kd[k] * (vl[k] - vF[k]) + al[k]) - aF[k];
    b6[3 + k] = (kp[3 + k] * pe[3 + k] + kd[3 + k] * (va[k] - vF[3 + k]) + aa[k]) - aF[3 + k];
  }
}

/* Task right-hand sides -> sm[oBv]; Hessian dv block -> SM_oH (factored by the elimination kernel);
 * gradient -> column nEq of B (it rides through the QR as an extra column). */
template <int NV>
TSIDB_DEV void k2_assemble(const DevConst& C, const double* mdl, double* sm, const TickArgs& a, int env, int lane, int mask, int neq, int n) {
  constexpr int nv = NV, na = NV - 6;
  double* bv = sm + SM_oBv;
  const double* fr = sm + SM_oFr;
  const double* qs = sm + SM_oQV;
  const double* vs = sm + SM_oQV + 32;
  /* lanes 0..3: the four SE3 laws (contact LF, contact RF, foot LF, foot RF); the references were staged in shared
   * memory by asynchronous copies issued before K1 (stage_refs) */
  const double* rf = sm + SM_oRef;
  if (lane < 4) {
    /* one pass for all four laws: the contact and the foot-task lanes differ only in their gains, their reference and
     * in the reference velocity / acceleration (zero for a contact), so they run the same instructions (two divergent
     * calls did the SE3 logarithm twice) */
    const int f = lane & 1;
    const bool is_contact = lane < 2;
    double b6[6], kp[6], kd[6];
    /* kp_contact[6], kd_contact[6], kp_foot[6], kd_foot[6] are consecutive in DevConst: one lane-indexed constant read
     * per gain instead of two reads and a select */
    static_assert(offsetof(DevConst, kd_contact) == offsetof(DevConst, kp_contact) + 48 &&
                  offsetof(DevConst, kp_foot) == offsetof(DevConst, kp_contact) + 96 &&
                  offsetof(DevConst, kd_foot) == offsetof(DevConst, kp_contact) + 144, "gain tables are consecutive");
    const double* gains = C.kp_contact + (is_contact ? 0 : 12);
#pragma unroll
    for (int k = 0; k < 6; k++) { kp[k] = gains[k]; kd[k] = gains[6 + k]; }
    const double* ref = is_contact ? rf + RF_CONTACT + 12 * f : rf + RF_FOOT + 24 * f;
    se3_rhs(fr, f, kp, kd, ref, is_contact ? nullptr : ref + 12, is_contact ? nullptr : ref + 18, b6);
    double* dst = bv + (is_contact ? BV_MOT : BV_FOOT) + 6 * f;
#pragma unroll
    for (int k = 0; k < 6; k++) dst[k] = b6[k];
  } else if (lane < 7) {
    /* tsid::TaskComEquality */
    const int r = lane - 4;
    const double rp = rf[RF_COM + r], rv = rf[RF_COM + 3 + r], ra = rf[RF_COM + 6 + r];
    double ades = -C.kp_com[r] * (fr[FR_COM + r] - rp) - C.kd_com[r] * (fr[FR_COM + 3 + r] - rv) + ra;
    bv[BV_COM + r] = ades - fr[FR_COM + 6 + r];
  } else if (lane < 10) {
    /* legacy tsid::TaskAMEquality: -Kp (L - 0) + 0 - drift */
    const int r = lane - 7;
    bv[BV_AM + r] = -C.kp_am[r] * fr[FR_L + r] - fr[FR_L + 3 + r];
  }
  /* tsid::TaskJointPosture */
  if (lane < na) {
    const double rp = rf[RF_POST + lane];
    bv[BV_POST + lane] = -mdl[MDL_oPOST + lane] * (qs[7 + lane] - rp) - mdl[MDL_oPOST + 23 + lane] * vs[6 + lane];
  }
  __syncwarp();
  /* H_dv = w_foot (JF0^T JF0 + JF1^T JF1) + w_com Jcom^T Jcom + w_post S^T S (+ w_am Ag^T Ag) + hreg I
   * g_dv = -(w_foot JF^T b_foot + w_com Jcom^T b_com + w_post S^T b_post + w_am Ag^T b_am)          */
  const double* JF = sm + SM_oJF;
  const double* Jcom = sm + SM_oJcom;
  const double* Ag = sm + SM_oAg;
  double* H = sm + SM_oH;
  double* gv = sm + SM_oGv;
  const int j = lane;
  if (j < nv) {
    double jf[12], jc[3], ja[3] = {0, 0, 0};
#pragma unroll
    for (int r = 0; r < 12; r++) jf[r] = JF[r * TSIDB_NVX + j];
#pragma unroll
    for (int r = 0; r < 3; r++) jc[r] = Jcom[r * TSIDB_NVX + j];
    if (C.use_am) {
#pragma unroll
      for (int r = 0; r < 3; r++) ja[r] = Ag[r * TSIDB_NVX + j];
    }
    /* Lane j keeps column j of the stacked task matrix [JF; Jcom; Ag] in registers and forms H[t][j] for two rows t
     * at a time: the other factor, column t, is the same for every lane, so it arrives as 16-byte BROADCAST reads (one
     * shared-memory wavefront each) and a row of H leaves as one contiguous store.  The symmetric half-matrix
     * scheme of round 1 (rows j+t cyclic) did half the FMAs but read 15 lane-strided values per entry and
     * scattered its stores at stride 28 (8-way bank conflicts): 2.5x the shared-memory wavefronts of this loop,
     * in a kernel that runs at two thirds of the shared-memory pipe's rate. */
    static_assert((NV & 1) == 0 && (TSIDB_NVX & 1) == 0, "rows of H come in pairs");
    /* Columns t, t+1 of a foot's Jacobian are exactly zero unless their joints lie on the chain root -> foot (the base
     * columns always do): the six rows of a foot are skipped for the column pairs off its chain — the arms' and the head's
     * pairs take neither foot, a leg's pairs one (the test is warp-uniform: t is the loop variable; adding the skipped
     * terms would add exact zeros, so the sums are unchanged bit for bit). */
    /* bit t of pm0 / pm1 (t even): the column pair t, t+1 meets the chain of foot 0 / 1 (columns t >= 6 are the joints of
     * bodies t-5, t-4; the base pairs always do) */
    const unsigned pm0 = ((C.foot_support[0] | (C.foot_support[0] >> 1)) << 5) | 63u;
    const unsigned pm1 = ((C.foot_support[1] | (C.foot_support[1] >> 1)) << 5) | 63u;
#pragma unroll 1
    for (int t = 0; t < nv; t += 2) {
      double sa0 = 0.0, sa1 = 0.0, sb0 = 0.0, sb1 = 0.0, ca = 0.0, cb = 0.0, ma = 0.0, mb = 0.0;
      const bool on0 = (pm0 >> t) & 1u, on1 = (pm1 >> t) & 1u;
#define TSIDB_HFOOT(R0_)                                                                       \
  _Pragma("unroll") for (int r = (R0_); r < (R0_) + 6; r += 2) {                                 \
    const double2 p = *reinterpret_cast<const double2*>(JF + r * TSIDB_NVX + t);                 \
    const double2 q = *reinterpret_cast<const double2*>(JF + (r + 1) * TSIDB_NVX + t);           \
    sa0 += p.x * jf[r]; sb0 += p.y * jf[r];                                                      \
    sa1 += q.x * jf[r + 1]; sb1 += q.y * jf[r + 1];                                              \
  }
      if (on0) { TSIDB_HFOOT(0) } /* one test per foot and trip (six, one per row pair, cost 145 instructions per env) */
      if (on1) { TSIDB_HFOOT(6) }
#undef TSIDB_HFOOT
#pragma unroll
      for (int r = 0; r < 3; r++) {
        const double2 p = *reinterpret_cast<const double2*>(Jcom + r * TSIDB_NVX + t);
        ca += p.x * jc[r]; cb += p.y * jc[r];
      }
      double ha = C.w_foot * (sa0 + sa1) + C.w_com * ca, hb = C.w_foot * (sb0 + sb1) + C.w_com * cb;
      if (C.use_am) {
#pragma unroll
        for (int r = 0; r < 3; r++) {
          const double2 p = *reinterpret_cast<const double2*>(Ag + r * TSIDB_NVX + t);
          ma += p.x * ja[r]; mb += p.y * ja[r];
        }
        ha += C.w_am * ma; hb += C.w_am * mb;
      }
      H[t * SM_LDM + j] = ha;
      H[(t + 1) * SM_LDM + j] = hb;
    }
    /* the diagonal terms (posture weight on the joints, regulariser) go in after the loop: the lane that wrote H[j][j]
     * adds them (inside the loop the two tests cost 28 instructions per trip, 7 % of the kernel) */
    H[j * SM_LDM + j] += (j >= 6 ? C.w_post : 0.0) + C.hreg;
    double gf = 0.0, gc = 0.0, ga = 0.0;
#pragma unroll
    for (int r = 0; r < 12; r++) gf += jf[r] * bv[BV_FOOT + r];
#pragma unroll
    for (int r = 0; r < 3; r++) gc += jc[r] * bv[BV_COM + r];
    double g = C.w_foot * gf + C.w_com * gc;
    if (C.use_am) {
#pragma unroll
      for (int r = 0; r < 3; r++) ga += ja[r] * bv[BV_AM + r];
      g += C.w_am * ga;
    }
    if (j >= 6) g += C.w_post * bv[BV_POST + j - 6];
    gv[j] = -g; /* the QP gradient: g = -sum w A^T b */
  }
  /* force part of g is zero (force regularisation has zero reference) */
  for (int k = nv + lane; k < TSIDB_NX; k += 32) gv[k] = 0.0;
  __syncwarp();
}

/* ================================================================= K3: the QP */
/* ---- register-blocked building blocks of the equality elimination (template on nv) ----
 * Each lane keeps ONE column (of B, of Q2/J2) or ONE row (of the Cholesky factor) in registers; all
 * register-array indices are compile-time constants (fully unrolled loops), the operands shared by the
 * warp (factor entries, Householder vectors) are broadcast reads from shared memory. */

/* b <- L^-1 b (dv block, axpy form) and b_f <- Lf^-1 b_f */
template <int NV, int NC>
TSIDB_DEV void fwdsub_L(double (&b)[NV + 12 * NC], const double* L, const double* ild, const DevConst& C) {
#pragma unroll
  for (int k = 0; k < NV; k++) {
    SCHED_FENCE();
    b[k] *= ild[k];
#pragma unroll
    for (int i = k + 1; i < NV; i++) b[i] -= L[i * SM_LDM + k] * b[k];
  }
#pragma unroll
  for (int s = 0; s < NC; s++) {
    {
      double t[12];
#pragma unroll
      for (int i = 0; i < 12; i++) t[i] = b[NV + 12 * s + i];
#pragma unroll
      for (int i = 0; i < 12; i++) {
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k <= i; k++) acc += C.Lfinv[i][k] * t[k];
        b[NV + 12 * s + i] = acc;
      }
    }
  }
}

/* c[K0:K) <- (I - tau v v^T) c[K0:K) with the dense reflector v (explicit zeros above its head, the unscaled head
 * entry at the head); rows below K0 and from K on are zero in v by construction and are not visited */
template <int N, int K0, int K, bool RELOAD>
TSIDB_DEV void reflect(double (&c)[N], const double* v, double tau) {
  static_assert((K & 1) == 0 && (K0 & 1) == 0, "rows come in pairs");
  /* the reflector is read as 16-byte pairs (broadcast): half the shared-memory instructions */
  const double2* v2 = reinterpret_cast<const double2*>(v);
  double w0 = 0.0, w1 = 0.0, w2 = 0.0, w3 = 0.0;
  if (RELOAD) {
#pragma unroll
    for (int k = K0; k < K; k += 4) {
      const double2 p = v2[k >> 1];
      w0 += p.x * c[k];
      w1 += p.y * c[k + 1];
      if (k + 2 < K) {
        const double2 q = v2[(k >> 1) + 1];
        w2 += q.x * c[k + 2];
        w3 += q.y * c[k + 3];
      }
    }
    const double w = tau * ((w0 + w1) + (w2 + w3));
    SCHED_FENCE(); /* reload v for the update instead of keeping 50 more values live (spills otherwise) */
#pragma unroll
    for (int k = K0; k < K; k += 2) {
      const double2 p = v2[k >> 1];
      c[k] -= w * p.x;
      c[k + 1] -= w * p.y;
    }
  } else {
    /* the lighter classes have the registers to keep the reflector between the two passes */
    double2 p[(K - K0) / 2];
#pragma unroll
    for (int k = 0; k < (K - K0) / 2; k++) p[k] = v2[(K0 >> 1) + k];
#pragma unroll
    for (int k = 0; k < K - K0; k += 4) {
      w0 += p[k >> 1].x * c[K0 + k];
      w1 += p[k >> 1].y * c[K0 + k + 1];
      if (k + 2 < K - K0) {
        w2 += p[(k >> 1) + 1].x * c[K0 + k + 2];
        w3 += p[(k >> 1) + 1].y * c[K0 + k + 3];
      }
    }
    const double w = tau * ((w0 + w1) + (w2 + w3));
#pragma unroll
    for (int k = 0; k < K - K0; k += 2) {
      c[K0 + k] -= w * p[k >> 1].x;
      c[K0 + k + 1] -= w * p[k >> 1].y;
    }
  }
}

template <bool B>
struct BoolTag { static constexpr bool value = B; };
/* head row of reflector k for a class with NCM contact-motion equalities (see k3_eliminate) */
template <int NV, int NCM>
TSIDB_DEV constexpr int head_row(int k) { return (k < NCM || NCM == 0) ? k : NV + (k - NCM); }

template <int N, int NV, int NCM, int NEQ>
TSIDB_DEV void store_R1(double* R1, const double (&b)[N], int lane) {
#pragma unroll
  for (int k = 0; k < NEQ; k++) R1[k * SM_LDB + lane] = b[head_row<NV, NCM>(k)];
}

/* shared-memory layout of one env in the elimination kernel per contact class: the assembly image (SE_*, the same
 * for every class) followed by class-sized work arrays; the reflector rows have the class's own stride N */
TSIDB_HD constexpr int e_per_env(int nv, int nc) {
  const int n = nv + 12 * nc, neq = 6 + 6 * nc;
  const int vt_own = (neq * n <= 162 + 312) ? 0 : neq * n; /* the reflectors of the light classes reuse the M_u | JF part of the image */
  return SE_IMAGE + 26 + 18 + 18 + vt_own + neq * SM_LDB + n + 64 + n + 2;
}
template <int NV, int NC>
struct EL {
  enum : int {
    N = NV + 12 * NC, NEQ = 6 + 6 * NC,
    VT_ALIAS = (NEQ * N <= 162 + 312) ? 1 : 0, /* M_u and JF are dead once B is built; the reflectors are written after that */
    oILD = SE_IMAGE,          /* 1/L_ii                           26 */
    oTAU = oILD + 26,         /* Householder coefficients         18 */
    oRD = oTAU + 18,          /* diagonal of R1, then its inverse 18 */
    oVT = VT_ALIAS ? SE_oMu : oRD + 18,                 /* reflectors [NEQ][N] */
    oR1 = VT_ALIAS ? oRD + 18 : oRD + 18 + NEQ * N,     /* R1 [NEQ][SM_LDB]    */
    oCOL = oR1 + NEQ * SM_LDB, /* published column                 N */
    oW0 = oCOL + N,           /* w0                               64 */
    oX = oW0 + 64,            /* x0                                N */
    oBar = oX + N,            /* mbarrier of the image load        2 */
    per_env = oBar + 2
  };
  static_assert(per_env == e_per_env(NV, NC) && (oVT % 2) == 0 && (oCOL % 2) == 0, "layout");
};

/* The equality elimination.  In: the assembly image (SE_*: H dv block, gradient, base rows of M, JF, base nle,
 * contact-motion rhs).  Out: x = x0 (the equality-constrained minimiser), the Cholesky factor L (in place of H,
 * EL::oILD) and the Householder reflectors of B = L^-1 CE^T (EL::oVT, EL::oTAU) from which the J2 kernel builds
 * the null-space basis, the c1*c2
 * product and R_norm; returns 0 or an HQP error status.
 *
 * Column order of B: the 6*nc contact-motion rows first, then the 6 base-dynamics rows.  Any order yields the
 * same null space, x0 and projector; this one keeps the first 6*nc reflectors inside the dv rows (a contact-motion
 * row has no force entries), which halves their cost here and in the J2 kernel. */
template <int NV, int NC>
TSIDB_DEV int k3_eliminate(const DevConst& C, const double* lfinv_sm, double* sm, int lane, int mask, double& c1c2, double& c1_out, double& R_norm_out) {
  constexpr int N = NV + 12 * NC;   /* n: the contact class fixes every size at compile time */
  constexpr int nc = NC, ncm = 6 * NC, neq = 6 + 6 * NC, n = N;
  typedef EL<NV, NC> LE;
  constexpr int LDV = N;            /* reflector row stride in shared memory */
  double* L = sm + SE_oH;
  double* ild = sm + LE::oILD;
  double* tauq = sm + LE::oTAU;
  double* Rd = sm + LE::oRD;
  double* Vt = sm + LE::oVT;   /* [neq][N] dense reflectors */
  double* R1 = sm + LE::oR1;   /* [18][SM_LDB] */
  double* gv = sm + SE_oG;    /* gradient, later Q^T w_unc / w_hat */
  double* colp = sm + LE::oCOL;
  double* w0v = sm + LE::oW0;
  double* x = sm + LE::oX;
  const double* Mm = sm + SE_oMu;
  const double* JF = sm + SE_oJF;
  const double* bmot = sm + SE_oBm;
  const int f0 = (mask & 1) ? 0 : 1; /* foot of force block 0 */

  int err = ST_OPTIMAL; /* an error status is carried to the end: every warp must reach every PHASE_SYNC_E */
  PHASE_SYNC_E();
  /* ---- Cholesky of the dv block: lane i keeps row i; c1 = trace(H), c2 = trace(L^-T) ---- */
  double c1, c2;
  {
    const int i = lane < NV ? lane : NV - 1;
    double l[NV];
#pragma unroll
    for (int k = 0; k < NV; k++) l[k] = L[i * SM_LDM + k];
    c1 = warp_sum(lane < NV ? L[i * SM_LDM + i] : 0.0) + nc * C.Hf_trace;
    bool bad = false;
    double c2p = 0.0;
#pragma unroll
    for (int j = 0; j < NV; j++) {
      double a0 = l[j], a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
      for (int k = 0; k < j; k++) {
        const double ljk = L[j * SM_LDM + k];
        if ((k & 3) == 0) a0 -= l[k] * ljk;
        else if ((k & 3) == 1) a1 -= l[k] * ljk;
        else if ((k & 3) == 2) a2 -= l[k] * ljk;
        else a3 -= l[k] * ljk;
      }
      const double s = (a0 + a1) + (a2 + a3);
      const double sj = shfl(s, j);
      if (!(sj > 0.0)) bad = true;
      const double inv = rsqrt(sj);
      l[j] = (lane == j) ? sj * inv : s * inv;
      c2p += inv;
      __syncwarp();
      if (lane >= j && lane < NV) L[lane * SM_LDM + j] = l[j];
      if (lane == j) ild[j] = inv;
      __syncwarp();
    }
    if (bad) err = ST_INFEASIBLE; /* eiquadprog: Cholesky failure -> UNBOUNDED -> HQP_STATUS_INFEASIBLE */
    c2 = c2p + nc * C.Lfinv_trace;
  }
  c1c2 = c1 * c2;
  c1_out = c1;

  PHASE_SYNC_E();
  /* ---- B = L^-1 [CE^T | g]: lane e keeps column e; Householder QR; the last column becomes Q^T w_unc ---- */
  double R_norm = 1.0;
  {
    double b[N];
    const int e = lane;
#pragma unroll
    for (int k = 0; k < N; k++) b[k] = 0.0;
    if (e < ncm) {
      /* contact motion row: [JF_f(r,:) | 0], contacts in x order */
      const int s = e / 6, r = e % 6;
      const int f = (s == 0) ? f0 : 1;
#pragma unroll
      for (int k = 0; k < NV; k++) b[k] = JF[(f * 6 + r) * TSIDB_NVX + k];
    } else if (e < neq) {
      /* base dynamics row u: [M(u,:) | -Jc(:,u)^T] */
      const int u = e - ncm;
#pragma unroll
      for (int k = 0; k < NV; k++) b[k] = Mm[u * SM_LDM + k];
#pragma unroll
      for (int s = 0; s < NC; s++) {
        {
          const int f = (s == 0) ? f0 : 1;
          double jf[6];
#pragma unroll
          for (int r = 0; r < 6; r++) jf[r] = JF[(f * 6 + r) * TSIDB_NVX + u];
#pragma unroll
          for (int o = 0; o < 12; o++) {
            double acc = 0.0;
#pragma unroll
            for (int r = 0; r < 6; r++) acc += C.T[r][o] * jf[r];
            b[NV + 12 * s + o] = -acc;
          }
        }
      }
    } else if (e == neq) {
#pragma unroll
      for (int k = 0; k < N; k++) b[k] = gv[k];
    }
    fwdsub_L<NV, NC>(b, L, ild, C);
    if (e == neq) {
#pragma unroll
      for (int k = 0; k < N; k++) b[k] = -b[k]; /* w_unc = -L^-1 g */
    }
    PHASE_SYNC_E();
    /* Reflector i < ncm (contact motion): head row i, span = dv rows i..NV-1.  Reflector i >= ncm (base
     * dynamics): head = force row NV + (i - ncm), span = dv rows ncm..NV-1 and the force rows from the head
     * on.  The base-dynamics columns carry their largest entries in the force rows (scaled by Lf^-1), so
     * pivoting on those keeps the factorisation row-wise stable; with the head on a small dv row the
     * result is 40x further from the 80-bit truth (measured, DESIGN.md).  Without contacts there are no
     * force rows: head i, span i..NV-1.  The two kinds run in loops of their own (the kind is a compile-time
     * constant of the step: a contact-motion reflector lives in the rows below 32, one trip per lane). */
    auto qr_step = [&](const int i, auto top_tag) {
      constexpr bool top = decltype(top_tag)::value;
      PHASE_SYNC_E();
      const int head = top ? i : NV + (i - ncm);
      __syncwarp();
      if (lane == i) {
        /* only the rows a reflector of this kind can span are published */
        double2* c2 = reinterpret_cast<double2*>(colp);
#pragma unroll
        for (int k = (top ? 0 : ncm); k < (top ? NV : N); k += 2) c2[k >> 1] = make_double2(b[k], b[k + 1]);
      }
      __syncwarp();
      double part = 0.0;
      if (top) {
        if (lane > i && lane < NV) { const double t = colp[lane]; part = t * t; }
      } else {
        for (int k = lane; k < n; k += 32) {
          const bool in_span = (k >= ncm && k < NV) || k > head;
          if (in_span) { const double t = colp[k]; part += t * t; }
        }
      }
      const double sigma = warp_sum(part);
      const double alpha = colp[head];
      const double nrm = sqrt(alpha * alpha + sigma);
      const double beta = (alpha >= 0.0) ? -nrm : nrm;
      /* dependent equality row [eiquadprog add_constraint: |d(iq)| <= eps * R_norm] */
      if (fabs(beta) <= TS_EPS * R_norm && err == ST_OPTIMAL) err = ST_ERROR;
      R_norm = fmax(R_norm, fabs(beta));
      /* UNSCALED Householder vector u = x - beta e_head, H = I - kappa u u^T with kappa = -1 / (beta u_head):
       * the vector can be published as soon as beta is known, and the one reciprocal (instead of two divisions)
       * overlaps with the dot products of the reflection */
      const double uh = alpha - beta;
      if (top) {
        Vt[i * LDV + lane] = (lane == i) ? uh : ((lane > i && lane < NV) ? colp[lane] : 0.0);
        if (lane + 32 < N) Vt[i * LDV + lane + 32] = 0.0;
      } else {
        for (int k = lane; k < N; k += 32) {
          const bool in_span = (k >= ncm && k < NV) || k > head;
          Vt[i * LDV + k] = (k == head) ? uh : (in_span ? colp[k] : 0.0);
        }
      }
      const double tau = -1.0 / (beta * uh);
      if (lane == 0) { tauq[i] = tau; Rd[i] = beta; }
      __syncwarp();
      if (lane > i && lane <= neq) {
        if (top) reflect<N, 0, NV, (NC == 2)>(b, Vt + i * LDV, tau);
        else reflect<N, ncm, N, (NC == 2)>(b, Vt + i * LDV, tau); /* a base-dynamics reflector is zero in the dv rows above ncm */
      }
    };
    constexpr int n_top = (nc == 0) ? neq : ncm;
    for (int i = 0; i < n_top; i++) qr_step(i, BoolTag<true>());
    for (int i = n_top; i < neq; i++) qr_step(i, BoolTag<false>());
    __syncwarp();
    /* R1 (strictly upper part; the diagonal is Rd) and the carried column */
    if (lane <= neq) {
      /* R1[k][j] = entry of column j at the head row of reflector k */
      store_R1<N, NV, ncm, neq>(R1, b, lane);
    }
    if (lane == neq) {
#pragma unroll
      for (int k = 0; k < N; k++) gv[k] = b[k];
    }
    __syncwarp();
  }
  PHASE_SYNC_E();
  /* ---- w_hat[0:neq] = R1^-T rhs (forward substitution, lane <-> equation); rhs = -ce0 ---- */
  {
    double rhs = 0.0;
    if (lane < ncm) {
      const int s = lane / 6, r = lane % 6;
      const int f = (s == 0) ? f0 : 1;
      rhs = bmot[6 * f + r];
    } else if (lane < neq) {
      rhs = -sm[SE_oNle + lane - ncm];
    }
    /* equation `lane` scaled by 1 / R_ll up front: a step of the chain is one shuffle and one FMA */
    const double ird = (lane < neq) ? 1.0 / Rd[lane] : 0.0;
    double accv = rhs * ird;
#pragma unroll
    for (int i = 0; i < neq - 1; i++) {
      const double wi = shfl(accv, i);
      if (lane > i && lane < neq) accv -= (R1[i * SM_LDB + lane] * ird) * wi;
    }
    __syncwarp();
    if (lane < neq) gv[(lane < ncm || nc == 0) ? lane : NV + (lane - ncm)] = accv; /* head row of reflector `lane` */
    __syncwarp();
  }
  /* ---- w0 = Q w_hat: reflectors in reverse, lanes over rows ---- */
  double y0 = (lane < n) ? gv[lane] : 0.0;
  double y1 = (lane + 32 < n) ? gv[lane + 32] : 0.0;
#pragma unroll
  for (int i = neq - 1; i >= 0; i--) {
    const double v0 = (lane < N) ? Vt[i * LDV + lane] : 0.0; /* a reflector row holds N entries */
    /* a contact-motion reflector (i < ncm, or any reflector without contacts) is zero in the rows from 32 on */
    const double v1 = (i >= ((nc == 0) ? neq : ncm) && lane + 32 < N) ? Vt[i * LDV + lane + 32] : 0.0;
    const double w = tauq[i] * warp_sum(v0 * y0 + v1 * y1);
    y0 -= w * v0;
    y1 -= w * v1;
  }
  /* ---- x0 = L^-T w0: force rows through the constant Lf^-T, dv rows by a column-oriented back substitution
   *      (lane <-> row; one broadcast and one FMA per step) ---- */
  w0v[lane] = y0;
  if (lane + 32 < N) w0v[lane + 32] = y1;
  __syncwarp();
  if (lane < 12 * nc) {
    const int s = lane / 12, i = lane % 12;
    double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
    for (int k = 0; k < 12; k += 2) { /* Lf^-1 is lower triangular: entries above the diagonal are stored as zeros */
      acc0 += lfinv_sm[k * 12 + i] * w0v[NV + 12 * s + k];
      acc1 += lfinv_sm[(k + 1) * 12 + i] * w0v[NV + 12 * s + k + 1];
    }
    x[NV + lane] = acc0 + acc1;
  }
  {
    /* row `lane` scaled by 1 / L_ll up front; unrolled, so the scaled coefficients are formed off the chain and a
     * step is one shuffle and one FMA */
    const double il = (lane < NV) ? ild[lane] : 0.0;
    y0 *= il;
#pragma unroll
    for (int k = NV - 1; k > 0; k--) {
      const double xk = shfl(y0, k);
      if (lane < k) y0 -= (L[k * SM_LDM + lane] * il) * xk;
    }
  }
  if (lane < NV) x[lane] = y0;
  __syncwarp();
  R_norm_out = R_norm;
  return err;
}

/* ================================================================= hand-off between the kernels */
/* The dynamics kernel leaves the assembly image (SE_*) for the elimination kernel, and both of them fill the
 * solver image (SA_*) that the active-set kernel pulls from a work counter with one linear bulk copy (the image is
 * that kernel's shared-memory layout).  What the hand-off buys is that every stage runs at the occupancy and the
 * thread mapping that suit it, and that the active set balances its data-dependent iteration counts (1..40)
 * dynamically. */
#define SA_LDJA 20                        /* JFa row stride                                  */
#define SA_LDM 26                         /* M_a row stride: even with SA_LDM/2 odd, 16-byte lane-strided reads are conflict-free */
/* Solver image / active-set shared-memory layout of one env, per contact class (nc = 2, 1, 0).  The first
 * `image` doubles are what the producer kernels write to HBM and what one bulk copy brings in; the work arrays
 * follow.  J2's row stride ldj (m or m + 2) is even (16-byte row accesses) with ldj/2 odd, which keeps both the row-wise
 * 16-byte accesses (lane <-> row) and the column-wise 8-byte ones (lane <-> column) free of bank conflicts.
 * The status block comes first so that it sits at the same place for every class. */
struct ALayout {
  int n, m, ldj;
  int oSc, oJ2, oMa, oJFa, oNle, oVj, oX, image;
  int oWr, oR, oNP, oD, oBar, per_env;
};
TSIDB_HD constexpr int even_up(int x) { return (x + 1) & ~1; }
TSIDB_HD constexpr ALayout a_layout(int nv, int nc) {
  ALayout L{};
  const int na = nv - 6;
  L.n = nv + 12 * nc;
  L.m = na + 6 * nc;
  L.ldj = (((L.m / 2) & 1) != 0) ? L.m : L.m + 2;
  L.oSc = 0;                              /* c1*c2, R_norm, error status, contact mask */
  L.oJ2 = 4;                              /* J2  n x ldj                               */
  L.oMa = L.oJ2 + L.n * L.ldj;            /* M_a na x SA_LDM (rows 6.. of M)           */
  L.oJFa = L.oMa + na * SA_LDM;           /* JF columns 6.. of the feet in contact, in force-block order: 6 nc x SA_LDJA */
  L.oNle = L.oJFa + 6 * nc * SA_LDJA;     /* nle_a                                     */
  L.oX = L.oNle + even_up(na);            /* x                                         */
  L.oVj = L.oX + even_up(L.n);            /* joint velocities: only read when the env is loaded (joint-bound limits
                                           * into registers), so the work arrays start on top of them */
  L.image = L.oVj + even_up(na);
  L.oWr = L.oVj;                          /* wrenches 12                               */
  L.oR = L.oWr + 12;                      /* R packed by columns: col j at j(j+1)/2    */
  L.oNP = L.oR + even_up(L.m * (L.m + 1) / 2);  /* dense constraint normal (actuation rows) */
  L.oD = L.oNP + even_up(L.n);            /* d (free columns), zero padded to m + 2; doubles as the Householder vector */
  L.oBar = L.oD + L.m + 2;                /* mbarrier of the image load                */
  L.per_env = L.oBar + 2;
  if (L.per_env < L.image + 2) L.per_env = L.image + 2;
  return L;
}
/* the same numbers as enumerators (pure compile-time constants in device code) */
template <int NV, int NC>
struct AL {
  enum : int { n = a_layout(NV, NC).n, m = a_layout(NV, NC).m, ldj = a_layout(NV, NC).ldj, oSc = a_layout(NV, NC).oSc, oJ2 = a_layout(NV, NC).oJ2, oMa = a_layout(NV, NC).oMa, oJFa = a_layout(NV, NC).oJFa, oNle = a_layout(NV, NC).oNle, oVj = a_layout(NV, NC).oVj, oX = a_layout(NV, NC).oX, image = a_layout(NV, NC).image, oWr = a_layout(NV, NC).oWr, oR = a_layout(NV, NC).oR, oNP = a_layout(NV, NC).oNP, oD = a_layout(NV, NC).oD, oBar = a_layout(NV, NC).oBar, per_env = a_layout(NV, NC).per_env };
};
#define SA_IMAGE (a_layout(TSIDB_NVX, 2).image)   /* slot stride of the solver images in HBM (largest class) */
#define SA_oSc 0
/* warps per CTA of the active-set kernel per contact class (shared memory: 27.4 / 18.7 / 12.6 KB per env);
 * multiples of 4 keep the four schedulers of an SM evenly loaded */
#define TSIDB_AS_WARPS_DS 8
#define TSIDB_AS_WARPS_SS 12
#define TSIDB_AS_WARPS_FL 12

/* ---- bulk asynchronous copy global -> shared (TMA, 1-D) completed through an mbarrier ---- */
#ifndef TSIDB_EMU
TSIDB_DEV unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
TSIDB_DEV void mbar_init(void* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
/* issued by ONE lane: every generic-proxy access of the destination by this warp must be ordered before
 * (caller: __syncwarp) */
TSIDB_DEV void bulk_load(void* dst, const void* src, unsigned bytes, void* bar) {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
/* bulk asynchronous store shared -> global (issued by ONE lane after a __syncwarp that makes the warp's
 * shared-memory writes visible); bulk_store_commit closes the group, bulk_store_wait_read returns when the
 * stores of all committed groups have finished READING shared memory (the source may then be overwritten) */
TSIDB_DEV void bulk_store(void* dst, const void* src, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
TSIDB_DEV void bulk_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
TSIDB_DEV void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
/* pull a region into L2 ahead of the bulk load that will fetch it (bytes: multiple of 16) */
TSIDB_DEV void bulk_prefetch_l2(const void* src, unsigned bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
TSIDB_DEV void mbar_wait(void* bar, unsigned parity) {
  unsigned ok = 0;
  const unsigned addr = smem_u32(bar);
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok)
                 : "r"(addr), "r"(parity)
                 : "memory");
  } while (!ok);
}
#endif

/* order-preserving map double -> uint64 (smaller double <-> smaller key) */
TSIDB_DEV unsigned long long sortable(double v) {
  unsigned long long b;
  memcpy(&b, &v, 8);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
/* per-lane constants of one env, kept in registers across the iterations */
struct LaneConst {
  double lb, ub;     /* joint-bound row `lane`: lb <= dv_j <= ub */
  double tmin, tmax; /* actuation row `lane`: tmin <= tau <= tmax */
  double vmin, vmax; /* joint velocity limits of joint `lane` */
  double fric[3];    /* friction pyramid row lane % 4 */
  double Trow[12];   /* row lane%6 of the force generator */
};

struct ASCtx {
  int na, nv;         /* compile-time in the per-class kernels (constant-propagated through the inlined solver) */
  int ldj;            /* row stride of J2 */
  double* J2;
  const double* Ma;
  const double* JFa;  /* rows of the feet in contact, in force-block order */
  int nfr;            /* 6 * (feet in contact) rows of JFa */
  int wro;            /* wrench of force block 0 starts at wr[wro] (wr is per foot: LF 0..5, RF 6..11) */
  const double* nle_a;
  const double* vj;
  double* x;
  double* wr;
  double *Rp, *np, *dd;
};

/* x index of foot f's first force variable */
TSIDB_DEV int fvar0(int nv, int mask, int f) { return nv + ((f == 1 && (mask & 1)) ? 12 : 0); }

/* one-sided candidate rows ("cid"), fixed numbering:
 *   0..31   friction pyramid upper sides: f = cid/16, corner = (cid%16)/4, k = cid%4
 *   32..35  normal force: f = (cid-32)/2, side = (cid-32)%2  (0: >= fmin, 1: <= fmax)
 *   36..36+2na-1        actuation, side-major
 *   36+2na..36+4na-1    joint (velocity) bounds, side-major
 * The never-active sides of the reference's two-sided blocks (friction lower side at -1e10, the six
 * base rows of the joint-bounds block at +-1e10) are not enumerated: they can neither be violated
 * nor change the violation sum.
 * Lane ownership: lane l evaluates "slot" 0: cid l (friction), 1: cid 32+(l-12) (lanes 12..15: they form the normal
 * force in the same pass in which lanes 0..11 form the wrenches), 2/3: actuation row l lower/upper, 4/5: joint-bound
 * row l lower/upper (l < na). */
#define NRM_LANE0 12
TSIDB_DEV int cid_of(int na, int lane, int slot) {
  return slot == 0 ? lane : (slot == 1 ? 32 + lane - NRM_LANE0 : 36 + (slot - 2) * na + lane);
}
TSIDB_DEV void cid_owner(int na, int cid, int& lane, int& slot) {
  if (cid < 32) { lane = cid; slot = 0; }
  else if (cid < 36) { lane = cid - 32 + NRM_LANE0; slot = 1; }
  else { const int k = cid - 36; slot = 2 + k / na; lane = k - (slot - 2) * na; }
}
/* bit index in the 192-bit active-set word = row numbering of tsidb_ci_row() */
TSIDB_DEV int cid_bit(int na, int nv, int cid) {
  if (cid < 32) return 34 * (cid >> 4) + 17 + (cid & 15);
  if (cid < 36) return 34 * ((cid - 32) >> 1) + (((cid - 32) & 1) ? 33 : 16);
  if (cid < 36 + 2 * na) { int k = cid - 36; return 68 + k; }
  int k = cid - 36 - 2 * na;
  int side = k >= na ? 1 : 0, i = k - side * na;
  return 68 + 2 * na + side * nv + 6 + i;
}

/* the part of LaneConst that depends on the lane only: read once per kernel (lane-indexed reads of __constant__
 * memory are served one address at a time) */
TSIDB_DEV void lane_const_init(const DevConst& C, LaneConst& K, int lane) {
  const int na = C.na;
  /* lanes 0..11: row lane % 6 of the force generator; lanes 12..15: the normal-force row [n n n n] */
#pragma unroll
  for (int j = 0; j < 12; j++) K.Trow[j] = (lane >= NRM_LANE0 && lane < NRM_LANE0 + 4) ? C.nrm[j % 3] : C.T[lane % 6][j];
#pragma unroll
  for (int j = 0; j < 3; j++) K.fric[j] = C.fric[lane & 3][j];
  K.tmin = (lane < na) ? C.tau_min[lane] : 0.0;
  K.tmax = (lane < na) ? C.tau_max[lane] : 0.0;
  K.vmin = (lane < na) ? C.v_min[lane] : 0.0;
  K.vmax = (lane < na) ? C.v_max[lane] : 0.0;
  K.lb = K.ub = 0.0;
}

/* the same from the handle's table (TBL_oLANE): coalesced */
TSIDB_DEV void lane_const_load(const double* tables, LaneConst& K, int lane) {
  const double* t = tables + TBL_oLANE + lane;
#pragma unroll
  for (int j = 0; j < 12; j++) K.Trow[j] = t[j * 32];
#pragma unroll
  for (int j = 0; j < 3; j++) K.fric[j] = t[(12 + j) * 32];
  K.tmin = t[15 * 32]; K.tmax = t[16 * 32]; K.vmin = t[17 * 32]; K.vmax = t[18 * 32];
  K.lb = K.ub = 0.0;
}

/* s = CI x + ci0 for the rows this lane owns; invalid rows get +inf */
TSIDB_DEV void eval_rows(const DevConst& C, const ASCtx& S, const LaneConst& K, int lane, int mask, double (&s)[6]) {
  const int na = S.na, nv = S.nv;
  const double* x = S.x;
#pragma unroll
  for (int k = 0; k < 6; k++) s[k] = TS_INF;
  {
    const int f = lane >> 4, c = (lane & 15) >> 2;
    if ((mask >> f) & 1) {
      const double* ff = x + fvar0(nv, mask, f) + 3 * c;
      s[0] = -(K.fric[0] * ff[0] + K.fric[1] * ff[1] + K.fric[2] * ff[2]);
    }
  }
  if (lane < 4) {
    const int f = lane >> 1, side = lane & 1;
    if ((mask >> f) & 1) {
      const double* ff = x + fvar0(nv, mask, f);
      double t = 0.0;
#pragma unroll
      for (int c = 0; c < 4; c++) t += C.nrm[0] * ff[3 * c] + C.nrm[1] * ff[3 * c + 1] + C.nrm[2] * ff[3 * c + 2];
      s[1] = side ? (C.fmax - t) : (t - C.fmin);
    }
  }
  if (lane < na) {
    if (C.use_tb) {
      /* tau_r = h_r + M_a(r,:) dv - sum_f JF_f(:,6+r)^T (T f_f); 16-byte reads of the row and of x */
      const double2* Mr = reinterpret_cast<const double2*>(S.Ma + lane * SA_LDM);
      const double2* x2 = reinterpret_cast<const double2*>(x);
      double t0 = S.nle_a[lane], t1 = 0.0, t2 = 0.0, t3 = 0.0;
      int j = 0;
      for (; j + 1 < nv / 2; j += 2) {
        const double2 m0 = Mr[j], m1 = Mr[j + 1], x0 = x2[j], x1 = x2[j + 1];
        t0 += m0.x * x0.x; t1 += m0.y * x0.y; t2 += m1.x * x1.x; t3 += m1.y * x1.y;
      }
      for (; j < nv / 2; j++) { const double2 m0 = Mr[j], x0 = x2[j]; t0 += m0.x * x0.x; t1 += m0.y * x0.y; }
      double u0 = 0.0, u1 = 0.0, u2 = 0.0;
      const double* wb = S.wr + S.wro;
#pragma unroll
      for (int q = 0; q < 12; q += 3) {
        if (q < S.nfr) {
          u0 += S.JFa[q * SA_LDJA + lane] * wb[q];
          u1 += S.JFa[(q + 1) * SA_LDJA + lane] * wb[q + 1];
          u2 += S.JFa[(q + 2) * SA_LDJA + lane] * wb[q + 2];
        }
      }
      const double t = ((t0 + t1) + (t2 + t3)) - ((u0 + u1) + u2);
      s[2] = t - K.tmin;
      s[3] = K.tmax - t;
    }
    if (C.use_jb) {
      s[4] = x[6 + lane] - K.lb;
      s[5] = K.ub - x[6 + lane];
    }
  }
}
/* s of one row (after a partial step) — lane-uniform call, every lane computes the same value */
TSIDB_DEV double eval_one(const DevConst& C, const ASCtx& S, const LaneConst& K, int cid, int mask) {
  const int na = S.na, nv = S.nv;
  const double* x = S.x;
  if (cid < 32) {
    const int f = cid >> 4, c = (cid & 15) >> 2, k = cid & 3;
    const double* ff = x + fvar0(nv, mask, f) + 3 * c;
    return -(C.fric[k][0] * ff[0] + C.fric[k][1] * ff[1] + C.fric[k][2] * ff[2]);
  }
  if (cid < 36) {
    const int f = (cid - 32) >> 1, side = (cid - 32) & 1;
    const double* ff = x + fvar0(nv, mask, f);
    double t = 0.0;
#pragma unroll
    for (int c = 0; c < 4; c++) t += C.nrm[0] * ff[3 * c] + C.nrm[1] * ff[3 * c + 1] + C.nrm[2] * ff[3 * c + 2];
    return side ? (C.fmax - t) : (t - C.fmin);
  }
  if (cid < 36 + 2 * na) {
    const int k = cid - 36, side = k >= na ? 1 : 0, r = k - side * na;
    const double* Mr = S.Ma + r * SA_LDM;
    double t = S.nle_a[r];
    for (int j = 0; j < nv; j++) t += Mr[j] * x[j];
#pragma unroll
    for (int q = 0; q < 12; q++)
      if (q < S.nfr) t -= S.JFa[q * SA_LDJA + r] * S.wr[S.wro + q];
    return side ? (C.tau_max[r] - t) : (t - C.tau_min[r]);
  }
  {
    const int k = cid - 36 - 2 * na, side = k >= na ? 1 : 0, i = k - side * na;
    /* the limits of joint i live in lane i's registers (the call is warp-uniform) */
    const double lim = shfl(side ? K.ub : K.lb, i);
    return side ? lim - x[6 + i] : x[6 + i] - lim;
  }
}

/* d_c = n_cid^T J2[:, c] for this lane's column c, using the sparsity of the row: 3 entries for a pyramid
 * row, 12 for a normal-force row, 1 for a joint bound; actuation rows are dense (normal built in np). */
TSIDB_DEV double row_dot_col(const DevConst& C, const ASCtx& S, int cid, int mask, int n, int lane, double* np) {
  const int na = S.na, nv = S.nv;
  const double* Jc = S.J2 + lane;
  if (cid < 32) {
    const int f = cid >> 4, c = (cid & 15) >> 2, k = cid & 3;
    const int r0 = fvar0(nv, mask, f) + 3 * c;
    return -(C.fric[k][0] * Jc[r0 * S.ldj] + C.fric[k][1] * Jc[(r0 + 1) * S.ldj] + C.fric[k][2] * Jc[(r0 + 2) * S.ldj]);
  }
  if (cid < 36) {
    const int f = (cid - 32) >> 1, side = (cid - 32) & 1;
    const int r0 = fvar0(nv, mask, f);
    double t = 0.0;
#pragma unroll
    for (int o = 0; o < 12; o++) t += C.nrm[o % 3] * Jc[(r0 + o) * S.ldj];
    return side ? -t : t;
  }
  if (cid >= 36 + 2 * na) {
    const int k = cid - 36 - 2 * na, side = k >= na ? 1 : 0, i = k - side * na;
    const double t = Jc[(6 + i) * S.ldj];
    return side ? -t : t;
  }
  /* actuation row r: n = +-[M_a(r,:) | -Jc(:,6+r)^T]; every lane reads the normal from np */
  double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
  int k = 0;
  for (; k + 3 < n; k += 4) {
    d0 += np[k] * Jc[k * S.ldj]; d1 += np[k + 1] * Jc[(k + 1) * S.ldj];
    d2 += np[k + 2] * Jc[(k + 2) * S.ldj]; d3 += np[k + 3] * Jc[(k + 3) * S.ldj];
  }
  for (; k < n; k++) d0 += np[k] * Jc[k * S.ldj];
  return (d0 + d1) + (d2 + d3);
}
/* dense normal of an actuation row into np[0..n) (all lanes cooperate) */
TSIDB_DEV void actuation_normal(const DevConst& C, const ASCtx& S, int cid, int mask, int n, double* np, int lane) {
  const int na = S.na, nv = S.nv;
  const int q = cid - 36, side = q >= na ? 1 : 0, r = q - side * na;
  for (int k = lane; k < n; k += 32) {
    double val;
    if (k < nv) val = S.Ma[r * SA_LDM + k];
    else {
      const int o = k - nv;
      const int blk = o / 12, j = o % 12; /* force block = row block of JFa */
      double t = 0.0;
#pragma unroll
      for (int kk = 0; kk < 6; kk++) t += C.T[kk][j] * S.JFa[(blk * 6 + kk) * SA_LDJA + r];
      val = -t;
    }
    np[k] = side ? -val : val;
  }
}

/* wrench T f of both feet -> wr[12] (zero for a foot not in contact), lanes 0..11; in the same pass lanes 12..15 form
 * the total normal force of foot (lane - 12) / 2 (K.Trow holds [n n n n] there).  Returns the lane's own sum. */
TSIDB_DEV double wrench_of(int nv, const LaneConst& K, const double* x, int mask, double* wr, int lane) {
  double s = 0.0;
  if (lane < NRM_LANE0 + 4) {
    const int f = (lane < NRM_LANE0) ? lane / 6 : (lane - NRM_LANE0) >> 1;
    if ((mask >> f) & 1) {
      const double* ff = x + fvar0(nv, mask, f);
      /* three independent chains (the solver is bound by dependent fp64 latency, not by throughput) */
      double s0 = 0.0, s1 = 0.0, s2 = 0.0;
#pragma unroll
      for (int j = 0; j < 12; j += 3) { s0 += K.Trow[j] * ff[j]; s1 += K.Trow[j + 1] * ff[j + 1]; s2 += K.Trow[j + 2] * ff[j + 2]; }
      s = (s0 + s1) + s2;
    }
    if (lane < NRM_LANE0) wr[lane] = s;
  }
  return s;
}

/* ---- Active-set iterations on the reduced basis [eiquadprog-fast solve_quadprog, after the equality phase] ----
 * The working set's state lives in registers (round 1 kept u, A, r, 1/R_jj, the saved copies and the Householder
 * vector in shared memory: every scalar update was "lane 0 writes, __syncwarp, everybody reads"; -1.7 KB of shared
 * memory per env and a third of the instructions per iteration).  Lane l owns position l of the working set — its
 * multiplier u_l, constraint id A_l, r_l = (R^-1 d)_l and 1/R_ll live in lane l's registers, like the two rows of x
 * the lane owns; the pending constraint's multiplier is a warp-uniform scalar (the reference's u[iq]); the saved copies
 * for the degenerate-add restore are register moves.  The two one-sided rows of an actuation or joint-bound pair
 * (lb <= . <= ub) cannot be violated together, so each pair is ONE candidate (the more negative side): four
 * candidates per lane instead of six, with the rows' reference indices (tie-break keys) precomputed per lane.  The
 * arg-min takes one REDUX on the high words and only falls back to the 64-bit + tie-break path when two lanes
 * share the high word.  The Householder vector is d itself with its head replaced.  All pivot rules are unchanged
 * (most violated row, lowest reference index on ties; min-ratio drop, lowest position on ties; degenerate add ->
 * exclude and restore) [eiquadprog-fast solve_quadprog after the equality phase]. */
TSIDB_DEV int warp_argmin_fast(double val, bool valid, int tiebreak) {
  const unsigned long long key = sortable(val);
  const unsigned hi = valid ? (unsigned)(key >> 32) : 0xffffffffu;
  const unsigned mhi = __reduce_min_sync(FULL, hi);
  const bool v1 = valid && hi == mhi;
  const unsigned b1 = __ballot_sync(FULL, v1);
  if (b1 == 0u) return -1;
  if ((b1 & (b1 - 1u)) == 0u) return __ffs(b1) - 1; /* a single lane holds the smallest high word */
  const unsigned lo = v1 ? (unsigned)key : 0xffffffffu;
  const unsigned mlo = __reduce_min_sync(FULL, lo);
  const bool v2 = v1 && lo == mlo;
  const unsigned tb = v2 ? (unsigned)tiebreak : 0xffffffffu;
  const unsigned mtb = __reduce_min_sync(FULL, tb);
  const unsigned win = __ballot_sync(FULL, v2 && tb == mtb);
  return win ? (__ffs(win) - 1) : -1;
}

template <int NV, int NC>
TSIDB_DEV int as_solve2(const DevConst& C, const ASCtx& S, const LaneConst& K, int lane, int mask, double c1c2, double trH,
                        double R_norm, int& iters_out, uint64_t* act_words, double& lam_out, int& lam_row_out) {
  typedef AL<NV, NC> LA;
  constexpr int nv = NV, na = NV - 6, n = LA::n, m = LA::m, ldj = LA::ldj;
  double* J2 = S.J2;
  double* x = S.x;
  double* wr = S.wr;
  double* Rp = S.Rp;
  double* np = S.np;
  double* dd = S.dd;   /* d with the entries of the active columns zeroed, zero padded to m + 2; doubles as the Householder vector */
  iters_out = 0;
  act_words[0] = act_words[1] = act_words[2] = 0;
  if (lane < 2) dd[m + lane] = 0.0;

  const int nin_ref = C.nin_ref_fixed + 34 * NC;
  const double psi_thresh = (double)nin_ref * TS_EPS * c1c2 * 100.0;
  /* reference row indices (tie-break keys) of the rows this lane owns */
  const int bit_f = 34 * (lane >> 4) + 17 + (lane & 15);
  const int bit_n = 34 * ((lane & 3) >> 1) + ((lane & 1) ? 33 : 16); /* lanes 12..15: (lane - 12) = lane & 3 */
  const int bit_a = 68 + lane;                 /* lower side; upper side + na */
  const int bit_j = 68 + 2 * na + 6 + lane;    /* lower side; upper side + nv */
  const bool has0 = lane < n, has1 = lane + 32 < n;
  /* state in registers: this lane's rows of x, position `lane` of the working set */
  double xr0 = has0 ? x[lane] : 0.0, xr1 = has1 ? x[lane + 32] : 0.0;
  double xo0 = xr0, xo1 = xr1;
  double ur = 0.0, uo = 0.0, irl = 0.0;
  int Ar = 0, Ao = 0;
  int iq = 0, iter = 0, status = ST_OPTIMAL;
  unsigned actbits = 0;  /* bit k: the row of slot k owned by this lane is in the working set */
  unsigned exclbits = 0;

  for (;;) { /* l1 */
    iter++;
    if (iter >= C.max_iter) { status = ST_MAX_ITER; break; }
    const double nf = wrench_of(nv, K, x, mask, wr, lane);
    __syncwarp();
    /* s = CI x + ci0 for the rows this lane owns, one candidate per two-sided pair */
    double c0 = TS_INF, c1 = TS_INF, c2 = TS_INF, c3 = TS_INF;
    int side2 = 0, side3 = 0;
    {
      const int f = lane >> 4, c = (lane & 15) >> 2;
      if ((mask >> f) & 1) {
        const double* ff = x + fvar0(nv, mask, f) + 3 * c;
        c0 = -(K.fric[0] * ff[0] + K.fric[1] * ff[1] + K.fric[2] * ff[2]);
      }
    }
    if (lane >= NRM_LANE0 && lane < NRM_LANE0 + 4) {
      const int f = (lane - NRM_LANE0) >> 1, side = lane & 1;
      if ((mask >> f) & 1) c1 = side ? (C.fmax - nf) : (nf - C.fmin);
    }
    if (lane < na) {
      if (C.use_tb) {
        const double2* Mr = reinterpret_cast<const double2*>(S.Ma + lane * SA_LDM);
        const double2* x2 = reinterpret_cast<const double2*>(x);
        double t0 = S.nle_a[lane], t1 = 0.0, t2 = 0.0, t3 = 0.0;
#pragma unroll
        for (int j = 0; j + 1 < nv / 2; j += 2) {
          const double2 m0 = Mr[j], m1 = Mr[j + 1], x0 = x2[j], x1 = x2[j + 1];
          t0 += m0.x * x0.x; t1 += m0.y * x0.y; t2 += m1.x * x1.x; t3 += m1.y * x1.y;
        }
        if ((nv / 2) & 1) { const double2 m0 = Mr[nv / 2 - 1], x0 = x2[nv / 2 - 1]; t0 += m0.x * x0.x; t1 += m0.y * x0.y; }
        double u0 = 0.0, u1 = 0.0, u2 = 0.0;
        const double* wb = wr + S.wro;
#pragma unroll
        for (int q = 0; q < 6 * NC; q += 3) {
          u0 += S.JFa[q * SA_LDJA + lane] * wb[q];
          u1 += S.JFa[(q + 1) * SA_LDJA + lane] * wb[q + 1];
          u2 += S.JFa[(q + 2) * SA_LDJA + lane] * wb[q + 2];
        }
        const double t = ((t0 + t1) + (t2 + t3)) - ((u0 + u1) + u2);
        const double slo = t - K.tmin, sup = K.tmax - t;
        side2 = sup < slo;
        c2 = side2 ? sup : slo;
      }
      if (C.use_jb) {
        const double xv = x[6 + lane];
        const double slo = xv - K.lb, sup = K.ub - xv;
        side3 = sup < slo;
        c3 = side3 ? sup : slo;
      }
    }
    /* violation sum: the other side of a pair is positive and adds nothing */
    double part = (c0 < 0.0) ? c0 : 0.0;
    part += (c1 < 0.0) ? c1 : 0.0;
    part += (c2 < 0.0) ? c2 : 0.0;
    part += (c3 < 0.0) ? c3 : 0.0;
    exclbits = 0;
    double best;
    int bslot, bbit;
    auto pick = [&]() {
      best = 0.0; bslot = -1; bbit = 1 << 30;
      const unsigned blocked = actbits | exclbits;
      auto consider = [&](double val, int slot, int bit) {
        if (val < 0.0 && !((blocked >> slot) & 1u) && (val < best || (val == best && bit < bbit))) { best = val; bslot = slot; bbit = bit; }
      };
      consider(c0, 0, bit_f);
      consider(c1, 1, bit_n);
      consider(c2, 2 + side2, bit_a + side2 * na);
      consider(c3, 4 + side3, bit_j + side3 * nv);
    };
    pick();
    int src = warp_argmin_fast(best, bslot >= 0, bbit);
    const double psi = warp_sum(part);
    if (fabs(psi) <= psi_thresh) { status = ST_OPTIMAL; break; }
    /* save x, u, A: register moves */
    xo0 = xr0; xo1 = xr1; uo = ur; Ao = Ar;
    bool done = false, restart_l1 = false, first_pick = true;
    for (;;) { /* l2 */
      if (!first_pick) {
        pick();
        src = warp_argmin_fast(best, bslot >= 0, bbit);
      }
      first_pick = false;
      if (src < 0) { status = ST_OPTIMAL; done = true; break; }
      const int ip_slot = __shfl_sync(FULL, bslot, src); /* the owner of the picked row is the lane that proposed it */
      const int ip = cid_of(na, src, ip_slot);
      double s_ip = shfl(best, src);
      const bool dense_row = (ip_slot == 2 || ip_slot == 3);
#ifdef TSIDB_EMU_TRACE
      if (lane == 0) printf("[emu] iter %d pick bit %d s=%.17g iq=%d\n", iter, cid_bit(na, nv, ip), s_ip, iq);
#endif
      if (dense_row) { actuation_normal(C, S, ip, mask, n, np, lane); __syncwarp(); }
      double up = 0.0; /* multiplier of the pending constraint (the reference's u[iq]) */
      for (;;) { /* l2a */
        /* d = J2^T n_ip (lane <-> column) */
        double dl = 0.0;
        if (lane < m) dl = row_dot_col(C, S, ip, mask, n, lane, np);
        if (lane < m) dd[lane] = (lane >= iq) ? dl : 0.0;
        __syncwarp();
        /* z = J2[:, iq:] d[iq:] (lanes over rows, 16-byte reads of the row and of d); zero if no free direction is left */
        double z0 = 0.0, z1 = 0.0;
        const double2* Jr0 = reinterpret_cast<const double2*>(J2 + (has0 ? lane : 0) * ldj);
        const double2* Jr1 = reinterpret_cast<const double2*>(J2 + (has1 ? lane + 32 : 0) * ldj);
        if (iq < m) {
          /* column pairs in static segments of four (every offset an immediate, the loads of a segment issue ahead of
           * its FMAs); a segment that lies entirely below iq is skipped, the pairs of the first live segment that lie
           * below iq multiply by the zeros of dd */
          const int cb = iq >> 1;
          constexpr int ce = (m + 1) >> 1;
          const double2* d2 = reinterpret_cast<const double2*>(dd);
          double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0, a2 = 0.0, a3 = 0.0, b2 = 0.0, b3 = 0.0;
#define TSIDB_ZPAIR(c)                                                                       \
  if ((c) < ce) {                                                                            \
    const double2 j0 = Jr0[c], j1 = Jr1[c], dv = d2[c];                                      \
    if ((c) & 1) { a2 += j0.x * dv.x; a3 += j0.y * dv.y; b2 += j1.x * dv.x; b3 += j1.y * dv.y; } \
    else { a0 += j0.x * dv.x; a1 += j0.y * dv.y; b0 += j1.x * dv.x; b1 += j1.y * dv.y; }     \
  }
#define TSIDB_ZSEG(s) if (cb < 4 * (s) + 4 && 4 * (s) < ce) { TSIDB_ZPAIR(4 * (s)) TSIDB_ZPAIR(4 * (s) + 1) TSIDB_ZPAIR(4 * (s) + 2) TSIDB_ZPAIR(4 * (s) + 3) }
          TSIDB_ZSEG(0) TSIDB_ZSEG(1) TSIDB_ZSEG(2) TSIDB_ZSEG(3)
#undef TSIDB_ZSEG
#undef TSIDB_ZPAIR
          static_assert(ce <= 16, "four segments of four column pairs");
          z0 = has0 ? (a0 + a1) + (a2 + a3) : 0.0;
          z1 = has1 ? (b0 + b1) + (b2 + b3) : 0.0;
        }
        /* r = R^-1 d[0:iq] (back substitution, lane <-> row; row l scaled by 1/R_ll, so a step of the chain is one
         * shuffle and one FMA; the column pointer walks down the packed storage) */
        double rl;
        {
          double accv = dl * irl; /* irl is zero for the lanes >= iq */
          const double* col = Rp + (iq - 1) * iq / 2 + lane;
          for (int i = iq - 1; i > 0; i--) {
            const double ri = shfl(accv, i);
            if (lane < i) accv -= (col[0] * irl) * ri;
            col -= i;
          }
          rl = accv;
        }
        /* partial step t1 = min u_k / r_k over r_k > 0, first position on ties */
        double t1 = TS_INF;
        const bool t1_valid = lane < iq && rl > 0.0;
        if (t1_valid) t1 = ur / rl;
        const int lpos = (__ballot_sync(FULL, t1_valid) != 0u) ? warp_argmin_fast(t1, t1_valid, lane) : -1;
        t1 = (lpos >= 0) ? shfl(t1, lpos) : TS_INF;
        /* full step t2 = -s_ip / z.n_ip, with z.n_ip = |d[iq:]|^2 (z = J2 d2, d2 = J2^T n) */
        /* The reference tests |z|^2 > eps.  z = J2 d with J2^T H J2 = I, so |z|^2 >= |d[iq:]|^2 / lambda_max(H) >=
         * |d[iq:]|^2 / trace(H): when that bound clears eps by a wide margin the sum over z is not needed */
        const double d2sum = warp_sum((lane >= iq && lane < m) ? dl * dl : 0.0);
        bool z_nonzero = d2sum > 64.0 * TS_EPS * trH;
        if (!z_nonzero) z_nonzero = fabs(warp_sum(z0 * z0 + z1 * z1)) > TS_EPS;
        const double t2 = z_nonzero ? (-s_ip / d2sum) : TS_INF;
        const double t = fmin(t1, t2);
#ifdef TSIDB_EMU_TRACE
        if (lane == 0) printf("[emu]   t1=%.17g (pos %d) t2=%.17g znp=%.6g\n", t1, lpos, t2, d2sum);
#endif
        if (t >= TS_INF) { status = ST_INFEASIBLE; done = true; break; } /* eiquadprog UNBOUNDED -> HQP INFEASIBLE */
        /* step in dual space, and in primal space unless no direction is left */
        if (lane < iq) ur -= t * rl;
        up += t;
        if (t2 < TS_INF) {
          xr0 += t * z0;
          xr1 += t * z1;
          if (has0) x[lane] = xr0;
          if (has1) x[lane + 32] = xr1;
        }
        if (t2 < TS_INF && t == t2) {
          /* full step: add ip.  Householder on the free columns iq..m-1 maps d[iq:] to beta e_iq; the
           * row sums needed for the update are z and column iq (already known). */
          bool degenerate = true; /* iq >= m: no free direction, |d(iq)| = 0 */
          if (iq < m) {
            const double nrm = sqrt(d2sum);
            const double d0 = shfl(dl, iq);
            const double beta = (d0 >= 0.0) ? -nrm : nrm;
            degenerate = !(fabs(beta) > TS_EPS * R_norm);
            if (!degenerate) {
              /* H = I - tau v v^T with the unscaled vector u = (d0 - beta, d_c) and rho = 1 / (beta (d0 - beta)):
               *   J2[k][c] += rho (z_k - beta J2[k][iq]) u_c   (sum_c' J2[k][c'] d_c' = z_k)
               * u is dd with its head replaced: one store, no second vector */
              const double rho = 1.0 / (beta * (d0 - beta));
              if (lane == iq) dd[iq] = d0 - beta;
              const double w0 = has0 ? -rho * (z0 - beta * J2[lane * ldj + iq]) : 0.0;
              const double w1 = has1 ? -rho * (z1 - beta * J2[(lane + 32) * ldj + iq]) : 0.0;
              __syncwarp();
              {
                const int cb = iq >> 1;
                constexpr int ce = (m + 1) >> 1;
                const double2* v2 = reinterpret_cast<const double2*>(dd);
                double2* W0 = const_cast<double2*>(Jr0);
                double2* W1 = const_cast<double2*>(Jr1);
                /* static segments of four column pairs as in the z pass; all loads of a segment ahead of its stores
                 * (the rows alias the store targets, so the compiler cannot move them itself) */
#define TSIDB_HSEG(s)                                                                                          \
  if (cb < 4 * (s) + 4 && 4 * (s) < ce) {                                                                      \
    constexpr int c_ = 4 * (s);                                                                                \
    double2 vq[4], p0[4], p1[4];                                                                               \
    _Pragma("unroll") for (int k = 0; k < 4; k++) if (c_ + k < ce) { vq[k] = v2[c_ + k]; p0[k] = Jr0[c_ + k]; p1[k] = Jr1[c_ + k]; } \
    _Pragma("unroll") for (int k = 0; k < 4; k++) if (c_ + k < ce) {                                           \
      p0[k].x -= w0 * vq[k].x; p0[k].y -= w0 * vq[k].y; p1[k].x -= w1 * vq[k].x; p1[k].y -= w1 * vq[k].y;       \
    }                                                                                                          \
    _Pragma("unroll") for (int k = 0; k < 4; k++) if (c_ + k < ce) { if (has0) W0[c_ + k] = p0[k]; if (has1) W1[c_ + k] = p1[k]; } \
  }
                TSIDB_HSEG(0) TSIDB_HSEG(1) TSIDB_HSEG(2) TSIDB_HSEG(3)
#undef TSIDB_HSEG
              }
              /* new column of R: [d[0:iq]; beta]; position iq of the working set */
              if (lane < iq) Rp[iq * (iq + 1) / 2 + lane] = dl;
              if (lane == iq) { Rp[iq * (iq + 1) / 2 + iq] = beta; irl = rho * (d0 - beta); ur = up; Ar = ip; }
              R_norm = fmax(R_norm, fabs(beta));
              if (lane == src) actbits |= 1u << ip_slot;
              iq++;
              __syncwarp();
            }
          }
#ifdef TSIDB_EMU_TRACE
          if (lane == 0) printf("[emu]   add -> %s Rnorm=%.6g\n", degenerate ? "DEGENERATE" : "ok", R_norm);
#endif
          if (degenerate) {
            /* eiquadprog: exclude ip, restore the saved x, u, A for the first iq entries, retry l2 */
            if (lane == src) exclbits |= 1u << ip_slot;
            actbits = 0;
            if (lane < iq) { Ar = Ao; ur = uo; }
            xr0 = xo0; xr1 = xo1;
            if (has0) x[lane] = xr0;
            if (has1) x[lane + 32] = xr1;
            __syncwarp();
            for (int i = 0; i < iq; i++) {
              int ol, os;
              cid_owner(na, __shfl_sync(FULL, Ar, i), ol, os);
              if (lane == ol) actbits |= 1u << os;
            }
            break; /* back to l2 with the same s */
          }
          restart_l1 = true;
          break;
        }
        /* dual-only step or partial step: drop the blocking constraint at position lpos
         * [eiquadprog-fast delete_constraint]: shift A, u and the columns of R, restore R to upper triangular with
         * Givens rotations of rows (j, j+1) and apply them to columns j, j+1 of J2 */
        {
          int ol, os;
          cid_owner(na, __shfl_sync(FULL, Ar, lpos), ol, os);
          if (lane == ol) actbits &= ~(1u << os);
        }
        {
          const int qq = lpos;
          __syncwarp(); /* every lane has finished reading R of the current working set */
          /* a column keeps its length when it moves one slot to the left: column c + 1 (length c + 2) goes into slot c
           * (capacity c + 1); its last element sits on the sub-diagonal and is carried in `sub` until the rotation
           * that annihilates it */
          double sub = 0.0;
          for (int c = qq; c < iq - 1; c++) {
            const double v0 = (lane <= c + 1) ? Rp[(c + 1) * (c + 2) / 2 + lane] : 0.0;
            __syncwarp();
            if (lane <= c) Rp[c * (c + 1) / 2 + lane] = v0;
            const double sd = shfl(v0, c + 1);
            if (lane == c) sub = sd;
            __syncwarp();
          }
          {
            const int An = __shfl_down_sync(FULL, Ar, 1);
            const double un = __shfl_down_sync(FULL, ur, 1);
            if (lane >= qq && lane < iq - 1) { Ar = An; ur = un; }
            if (lane == iq - 1) { Ar = 0; ur = 0.0; }
          }
          iq--;
          for (int j = qq; j < iq; j++) {
            double cc = Rp[j * (j + 1) / 2 + j];
            double ss = shfl(sub, j);
            /* eiquadprog distance() */
            const double a1 = fabs(cc), b1 = fabs(ss);
            double h;
            if (a1 > b1) { const double tq = b1 / a1; h = a1 * sqrt(1.0 + tq * tq); }
            else if (b1 > a1) { const double tq = a1 / b1; h = b1 * sqrt(1.0 + tq * tq); }
            else h = a1 * sqrt(2.0);
            if (h == 0.0) continue;
            cc = cc / h; ss = ss / h;
            double dj = h;
            if (cc < 0.0) { dj = -h; cc = -cc; ss = -ss; }
            const double xny = ss / (1.0 + cc);
            __syncwarp();
            if (lane == j) Rp[j * (j + 1) / 2 + j] = dj;
            /* rows j, j+1 of columns k > j: lane k owns column k (both rows are regular stored entries) */
            if (lane > j && lane < iq) {
              const double q1 = Rp[lane * (lane + 1) / 2 + j];
              const double q2 = Rp[lane * (lane + 1) / 2 + j + 1];
              const double n1 = q1 * cc + q2 * ss;
              Rp[lane * (lane + 1) / 2 + j] = n1;
              Rp[lane * (lane + 1) / 2 + j + 1] = xny * (q1 + n1) - q2;
            }
            /* columns j, j+1 of J2: lanes over rows */
            if (has0) {
              const double q1 = J2[lane * ldj + j], q2 = J2[lane * ldj + j + 1];
              const double n1 = q1 * cc + q2 * ss;
              J2[lane * ldj + j] = n1;
              J2[lane * ldj + j + 1] = xny * (n1 + q1) - q2;
            }
            if (has1) {
              const double q1 = J2[(lane + 32) * ldj + j], q2 = J2[(lane + 32) * ldj + j + 1];
              const double n1 = q1 * cc + q2 * ss;
              J2[(lane + 32) * ldj + j] = n1;
              J2[(lane + 32) * ldj + j + 1] = xny * (n1 + q1) - q2;
            }
            __syncwarp();
          }
          irl = (lane < iq) ? 1.0 / Rp[lane * (lane + 1) / 2 + lane] : 0.0;
          __syncwarp();
        }
        if (t2 < TS_INF) {
          /* partial step: recompute s(ip) at the new x and try again */
          wrench_of(nv, K, x, mask, wr, lane);
          __syncwarp();
          s_ip = eval_one(C, S, K, ip, mask);
        }
      } /* l2a */
      if (done || restart_l1) break;
    } /* l2 */
    if (done) break;
  } /* l1 */
  iters_out = iter;
  lam_out = 0.0;
  lam_row_out = -1;
  if (status == ST_OPTIMAL || status == ST_MAX_ITER) {
    if (lane < iq) { lam_out = ur; lam_row_out = cid_bit(na, nv, Ar); } /* sol.lambda: position `lane` of the working set */
    uint64_t w0 = 0, w1 = 0, w2 = 0;
    for (int i = 0; i < iq; i++) {
      const int bit = cid_bit(na, nv, __shfl_sync(FULL, Ar, i));
      if (bit < 64) w0 |= 1ull << bit;
      else if (bit < 128) w1 |= 1ull << (bit - 64);
      else w2 |= 1ull << (bit - 128);
    }
    act_words[0] = w0; act_words[1] = w1; act_words[2] = w2;
  }
  return status;
}

/* ================================================================= kernel D: dynamics + assembly of one env */
/* This env's references -> shared memory, one element per lane and array, as asynchronous copies (cp.async: no
 * register, no wait): they are issued before K1 and waited for after it, so the tick never stalls on them.  An
 * array the caller did not pass (null) takes the handle's default reference. */
TSIDB_DEV void stage_one(double* dst, const double* src, const TickArgs& a, int env, int k, int nd, const double* dflt) {
  if (!src) { *dst = dflt[k]; return; } /* lane-indexed read of the constants: default path only */
#ifndef TSIDB_EMU
  const double* g = src + eidx(a, env, k, nd);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(g) : "memory");
#else
  *dst = src[eidx(a, env, k, nd)];
#endif
}
TSIDB_DEV void stage_refs(const DevConst& C, const double* mdl, double* sm, const TickArgs& a, int env, int lane, int na) {
  double* rf = sm + SM_oRef;
  if (lane < 24) {
    stage_one(rf + RF_FOOT + lane, a.r_foot[0], a, env, lane, 24, C.ref_foot[0]);
    stage_one(rf + RF_FOOT + 24 + lane, a.r_foot[1], a, env, lane, 24, C.ref_foot[1]);
  }
  if (lane < 12) {
    stage_one(rf + RF_CONTACT + lane, a.r_contact[0], a, env, lane, 12, C.ref_contact[0]);
    stage_one(rf + RF_CONTACT + 12 + lane, a.r_contact[1], a, env, lane, 12, C.ref_contact[1]);
  }
  if (lane < 9) stage_one(rf + RF_COM + lane, a.r_com, a, env, lane, 9, C.ref_com);
  if (lane < na) stage_one(rf + RF_POST + lane, a.r_posture, a, env, lane, na, mdl + MDL_oPOST + 46);
#ifndef TSIDB_EMU
  asm volatile("cp.async.commit_group;" ::: "memory");
#endif
}
/* ... and waited for; the five reference positions (CoM, the two foot tasks, the two contacts) are then taken relative
 * to the env's reference point c (ref_point of q[0:3] staged at SM_oQV), as K1's frames and CoM are: nothing rounds at
 * the size of the distance from the origin.  Lane k staged coordinate k of q and of each of the five (stage_refs, the q
 * staging of every caller), so it shifts them after its own wait, with no extra barrier. */
TSIDB_DEV void stage_refs_wait(double* sm, int lane) {
#ifndef TSIDB_EMU
  asm volatile("cp.async.wait_group 0;" ::: "memory");
#endif
  if (lane < 3) {
    const double c = ref_point(sm[SM_oQV + lane]);
    double* rf = sm + SM_oRef + lane;
    rf[RF_COM] -= c; rf[RF_FOOT] -= c; rf[RF_FOOT + 24] -= c; rf[RF_CONTACT] -= c; rf[RF_CONTACT + 12] -= c;
  }
  __syncwarp();
}

/* `prefetched`: q, v of this env already sit in the warp's next-env buffer (the previous call asked for them);
 * `env_next` >= 0: ask for that env's q, v now — the copies travel with this env's references (one cp.async group, waited
 * for after K1), so the next call finds them without waiting on HBM (17.9 % of the kernel's samples were long-scoreboard
 * stalls, a third of them on these two loads at the head of an env). */
/* LOCAL (single-launch small-batch kernel): a.ws / a.ws3 point at shared memory of the same CTA — the images are
 * written with ordinary stores and the next stage works on them in place */
template <int NV, bool LOCAL = false>
TSIDB_DEV void dynamics_env(const DevConst& C, const double* mdl, double* sm, const TickArgs& a, int env, int slot, int lane,
                            bool prefetched = false, int env_next = -1) {
  constexpr int nv = NV, na = NV - 6, nq = NV + 1;
  PHASE_SYNC_D();
#ifndef TSIDB_EMU
  if (!LOCAL) {
    if (lane == 0) bulk_store_wait_read(); /* the previous env's image stores are done with this warp's shared memory */
    __syncwarp();
  }
#endif
  /* stage q, v */
  if (prefetched) {
    sm[SM_oQV + lane] = sm[SM_oQVn + lane];
    sm[SM_oQV + 32 + lane] = sm[SM_oQVn + 32 + lane];
    __syncwarp();
  } else {
    if (lane < nq) sm[SM_oQV + lane] = ldin(a.q, a, env, lane, nq);
    if (lane < nv) sm[SM_oQV + 32 + lane] = a.v ? ldin(a.v, a, env, lane, nv) : 0.0;
  }
  if (!a.kin_only) {
    if (env_next >= 0) {
      if (lane < nq) stage_one(sm + SM_oQVn + lane, a.q, a, env_next, lane, nq, nullptr);
      if (lane < nv) { if (a.v) stage_one(sm + SM_oQVn + 32 + lane, a.v, a, env_next, lane, nv, nullptr); else sm[SM_oQVn + 32 + lane] = 0.0; }
    }
    stage_refs(C, mdl, sm, a, env, lane, na);
  }
  __syncwarp();
  k1_dynamics<NV>(C, mdl, sm, lane);
  const double* fr = sm + SM_oFr;
  /* world positions again: K1's CoM and soles are relative to the reference point c */
  const double cw = lane < 3 ? ref_point(sm[SM_oQV + lane]) : 0.0;
  if (a.o_com && lane < 9) a.o_com[eidx(a, env, lane, 9)] = fr[FR_COM + lane] + cw;
#pragma unroll
  for (int f = 0; f < 2; f++)
    if (a.o_foot[f] && lane < 12) {
      /* (p, R column-major) */
      double val = (lane < 3) ? fr[FR_OMF + f * 12 + lane] + cw : fr[FR_OMF + f * 12 + 3 + 3 * ((lane - 3) % 3) + (lane - 3) / 3];
      a.o_foot[f][eidx(a, env, lane, 12)] = val;
    }
  if (a.kin_only) return;

  const int mask = a.mask ? (a.mask[env] & 3) : 3;
  const int nc = (mask & 1) + ((mask >> 1) & 1);
  const int n = nv + 12 * nc, neq = 6 + 6 * nc;
  /* M shares its shared-memory region with the Hessian block that K2 is about to write: the rows of M that the
   * later stages need leave for their images now */
  /* offsets of the class's solver-image layout (compile-time per class; the class of the env is data) */
  const int oMa_c = (nc == 2) ? AL<NV, 2>::oMa : ((nc == 1) ? AL<NV, 1>::oMa : AL<NV, 0>::oMa);
  const int oJFa_c = (nc == 2) ? AL<NV, 2>::oJFa : ((nc == 1) ? AL<NV, 1>::oJFa : AL<NV, 0>::oJFa);
  const int oNle_c = (nc == 2) ? AL<NV, 2>::oNle : ((nc == 1) ? AL<NV, 1>::oNle : AL<NV, 0>::oNle);
  const int oVj_c = (nc == 2) ? AL<NV, 2>::oVj : ((nc == 1) ? AL<NV, 1>::oVj : AL<NV, 0>::oVj);
  double* img = a.ws + (size_t)slot * SA_IMAGE;
  double* eimg = a.ws3 + (size_t)slot * SE_IMAGE;
  /* M_a row by row (lanes over the columns): no index arithmetic per element */
  if (lane < SA_LDM) {
    double* dst = img + oMa_c + lane;
    const double* srcm = sm + SM_oM + 6 * SM_LDM + lane;
#pragma unroll
    for (int r = 0; r < na; r++) dst[r * SA_LDM] = (lane < nv) ? srcm[r * SM_LDM] : 0.0;
  }
  for (int k = lane; k < 162; k += 32) eimg[SE_oMu + k] = sm[SM_oM + k];
  __syncwarp();
  PHASE_SYNC_D();
  stage_refs_wait(sm, lane);
  k2_assemble<NV>(C, mdl, sm, a, env, lane, mask, neq, n);
  /* solver image (layout a_layout(nv, nc)): the parts that do not depend on the elimination */
  /* rows of the feet in contact, in force-block order (block 0 = LF if it is in contact, else RF), row by row */
  if (lane < SA_LDJA) {
    const int f0 = (mask & 1) ? 0 : 1;
#pragma unroll
    for (int q = 0; q < 12; q++) {
      if (q < 6 * nc) {
        const int f = (q < 6) ? f0 : 1;
        img[oJFa_c + q * SA_LDJA + lane] = (lane < na) ? sm[SM_oJF + (f * 6 + q % 6) * TSIDB_NVX + 6 + lane] : 0.0;
      }
    }
  }
  if (lane < na) { img[oNle_c + lane] = sm[SM_oNle + 6 + lane]; img[oVj_c + lane] = sm[SM_oQV + 32 + 6 + lane]; }
  /* assembly image (layout SE_*) for the elimination kernel */
#ifndef TSIDB_EMU
  /* the two contiguous pieces (H | g, JF) leave as bulk asynchronous stores (TMA); the next env
   * of this warp waits for them to have read shared memory before it overwrites it */
  __syncwarp();
  if (LOCAL) {
    static_assert((SE_oH % 2) == 0 && (SM_oH % 2) == 0 && (SE_oJF % 2) == 0 && (SM_oJF % 2) == 0 && (TSIDB_NX % 2) == 0, "16-byte copies");
    const double2* s0 = reinterpret_cast<const double2*>(sm + SM_oH);
    double2* d0 = reinterpret_cast<double2*>(eimg + SE_oH);
    for (int k = lane; k < (702 + TSIDB_NX) / 2; k += 32) d0[k] = s0[k];
    const double2* s1 = reinterpret_cast<const double2*>(sm + SM_oJF);
    double2* d1 = reinterpret_cast<double2*>(eimg + SE_oJF);
    for (int k = lane; k < 312 / 2; k += 32) d1[k] = s1[k];
  } else if (lane == 0) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    bulk_store(eimg + SE_oH, sm + SM_oH, (702 + TSIDB_NX) * sizeof(double)); /* SM_oGv follows SM_oH, SE_oG follows SE_oH */
    bulk_store(eimg + SE_oJF, sm + SM_oJF, 312 * sizeof(double));
    bulk_store_commit();
  }
#else
  for (int k = lane; k < 702; k += 32) eimg[SE_oH + k] = sm[SM_oH + k];
  for (int k = lane; k < TSIDB_NX; k += 32) eimg[SE_oG + k] = sm[SM_oGv + k];
  for (int k = lane; k < 312; k += 32) eimg[SE_oJF + k] = sm[SM_oJF + k];
#endif
  if (lane < 8) eimg[SE_oNle + lane] = (lane < 6) ? sm[SM_oNle + lane] : 0.0;
  if (lane < 12) eimg[SE_oBm + lane] = sm[SM_oBv + BV_MOT + lane];
  if (lane < 2) eimg[SE_oSc + lane] = (lane == 0) ? (double)mask : 0.0;
  __syncwarp();
}

/* ================================================================= kernel E: equality elimination of one env */
template <int NV, int NC>
TSIDB_DEV void j2_from_factor(const DevConst& C, const double* L, const double* ild, const double* tauq, const double* Vt,
                              double* img, int lane);
template <int NV, int NC, bool LOCAL = false>
TSIDB_DEV void eliminate_env(const DevConst& C, const double* lfinv_sm, double* sm, const TickArgs& a, int slot, int lane, unsigned& parity) {
  typedef EL<NV, NC> LE;
  __syncwarp(); /* every lane is done with the previous env's shared memory */
#ifndef TSIDB_EMU
  if (!LOCAL) { /* LOCAL: sm IS the assembly image the dynamics stage left */
    if (lane == 0) bulk_load(sm, a.ws3 + (size_t)slot * SE_IMAGE, SE_IMAGE * sizeof(double), sm + LE::oBar);
    mbar_wait(sm + LE::oBar, parity);
    parity ^= 1u;
  }
#else
  for (int k = lane; k < SE_IMAGE; k += 32) sm[k] = a.ws3[(size_t)slot * SE_IMAGE + k];
#endif
  __syncwarp();
  const int mask = (int)sm[SE_oSc]; /* its contact count is NC: the slots are class-sorted */
  constexpr int n = NV + 12 * NC;
  double c1c2 = 0.0, c1 = 0.0, R_norm = 1.0;
  const int err = k3_eliminate<NV, NC>(C, lfinv_sm, sm, lane, mask, c1c2, c1, R_norm);
  typedef AL<NV, NC> LA;
  double* img = a.ws + (size_t)slot * SA_IMAGE;
  for (int k = lane; k < even_up(n); k += 32) img[LA::oX + k] = (k < n) ? sm[LE::oX + k] : 0.0;
  /* scalars of the solver image: c1 c2, R_norm, (status, contact mask) packed, trace(H) */
  if (lane == 0) { img[SA_oSc] = c1c2; img[SA_oSc + 1] = R_norm; img[SA_oSc + 2] = (double)(4 * err + mask); img[SA_oSc + 3] = c1; }
  /* the null-space basis goes straight from the factor in shared memory to the solver image */
  __syncwarp();
  if (err == ST_OPTIMAL) j2_from_factor<NV, NC>(C, sm + SE_oH, sm + LE::oILD, sm + LE::oTAU, sm + LE::oVT, img, lane);
  __syncwarp();
}

/* ================================================================= null-space basis of one env (tail of kernel E) */
/* J2[:, c] = L^-T Q [0; e_c], one lane per column c < m = n - neq, the column in registers, every index a
 * compile-time constant.  The reflectors are applied in reverse: the base-dynamics ones (rows i..n-1) first,
 * after which the force rows are final and leave through the constant Lf^-T; then the contact-motion ones
 * (rows i..nv-1) and the back substitution with L on the dv rows.  Operands shared by the warp (reflector and
 * factor entries) are broadcast reads of the elimination's own shared memory: the factor never travels through
 * HBM (round 1 ran this as a kernel of its own behind a 13 KB factor image per env; that image and its round
 * trip — 1.8 GB per 65536-env tick, 94 % of the HBM rate inside the single-support launch — are gone). */
template <int NV, int NC>
TSIDB_DEV void j2_from_factor(const DevConst& C, const double* L, const double* ild, const double* tauq, const double* Vt,
                              double* img, int lane) {
  constexpr int N = NV + 12 * NC, NEQ = 6 + 6 * NC, NCM = 6 * NC, M = N - NEQ;
  constexpr int NS = N; /* reflector row stride in the elimination's shared memory (EL::oVT) */
  typedef AL<NV, NC> LA;
  if (lane >= M) return;
  /* column c starts as the unit vector of the c-th row that is not a reflector head: dv rows NCM..NV-1, then
   * the force rows NV+6.. (without contacts: rows 6..NV-1) */
  double q[N];
#pragma unroll
  for (int k = 0; k < N; k++) {
    const int col = (NC == 0) ? k - 6 : ((k < NV) ? k - NCM : ((k >= NV + 6) ? (NV - NCM) + (k - NV - 6) : -1));
    q[k] = (col >= 0 && col == lane) ? 1.0 : 0.0;
  }
#pragma unroll
  for (int i = NEQ - 1; i >= 0; i--) {
    const bool top = (i < NCM) || NC == 0;
    const int head = top ? i : NV + (i - NCM);
    const int lo = top ? i + 1 : NCM;            /* dv rows lo..NV-1 */
    const int flo = top ? N : head + 1;          /* force rows flo..N-1 */
    const double2* v2 = reinterpret_cast<const double2*>(Vt + i * NS);
    /* the head row is still zero here (no reflector applied so far touches it); the reflectors are unscaled
     * (H = I - kappa u u^T, u_head = alpha - beta); entries come in pairs (16-byte broadcast reads) */
    double w0 = 0.0, w1 = 0.0, w2 = 0.0, w3 = 0.0;
#pragma unroll
    for (int kk = (lo & ~1); kk < NV; kk += 2) {
      const double2 p = v2[kk >> 1];
      if (kk >= lo) { if (kk & 2) w2 += p.x * q[kk]; else w0 += p.x * q[kk]; }
      if (kk & 2) w3 += p.y * q[kk + 1]; else w1 += p.y * q[kk + 1];
    }
#pragma unroll
    for (int kk = (flo & ~1); kk < N; kk += 2) {
      const double2 p = v2[kk >> 1];
      if (kk >= flo) { if (kk & 2) w2 += p.x * q[kk]; else w0 += p.x * q[kk]; }
      if (kk & 2) w3 += p.y * q[kk + 1]; else w1 += p.y * q[kk + 1];
    }
    const double w = tauq[i] * ((w0 + w1) + (w2 + w3));
    q[head] = -w * Vt[i * NS + head];
#pragma unroll
    for (int kk = (lo & ~1); kk < NV; kk += 2) {
      const double2 p = v2[kk >> 1];
      if (kk >= lo) q[kk] -= w * p.x;
      q[kk + 1] -= w * p.y;
    }
#pragma unroll
    for (int kk = (flo & ~1); kk < N; kk += 2) {
      const double2 p = v2[kk >> 1];
      if (kk >= flo) q[kk] -= w * p.x;
      q[kk + 1] -= w * p.y;
    }
    if (i == NCM) {
      /* force rows are final: J2_f = Lf^-T q_f, stored right away */
#pragma unroll
      for (int s = 0; s < NC; s++) {
#pragma unroll
        for (int r = 0; r < 12; r++) {
          double acc = 0.0;
#pragma unroll
          for (int k = r; k < 12; k++) acc += C.Lfinv[k][r] * q[NV + 12 * s + k];
          img[LA::oJ2 + (NV + 12 * s + r) * LA::ldj + lane] = acc;
        }
      }
    }
  }
  /* dv rows: q <- L^-T q (column-oriented back substitution; row k of L is a broadcast read) */
#pragma unroll
  for (int k = NV - 1; k >= 0; k--) {
    q[k] *= ild[k];
    /* row k of L as 16-byte broadcast reads wherever the (odd) row stride leaves a pair aligned */
    const int i0 = (k * SM_LDM) & 1;
    if (i0 && k > 0) q[0] -= L[k * SM_LDM] * q[k];
#pragma unroll
    for (int ii = i0; ii < k; ii += 2) {
      if (ii + 1 < k) {
        const double2 p = *reinterpret_cast<const double2*>(L + k * SM_LDM + ii);
        q[ii] -= p.x * q[k];
        q[ii + 1] -= p.y * q[k];
      } else {
        q[ii] -= L[k * SM_LDM + ii] * q[k];
      }
    }
  }
#pragma unroll
  for (int k = 0; k < NV; k++) img[LA::oJ2 + k * LA::ldj + lane] = q[k];
}

/* ================================================================= kernel A: active set + decode of one env */
template <int NV, int NC, bool LOCAL = false>
TSIDB_DEV void activeset_env(const DevConst& C, LaneConst& K, double* sm, const TickArgs& a, int env, int slot, int lane, unsigned& parity) {
  typedef AL<NV, NC> LA;
  constexpr int nv = NV, na = NV - 6;
  __syncwarp(); /* every lane is done with the previous env's shared memory */
#ifndef TSIDB_EMU
  if (!LOCAL) { /* LOCAL: sm IS the solver image the two earlier stages filled */
    /* the 21 KB solver image arrives as ONE bulk asynchronous copy (TMA); the warp waits on its mbarrier */
    if (lane == 0) bulk_load(sm, a.ws + (size_t)slot * SA_IMAGE, LA::image * sizeof(double), sm + LA::oBar);
    mbar_wait(sm + LA::oBar, parity);
    parity ^= 1u;
  }
#else
  for (int k = lane; k < LA::image; k += 32) sm[k] = a.ws[(size_t)slot * SA_IMAGE + k];
#endif
  __syncwarp();
  ASCtx S;
  S.na = na; S.nv = nv; S.ldj = LA::ldj; S.nfr = 6 * NC;
  S.J2 = sm + LA::oJ2; S.Ma = sm + LA::oMa; S.JFa = sm + LA::oJFa; S.nle_a = sm + LA::oNle; S.vj = sm + LA::oVj;
  S.x = sm + LA::oX; S.wr = sm + LA::oWr;
  S.Rp = sm + LA::oR; S.np = sm + LA::oNP; S.dd = sm + LA::oD;
  const double c1c2 = sm[SA_oSc], R_norm = sm[SA_oSc + 1], c1 = sm[SA_oSc + 3];
  const int em = (int)sm[SA_oSc + 2], err = em >> 2, mask = em & 3; /* its contact count is NC (class-sorted slots) */
  S.wro = (NC == 1 && !(mask & 1)) ? 6 : 0;
  K.lb = K.ub = 0.0;
  if (lane < na && C.use_jb) {
    /* [tsid TaskJointBounds] (v_min - v)/dt <= dv <= (v_max - v)/dt, clipped to +-1e10 */
    const double vj = S.vj[lane];
    K.ub = fmin((K.vmax - vj) / C.jb_dt, 1e10);
    K.lb = fmax((K.vmin - vj) / C.jb_dt, -1e10);
  }
  __syncwarp(); /* the joint velocities are dead from here on: the work arrays take their place */
  int iters = 0;
  uint64_t words[3] = {0, 0, 0};
  int status = err;
  double lam = 0.0;
  int lam_row = -1;
  if (err == ST_OPTIMAL) status = as_solve2<NV, NC>(C, S, K, lane, mask, c1c2, c1, R_norm, iters, words, lam, lam_row);
  const bool ok = (status == ST_OPTIMAL || status == ST_MAX_ITER);
  const double* x = S.x;
  double* wr = S.wr;
  if (ok) wrench_of(nv, K, x, mask, wr, lane);
  __syncwarp();
  /* decode: dv = x[:nv], f = x[nv:], tau = h_a + M_a dv - J_a^T f  (ref:main.py:126-127) */
  if (lane < nv) a.ddq[eidx(a, env, lane, nv)] = ok ? x[lane] : 0.0;
  if (lane < 24) {
    const int f = lane / 12;
    double val = 0.0;
    if (ok && ((mask >> f) & 1)) val = x[fvar0(nv, mask, f) + lane % 12];
    a.f[eidx(a, env, lane, 24)] = val;
  }
  if (lane < na) {
    double val = 0.0;
    if (ok) {
      const double* Mr = S.Ma + lane * SA_LDM;
      double s0 = S.nle_a[lane], s1 = 0.0;
      for (int j = 0; j < nv; j += 2) { s0 += Mr[j] * x[j]; s1 += (j + 1 < nv) ? Mr[j + 1] * x[j + 1] : 0.0; }
      double s = s0 + s1;
#pragma unroll
      for (int q = 0; q < 6 * NC; q++) s -= S.JFa[q * SA_LDJA + lane] * wr[S.wro + q];
      val = s;
    }
    a.tau[eidx(a, env, lane, na)] = val;
  }
  if (a.o_wrench && lane < 12) a.o_wrench[eidx(a, env, lane, 12)] = ok ? wr[lane] : 0.0;
  if (a.o_lambda) a.o_lambda[(size_t)env * 32 + lane] = lam;
  if (a.o_lambda_row) a.o_lambda_row[(size_t)env * 32 + lane] = lam_row;
  if (lane == 0) {
    a.status[env] = status;
    a.iters[env] = iters;
    if (a.pred) a.pred[env] = iters; /* next tick's longest-first order (tsidb_classify_kernel) */
    if (a.active) {
      a.active[env] = words[0];
      a.active[(size_t)a.n_envs + env] = words[1];
      a.active[2 * (size_t)a.n_envs + env] = words[2];
    }
  }
  __syncwarp();
}

/* ================================================================= QP export of one env (tsidb_problem_data) */
/* The problem SolverHQuadProgFast hands to eiquadprog for this env, in the compact variables x = [dv; f of the feet in
 * contact, LF first], written row-major and zero padded to the handle's maxima (include/tsidb.h).  Everything comes from
 * the images the dynamics kernel left for this env (slot == env) and from the handle's constants; nothing is solved.
 * Lanes run over the column pairs of a row and every row leaves as one 16-byte store per lane. */
template <int NV>
struct PB {
  enum : int {
    oE = 0,                                  /* assembly image                          SE_IMAGE */
    oMa = SE_IMAGE,                          /* M_a (rows 6.. of M)                  na x SA_LDM */
    oNle = oMa + (NV - 6) * SA_LDM,          /* nle_a                                          na */
    oVj = oNle + even_up(NV - 6),            /* joint velocities                               na */
    oJc = oVj + even_up(NV - 6),             /* Jc = T^T JF of the feet in contact, transposed: [j][12 s + k], nv x 24 */
    per_env = oJc + NV * 24
  };
};
TSIDB_DEV void st_pair(double* p, double x, double y) { *reinterpret_cast<double2*>(p) = make_double2(x, y); }

/* CI row ri of an env -> (block 0 force / 2 actuation / 3 joint bounds / -1 padding, side, row i, force slot) */
TSIDB_DEV int ci_block(const DevConst& C, int ri, int nc, int na, int nv, int& side, int& i, int& slot) {
  int r = ri;
  for (int s = 0; s < nc; s++) {
    if (r < 34) { slot = s; side = r >= 17; i = r - 17 * side; return 0; }
    r -= 34;
  }
  if (C.use_tb) {
    if (r < 2 * na) { side = r >= na; i = r - na * side; return 2; }
    r -= 2 * na;
  }
  if (C.use_jb && r < 2 * nv) { side = r >= nv; i = r - nv * side; return 3; }
  return -1;
}

template <int NV>
TSIDB_DEV void problem_env(const DevConst& C, const double* pt, double* sm, const TickArgs& a, const ProblemOut& o, int env,
                           int lane) {
  typedef PB<NV> P;
  constexpr int nv = NV, na = NV - 6, NX = NV + 24, NEQX = 18;
  const double BIG = 1e10; /* [UPSTREAM TaskJointBounds] unbounded base rows; Contact6d's open pyramid side */
  const int nin_x = 2 * (34 + (C.use_tb ? na : 0) + (C.use_jb ? nv : 0));
  __syncwarp(); /* every lane is done with the previous env's shared memory */
  {
    const double2* s = reinterpret_cast<const double2*>(a.ws3 + (size_t)env * SE_IMAGE);
    double2* d = reinterpret_cast<double2*>(sm + P::oE);
    for (int k = lane; k < SE_IMAGE / 2; k += 32) d[k] = s[k];
  }
  const int mask = a.mask ? (a.mask[env] & 3) : 3;
  const int nc = (mask & 1) + ((mask >> 1) & 1);
  const int n = nv + 12 * nc, neq = 6 + 6 * nc;
  const int nin = 2 * (17 * nc + (C.use_tb ? na : 0) + (C.use_jb ? nv : 0));
  const int f0 = (mask & 1) ? 0 : 1; /* foot of force slot 0; slot 1 is RF */
  {
    const ALayout L = a_layout(nv, nc);
    const double* img = a.ws + (size_t)env * SA_IMAGE;
    const double2* s = reinterpret_cast<const double2*>(img + L.oMa);
    double2* d = reinterpret_cast<double2*>(sm + P::oMa);
    for (int k = lane; k < na * SA_LDM / 2; k += 32) d[k] = s[k];
    if (lane < na) { sm[P::oNle + lane] = img[L.oNle + lane]; sm[P::oVj + lane] = img[L.oVj + lane]; }
  }
  __syncwarp();
  const double* E = sm + P::oE;
  const double* Ma = sm + P::oMa;
  double* Jc = sm + P::oJc;
  if (lane < nv) {
    for (int s = 0; s < nc; s++) {
      const int f = s == 0 ? f0 : 1;
      double jf[6];
#pragma unroll
      for (int m = 0; m < 6; m++) jf[m] = E[SE_oJF + (f * 6 + m) * TSIDB_NVX + lane];
#pragma unroll
      for (int k = 0; k < 12; k++) {
        double acc = 0.0;
#pragma unroll
        for (int m = 0; m < 6; m++) acc += pt[PT_oT + m * 12 + k] * jf[m];
        Jc[lane * 24 + 12 * s + k] = acc;
      }
    }
  }
  __syncwarp();
  const bool cols = lane < NX / 2; /* this lane's columns 2 lane, 2 lane + 1 */
  if (o.H && cols) {
    double* out = o.H + (size_t)env * NX * NX + 2 * lane;
    for (int i = 0; i < NX; i++) {
      double x[2];
#pragma unroll
      for (int u = 0; u < 2; u++) {
        const int j = 2 * lane + u;
        double val = 0.0;
        if (i < n && j < n) {
          if (i < nv && j < nv) val = E[SE_oH + (i >= j ? i * SM_LDM + j : j * SM_LDM + i)]; /* lower triangle */
          else if (i >= nv && j >= nv && (i - nv) / 12 == (j - nv) / 12) val = pt[PT_oHF + ((i - nv) % 12) * 12 + (j - nv) % 12];
        }
        x[u] = val;
      }
      st_pair(out + i * NX, x[0], x[1]);
    }
  }
  if (o.g)
    for (int k = lane; k < NX; k += 32) o.g[(size_t)env * NX + k] = k < nv ? E[SE_oG + k] : 0.0;
  if (o.CE && cols) {
    double* out = o.CE + (size_t)env * NEQX * NX + 2 * lane;
    for (int r = 0; r < NEQX; r++) {
      double x[2];
#pragma unroll
      for (int u = 0; u < 2; u++) {
        const int j = 2 * lane + u;
        double val = 0.0;
        if (r < 6) { /* base dynamics: [M_u | -Jc^T] x + h_u = 0 */
          if (j < nv) val = E[SE_oMu + r * SM_LDM + j];
          else if (j < n) val = -Jc[r * 24 + j - nv];
        } else if (r < neq && j < nv) { /* contact motion: JF x - a_des = 0 */
          const int f = (r < 12) ? f0 : 1;
          val = E[SE_oJF + (f * 6 + (r - 6) % 6) * TSIDB_NVX + j];
        }
        x[u] = val;
      }
      st_pair(out + r * NX, x[0], x[1]);
    }
  }
  if (o.ce0 && lane < NEQX) {
    double val = 0.0;
    if (lane < 6) val = E[SE_oNle + lane];
    else if (lane < neq) val = -E[SE_oBm + ((lane < 12) ? f0 : 1) * 6 + (lane - 6) % 6];
    o.ce0[(size_t)env * NEQX + lane] = val;
  }
  if (o.CI && cols) {
    double* out = o.CI + (size_t)env * nin_x * NX + 2 * lane;
    for (int ri = 0; ri < nin_x; ri++) {
      int side = 0, i = 0, slot = 0;
      const int blk = ci_block(C, ri, nc, na, nv, side, i, slot);
      double x[2];
#pragma unroll
      for (int u = 0; u < 2; u++) {
        const int j = 2 * lane + u;
        double val = 0.0;
        if (blk == 0) {
          const int k = j - nv - 12 * slot;
          if (k >= 0 && k < 12) val = pt[PT_oB + i * 12 + k];
        } else if (blk == 2) { /* [M_a | -Jc_a^T] x + h_a in [tau_min, tau_max] */
          if (j < nv) val = Ma[i * SA_LDM + j];
          else if (j < n) val = -Jc[(6 + i) * 24 + j - nv];
        } else if (blk == 3) {
          val = (j == i) ? 1.0 : 0.0;
        }
        x[u] = side ? -val : val; /* [lower rows: A x - lb >= 0; upper rows: -A x + ub >= 0] */
      }
      st_pair(out + ri * NX, x[0], x[1]);
    }
  }
  if (o.ci0) {
    for (int ri = lane; ri < nin_x; ri += 32) {
      int side = 0, i = 0, slot = 0;
      const int blk = ci_block(C, ri, nc, na, nv, side, i, slot);
      double lb = 0.0, ub = 0.0;
      if (blk == 0) {
        lb = (i < 16) ? -BIG : C.fmin;
        ub = (i < 16) ? 0.0 : C.fmax;
      } else if (blk == 2) {
        lb = pt[PT_oTMIN + i] - sm[P::oNle + i];
        ub = pt[PT_oTMAX + i] - sm[P::oNle + i];
      } else if (blk == 3) {
        lb = -BIG; ub = BIG;
        if (i >= 6) {
          const double vj = sm[P::oVj + i - 6];
          const double hi = (pt[PT_oVMAX + i - 6] - vj) / C.jb_dt, lo = (pt[PT_oVMIN + i - 6] - vj) / C.jb_dt;
          ub = hi < BIG ? hi : BIG;
          lb = lo > -BIG ? lo : -BIG;
        }
      }
      o.ci0[(size_t)env * nin_x + ri] = (blk < 0) ? 0.0 : (side ? ub : -lb);
    }
  }
  if (o.TA && cols) { /* getActuatorForces: tau = [M_a | -Jc_a^T] x + h_a */
    double* out = o.TA + (size_t)env * na * NX + 2 * lane;
    for (int r = 0; r < na; r++) {
      double x[2];
#pragma unroll
      for (int u = 0; u < 2; u++) {
        const int j = 2 * lane + u;
        x[u] = (j < nv) ? Ma[r * SA_LDM + j] : ((j < n) ? -Jc[(6 + r) * 24 + j - nv] : 0.0);
      }
      st_pair(out + r * NX, x[0], x[1]);
    }
  }
  if (o.ta0)
    for (int r = lane; r < na; r += 32) o.ta0[(size_t)env * na + r] = sm[P::oNle + r];
  if (o.sizes && lane < 3) o.sizes[(size_t)env * 3 + lane] = (lane == 0) ? n : ((lane == 1) ? neq : nin);
}

/* ================================================================= adjoint of the reference terms (tsidb_refs_grad) */
/* Reverse mode of log6_dev, branch for branch as log6_dev computes it: given (ol, oa) = dL/d(out lin, out ang), adds
 * dL/dR (9, row-major, R taken as 9 free entries: the formulas are differentiated as written, not on SO(3)) to Rb and
 * dL/dp to pb.  theta enters through the trace only, tr = R0 + R4 + R8:
 *   small angle (theta < prec3): w = (R - R^T)^vee / 2 has no theta term; alpha and beta are series in s = theta^2, whose
 *     derivative in the trace is -theta / sin(theta) = -(1 + s/6) to rounding; at the clamp tr >= 3 (theta = 0) that is the
 *     interior limit -1.  Nothing is differentiated through acos or the clamp, so theta = 0 gives a finite gradient.
 *   generic: dtheta/dtr = -1 / (2 sin theta); t = theta / (2 sin theta), alpha = theta sin / (2 (1 - cos)),
 *     beta = (1 - alpha) / theta^2, differentiated in closed form.
 *   near pi (theta >= pi - 1e-2): w_k = sign_k sqrt((R_kk + cphi) theta^2 / (1 + cphi)), cphi = -(tr - 1)/2; the signs are
 *     piecewise constant, and a component whose sqrt argument is <= 0 (w_k = 0) contributes zero.  At tr <= -1
 *     (theta = pi) dtheta/dtr is unbounded and the theta terms contribute zero. */
TSIDB_DEV void log6_adj(const double* R, const double* p, const double* ol, const double* oa, double* Rb, double* pb) {
  const double PI = 3.14159265358979323846;
  const double prec3 = 1.220703125e-4;
  const double tr = R[0] + R[4] + R[8];
  double th;
  if (tr >= 3.0) th = 0.0;
  else if (tr <= -1.0) th = PI;
  else th = acos((tr - 1.0) / 2.0);
  const double ct = (tr >= 3.0) ? 1.0 : ((tr <= -1.0) ? -1.0 : (tr - 1.0) / 2.0);
  const double st = sqrt(fmax((1.0 - ct) * (1.0 + ct), 0.0));
  const double dth = st > 0.0 ? -0.5 / st : 0.0; /* dtheta/dtr */
  const bool near_pi = th >= PI - 1e-2;
  double w[3], v[3] = {R[7] - R[5], R[2] - R[6], R[3] - R[1]}, tk[3] = {0, 0, 0}, bpi = 0.0, cphi = 0.0, t = 0.5;
  if (near_pi) {
    cphi = -(tr - 1.0) / 2.0;
    bpi = th * th / (1.0 + cphi);
    tk[0] = (R[0] + cphi) * bpi; tk[1] = (R[4] + cphi) * bpi; tk[2] = (R[8] + cphi) * bpi;
    w[0] = (R[7] > R[5] ? 1.0 : -1.0) * (tk[0] > 0 ? sqrt(tk[0]) : 0.0);
    w[1] = (R[2] > R[6] ? 1.0 : -1.0) * (tk[1] > 0 ? sqrt(tk[1]) : 0.0);
    w[2] = (R[3] > R[1] ? 1.0 : -1.0) * (tk[2] > 0 ? sqrt(tk[2]) : 0.0);
  } else {
    t = ((th > prec3) ? th / st : 1.0) / 2.0;
    w[0] = t * v[0]; w[1] = t * v[1]; w[2] = t * v[2];
  }
  const double s = th * th;
  double alpha, beta;
  if (th < prec3) {
    alpha = 1.0 - s / 12.0 - s * s / 720.0;
    beta = 1.0 / 12.0 + s / 720.0;
  } else {
    alpha = th * st / (2.0 * (1.0 - ct));
    beta = 1.0 / s - st / (2.0 * th * (1.0 - ct));
  }
  /* out_lin = alpha p - w x p / 2 + beta (w.p) w, out_ang = w */
  const double wdp = dot3(w, p), wdo = dot3(w, ol);
  double lxw[3], pxl[3], wb[3];
  cross3(ol, w, lxw);
  cross3(p, ol, pxl);
#pragma unroll
  for (int k = 0; k < 3; k++) {
    pb[k] += alpha * ol[k] - 0.5 * lxw[k] + (beta * wdo) * w[k];
    wb[k] = oa[k] - 0.5 * pxl[k] + beta * (wdo * p[k] + wdp * ol[k]);
  }
  const double ab = dot3(ol, p), bb = wdp * wdo; /* dL/dalpha, dL/dbeta */
  double trb;
  if (th < prec3) {
    const double ds = (tr >= 3.0) ? -1.0 : -(1.0 + s / 6.0); /* ds/dtr */
    trb = (ab * (-1.0 / 12.0 - s / 360.0) + bb / 720.0) * ds;
  } else {
    const double da = (st - th) / (2.0 * (1.0 - ct)); /* dalpha/dtheta */
    const double db = -(da + 2.0 * th * beta) / s;     /* dbeta/dtheta */
    trb = (ab * da + bb * db) * dth;
  }
  if (near_pi) {
    double cb = 0.0, bpib = 0.0;
    const double dd[3] = {R[0], R[4], R[8]};
#pragma unroll
    for (int k = 0; k < 3; k++) {
      if (tk[k] > 0) {
        const double tb = wb[k] * (w[k] > 0 ? 1.0 : -1.0) * 0.5 / sqrt(tk[k]);
        Rb[4 * k] += tb * bpi;
        cb += tb * bpi;
        bpib += tb * (dd[k] + cphi);
      }
    }
    cb -= bpib * s / ((1.0 + cphi) * (1.0 + cphi));
    trb += -0.5 * cb + bpib * 2.0 * th / (1.0 + cphi) * dth;
  } else {
    const double vb[3] = {t * wb[0], t * wb[1], t * wb[2]};
    Rb[7] += vb[0]; Rb[5] -= vb[0];
    Rb[2] += vb[1]; Rb[6] -= vb[1];
    Rb[3] += vb[2]; Rb[1] -= vb[2];
    if (th > prec3) {
      const double dt = (st - th * ct) / (2.0 * st * st); /* dt/dtheta */
      trb += dot3(wb, v) * dt * dth;
    }
  }
  Rb[0] += trb; Rb[4] += trb; Rb[8] += trb;
}

/* dL/d(references) of one env after K1 (frames, JF, Jcom in shared memory; references staged): the adjoint of the task
 * right-hand sides (k2_assemble / se3_rhs) that g and the contact-motion rows of ce0 carry.
 *   g_dv = -(w_foot JF^T b_foot + w_com Jcom^T b_com + w_post S^T b_post + w_am Ag^T b_am), ce0[6 + 6s + k] = -b_mot[f][k],
 * so bb_foot = -w_foot JF gb, bb_com = -w_com Jcom gb, bb_post = -w_post gb[6:], bb_mot = -ce0b[contact rows]; the AM task
 * has no reference.  lanes 0..3: the SE3 laws (contact LF, contact RF, foot LF, foot RF), 4..6: CoM, lanes < na: posture. */
template <int NV>
TSIDB_DEV void refs_adjoint_env(const DevConst& C, const double* mdl, double* sm, const TickArgs& a, const RefsGradArgs& r,
                                int env, int lane, int mask) {
  constexpr int nv = NV, na = NV - 6;
  const int f0 = (mask & 1) ? 0 : 1; /* foot of contact slot 0; slot 1 is RF */
  double* gb = sm + SM_oBv;       /* dL/dg_dv at [0, nv), bb_foot at [32, 44), bb_com at [44, 47) */
  const double* fr = sm + SM_oFr;
  const double* rf = sm + SM_oRef;
  if (lane < nv) gb[lane] = r.dg ? r.dg[(size_t)env * r.n_max + lane] : 0.0;
  __syncwarp();
  double acc = 0.0;
  if (lane < 12) {
#pragma unroll 2
    for (int j = 0; j < nv; j++) acc += sm[SM_oJF + lane * TSIDB_NVX + j] * gb[j];
    acc *= -C.w_foot;
  } else if (lane < 15) {
#pragma unroll 2
    for (int j = 0; j < nv; j++) acc += sm[SM_oJcom + (lane - 12) * TSIDB_NVX + j] * gb[j];
    acc *= -C.w_com;
  }
  double postb = 0.0;
  if (lane < na) postb = -C.w_post * gb[6 + lane];
  __syncwarp();
  if (lane < 15) gb[32 + lane] = acc;
  __syncwarp();
  if (lane < 4) {
    const int f = lane & 1;
    const bool is_contact = lane < 2;
    double* out = is_contact ? r.out[3 + f] : r.out[1 + f];
    const int nd = is_contact ? 12 : 24;
    if (out) {
      double bb[6];
      const bool live = !is_contact || ((mask >> f) & 1);
      if (is_contact) {
        const int row = 6 + 6 * ((f == f0) ? 0 : 1);
#pragma unroll
        for (int k = 0; k < 6; k++) bb[k] = (live && r.dce0) ? -r.dce0[(size_t)env * r.neq_max + row + k] : 0.0;
      } else {
#pragma unroll
        for (int k = 0; k < 6; k++) bb[k] = gb[32 + 6 * f + k];
      }
      const double* gains = C.kp_contact + (is_contact ? 0 : 12);
      const double* ref = is_contact ? rf + RF_CONTACT + 12 * f : rf + RF_FOOT + 24 * f;
      const double* pf = fr + FR_OMF + f * 12;
      const double* Rf = pf + 3;
      /* the 3 x 3 work of the lane lives in K1's scratch region (dead after K1), not in registers: E, dL/dE, ep, dL/dep */
      double* E = sm + SM_oM + 32 * lane;
      double* ep = E + 9;
      double* Eb = E + 12;
      double* epb = E + 21;
      {
        double Rr[9], dp[3];
#pragma unroll
        for (int c = 0; c < 3; c++)
#pragma unroll
          for (int q = 0; q < 3; q++) Rr[3 * q + c] = ref[3 + 3 * c + q];
        dp[0] = ref[0] - pf[0]; dp[1] = ref[1] - pf[1]; dp[2] = ref[2] - pf[2];
#pragma unroll
        for (int i = 0; i < 3; i++)
#pragma unroll
          for (int j = 0; j < 3; j++) E[3 * i + j] = Rf[i] * Rr[j] + Rf[3 + i] * Rr[3 + j] + Rf[6 + i] * Rr[6 + j];
        mtv3(Rf, dp, ep);
      }
#pragma unroll
      for (int k = 0; k < 12; k++) Eb[k] = 0.0; /* Eb and epb */
      {
        double ol[3], oa[3];
#pragma unroll
        for (int k = 0; k < 3; k++) { ol[k] = gains[k] * bb[k]; oa[k] = gains[3 + k] * bb[3 + k]; }
        log6_adj(E, ep, ol, oa, Eb, epb);
      }
      auto put = [&](int k, double val) { out[eidx(a, env, k, nd)] = live ? val : 0.0; }; /* not in contact: exact zeros */
      double t3[3];
      mv3(Rf, epb, t3); /* ep = Rf^T (p_ref - p_f) */
      put(0, t3[0]); put(1, t3[1]); put(2, t3[2]);
#pragma unroll
      for (int c = 0; c < 3; c++) /* E = Rf^T R_ref: dL/dR_ref = Rf dL/dE, column c of it to ref[3 + 3c ..] */
#pragma unroll
        for (int q = 0; q < 3; q++) put(3 + 3 * c + q, Rf[3 * q] * Eb[c] + Rf[3 * q + 1] * Eb[3 + c] + Rf[3 * q + 2] * Eb[6 + c]);
      if (!is_contact) { /* vl = Rf^T v_ref, al = Rf^T a_ref */
        double kb[6];
#pragma unroll
        for (int k = 0; k < 6; k++) kb[k] = gains[6 + k] * bb[k];
        mv3(Rf, kb, t3);     put(12, t3[0]); put(13, t3[1]); put(14, t3[2]);
        mv3(Rf, kb + 3, t3); put(15, t3[0]); put(16, t3[1]); put(17, t3[2]);
        mv3(Rf, bb, t3);     put(18, t3[0]); put(19, t3[1]); put(20, t3[2]);
        mv3(Rf, bb + 3, t3); put(21, t3[0]); put(22, t3[1]); put(23, t3[2]);
      }
    }
  } else if (lane < 7) {
    const int q = lane - 4;
    const double bb = gb[44 + q];
    if (r.out[0]) {
      r.out[0][eidx(a, env, q, 9)] = C.kp_com[q] * bb;
      r.out[0][eidx(a, env, 3 + q, 9)] = C.kd_com[q] * bb;
      r.out[0][eidx(a, env, 6 + q, 9)] = bb;
    }
  }
  if (lane < na && r.out[5]) r.out[5][eidx(a, env, lane, na)] = mdl[MDL_oPOST + lane] * postb;
}

/* one env of tsidb_refs_grad: q, v and the references staged as the dynamics kernel stages them, K1, then the adjoint.
 * Nothing is written to the handle's images. */
template <int NV>
TSIDB_DEV void refs_grad_env(const DevConst& C, const double* mdl, double* sm, const TickArgs& a, const RefsGradArgs& r,
                             int env, int lane) {
  constexpr int nv = NV, na = NV - 6, nq = NV + 1;
  __syncwarp(); /* every lane is done with the previous env's shared memory */
  if (lane < nq) sm[SM_oQV + lane] = ldin(a.q, a, env, lane, nq);
  if (lane < nv) sm[SM_oQV + 32 + lane] = ldin(a.v, a, env, lane, nv);
  stage_refs(C, mdl, sm, a, env, lane, na);
  __syncwarp();
  k1_dynamics<NV>(C, mdl, sm, lane);
  stage_refs_wait(sm, lane);
  const int mask = a.mask ? (a.mask[env] & 3) : 3;
  refs_adjoint_env<NV>(C, mdl, sm, a, r, env, lane, mask);
}

/* ================================================================= adjoint of the export in the gains (tsidb_gains_grad) */
/* dL/d(gains and weights) of one env after K1 (frames, JF, Jcom, Ag in shared memory; references staged), in tsidb_gains
 * order (TSIDB_GAINS_LEN).  The gains and weights enter
 *   H_dv  = w_foot JF^T JF + w_com Jcom^T Jcom + w_post S^T S (+ w_am Ag^T Ag) + hreg I,
 *   H_ff  = w_freg G + hreg I per foot in contact (G = (W T)^T (W T), r.frg),
 *   g_dv  = -(w_foot JF^T b_foot + w_com Jcom^T b_com + w_post S^T b_post + w_am Ag^T b_am),  ce0[6 + 6s + k] = -b_mot,
 * so with y_r = J_r gb:  wb = <Hb, J^T J> - sum_r b_r y_r,  bb = -w y (bb_post = -w_post gb[6:], bb_mot = -ce0b), and the
 * gradient of each gain is bb times the term it multiplies in the task law.  <Hb, J_r^T J_r> = J_r Hb J_r^T: lane j forms
 * column j of J Hb from the rows of Hb (coalesced) and the warp reduces.  Lanes 0..3: the SE3 laws (contact LF, contact
 * RF, foot LF, foot RF), 4..6: CoM, 7..9: AM, lanes < na: posture. */
template <int NV>
TSIDB_DEV void gains_adjoint_env(const DevConst& C, const double* mdl, double* sm, const TickArgs& a, const GainsGradArgs& r,
                                 int env, int lane, int mask) {
  constexpr int nv = NV, na = NV - 6;
  const int nc = (mask & 1) + ((mask >> 1) & 1);
  const int f0 = (mask & 1) ? 0 : 1; /* foot of contact slot 0; slot 1 is RF */
  const size_t nx = (size_t)r.n_max;
  const double* Hb = r.dH ? r.dH + (size_t)env * nx * nx : nullptr;
  const double* JF = sm + SM_oJF;
  const double* Jcom = sm + SM_oJcom;
  const double* Ag = sm + SM_oAg;
  const double* fr = sm + SM_oFr;
  const double* rf = sm + SM_oRef;
  const double* qs = sm + SM_oQV;
  const double* vs = sm + SM_oQV + 32;
  double* gb = sm + SM_oBv;      /* dL/dg_dv at [0, nv), y = J gb at [32, 50): foot 12, CoM 3, AM 3 */
  double* res = sm + SM_oM;      /* the gradient in tsidb_gains order; K1's scratch region is dead after K1 */
  double* part = sm + SM_oM + 96; /* lane l < 4 of the SE3 laws: its kp and kd terms at [12 l, 12 l + 12) */
  if (lane < nv) gb[lane] = r.dg ? r.dg[(size_t)env * nx + lane] : 0.0;
  __syncwarp();
  if (lane < 18) {
    const double* A = lane < 12 ? JF + lane * TSIDB_NVX : (lane < 15 ? Jcom + (lane - 12) * TSIDB_NVX : Ag + (lane - 15) * TSIDB_NVX);
    double acc = 0.0;
    if (lane < 15 || C.use_am) {
#pragma unroll 2
      for (int j = 0; j < nv; j++) acc += A[j] * gb[j];
    }
    gb[32 + lane] = acc;
  }
  /* <Hb, J^T J> of the foot, CoM and AM tasks, the posture's sum of Hb_jj (j >= 6) and <Hb_ff, G> of the feet in contact */
  double hf = 0.0, hc = 0.0, ha = 0.0, hp = 0.0, hr = 0.0;
  if (Hb && lane < nv) {
    const int j = lane;
    double uf[12], uc[3], ua[3];
#pragma unroll
    for (int q = 0; q < 12; q++) uf[q] = 0.0;
#pragma unroll
    for (int q = 0; q < 3; q++) { uc[q] = 0.0; ua[q] = 0.0; }
#pragma unroll 1
    for (int i = 0; i < nv; i++) {
      const double h = Hb[i * nx + j];
#pragma unroll
      for (int q = 0; q < 12; q++) uf[q] += JF[q * TSIDB_NVX + i] * h;
#pragma unroll
      for (int q = 0; q < 3; q++) uc[q] += Jcom[q * TSIDB_NVX + i] * h;
      if (C.use_am) {
#pragma unroll
        for (int q = 0; q < 3; q++) ua[q] += Ag[q * TSIDB_NVX + i] * h;
      }
    }
#pragma unroll
    for (int q = 0; q < 12; q++) hf += uf[q] * JF[q * TSIDB_NVX + j];
#pragma unroll
    for (int q = 0; q < 3; q++) hc += uc[q] * Jcom[q * TSIDB_NVX + j];
    if (C.use_am) {
#pragma unroll
      for (int q = 0; q < 3; q++) ha += ua[q] * Ag[q * TSIDB_NVX + j];
    }
    if (j >= 6) hp = Hb[j * nx + j];
    if (j < 12)
      for (int s = 0; s < nc; s++) {
        const double* blk = Hb + (nv + 12 * s) * (nx + 1);
#pragma unroll 4
        for (int i = 0; i < 12; i++) hr += blk[i * nx + j] * r.frg[i * 12 + j];
      }
  }
  __syncwarp();
  const double* y = gb + 32;
  double wf = 0.0, wc = 0.0, wa = 0.0, wp = 0.0; /* - b_r y_r of the foot, CoM, AM and posture tasks */
  if (lane < 4) {
    const int f = lane & 1;
    const bool is_contact = lane < 2;
    double kpb[6], kdb[6];
#pragma unroll
    for (int k = 0; k < 6; k++) { kpb[k] = 0.0; kdb[k] = 0.0; }
    if (!is_contact || ((mask >> f) & 1)) { /* a contact not in contact: exact zeros */
      /* se3_rhs's law, restated with its intermediate terms kept (log6 pe, velocity error ve), which the gains'
       * gradients multiply; se3_rhs itself stays as the tick's kernels compile it.  The two must stay in step. */
      const double* gains = C.kp_contact + (is_contact ? 0 : 12);
      const double* ref = is_contact ? rf + RF_CONTACT + 12 * f : rf + RF_FOOT + 24 * f;
      const double* pf = fr + FR_OMF + f * 12;
      const double* Rf = pf + 3;
      const double* vF = fr + FR_VF + f * 6;
      const double* aF = fr + FR_AF + f * 6;
      double Rr[9], dp[3], E[9], ep[3], pe[6];
#pragma unroll
      for (int c = 0; c < 3; c++)
#pragma unroll
        for (int q = 0; q < 3; q++) Rr[3 * q + c] = ref[3 + 3 * c + q];
      dp[0] = ref[0] - pf[0]; dp[1] = ref[1] - pf[1]; dp[2] = ref[2] - pf[2];
#pragma unroll
      for (int i = 0; i < 3; i++)
#pragma unroll
        for (int q = 0; q < 3; q++) E[3 * i + q] = Rf[i] * Rr[q] + Rf[3 + i] * Rr[3 + q] + Rf[6 + i] * Rr[6 + q];
      mtv3(Rf, dp, ep);
      log6_dev(E, ep, pe);
      double ve[6], bb[6]; /* velocity error Rf^T v_ref - v_F (v_ref = 0 for a contact), bb = dL/db */
      if (is_contact) {
        const int row = 6 + 6 * ((f == f0) ? 0 : 1);
#pragma unroll
        for (int k = 0; k < 6; k++) {
          ve[k] = -vF[k];
          bb[k] = r.dce0 ? -r.dce0[(size_t)env * r.neq_max + row + k] : 0.0;
        }
      } else {
        double vl[3], va[3], al[3], aa[3];
        mtv3(Rf, ref + 12, vl); mtv3(Rf, ref + 15, va);
        mtv3(Rf, ref + 18, al); mtv3(Rf, ref + 21, aa);
#pragma unroll
        for (int k = 0; k < 3; k++) { ve[k] = vl[k] - vF[k]; ve[3 + k] = va[k] - vF[3 + k]; }
#pragma unroll
        for (int k = 0; k < 6; k++) {
          bb[k] = -C.w_foot * y[6 * f + k];
          const double b = (gains[k] * pe[k] + gains[6 + k] * ve[k] + (k < 3 ? al[k] : aa[k - 3])) - aF[k]; /* se3_rhs */
          wf -= b * y[6 * f + k];
        }
      }
#pragma unroll
      for (int k = 0; k < 6; k++) { kpb[k] = bb[k] * pe[k]; kdb[k] = bb[k] * ve[k]; }
    }
#pragma unroll
    for (int k = 0; k < 6; k++) { part[12 * lane + k] = kpb[k]; part[12 * lane + 6 + k] = kdb[k]; }
  } else if (lane < 7) { /* CoM: b = -Kp (c - c_ref) - Kd (vc - vc_ref) + ac_ref - drift */
    const int q = lane - 4;
    const double e = fr[FR_COM + q] - rf[RF_COM + q], ed = fr[FR_COM + 3 + q] - rf[RF_COM + 3 + q];
    const double bb = -C.w_com * y[12 + q];
    res[24 + q] = -bb * e;
    res[27 + q] = -bb * ed;
    const double b = (-C.kp_com[q] * e - C.kd_com[q] * ed + rf[RF_COM + 6 + q]) - fr[FR_COM + 6 + q];
    wc = -b * y[12 + q];
  } else if (lane < 10) { /* legacy AM: b = -Kp L - drift */
    const int q = lane - 7;
    double g = 0.0;
    if (C.use_am) {
      const double bb = -C.w_am * y[15 + q];
      g = -bb * fr[FR_L + q];
      wa = (C.kp_am[q] * fr[FR_L + q] + fr[FR_L + 3 + q]) * y[15 + q];
    }
    res[76 + q] = g;
  }
  if (lane < 23) { /* posture: b = -Kp (q_j - q_ref) - Kd v_j; columns past na are exact zeros */
    double gp = 0.0, gd = 0.0;
    if (lane < na) {
      const double e = qs[7 + lane] - rf[RF_POST + lane], gj = gb[6 + lane];
      const double bb = -C.w_post * gj;
      gp = -bb * e;
      gd = -bb * vs[6 + lane];
      wp = (mdl[MDL_oPOST + lane] * e + mdl[MDL_oPOST + 23 + lane] * vs[6 + lane]) * gj;
    }
    res[30 + lane] = gp;
    res[53 + lane] = gd;
  }
  const double sf = warp_sum(hf + wf), sc = warp_sum(hc + wc), sa = warp_sum(ha + wa), sp = warp_sum(hp + wp);
  const double sr = warp_sum(hr);
  __syncwarp();
  if (lane < 24) { /* both contacts share kp_contact / kd_contact, both feet kp_foot / kd_foot */
    const int o = lane + (lane >= 12 ? 12 : 0);
    res[lane] = part[o] + part[o + 12];
  } else if (lane == 24) {
    res[79] = sf; res[80] = sc; res[81] = sp; res[82] = C.use_am ? sa : 0.0; res[83] = sr;
  }
  __syncwarp();
  for (int k = lane; k < TSIDB_GAINS_LEN; k += 32) r.out[eidx(a, env, k, TSIDB_GAINS_LEN)] = res[k];
}

/* one env of tsidb_gains_grad: q, v and the references staged as the dynamics kernel stages them, K1, then the adjoint.
 * Nothing is written to the handle's images. */
template <int NV>
TSIDB_DEV void gains_grad_env(const DevConst& C, const double* mdl, double* sm, const TickArgs& a, const GainsGradArgs& r,
                              int env, int lane) {
  constexpr int nv = NV, na = NV - 6, nq = NV + 1;
  __syncwarp(); /* every lane is done with the previous env's shared memory */
  if (lane < nq) sm[SM_oQV + lane] = ldin(a.q, a, env, lane, nq);
  if (lane < nv) sm[SM_oQV + 32 + lane] = ldin(a.v, a, env, lane, nv);
  stage_refs(C, mdl, sm, a, env, lane, na);
  __syncwarp();
  k1_dynamics<NV>(C, mdl, sm, lane);
  stage_refs_wait(sm, lane);
  const int mask = a.mask ? (a.mask[env] & 3) : 3;
  gains_adjoint_env<NV>(C, mdl, sm, a, r, env, lane, mask);
}

/* ================================================================= adjoint of the export in q and v (tsidb_state_grad) */
/* Stage 1 of one env, after K1 and K2 ran on this env in `sm`: the cotangent of the export (the parts of r, NULL = zero)
 * pulled back onto K1's outputs.  It lands in `cb` at K1's own offsets (M, JF, Jcom, Ag, nle, frames; zero where the
 * export does not depend on them), and the terms that depend on q and v directly (posture task, joint-bound rows) land in
 * cb[SM_oQV + k] (q) and cb[SM_oQV + 32 + k] (v).  Of an env with sizes (n, neq, nin) it reads only what depends on
 * the state:
 *   H    rows and columns 0..nv (the dv block; dL/dH_ij + dL/dH_ji multiplies dH_ij); the force block is constant
 *   g    0..nv
 *   CE   rows 0..6, columns 0..n ([M_u | -Jc_u^T]); rows 6..neq, columns 0..nv (JF of the feet in contact)
 *   ce0  0..neq (h_u, -b_mot)
 *   CI   the actuation rows (torque bounds), columns 0..n; the force and joint-bound rows are constant
 *   ci0  the actuation rows (h_a) and the joint-bound rows of the joints (v_j); the force rows and base rows are constant
 *   TA   rows 0..na, columns 0..n;  ta0  0..na
 * A joint-bound entry of ci0 is clipped to +-1e10 by the export; where the clip binds its derivative is zero. */
template <int NV>
TSIDB_DEV void state_adjoint_env(const DevConst& C, const double* mdl, double* sm, double* cb, const StateGradArgs& r,
                                 int env, int lane, int mask) {
  constexpr int nv = NV, na = NV - 6;
  const double BIG = 1e10; /* the export's clip of the joint-bound rows */
  const int nc = (mask & 1) + ((mask >> 1) & 1);
  const int neq = 6 + 6 * nc;
  const int f0 = (mask & 1) ? 0 : 1; /* foot of force slot 0; slot 1 is RF */
  const int oAct = 34 * nc, oJb = 34 * nc + (C.use_tb ? 2 * na : 0); /* first actuation and joint-bound row of CI */
  const double* JF = sm + SM_oJF;
  const double* Jcom = sm + SM_oJcom;
  const double* Ag = sm + SM_oAg;
  const double* bv = sm + SM_oBv;
  const double* fr = sm + SM_oFr;
  const double* rf = sm + SM_oRef;
  const double* vs = sm + SM_oQV + 32;
  const size_t nx = (size_t)r.n_max;
  const double* H = r.H ? r.H + (size_t)env * nx * nx : nullptr;
  const double* g = r.g ? r.g + (size_t)env * nx : nullptr;
  const double* CE = r.CE ? r.CE + (size_t)env * r.neq_max * nx : nullptr;
  const double* ce0 = r.ce0 ? r.ce0 + (size_t)env * r.neq_max : nullptr;
  const double* CI = (r.CI && C.use_tb) ? r.CI + (size_t)env * r.nin_max * nx : nullptr;
  const double* ci0 = r.ci0 ? r.ci0 + (size_t)env * r.nin_max : nullptr;
  const double* TA = r.TA ? r.TA + (size_t)env * na * nx : nullptr;
  const double* ta0 = r.ta0 ? r.ta0 + (size_t)env * na : nullptr;
  for (int k = lane; k < SM_oRef; k += 32) cb[k] = 0.0;
  double* gb = cb + SM_oGv; /* dL/dg_dv */
  double* bb = cb + SM_oBv; /* dL/d of the task right-hand sides, at the BV_* offsets */
  __syncwarp();
  if (lane < nv) gb[lane] = g ? g[lane] : 0.0;
  __syncwarp();
  /* g_dv = -(w_foot JF^T b_foot + w_com Jcom^T b_com + w_am Ag^T b_am + w_post S^T b_post), ce0[6 + 6s + k] = -b_mot[f_s][k] */
  if (lane < 18) {
    const double* A = lane < 12 ? JF + lane * TSIDB_NVX : (lane < 15 ? Jcom + (lane - 12) * TSIDB_NVX : Ag + (lane - 15) * TSIDB_NVX);
    double acc = 0.0;
#pragma unroll 2
    for (int j = 0; j < nv; j++) acc += A[j] * gb[j];
    if (lane < 12) bb[BV_FOOT + lane] = -C.w_foot * acc;
    else if (lane < 15) bb[BV_COM + lane - 12] = -C.w_com * acc;
    else bb[BV_AM + lane - 15] = C.use_am ? -C.w_am * acc : 0.0;
  }
  if (lane < 12) {
    const int f = lane / 6;
    bb[BV_MOT + lane] = (ce0 && ((mask >> f) & 1)) ? -ce0[6 + 6 * (f == f0 ? 0 : 1) + lane % 6] : 0.0;
  }
  if (lane < na) {
    bb[BV_POST + lane] = -C.w_post * gb[6 + lane];
    /* posture task: b_post = -Kp (q_j - q_ref) - Kd v_j */
    cb[SM_oQV + 7 + lane] = -mdl[MDL_oPOST + lane] * bb[BV_POST + lane];
    cb[SM_oQV + 32 + 6 + lane] = -mdl[MDL_oPOST + 23 + lane] * bb[BV_POST + lane];
  }
  __syncwarp();
  /* joint-bound rows: ub = min((v_max - v_j) / dt, 1e10), lb = max((v_min - v_j) / dt, -1e10), ci0 = (-lb, ub) */
  if (ci0 && C.use_jb && lane >= 6 && lane < nv) {
    const double vj = vs[lane];
    const double hi = (C.v_max[lane - 6] - vj) / C.jb_dt, lo = (C.v_min[lane - 6] - vj) / C.jb_dt;
    double d = 0.0;
    if (lo > -BIG) d += ci0[oJb + lane] / C.jb_dt;
    if (hi < BIG) d -= ci0[oJb + nv + lane] / C.jb_dt;
    cb[SM_oQV + 32 + lane] += d;
  }
  /* column j of M, JF, Jcom, Ag and entry j of nle, one lane each */
  if (lane < nv) {
    const int j = lane;
    double jfb[12], jcb[3], agb[3];
#pragma unroll
    for (int q = 0; q < 12; q++) jfb[q] = 0.0;
#pragma unroll
    for (int q = 0; q < 3; q++) { jcb[q] = 0.0; agb[q] = 0.0; }
    /* H_dv = w_foot JF^T JF + w_com Jcom^T Jcom (+ w_am Ag^T Ag) + constant diagonal: dL/dA = w A (Hb + Hb^T) */
    if (H) {
#pragma unroll 1
      for (int m = 0; m < nv; m++) {
        const double s = H[j * nx + m] + H[m * nx + j];
#pragma unroll
        for (int q = 0; q < 12; q++) jfb[q] += s * JF[q * TSIDB_NVX + m];
#pragma unroll
        for (int q = 0; q < 3; q++) jcb[q] += s * Jcom[q * TSIDB_NVX + m];
        if (C.use_am) {
#pragma unroll
          for (int q = 0; q < 3; q++) agb[q] += s * Ag[q * TSIDB_NVX + m];
        }
      }
    }
    const double gj = gb[j];
#pragma unroll
    for (int q = 0; q < 12; q++) jfb[q] = C.w_foot * (jfb[q] - gj * bv[BV_FOOT + q]);
#pragma unroll
    for (int q = 0; q < 3; q++) {
      jcb[q] = C.w_com * (jcb[q] - gj * bv[BV_COM + q]);
      agb[q] = C.use_am ? C.w_am * (agb[q] - gj * bv[BV_AM + q]) : 0.0;
    }
#pragma unroll
    for (int q = 0; q < 12; q++) cb[SM_oJF + q * TSIDB_NVX + j] = jfb[q];
#pragma unroll
    for (int q = 0; q < 3; q++) { cb[SM_oJcom + q * TSIDB_NVX + j] = jcb[q]; cb[SM_oAg + q * TSIDB_NVX + j] = agb[q]; }
    /* CE: rows 0..6 are [M_u | -Jc_u^T], rows 6..neq the JF rows of the feet in contact */
    if (CE) {
      for (int q = 0; q < 6; q++) cb[SM_oM + q * SM_LDM + j] = CE[q * nx + j];
      for (int q = 6; q < neq; q++) cb[SM_oJF + (((q < 12) ? f0 : 1) * 6 + (q - 6) % 6) * TSIDB_NVX + j] += CE[q * nx + j];
    }
    /* CI actuation rows ([M_a | -Jc_a^T], lower side +, upper side -) and TA ([M_a | -Jc_a^T]) */
    for (int q = 6; q < nv; q++) {
      double x = 0.0;
      if (CI) x += CI[(oAct + q - 6) * nx + j] - CI[(oAct + na + q - 6) * nx + j];
      if (TA) x += TA[(q - 6) * nx + j];
      cb[SM_oM + q * SM_LDM + j] = x;
    }
    /* Jc = T^T JF_f of force slot s: row j of Jc enters CE row j (j < 6), the actuation rows and TA row j - 6 (j >= 6) */
    for (int s = 0; s < nc; s++) {
      const int f = s == 0 ? f0 : 1;
      double jc[12];
#pragma unroll
      for (int k = 0; k < 12; k++) {
        const int col = nv + 12 * s + k;
        double x = 0.0;
        if (j < 6) {
          if (CE) x -= CE[j * nx + col];
        } else {
          if (CI) x += CI[(oAct + na + j - 6) * nx + col] - CI[(oAct + j - 6) * nx + col];
          if (TA) x -= TA[(j - 6) * nx + col];
        }
        jc[k] = x;
      }
#pragma unroll
      for (int m = 0; m < 6; m++) {
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < 12; k++) acc += C.T[m][k] * jc[k];
        cb[SM_oJF + (f * 6 + m) * TSIDB_NVX + j] += acc;
      }
    }
    /* ce0 rows 0..6 are h_u; ci0's actuation rows h_a - tau_min and tau_max - h_a; ta0 = h_a */
    double nb = 0.0;
    if (j < 6) {
      if (ce0) nb = ce0[j];
    } else {
      if (ci0 && C.use_tb) nb += ci0[oAct + j - 6] - ci0[oAct + na + j - 6];
      if (ta0) nb += ta0[j - 6];
    }
    cb[SM_oNle + j] = nb;
  }
  /* the four SE3 laws (contact LF, contact RF, foot LF, foot RF): b = Kp log6(Rf^T R_ref, Rf^T (p_ref - p_f))
   * + Kd (Rf^T v_ref - v_F) + Rf^T a_ref - a_F, each lane's frame cotangent to its own scratch, summed per foot below */
  double* wk = sm + SM_oM + 64 * lane; /* K2's Hessian block, dead: E 9, ep 3, dL/dE 9, dL/dep 3, then p 3, R 9, vF 6, aF 6 */
  if (lane < 4) {
    const int f = lane & 1;
    const bool is_contact = lane < 2;
    double* E = wk;
    double* ep = wk + 9;
    double* Eb = wk + 12;
    double* epb = wk + 21;
    double* o = wk + 24;
#pragma unroll
    for (int k = 0; k < 36; k++) wk[12 + k] = 0.0; /* Eb, epb, o */
    if (!is_contact || ((mask >> f) & 1)) {
      double b6[6], kp[6], kd[6], Rr[9], dp[3];
      const double* gains = C.kp_contact + (is_contact ? 0 : 12);
#pragma unroll
      for (int k = 0; k < 6; k++) {
        b6[k] = bb[(is_contact ? BV_MOT : BV_FOOT) + 6 * f + k];
        kp[k] = gains[k];
        kd[k] = gains[6 + k];
      }
      const double* ref = is_contact ? rf + RF_CONTACT + 12 * f : rf + RF_FOOT + 24 * f;
      const double* pf = fr + FR_OMF + f * 12;
      const double* Rf = pf + 3;
#pragma unroll
      for (int c = 0; c < 3; c++)
#pragma unroll
        for (int q = 0; q < 3; q++) Rr[3 * q + c] = ref[3 + 3 * c + q];
      dp[0] = ref[0] - pf[0]; dp[1] = ref[1] - pf[1]; dp[2] = ref[2] - pf[2];
#pragma unroll
      for (int i = 0; i < 3; i++)
#pragma unroll
        for (int q = 0; q < 3; q++) E[3 * i + q] = Rf[i] * Rr[q] + Rf[3 + i] * Rr[3 + q] + Rf[6 + i] * Rr[6 + q];
      mtv3(Rf, dp, ep);
      {
        double ol[3], oa[3];
#pragma unroll
        for (int k = 0; k < 3; k++) { ol[k] = kp[k] * b6[k]; oa[k] = kp[3 + k] * b6[3 + k]; }
        log6_adj(E, ep, ol, oa, Eb, epb);
      }
      /* E = Rf^T R_ref, ep = Rf^T dp, dp = p_ref - p_f; foot task: v = Rf^T v_ref, a = Rf^T a_ref */
#pragma unroll
      for (int q = 0; q < 3; q++)
#pragma unroll
        for (int i = 0; i < 3; i++) {
          double x = Rr[3 * q] * Eb[3 * i] + Rr[3 * q + 1] * Eb[3 * i + 1] + Rr[3 * q + 2] * Eb[3 * i + 2] + dp[q] * epb[i];
          if (!is_contact)
            x += ref[12 + q] * kd[i] * b6[i] + ref[15 + q] * kd[3 + i] * b6[3 + i] + ref[18 + q] * b6[i] + ref[21 + q] * b6[3 + i];
          o[3 + 3 * q + i] = x;
        }
      double t3[3];
      mv3(Rf, epb, t3);
      o[0] = -t3[0]; o[1] = -t3[1]; o[2] = -t3[2];
#pragma unroll
      for (int k = 0; k < 6; k++) { o[12 + k] = -kd[k] * b6[k]; o[18 + k] = -b6[k]; }
    }
  } else if (lane < 7) {
    const int q = lane - 4; /* CoM task: b = -Kp (c - c_ref) - Kd (vc - vc_ref) + ac_ref - drift */
    cb[SM_oFr + FR_COM + q] = -C.kp_com[q] * bb[BV_COM + q];
    cb[SM_oFr + FR_COM + 3 + q] = -C.kd_com[q] * bb[BV_COM + q];
    cb[SM_oFr + FR_COM + 6 + q] = -bb[BV_COM + q];
  } else if (lane < 10) {
    const int q = lane - 7; /* legacy AM task: b = -Kp L - drift */
    cb[SM_oFr + FR_L + q] = -C.kp_am[q] * bb[BV_AM + q];
    cb[SM_oFr + FR_L + 3 + q] = -bb[BV_AM + q];
  }
  __syncwarp();
  const double* w0 = sm + SM_oM + 24;
  if (lane < 24) { /* placements: foot f = lane / 12, contact lane f and foot-task lane 2 + f */
    const int f = lane / 12;
    cb[SM_oFr + FR_OMF + lane] = w0[64 * f + lane % 12] + w0[64 * (2 + f) + lane % 12];
  }
  if (lane < 12) { /* velocities and drifts */
    const int f = lane / 6;
    cb[SM_oFr + FR_VF + lane] = w0[64 * f + 12 + lane % 6] + w0[64 * (2 + f) + 12 + lane % 6];
    cb[SM_oFr + FR_AF + lane] = w0[64 * f + 18 + lane % 6] + w0[64 * (2 + f) + 18 + lane % 6];
  }
  __syncwarp();
}

/* one env of tsidb_state_grad.  q, v and the references staged and K1 + K2 run as the dynamics kernel runs them, stage 1
 * (state_adjoint_env), then stage 2: K1 again in tangent arithmetic once per raw input direction (nq components of q, nv
 * of v), each pass contracted with stage 1's cotangents.  The tangent passes overwrite `sm` (Dual, 2 SM_oRef doubles);
 * `cb` (SM_oRef doubles) holds the cotangents and the result. */
template <int NV>
TSIDB_DEV void state_grad_env(const DevConst& C, const double* mdl, double* sm, double* cb, const TickArgs& a,
                              const StateGradArgs& r, int env, int lane) {
  constexpr int nv = NV, na = NV - 6, nq = NV + 1;
  __syncwarp(); /* every lane is done with the previous env's shared memory */
  const double qv = lane < nq ? ldin(a.q, a, env, lane, nq) : 0.0;
  const double vv = lane < nv ? ldin(a.v, a, env, lane, nv) : 0.0;
  if (lane < nq) sm[SM_oQV + lane] = qv;
  if (lane < nv) sm[SM_oQV + 32 + lane] = vv;
  stage_refs(C, mdl, sm, a, env, lane, na);
  __syncwarp();
  k1_dynamics<NV>(C, mdl, sm, lane);
  stage_refs_wait(sm, lane);
  const int mask = a.mask ? (a.mask[env] & 3) : 3;
  const int nc = (mask & 1) + ((mask >> 1) & 1);
  k2_assemble<NV>(C, mdl, sm, a, env, lane, mask, 6 + 6 * nc, nv + 12 * nc);
  state_adjoint_env<NV>(C, mdl, sm, cb, r, env, lane, mask);
  Dual* ds = reinterpret_cast<Dual*>(sm);
#pragma unroll 1
  for (int dir = 0; dir < nq + nv; dir++) {
    __syncwarp();
    if (lane < nq) ds[SM_oQV + lane] = Dual(qv, dir == lane ? 1.0 : 0.0);
    if (lane < nv) ds[SM_oQV + 32 + lane] = Dual(vv, dir == nq + lane ? 1.0 : 0.0);
    __syncwarp();
    k1_dynamics<NV>(C, mdl, ds, lane);
    /* the entries K1 writes: M (nv rows), JF, the nv columns of Jcom and Ag, nle, the frames */
    double acc = 0.0;
    for (int k = lane; k < nv * SM_LDM; k += 32) acc += cb[SM_oM + k] * ds[SM_oM + k].d;
    for (int k = lane; k < 12 * TSIDB_NVX; k += 32) acc += cb[SM_oJF + k] * ds[SM_oJF + k].d;
    for (int k = lane; k < 6 * TSIDB_NVX + nv; k += 32)
      if (k >= 6 * TSIDB_NVX || k % TSIDB_NVX < nv) acc += cb[SM_oJcom + k] * ds[SM_oJcom + k].d;
    for (int k = lane; k < FR_L + 6; k += 32) acc += cb[SM_oFr + k] * ds[SM_oFr + k].d;
    acc = warp_sum(acc);
    if (lane == 0) cb[SM_oQV + (dir < nq ? dir : 32 + dir - nq)] += acc;
  }
  __syncwarp();
  if (r.dq && lane < nq) r.dq[eidx(a, env, lane, nq)] = cb[SM_oQV + lane];
  if (r.dv && lane < nv) r.dv[eidx(a, env, lane, nv)] = cb[SM_oQV + 32 + lane];
}

/* ================================================================= generic QP solve of one env (tsidb_qp_solve) */
/* eiquadprog-fast solve_quadprog on a caller-supplied problem, min 1/2 x'Hx + g'x s.t. CE x + ce0 = 0, CI x + ci0 >= 0,
 * step for step as the oracle's eq_solve states it: LLT of H, J = L^-T, x0 = -H^-1 g, the equalities added one by one,
 * then the dual active-set passes (most violated row first, lowest index on ties; psi stopping test; Givens add/delete).
 * J, R and the per-row state live in shared memory; lanes run over rows or columns of J and R (row k / column c: lanes
 * k % 32, two per lane at n = 64), every scalar that steers the iteration is computed identically by all lanes, so the
 * control flow is warp-uniform.  Sums over k keep the oracle's order where a lane owns the whole sum (d = J'np,
 * z = J2 d2, the violation scan); the triangular solves run column-oriented and the dot products as warp sums. */
#define QP_SLOTS (TSIDB_QP_MAX_N / 32)
struct QpLayout {
  int ld;                                            /* row stride of J and R: odd, so column walks are conflict-free */
  int oJ, oR, ox, oxo, od, oz, or_, onp, ou, ouo, os; /* doubles */
  int oA, oAo, oiai, oix;                            /* int32, from sm + oI */
  int oI, per_env;
};
TSIDB_HD inline QpLayout qp_layout(int n_max, int nin_max) {
  QpLayout L;
  L.ld = n_max | 1;
  L.oJ = 0;
  L.oR = L.oJ + n_max * L.ld;
  L.ox = L.oR + n_max * L.ld;
  L.oxo = L.ox + n_max;
  L.od = L.oxo + n_max;
  L.oz = L.od + n_max;
  L.or_ = L.oz + n_max;
  L.onp = L.or_ + n_max;
  L.ou = L.onp + n_max;
  L.ouo = L.ou + n_max + 1;
  L.os = L.ouo + n_max + 1;
  L.oI = L.os + nin_max;
  L.oA = 0;
  L.oAo = n_max + 1;
  L.oiai = 2 * (n_max + 1);
  L.oix = L.oiai + nin_max;
  L.per_env = L.oI + (L.oix + nin_max + 1) / 2;
  L.per_env += L.per_env & 1; /* every env's area starts 16-byte aligned */
  return L;
}

TSIDB_DEV double eq_distance(double a, double b) {
  const double a1 = fabs(a), b1 = fabs(b);
  if (a1 > b1) { const double t = b1 / a1; return a1 * sqrt(1.0 + t * t); }
  if (b1 > a1) { const double t = a1 / b1; return b1 * sqrt(1.0 + t * t); }
  return a1 * sqrt(2.0);
}

/* (value, index) argmin over the warp: the smallest value, the lowest index among equal values; idx < 0 = no candidate.
 * The butterfly leaves the same pair in every lane. */
TSIDB_DEV void warp_argmin(double& val, int& idx) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(FULL, val, o);
    const int oi = __shfl_xor_sync(FULL, idx, o);
    if (oi >= 0 && (idx < 0 || ov < val || (ov == val && oi < idx))) { val = ov; idx = oi; }
  }
}

struct QpEnv {
  int n, nm, ld;
  double *J, *R, *x, *xo, *d, *z, *r, *np, *u, *uo, *s;
  int *A, *Ao, *iai, *iax;
};

/* d = J' np (lane per column, k ascending) */
TSIDB_DEV void qp_compute_d(const QpEnv& E, int lane) {
  for (int c = lane; c < E.n; c += 32) {
    double s = 0.0;
    for (int k = 0; k < E.n; k++) s += E.J[k * E.ld + c] * E.np[k];
    E.d[c] = s;
  }
}
/* z = J[:, iq:] d[iq:] (lane per row, k ascending; zero when iq >= n) */
TSIDB_DEV void qp_update_z(const QpEnv& E, int iq, int lane) {
  for (int i = lane; i < E.n; i += 32) {
    double s = 0.0;
    for (int k = iq; k < E.n; k++) s += E.J[i * E.ld + k] * E.d[k];
    E.z[i] = s;
  }
}
/* R[:iq, :iq] r = d[:iq], column-oriented back substitution */
TSIDB_DEV void qp_update_r(const QpEnv& E, int iq, int lane) {
  double acc[QP_SLOTS];
#pragma unroll
  for (int t = 0; t < QP_SLOTS; t++) acc[t] = (lane + 32 * t < iq) ? E.d[lane + 32 * t] : 0.0;
  for (int i = iq - 1; i >= 0; i--) {
    const double ri = __shfl_sync(FULL, (i >> 5) ? acc[QP_SLOTS - 1] : acc[0], i & 31) / E.R[i * E.ld + i];
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int m = lane + 32 * t;
      if (m < i) acc[t] -= E.R[m * E.ld + i] * ri;
      else if (m == i) acc[t] = ri;
    }
  }
#pragma unroll
  for (int t = 0; t < QP_SLOTS; t++)
    if (lane + 32 * t < iq) E.r[lane + 32 * t] = acc[t];
  __syncwarp();
}
/* add_constraint: Givens rotations that zero d[iq+1..n-1] into J, then the new column of R; false when the new column is
 * (numerically) dependent.  d is read by every lane and carried in registers; lane 0 writes it back. */
TSIDB_DEV bool qp_add_constraint(const QpEnv& E, int& iq, double& R_norm, int lane) {
  const int n = E.n, ld = E.ld;
  if (n - 1 >= iq + 1) {
    double cur = E.d[n - 1];
    for (int j = n - 1; j >= iq + 1; j--) {
      double cc = E.d[j - 1], ss = cur;
      const double h = eq_distance(cc, ss);
      if (h == 0.0) { cur = cc; continue; }
      ss = ss / h;
      cc = cc / h;
      if (cc < 0) { cc = -cc; ss = -ss; cur = -h; }
      else cur = h;
      const double xny = ss / (1.0 + cc);
      for (int k = lane; k < n; k += 32) {
        const double t1 = E.J[k * ld + j - 1], t2 = E.J[k * ld + j];
        const double a = t1 * cc + t2 * ss;
        E.J[k * ld + j - 1] = a;
        E.J[k * ld + j] = xny * (t1 + a) - t2;
      }
    }
    __syncwarp();
    if (lane == 0) {
      E.d[iq] = cur;
      for (int j = iq + 1; j < n; j++) E.d[j] = 0.0;
    }
    __syncwarp();
  }
  iq++;
  for (int i = lane; i < iq; i += 32) E.R[i * ld + iq - 1] = E.d[i];
  __syncwarp();
  const double dl = fabs(E.d[iq - 1]);
  if (dl <= TS_EPS * R_norm) return false;
  if (dl > R_norm) R_norm = dl;
  return true;
}
/* delete_constraint: drop inequality row l from the working set, restore R to triangular with Givens rotations */
TSIDB_DEV void qp_delete_constraint(const QpEnv& E, int neq, int& iq, int l, int lane) {
  const int n = E.n, ld = E.ld;
  int qq = 0;
  for (int i = neq; i < iq; i++)
    if (E.A[i] == l) { qq = i; break; }
  for (int k = lane; k < n; k += 32)
    for (int i = qq; i < iq - 1; i++) E.R[k * ld + i] = E.R[k * ld + i + 1];
  __syncwarp();
  if (lane == 0) {
    for (int i = qq; i < iq - 1; i++) { E.A[i] = E.A[i + 1]; E.u[i] = E.u[i + 1]; }
    E.A[iq - 1] = E.A[iq];
    E.u[iq - 1] = E.u[iq];
    E.A[iq] = 0;
    E.u[iq] = 0.0;
  }
  for (int j = lane; j < iq; j += 32) E.R[j * ld + iq - 1] = 0.0;
  __syncwarp();
  iq--;
  if (iq == 0) return;
  for (int j = qq; j < iq; j++) {
    double cc = E.R[j * ld + j], ss = E.R[(j + 1) * ld + j];
    const double h = eq_distance(cc, ss);
    if (h == 0.0) continue;
    cc = cc / h;
    ss = ss / h;
    __syncwarp(); /* every lane has read the pivot pair */
    if (lane == 0) E.R[(j + 1) * ld + j] = 0.0;
    if (cc < 0) {
      if (lane == 0) E.R[j * ld + j] = -h;
      cc = -cc;
      ss = -ss;
    } else if (lane == 0) E.R[j * ld + j] = h;
    const double xny = ss / (1.0 + cc);
    for (int k = j + 1 + lane; k < iq; k += 32) {
      const double t1 = E.R[j * ld + k], t2 = E.R[(j + 1) * ld + k];
      const double a = t1 * cc + t2 * ss;
      E.R[j * ld + k] = a;
      E.R[(j + 1) * ld + k] = xny * (t1 + a) - t2;
    }
    for (int k = lane; k < n; k += 32) {
      const double t1 = E.J[k * ld + j], t2 = E.J[k * ld + j + 1];
      const double a = t1 * cc + t2 * ss;
      E.J[k * ld + j] = a;
      E.J[k * ld + j + 1] = xny * (a + t1) - t2;
    }
    __syncwarp();
  }
}

/* eiquadprog-fast result codes (the oracle's eq_solve) */
enum { QP_OPTIMAL = 0, QP_INFEASIBLE = 1, QP_UNBOUNDED = 2, QP_MAX_ITER = 3, QP_REDUNDANT_EQ = 4 };

/* Eigen::LLT (lower) of the n x n matrix H (row stride nm; the strict upper triangle is never read) into L (row stride
 * ld): column j by the lanes that own rows i >= j.  False when H is not positive definite. */
TSIDB_DEV bool qp_llt(const double* H, int nm, double* L, int ld, int n, int lane) {
  for (int j = 0; j < n; j++) {
    double acc[QP_SLOTS];
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int i = lane + 32 * t;
      acc[t] = 0.0;
      if (i >= j && i < n) {
        double a = H[(size_t)i * nm + j];
        for (int k = 0; k < j; k++) a -= L[i * ld + k] * L[j * ld + k];
        acc[t] = a;
      }
    }
    const double sdiag = __shfl_sync(FULL, (j >> 5) ? acc[QP_SLOTS - 1] : acc[0], j & 31);
    if (!(sdiag > 0)) return false;
    const double ljj = sqrt(sdiag);
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int i = lane + 32 * t;
      if (i == j) L[i * ld + j] = ljj;
      else if (i > j && i < n) L[i * ld + j] = acc[t] / ljj;
    }
    __syncwarp();
  }
  return true;
}

/* one env; sm holds qp_layout(q.n_max, q.nin_max).per_env doubles of this warp */
TSIDB_DEV void qp_env(const QpArgs& q, double* sm, int env, int lane) {
  const QpLayout Ly = qp_layout(q.n_max, q.nin_max);
  const int nm = q.n_max, ld = Ly.ld;
  int* smi = reinterpret_cast<int*>(sm + Ly.oI);
  QpEnv E;
  E.nm = nm; E.ld = ld;
  E.J = sm + Ly.oJ; E.R = sm + Ly.oR; E.x = sm + Ly.ox; E.xo = sm + Ly.oxo; E.d = sm + Ly.od; E.z = sm + Ly.oz;
  E.r = sm + Ly.or_; E.np = sm + Ly.onp; E.u = sm + Ly.ou; E.uo = sm + Ly.ouo; E.s = sm + Ly.os;
  E.A = smi + Ly.oA; E.Ao = smi + Ly.oAo; E.iai = smi + Ly.oiai; E.iax = smi + Ly.oix;
  __syncwarp(); /* every lane is done with the previous env's shared memory */
  const int n = q.sizes[(size_t)env * 3], neq = q.sizes[(size_t)env * 3 + 1], nin = q.sizes[(size_t)env * 3 + 2];
  E.n = n;
  int res = QP_REDUNDANT_EQ, iter = 0, iq = 0;
  const bool valid = n >= 1 && n <= nm && neq >= 0 && neq <= n && neq <= q.neq_max && nin >= 0 && nin <= q.nin_max;
  if (valid) {
    const double* H = q.H + (size_t)env * nm * nm;
    const double* g = q.g + (size_t)env * nm;
    const double* CE = q.CE + (size_t)env * q.neq_max * nm;
    const double* ce0 = q.ce0 + (size_t)env * q.neq_max;
    const double* CI = q.CI + (size_t)env * q.nin_max * nm;
    const double* ci0 = q.ci0 + (size_t)env * q.nin_max;
    double* J = E.J;
    double* R = E.R;
    double* L = E.R; /* the factor lives where R goes; R is cleared once J and x0 are formed */
    double c1 = 0.0, c2 = 0.0, R_norm = 1.0;
    int ip = 0, l = 0;
    double ss = 0.0;
    for (int i = 0; i < n; i++) c1 += H[(size_t)i * nm + i];
    if (!qp_llt(H, nm, L, ld, n, lane)) { res = QP_UNBOUNDED; goto done; }
    /* J = L^-T: L' J = I column by column, a lane per column */
    for (int c = lane; c < n; c += 32)
      for (int i = n - 1; i >= 0; i--) {
        double a = (i == c) ? 1.0 : 0.0;
        for (int k = i + 1; k < n; k++) a -= L[k * ld + i] * J[k * ld + c];
        J[i * ld + c] = a / L[i * ld + i];
      }
    __syncwarp();
    for (int i = 0; i < n; i++) c2 += J[i * ld + i];
    /* x = -H^-1 g: L y = g, then L' x = y, column-oriented */
    {
      double acc[QP_SLOTS];
#pragma unroll
      for (int t = 0; t < QP_SLOTS; t++) acc[t] = (lane + 32 * t < n) ? g[lane + 32 * t] : 0.0;
      for (int i = 0; i < n; i++) {
        const double yi = __shfl_sync(FULL, (i >> 5) ? acc[QP_SLOTS - 1] : acc[0], i & 31) / L[i * ld + i];
#pragma unroll
        for (int t = 0; t < QP_SLOTS; t++) {
          const int m = lane + 32 * t;
          if (m > i && m < n) acc[t] -= L[m * ld + i] * yi;
          else if (m == i) acc[t] = yi;
        }
      }
      for (int i = n - 1; i >= 0; i--) {
        const double xi = __shfl_sync(FULL, (i >> 5) ? acc[QP_SLOTS - 1] : acc[0], i & 31) / L[i * ld + i];
#pragma unroll
        for (int t = 0; t < QP_SLOTS; t++) {
          const int m = lane + 32 * t;
          if (m < i) acc[t] -= L[i * ld + m] * xi;
          else if (m == i) acc[t] = xi;
        }
      }
#pragma unroll
      for (int t = 0; t < QP_SLOTS; t++)
        if (lane + 32 * t < n) E.x[lane + 32 * t] = -acc[t];
    }
    __syncwarp();
    for (int k = lane; k < n * ld; k += 32) R[k] = 0.0;
    for (int k = lane; k < n; k += 32) E.d[k] = 0.0;
    __syncwarp();
    /* equality constraints, in row order */
    for (int i = 0; i < neq; i++) {
      for (int k = lane; k < n; k += 32) E.np[k] = CE[(size_t)i * nm + k];
      __syncwarp();
      qp_compute_d(E, lane);
      __syncwarp();
      qp_update_z(E, iq, lane);
      qp_update_r(E, iq, lane);
      double zz = 0.0, znp = 0.0, npx = 0.0;
      for (int k = lane; k < n; k += 32) { zz += E.z[k] * E.z[k]; znp += E.z[k] * E.np[k]; npx += E.np[k] * E.x[k]; }
      zz = warp_sum(zz); znp = warp_sum(znp); npx = warp_sum(npx);
      double t2 = 0.0;
      if (fabs(zz) > TS_EPS) t2 = (-npx - ce0[i]) / znp;
      for (int k = lane; k < n; k += 32) E.x[k] += t2 * E.z[k];
      for (int k = lane; k < iq; k += 32) E.u[k] -= t2 * E.r[k];
      if (lane == 0) { E.u[iq] = t2; E.A[i] = -i - 1; }
      __syncwarp();
      if (!qp_add_constraint(E, iq, R_norm, lane)) { res = QP_REDUNDANT_EQ; goto done; }
    }
    for (int i = lane; i < nin; i += 32) E.iai[i] = i;
    __syncwarp();

  l1:
    iter++;
    if (iter >= q.max_iter) { res = QP_MAX_ITER; goto done; }
    for (int i = neq + lane; i < iq; i += 32) E.iai[E.A[i]] = -1;
    ss = 0.0;
    ip = 0;
    {
      /* violation scan: a lane per row, streaming the row from global memory with the oracle's k order */
      double psi = 0.0;
      for (int i = lane; i < nin; i += 32) {
        const double* row = CI + (size_t)i * nm;
        double a = 0.0;
        for (int k = 0; k < n; k++) a += row[k] * E.x[k];
        const double si = a + ci0[i];
        E.s[i] = si;
        E.iax[i] = 1;
        psi += si < 0 ? si : 0.0;
      }
      psi = warp_sum(psi);
      __syncwarp();
      if (fabs(psi) <= nin * TS_EPS * c1 * c2 * 100.0) { res = QP_OPTIMAL; goto done; }
    }
    for (int i = lane; i < iq; i += 32) { E.uo[i] = E.u[i]; E.Ao[i] = E.A[i]; }
    for (int k = lane; k < n; k += 32) E.xo[k] = E.x[k];
    __syncwarp();

  l2:
    {
      double best = ss;
      int bi = -1;
      for (int i = lane; i < nin; i += 32)
        if (E.s[i] < best && E.iai[i] != -1 && E.iax[i]) { best = E.s[i]; bi = i; }
      warp_argmin(best, bi);
      if (bi >= 0) { ss = best; ip = bi; }
    }
    if (ss >= 0) { res = QP_OPTIMAL; goto done; }
    for (int k = lane; k < n; k += 32) E.np[k] = CI[(size_t)ip * nm + k];
    if (lane == 0) { E.u[iq] = 0.0; E.A[iq] = ip; }
    __syncwarp();

  l2a:
    {
      qp_compute_d(E, lane);
      __syncwarp();
      if (iq >= n) {
        for (int k = lane; k < n; k += 32) E.z[k] = 0.0;
      } else {
        qp_update_z(E, iq, lane);
      }
      qp_update_r(E, iq, lane);
      /* partial step length t1: the smallest u/r over the inequalities of the working set with r > 0, first on ties */
      double t1 = TS_INF;
      {
        int bk = -1;
        for (int k = neq + lane; k < iq; k += 32) {
          double tmp;
          if (E.r[k] > 0 && ((tmp = E.u[k] / E.r[k]) < t1)) { t1 = tmp; bk = k; }
        }
        warp_argmin(t1, bk);
        l = bk >= 0 ? E.A[bk] : 0;
      }
      double zz = 0.0, znp = 0.0;
      for (int k = lane; k < n; k += 32) { zz += E.z[k] * E.z[k]; znp += E.z[k] * E.np[k]; }
      zz = warp_sum(zz); znp = warp_sum(znp);
      const double t2 = (fabs(zz) > TS_EPS) ? -E.s[ip] / znp : TS_INF;
      const double t = t1 < t2 ? t1 : t2;
      if (t >= TS_INF) { res = QP_UNBOUNDED; goto done; }
      if (t2 >= TS_INF) {
        for (int k = lane; k < iq; k += 32) E.u[k] -= t * E.r[k];
        __syncwarp();
        if (lane == 0) { E.u[iq] += t; E.iai[l] = l; }
        __syncwarp();
        qp_delete_constraint(E, neq, iq, l, lane);
        goto l2a;
      }
      for (int k = lane; k < n; k += 32) E.x[k] += t * E.z[k];
      for (int k = lane; k < iq; k += 32) E.u[k] -= t * E.r[k];
      __syncwarp();
      if (lane == 0) E.u[iq] += t;
      __syncwarp();
      if (t == t2) {
        if (!qp_add_constraint(E, iq, R_norm, lane)) {
          if (lane == 0) E.iax[ip] = 0;
          __syncwarp();
          qp_delete_constraint(E, neq, iq, ip, lane);
          for (int i = lane; i < nin; i += 32) E.iai[i] = i;
          __syncwarp();
          if (lane == 0)
            for (int i = 0; i < iq; i++) {
              E.A[i] = E.Ao[i];
              if (E.A[i] >= 0) E.iai[E.A[i]] = -1;
              E.u[i] = E.uo[i];
            }
          for (int k = lane; k < n; k += 32) E.x[k] = E.xo[k];
          __syncwarp();
          goto l2;
        }
        if (lane == 0) E.iai[ip] = -1;
        __syncwarp();
        goto l1;
      }
      if (lane == 0) E.iai[l] = l;
      __syncwarp();
      qp_delete_constraint(E, neq, iq, l, lane);
      {
        double a = 0.0;
        for (int k = lane; k < n; k += 32) a += CI[(size_t)ip * nm + k] * E.x[k];
        a = warp_sum(a);
        if (lane == 0) E.s[ip] = a + ci0[ip];
        __syncwarp();
      }
      goto l2a;
    }
  }
done:
  __syncwarp();
  /* SolverHQuadProgFast's status mapping; the solution and the working set are reported for OPTIMAL and MAX_ITER */
  const int status = !valid ? ST_ERROR
                     : (res == QP_OPTIMAL ? ST_OPTIMAL
                        : (res == QP_MAX_ITER ? ST_MAX_ITER
                           : ((res == QP_UNBOUNDED || res == QP_INFEASIBLE) ? ST_INFEASIBLE : ST_ERROR)));
  const bool out = status == ST_OPTIMAL || status == ST_MAX_ITER;
  const int nw = out ? iq : 0, ne = out ? neq : 0, nx = out ? n : 0;
  if (lane == 0) {
    q.status[env] = status;
    if (q.iters) q.iters[env] = valid ? iter : 0;
  }
  for (int k = lane; k < nm; k += 32) {
    q.x[(size_t)env * nm + k] = k < nx ? E.x[k] : 0.0;
    if (q.active) q.active[(size_t)env * nm + k] = k < nw - ne ? E.A[ne + k] : -1;
    if (q.lambda) q.lambda[(size_t)env * nm + k] = k < nw - ne ? E.u[ne + k] : 0.0;
  }
  if (q.lambda_eq)
    for (int k = lane; k < q.neq_max; k += 32) q.lambda_eq[(size_t)env * q.neq_max + k] = k < ne ? E.u[k] : 0.0;
  if (q.tau)
    for (int r = lane; r < q.na; r += 32) {
      double a = 0.0;
      if (out) {
        const double* row = q.TA + ((size_t)env * q.na + r) * nm;
        for (int k = 0; k < n; k++) a += row[k] * E.x[k];
        a += q.ta0[(size_t)env * q.na + r];
      }
      q.tau[(size_t)env * q.na + r] = a;
    }
}

/* ================================================================= adjoint of the QP solve of one env (tsidb_qp_grad) */
/* At an OPTIMAL solution with working set W, x and nu = [lambda_eq; lambda_W] solve the KKT system of the rows
 * G = [CE; CI_W], b = [ce0; ci0_W]:  H x + g = G' nu,  G x + b = 0.  Its adjoint for incoming xb (+ TA' taub) and nub is
 *   H p + G' q = xb,  G p = -nub,
 * from which gb = -p, Gb = nu p' - q x', bb = -q, TAb = taub x', ta0b = taub and, since the solve reads only the lower
 * triangle of H, Hb = tril(P + P', -1) + diag(P) with P = -p x'.  The system is solved through the factors of the
 * forward: H = L L', M = L^-1 G' = [Q1 Q2] [R; 0] (Householder), y = L^-1 xb:
 *   p~ = Q2 Q2' y - Q1 R^-T nub,  q = R^-1 (Q1' y + R^-T nub),  p = L^-T p~
 * (no normal equations G H^-1 G', which would square the conditioning of the contact rows). */
struct QgLayout {
  int ld;                     /* row stride of L and M: odd, so column walks are conflict-free */
  int oL, oM, ox, op, oq, onu, obeta, ordiag; /* doubles */
  int oW, opos;               /* int32, from sm + oI */
  int oI, per_env;
};
TSIDB_HD inline QgLayout qg_layout(int n_max, int nin_max) {
  QgLayout L;
  L.ld = n_max | 1;
  L.oL = 0;
  L.oM = L.oL + n_max * L.ld;
  L.ox = L.oM + n_max * L.ld;
  L.op = L.ox + n_max;
  L.oq = L.op + n_max;
  L.onu = L.oq + n_max;
  L.obeta = L.onu + n_max;
  L.ordiag = L.obeta + n_max;
  L.oI = L.ordiag + n_max;
  L.oW = 0;
  L.opos = n_max;
  L.per_env = L.oI + (n_max + nin_max + 1) / 2;
  L.per_env += L.per_env & 1;
  return L;
}

/* out[r * nm + c] = f(r, c) for the rows x nm block: the warp stores 32 consecutive doubles at a time */
template <class F>
TSIDB_DEV void qg_store(double* out, int rows, int nm, int lane, F f) {
  if (rows <= 0 || nm <= 0) return;
  int r = 0, c = lane;
  while (c >= nm) { c -= nm; r++; }
  const long total = (long)rows * nm;
  for (long k = lane; k < total; k += 32) {
    out[k] = f(r, c);
    c += 32;
    while (c >= nm) { c -= nm; r++; }
  }
}

/* y = Q' y (fwd) or Q y for the Householder reflectors in the columns 0..m-1 of M; y in the lane-owned registers */
TSIDB_DEV void qg_reflect(const double* M, int ld, const double* beta, int n, int m, bool fwd, double (&y)[QP_SLOTS], int lane) {
  for (int s = 0; s < m; s++) {
    const int k = fwd ? s : m - 1 - s;
    double d = 0.0;
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int i = lane + 32 * t;
      if (i >= k && i < n) d += M[i * ld + k] * y[t];
    }
    d = warp_sum(d) * beta[k];
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int i = lane + 32 * t;
      if (i >= k && i < n) y[t] -= d * M[i * ld + k];
    }
  }
}

TSIDB_DEV double qg_lane(const double (&v)[QP_SLOTS], int i) { return __shfl_sync(FULL, (i >> 5) ? v[QP_SLOTS - 1] : v[0], i & 31); }

/* The factorisation of the working-set KKT system and the solve through it, shared by the adjoint of the QP solve
 * (qp_grad_env) and the forward derivative of the tick (tick_jvp_env), called in this order:
 *   qg_working_set, qp_llt, qg_fill_G, qg_lsolve_cols, qg_qr, then per right-hand side qg_lsolve and qg_kkt_solve. */
/* the working set of an env from the solve's `active` row: W[k] = the CI row of entry k, pos[r] = its entry or -1 for
 * r < nin; false unless the entries >= 0 are a -1 padded prefix of distinct rows of [0, nin) with neq + |W| <= n.
 * m = neq + |W| */
TSIDB_DEV bool qg_working_set(const int32_t* active, int n, int neq, int nin, int* W, int* pos, int& m, int lane) {
  int act[QP_SLOTS];
  bool bad = false;
  for (int r = lane; r < nin; r += 32) pos[r] = -1;
#pragma unroll
  for (int t = 0; t < QP_SLOTS; t++) {
    const int k = lane + 32 * t;
    act[t] = k < n ? active[k] : -1;
    bad |= act[t] < -1 || act[t] >= nin;
  }
  unsigned long long used = 0;
#pragma unroll
  for (int t = 0; t < QP_SLOTS; t++) used |= (unsigned long long)__ballot_sync(FULL, act[t] >= 0) << (32 * t);
  int w = 0;
  while (w < 64 && ((used >> w) & 1ull)) w++;
  bad |= (used & (used + 1)) != 0 || neq + w > n; /* the entries >= 0 are a prefix */
  __syncwarp();
#pragma unroll
  for (int t = 0; t < QP_SLOTS; t++)
    if (!bad && act[t] >= 0) {
      pos[act[t]] = lane + 32 * t;
      W[lane + 32 * t] = act[t];
    }
  __syncwarp();
#pragma unroll
  for (int t = 0; t < QP_SLOTS; t++) bad |= !bad && act[t] >= 0 && pos[act[t]] != lane + 32 * t; /* duplicate row */
  m = neq + w;
  return __ballot_sync(FULL, bad) == 0;
}
/* M = G' (row j of G = [CE; CI_W] into column j) */
TSIDB_DEV void qg_fill_G(const double* CE, const double* CI, const int* W, int nm, int n, int neq, int m, double* M, int ld,
                         int lane) {
  for (int j = 0; j < m; j++) {
    const double* row = j < neq ? CE + (size_t)j * nm : CI + (size_t)W[j - neq] * nm;
    for (int i = lane; i < n; i += 32) M[i * ld + j] = row[i];
  }
}
/* M = L^-1 M: forward substitution, a lane per column */
TSIDB_DEV void qg_lsolve_cols(const double* L, double* M, int ld, int n, int m, int lane) {
  for (int j = lane; j < m; j += 32)
    for (int i = 0; i < n; i++) {
      double s = M[i * ld + j];
      for (int k = 0; k < i; k++) s -= L[i * ld + k] * M[k * ld + j];
      M[i * ld + j] = s / L[i * ld + i];
    }
}
/* y = L^-1 y, column-oriented; y in the lane-owned registers */
TSIDB_DEV void qg_lsolve(const double* L, int ld, int n, double (&y)[QP_SLOTS], int lane) {
  for (int i = 0; i < n; i++) {
    const double yi = qg_lane(y, i) / L[i * ld + i];
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int k = lane + 32 * t;
      if (k > i && k < n) y[t] -= L[k * ld + i] * yi;
      else if (k == i) y[t] = yi;
    }
  }
}
/* Householder QR of M: reflector k in column k (rows k..n-1), R above the diagonal, its diagonal in rdiag.  A diagonal at
 * or below eps times the largest so far is a dependent row (the solve's own test in add_constraint): false. */
TSIDB_DEV bool qg_qr(double* M, int ld, double* beta, double* rdiag, int n, int m, int lane) {
  double R_norm = 1.0;
  for (int k = 0; k < m; k++) {
    double s2 = 0.0;
    for (int i = k + lane; i < n; i += 32) s2 += M[i * ld + k] * M[i * ld + k];
    s2 = warp_sum(s2);
    const double x0 = M[k * ld + k], nrm = sqrt(s2);
    const double alpha = x0 > 0 ? -nrm : nrm;
    if (!(nrm > TS_EPS * R_norm)) return false;
    if (nrm > R_norm) R_norm = nrm;
    const double bk = 1.0 / (nrm * (nrm + fabs(x0))); /* 2 / v'v */
    __syncwarp();
    if (lane == 0) { M[k * ld + k] = x0 - alpha; beta[k] = bk; rdiag[k] = alpha; }
    __syncwarp();
    for (int j = k + 1 + lane; j < m; j += 32) {
      double d = 0.0;
      for (int i = k; i < n; i++) d += M[i * ld + k] * M[i * ld + j];
      d *= bk;
      for (int i = k; i < n; i++) M[i * ld + j] -= d * M[i * ld + k];
    }
    __syncwarp();
  }
  return true;
}
/* H p + G' q = xb, G p = -nub through the factors, with y = L^-1 xb and v = nub on entry (lane-owned registers):
 *   p~ = Q2 Q2' y - Q1 R^-T nub,  q = R^-1 (Q1' y + R^-T nub),  p = L^-T p~;  p is left in y, q in u. */
TSIDB_DEV void qg_kkt_solve(const double* L, const double* M, int ld, const double* beta, const double* rdiag, int n, int m,
                            double (&y)[QP_SLOTS], double (&v)[QP_SLOTS], double (&u)[QP_SLOTS], int lane) {
  qg_reflect(M, ld, beta, n, m, true, y, lane); /* y = Q' L^-1 xb = [z1; z2] */
  /* v = R^-T nub, column-oriented forward substitution */
  for (int i = 0; i < m; i++) {
    const double vi = qg_lane(v, i) / rdiag[i];
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int j = lane + 32 * t;
      if (j > i && j < m) v[t] -= M[i * ld + j] * vi;
      else if (j == i) v[t] = vi;
    }
  }
  /* q = R^-1 (z1 + v), back substitution; then y = [-v; z2] */
#pragma unroll
  for (int t = 0; t < QP_SLOTS; t++) {
    const int j = lane + 32 * t;
    u[t] = j < m ? y[t] + v[t] : 0.0;
    if (j < m) y[t] = -v[t];
  }
  for (int i = m - 1; i >= 0; i--) {
    const double qi = qg_lane(u, i) / rdiag[i];
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int j = lane + 32 * t;
      if (j < i) u[t] -= M[j * ld + i] * qi;
      else if (j == i) u[t] = qi;
    }
  }
  qg_reflect(M, ld, beta, n, m, false, y, lane); /* p~ */
  /* p = L^-T p~, column-oriented back substitution */
  for (int i = n - 1; i >= 0; i--) {
    const double pi = qg_lane(y, i) / L[i * ld + i];
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int k = lane + 32 * t;
      if (k < i) y[t] -= L[i * ld + k] * pi;
      else if (k == i) y[t] = pi;
    }
  }
}

/* one env; sm holds qg_layout(a.n_max, a.nin_max).per_env doubles of this warp */
TSIDB_DEV void qp_grad_env(const QpGradArgs& a, double* sm, int env, int lane) {
  const QgLayout Ly = qg_layout(a.n_max, a.nin_max);
  const int nm = a.n_max, ld = Ly.ld, na = a.na;
  double *L = sm + Ly.oL, *M = sm + Ly.oM, *x = sm + Ly.ox, *p = sm + Ly.op, *q = sm + Ly.oq, *nu = sm + Ly.onu;
  double *beta = sm + Ly.obeta, *rdiag = sm + Ly.ordiag;
  int* W = reinterpret_cast<int*>(sm + Ly.oI) + Ly.oW;
  int* pos = reinterpret_cast<int*>(sm + Ly.oI) + Ly.opos;
  __syncwarp(); /* every lane is done with the previous env's shared memory */
  const int n = a.sizes[(size_t)env * 3], neq = a.sizes[(size_t)env * 3 + 1], nin = a.sizes[(size_t)env * 3 + 2];
  bool ok = a.sol_status[env] == ST_OPTIMAL && n >= 1 && n <= nm && neq >= 0 && neq <= n && neq <= a.neq_max && nin >= 0 &&
            nin <= a.nin_max;
  int m = 0;
  if (ok) ok = qg_working_set(a.active + (size_t)env * nm, n, neq, nin, W, pos, m, lane);
  const double* H = a.H + (size_t)env * nm * nm;
  if (ok) ok = qp_llt(H, nm, L, ld, n, lane);
  double y[QP_SLOTS], v[QP_SLOTS];
  if (ok) {
    /* M = G', x, nu, y = xb + TA' taub */
    qg_fill_G(a.CE + (size_t)env * a.neq_max * nm, a.CI + (size_t)env * a.nin_max * nm, W, nm, n, neq, m, M, ld, lane);
    for (int i = lane; i < n; i += 32) x[i] = a.x[(size_t)env * nm + i];
    for (int j = lane; j < m; j += 32) nu[j] = j < neq ? a.lambda_eq[(size_t)env * a.neq_max + j] : a.lambda[(size_t)env * nm + j - neq];
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int i = lane + 32 * t;
      double s = 0.0;
      if (i < n) {
        if (a.gx) s = a.gx[(size_t)env * nm + i];
        if (a.gtau)
          for (int r = 0; r < na; r++) s += a.TA[((size_t)env * na + r) * nm + i] * a.gtau[(size_t)env * na + r];
      }
      y[t] = s;
      const int j = i;
      v[t] = 0.0;
      if (j < neq && a.glambda_eq) v[t] = a.glambda_eq[(size_t)env * a.neq_max + j];
      else if (j >= neq && j < m && a.glambda) v[t] = a.glambda[(size_t)env * nm + j - neq];
    }
    __syncwarp();
    qg_lsolve_cols(L, M, ld, n, m, lane);
    qg_lsolve(L, ld, n, y, lane);
    __syncwarp();
    ok = qg_qr(M, ld, beta, rdiag, n, m, lane);
  }
  if (ok) {
    double u[QP_SLOTS];
    qg_kkt_solve(L, M, ld, beta, rdiag, n, m, y, v, u, lane);
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int k = lane + 32 * t;
      if (k < n) p[k] = y[t];
      if (k < m) q[k] = u[t];
    }
  }
  __syncwarp();
  /* every byte of every requested part; zeros outside the env's sizes and for an env that was not differentiated */
  if (lane == 0) a.status[env] = ok ? ST_OPTIMAL : ST_ERROR;
  const int nx = ok ? n : 0, ne = ok ? neq : 0, ni = ok ? nin : 0;
  if (a.dH)
    qg_store(a.dH + (size_t)env * nm * nm, nm, nm, lane, [&](int i, int j) {
      return (i < nx && j <= i) ? (j < i ? -(p[i] * x[j] + p[j] * x[i]) : -(p[i] * x[i])) : 0.0;
    });
  if (a.dg) qg_store(a.dg + (size_t)env * nm, 1, nm, lane, [&](int, int j) { return j < nx ? -p[j] : 0.0; });
  if (a.dCE)
    qg_store(a.dCE + (size_t)env * a.neq_max * nm, a.neq_max, nm, lane, [&](int r, int j) {
      return (r < ne && j < nx) ? nu[r] * p[j] - q[r] * x[j] : 0.0;
    });
  if (a.dce0) qg_store(a.dce0 + (size_t)env * a.neq_max, 1, a.neq_max, lane, [&](int, int r) { return r < ne ? -q[r] : 0.0; });
  if (a.dCI)
    qg_store(a.dCI + (size_t)env * a.nin_max * nm, a.nin_max, nm, lane, [&](int r, int j) {
      const int k = r < ni ? pos[r] : -1;
      return (k >= 0 && j < nx) ? nu[neq + k] * p[j] - q[neq + k] * x[j] : 0.0;
    });
  if (a.dci0)
    qg_store(a.dci0 + (size_t)env * a.nin_max, 1, a.nin_max, lane, [&](int, int r) {
      const int k = r < ni ? pos[r] : -1;
      return k >= 0 ? -q[neq + k] : 0.0;
    });
  const double* gt = (ok && a.gtau) ? a.gtau + (size_t)env * na : nullptr;
  if (a.dTA)
    qg_store(a.dTA + (size_t)env * na * nm, na, nm, lane, [&](int r, int j) { return (gt && j < nx) ? gt[r] * x[j] : 0.0; });
  if (a.dta0) qg_store(a.dta0 + (size_t)env * na, 1, na, lane, [&](int, int r) { return gt ? gt[r] : 0.0; });
}

/* ================================================================= forward derivative of export + solve (tsidb_tick_jvp) */
/* Per warp: the tangent workspace (K1_DUAL_SIZE Duals), this env's primal workspace (SM_PER_ENV doubles: q, v, the
 * references, K1 and K2 in double as the tick runs them) followed by the JV_* vectors below, and the KKT factors of
 * qg_layout(n_max, nin_max). */
#define JV_oJL SM_PER_ENV          /* the four SE3 laws' log6 Jacobians in (E 9, ep 3), 6 x 12 per lane 0..3        288 */
#define JV_oA (JV_oJL + 288)       /* a = [JF; Jcom; Ag] x_dv                                                         18 */
#define JV_oPHI (JV_oA + 18)       /* T f_s of the force slots (6 per slot)                                           12 */
#define JV_oNUD (JV_oPHI + 12)     /* multiplier of each dynamics row (M | -Jc^T) summed over CE and the actuation rows 32 */
#define JV_oNUJ (JV_oNUD + 32)     /* multiplier of each contact-motion (JF) row, by foot                              12 */
#define JV_oDQV (JV_oNUJ + 12)     /* per direction: dq (32), dv (32)                                                 64 */
#define JV_oDRF (JV_oDQV + 64)     /* per direction: the references' tangents at the RF_* offsets                    106 */
#define JV_oAD (JV_oDRF + 106)     /* per direction: [JF; Jcom; Ag]' x_dv (18), then JF' nu_dyn (12)                    30 */
#define JV_oBD (JV_oAD + 30)       /* per direction: the task right-hand sides' tangents at the BV_* offsets           64 */
#define JV_oDD (JV_oBD + 64)       /* per direction: (M | -Jc^T)' x of the dynamics rows (32), then nle' (32)           64 */
#define JV_oDK (JV_oDD + 64)       /* the G rows: kind (int, 64), index (int, 64), as 64 doubles; coefficient (64)     128 */
#define JV_oXD (JV_oDK + 128)      /* per direction: x' (64)                                                          64 */
#define JV_oM (JV_oXD + 64)        /* m = neq + |W| (int)                                                              2 */
#define JV_SIZE (JV_oM + 2)
#define JV_DUALS (2 * K1_DUAL_SIZE)
#define TSIDB_J_PER_WARP(n_max, nin_max) (JV_DUALS + JV_SIZE + qg_layout(n_max, nin_max).per_env)
static_assert((JV_DUALS % 2) == 0 && (JV_SIZE % 2) == 0, "every region starts 16-byte aligned");

/* One env of tsidb_tick_jvp.  q, v and the references are staged and K1 + K2 run in double (sm); the working-set KKT
 * system of sol is factored as tsidb_qp_grad factors it.  Then per direction: K1 in tangent arithmetic seeded with the
 * direction's q and v parts (skipped when both are zero), the right-hand sides
 *   r1 = -(H' x + g' - G'^T nu),  r2 = -(G' x + b')    (G = [CE; CI_W], b = [ce0; ci0_W], nu = [lambda_eq; lambda_W])
 * formed from the tangents of K1's outputs, the task right-hand sides and the references, never from a tangent of the
 * export, and H x' - G^T nu' = r1, G x' = r2 solved through the factors (qp_grad's system with xb = r1, nub = -r2);
 * tau' = TA' x + ta0' + TA x'.  The tangent covers the entries state_adjoint_env and refs_adjoint_env read; the rest of
 * the export (and whatever a caller appended) is constant. */
/* the per-env part: staging, K1 and K2, the factors and what every direction reuses; false (status 4, zero outputs
 * written) when the env is not differentiated.  Not inlined, like tick_jvp_dir: the tangent K1 between them then keeps
 * the registers to itself. */
template <int NV>
TSIDB_DEVNI bool tick_jvp_setup(const DevConst& C, const double* mdl, double* sm, double* qs, const TickArgs& a,
                                const JvpArgs& j, int env, int lane) {
  constexpr int nv = NV, na = NV - 6, nq = NV + 1;
  const double BIG = 1e10; /* the export's clip of the joint-bound rows */
  const QgLayout Ly = qg_layout(j.n_max, j.nin_max);
  const int nm = j.n_max, ld = Ly.ld, D = j.n_dirs;
  double *L = qs + Ly.oL, *M = qs + Ly.oM, *x = qs + Ly.ox, *nu = qs + Ly.onu, *beta = qs + Ly.obeta, *rdiag = qs + Ly.ordiag;
  int* W = reinterpret_cast<int*>(qs + Ly.oI) + Ly.oW;
  int* pos = reinterpret_cast<int*>(qs + Ly.oI) + Ly.opos;
  int* dkind = reinterpret_cast<int*>(sm + JV_oDK);
  int* didx = dkind + 64;
  double* dcoef = sm + JV_oDK + 64;
  __syncwarp(); /* every lane is done with the previous env's shared memory */
  if (lane < nq) sm[SM_oQV + lane] = ldin(a.q, a, env, lane, nq);
  if (lane < nv) sm[SM_oQV + 32 + lane] = ldin(a.v, a, env, lane, nv);
  stage_refs(C, mdl, sm, a, env, lane, na);
  __syncwarp();
  k1_dynamics<NV>(C, mdl, sm, lane);
  stage_refs_wait(sm, lane);
  const int mask = a.mask ? (a.mask[env] & 3) : 3;
  const int nc = (mask & 1) + ((mask >> 1) & 1);
  const int f0 = (mask & 1) ? 0 : 1; /* foot of force slot 0; slot 1 is RF */
  const int nx_e = nv + 12 * nc, neq_e = 6 + 6 * nc;
  const int nin_e = 2 * (17 * nc + (C.use_tb ? na : 0) + (C.use_jb ? nv : 0));
  const int oAct = 34 * nc; /* first actuation row of CI */
  k2_assemble<NV>(C, mdl, sm, a, env, lane, mask, neq_e, nx_e);

  /* the KKT factors of the final working set; the export's own rows and variables must be there */
  const int n = j.sizes[(size_t)env * 3], neq = j.sizes[(size_t)env * 3 + 1], nin = j.sizes[(size_t)env * 3 + 2];
  bool ok = j.sol_status[env] == ST_OPTIMAL && n >= nx_e && n <= nm && neq >= neq_e && neq <= n && neq <= j.neq_max &&
            nin >= nin_e && nin <= j.nin_max;
  int m = 0;
  if (ok) ok = qg_working_set(j.active + (size_t)env * nm, n, neq, nin, W, pos, m, lane);
  if (ok) ok = qp_llt(j.H + (size_t)env * nm * nm, nm, L, ld, n, lane);
  if (ok) {
    qg_fill_G(j.CE + (size_t)env * j.neq_max * nm, j.CI + (size_t)env * j.nin_max * nm, W, nm, n, neq, m, M, ld, lane);
    for (int i = lane; i < n; i += 32) x[i] = j.x[(size_t)env * nm + i];
    for (int k = lane; k < m; k += 32) nu[k] = k < neq ? j.lambda_eq[(size_t)env * j.neq_max + k] : j.lambda[(size_t)env * nm + k - neq];
    __syncwarp();
    qg_lsolve_cols(L, M, ld, n, m, lane);
    __syncwarp();
    ok = qg_qr(M, ld, beta, rdiag, n, m, lane);
  }
  if (lane == 0) j.status[env] = ok ? ST_OPTIMAL : ST_ERROR;
  if (!ok) { /* every byte of every requested output */
    for (int d = 0; d < D; d++) {
      if (j.ox) for (int k = lane; k < nm; k += 32) j.ox[((size_t)env * D + d) * nm + k] = 0.0;
      if (j.otau && lane < na) j.otau[((size_t)env * D + d) * na + lane] = 0.0;
    }
    return false;
  }

  /* once per env: the log6 Jacobians, a, T f, the multipliers of the dynamics and contact-motion rows, the G rows */
  const double* JF = sm + SM_oJF; /* [JF; Jcom; Ag]: 18 rows of stride TSIDB_NVX */
  const double* fr = sm + SM_oFr;
  const double* rf = sm + SM_oRef;
  if (lane < 4) {
    const int f = lane & 1;
    const bool is_contact = lane < 2;
    const double* ref = is_contact ? rf + RF_CONTACT + 12 * f : rf + RF_FOOT + 24 * f;
    const double* pf = fr + FR_OMF + f * 12;
    const double* Rf = pf + 3;
    double Rr[9], dp[3], E[9], ep[3];
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int q = 0; q < 3; q++) Rr[3 * q + c] = ref[3 + 3 * c + q];
    dp[0] = ref[0] - pf[0]; dp[1] = ref[1] - pf[1]; dp[2] = ref[2] - pf[2];
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
      for (int q = 0; q < 3; q++) E[3 * i + q] = Rf[i] * Rr[q] + Rf[3 + i] * Rr[3 + q] + Rf[6 + i] * Rr[6 + q];
    mtv3(Rf, dp, ep);
    double* JL = sm + JV_oJL + 72 * lane;
    for (int k = 0; k < 6; k++) { /* row k of d log6 / d(E, ep): the adjoint with a unit cotangent */
      double ol[3] = {0, 0, 0}, oa[3] = {0, 0, 0};
      if (k < 3) ol[k] = 1.0; else oa[k - 3] = 1.0;
      double* row = JL + 12 * k;
      for (int i = 0; i < 12; i++) row[i] = 0.0;
      log6_adj(E, ep, ol, oa, row, row + 9);
    }
  }
  if (lane < 18) {
    double s = 0.0;
    for (int k = 0; k < nv; k++) s += JF[lane * TSIDB_NVX + k] * x[k];
    sm[JV_oA + lane] = s;
  }
  if (lane < 12) {
    const int s = lane / 6, mm = lane % 6;
    double t = 0.0;
    if (s < nc)
      for (int k = 0; k < 12; k++) t += C.T[mm][k] * x[nv + 12 * s + k];
    sm[JV_oPHI + lane] = t;
    const int f = lane / 6; /* contact-motion row of foot f: 6 + 6 s + k with s its force slot */
    sm[JV_oNUJ + lane] = ((mask >> f) & 1) ? nu[6 + 6 * (f == f0 ? 0 : 1) + lane % 6] : 0.0;
  }
  if (lane < nv) {
    double t = 0.0;
    if (lane < 6) t = nu[lane];
    else if (C.use_tb) {
      const int lo = pos[oAct + lane - 6], up = pos[oAct + na + lane - 6];
      if (lo >= 0) t += nu[neq + lo];
      if (up >= 0) t -= nu[neq + up];
    }
    sm[JV_oNUD + lane] = t;
  }
  /* G rows: kind 1 = dynamics row idx with sign coef, 2 = contact-motion row (JF row idx), 3 = joint-bound row of
   * joint idx (coef = d ci0 / d v_idx), 0 = constant */
  for (int r = lane; r < m; r += 32) {
    int kind = 0, idx = 0;
    double coef = 0.0;
    if (r < neq) {
      if (r < 6) { kind = 1; idx = r; coef = 1.0; }
      else if (r < neq_e) { kind = 2; idx = (((r < 12) ? f0 : 1) * 6) + (r - 6) % 6; }
    } else if (W[r - neq] < nin_e) {
      int side = 0, i = 0, slot = 0;
      const int blk = ci_block(C, W[r - neq], nc, na, nv, side, i, slot);
      if (blk == 2) { kind = 1; idx = 6 + i; coef = side ? -1.0 : 1.0; }
      else if (blk == 3 && i >= 6) {
        const double vj = sm[SM_oQV + 32 + i];
        const double hi = (C.v_max[i - 6] - vj) / C.jb_dt, lo = (C.v_min[i - 6] - vj) / C.jb_dt;
        kind = 3; idx = i;
        coef = side ? (hi < BIG ? -1.0 / C.jb_dt : 0.0) : (lo > -BIG ? 1.0 / C.jb_dt : 0.0);
      }
    }
    dkind[r] = kind; didx[r] = idx; dcoef[r] = coef;
  }
  if (lane == 0) *reinterpret_cast<int*>(sm + JV_oM) = m;
  __syncwarp();
  return true;
}

/* one direction d after its tangents are staged in sm (and, when kin, the tangent K1 ran in ds): the right-hand sides,
 * the solve through the factors and the stores of x' and tau' */
template <int NV>
TSIDB_DEVNI void tick_jvp_dir(const DevConst& C, const double* mdl, const Dual* ds, double* sm, const double* qs,
                              const TickArgs& a, const JvpArgs& j, int env, int d, bool kin, int lane) {
  constexpr int nv = NV, na = NV - 6;
  const QgLayout Ly = qg_layout(j.n_max, j.nin_max);
  const int nm = j.n_max, ld = Ly.ld, D = j.n_dirs;
  const double *L = qs + Ly.oL, *M = qs + Ly.oM, *x = qs + Ly.ox, *beta = qs + Ly.obeta, *rdiag = qs + Ly.ordiag;
  const int* dkind = reinterpret_cast<const int*>(sm + JV_oDK);
  const int* didx = dkind + 64;
  const double* dcoef = sm + JV_oDK + 64;
  const int n = j.sizes[(size_t)env * 3], m = *reinterpret_cast<const int*>(sm + JV_oM);
  const int mask = a.mask ? (a.mask[env] & 3) : 3;
  const int nc = (mask & 1) + ((mask >> 1) & 1);
  const int f0 = (mask & 1) ? 0 : 1;
  const int nx_e = nv + 12 * nc;
  const double* JF = sm + SM_oJF;
  const double* fr = sm + SM_oFr;
  const double* rf = sm + SM_oRef;
  const double* TA = j.TA + (size_t)env * na * nm;
  const size_t row = j.shared ? (size_t)d : (size_t)env * D + d;
  for (int k = lane; k < RF_POST + na; k += 32) { /* the references' tangents */
    const double* p;
    int nd, i;
    if (k < RF_FOOT) { p = j.dref[0]; nd = 9; i = k; }
    else if (k < RF_CONTACT) { p = j.dref[1 + (k - RF_FOOT) / 24]; nd = 24; i = (k - RF_FOOT) % 24; }
    else if (k < RF_POST) { p = j.dref[3 + (k - RF_CONTACT) / 12]; nd = 12; i = (k - RF_CONTACT) % 12; }
    else { p = j.dref[5]; nd = na; i = k - RF_POST; }
    sm[JV_oDRF + k] = (p && i < nd) ? p[row * nd + i] : 0.0;
  }
  __syncwarp();
  {
    auto T = [&](int k) -> double { return kin ? ds[k].d : 0.0; }; /* tangent of K1's output at sm offset k */
    const double* dq = sm + JV_oDQV;
    const double* dvv = sm + JV_oDQV + 32;
    const double* drf = sm + JV_oDRF;
    /* the task right-hand sides' tangents (k2_assemble / se3_rhs) */
    double* bd = sm + JV_oBD;
    if (lane < 4) {
      const int f = lane & 1;
      const bool is_contact = lane < 2;
      double b6[6] = {0, 0, 0, 0, 0, 0};
      if (!is_contact || ((mask >> f) & 1)) {
        const int oref = is_contact ? RF_CONTACT + 12 * f : RF_FOOT + 24 * f;
        const double* ref = rf + oref;
        const double* rd = drf + oref;
        const double* gains = C.kp_contact + (is_contact ? 0 : 12);
        Dual Rf[9], pf[3], Rr[9], dp[3], E[9], ep[3];
#pragma unroll
        for (int k = 0; k < 3; k++) pf[k] = Dual(fr[FR_OMF + 12 * f + k], T(SM_oFr + FR_OMF + 12 * f + k));
#pragma unroll
        for (int k = 0; k < 9; k++) Rf[k] = Dual(fr[FR_OMF + 12 * f + 3 + k], T(SM_oFr + FR_OMF + 12 * f + 3 + k));
#pragma unroll
        for (int c = 0; c < 3; c++)
#pragma unroll
          for (int q = 0; q < 3; q++) Rr[3 * q + c] = Dual(ref[3 + 3 * c + q], rd[3 + 3 * c + q]);
#pragma unroll
        for (int k = 0; k < 3; k++) dp[k] = Dual(ref[k], rd[k]) - pf[k];
#pragma unroll
        for (int i = 0; i < 3; i++)
#pragma unroll
          for (int q = 0; q < 3; q++) E[3 * i + q] = Rf[i] * Rr[q] + Rf[3 + i] * Rr[3 + q] + Rf[6 + i] * Rr[6 + q];
        mtv3(Rf, dp, ep);
        const double* JL = sm + JV_oJL + 72 * lane;
        Dual vl[6], al[6];
        if (!is_contact) {
          Dual vr[6], ar[6];
#pragma unroll
          for (int k = 0; k < 6; k++) { vr[k] = Dual(ref[12 + k], rd[12 + k]); ar[k] = Dual(ref[18 + k], rd[18 + k]); }
          mtv3(Rf, vr, vl); mtv3(Rf, vr + 3, vl + 3);
          mtv3(Rf, ar, al); mtv3(Rf, ar + 3, al + 3);
        }
#pragma unroll
        for (int k = 0; k < 6; k++) {
          double pe = 0.0;
#pragma unroll
          for (int i = 0; i < 9; i++) pe += JL[12 * k + i] * E[i].d;
#pragma unroll
          for (int i = 0; i < 3; i++) pe += JL[12 * k + 9 + i] * ep[i].d;
          const double vF = T(SM_oFr + FR_VF + 6 * f + k), aF = T(SM_oFr + FR_AF + 6 * f + k);
          b6[k] = gains[k] * pe + gains[6 + k] * ((is_contact ? 0.0 : vl[k].d) - vF) + (is_contact ? 0.0 : al[k].d) - aF;
        }
      }
#pragma unroll
      for (int k = 0; k < 6; k++) bd[(is_contact ? BV_MOT : BV_FOOT) + 6 * f + k] = b6[k];
    } else if (lane < 7) {
      const int r = lane - 4;
      bd[BV_COM + r] = -C.kp_com[r] * (T(SM_oFr + FR_COM + r) - drf[RF_COM + r]) -
                       C.kd_com[r] * (T(SM_oFr + FR_COM + 3 + r) - drf[RF_COM + 3 + r]) + drf[RF_COM + 6 + r] -
                       T(SM_oFr + FR_COM + 6 + r);
    } else if (lane < 10) {
      const int r = lane - 7;
      bd[BV_AM + r] = -C.kp_am[r] * T(SM_oFr + FR_L + r) - T(SM_oFr + FR_L + 3 + r);
    }
    if (lane < na)
      bd[BV_POST + lane] = -mdl[MDL_oPOST + lane] * (dq[7 + lane] - drf[RF_POST + lane]) - mdl[MDL_oPOST + 23 + lane] * dvv[6 + lane];
    /* [JF; Jcom; Ag]' x_dv, JF' nu_dyn, (M | -Jc^T)' x and nle' of the dynamics rows */
    const double* nud = sm + JV_oNUD;
    if (lane < 18) {
      double s = 0.0;
      if (kin)
        for (int k = 0; k < nv; k++) s += ds[SM_oJF + lane * TSIDB_NVX + k].d * x[k];
      sm[JV_oAD + lane] = s;
    } else if (lane < 30) {
      double s = 0.0;
      if (kin)
        for (int k = 0; k < nv; k++) s += ds[SM_oJF + (lane - 18) * TSIDB_NVX + k].d * nud[k];
      sm[JV_oAD + lane] = s;
    }
    if (lane < nv) {
      double s = 0.0;
      if (kin) {
        for (int k = 0; k < nv; k++) s += ds[SM_oM + lane * SM_LDM + k].d * x[k];
        for (int sl = 0; sl < nc; sl++) {
          const int f = sl == 0 ? f0 : 1;
          for (int mm = 0; mm < 6; mm++) s -= ds[SM_oJF + (f * 6 + mm) * TSIDB_NVX + lane].d * sm[JV_oPHI + 6 * sl + mm];
        }
      }
      sm[JV_oDD + lane] = s;
      sm[JV_oDD + 32 + lane] = T(SM_oNle + lane);
    }
    __syncwarp();
    /* r1 into y (xb), -r2 into v (nub) */
    const double* ad = sm + JV_oAD;
    const double* bv = sm + SM_oBv;
    const double* dd = sm + JV_oDD;
    const double* nuj = sm + JV_oNUJ;
    double y[QP_SLOTS], v[QP_SLOTS], u[QP_SLOTS];
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int c = lane + 32 * t;
      double r1 = 0.0;
      if (c < nv) {
        double hx = 0.0, gd = 0.0, gt = 0.0;
        for (int q = 0; q < 18; q++) {
          const double w = q < 12 ? C.w_foot : (q < 15 ? C.w_com : (C.use_am ? C.w_am : 0.0));
          const double Jq = JF[q * TSIDB_NVX + c], Jd = T(SM_oJF + q * TSIDB_NVX + c);
          hx += w * (Jd * sm[JV_oA + q] + Jq * ad[q]);
          gd += w * (Jd * bv[BV_FOOT + q] + Jq * bd[BV_FOOT + q]);
        }
        gd = -gd - (c >= 6 ? C.w_post * bd[BV_POST + c - 6] : 0.0);
        if (kin) {
          for (int i = 0; i < nv; i++) gt += nud[i] * ds[SM_oM + i * SM_LDM + c].d;
          for (int q = 0; q < 12; q++) gt += nuj[q] * ds[SM_oJF + q * TSIDB_NVX + c].d;
        }
        r1 = -(hx + gd - gt);
      } else if (c < nx_e) {
        const int sl = (c - nv) / 12, k = (c - nv) % 12, f = sl == 0 ? f0 : 1;
        double s = 0.0;
        for (int mm = 0; mm < 6; mm++) s += C.T[mm][k] * ad[18 + f * 6 + mm];
        r1 = -s;
      }
      y[t] = r1;
      double r2 = 0.0;
      if (c < m) {
        const int kind = dkind[c], i = didx[c];
        if (kind == 1) r2 = -dcoef[c] * (dd[i] + dd[32 + i]);
        else if (kind == 2) r2 = -(ad[i] - bd[BV_MOT + i]);
        else if (kind == 3) r2 = -dcoef[c] * dvv[i];
      }
      v[t] = -r2;
    }
    qg_lsolve(L, ld, n, y, lane);
    qg_kkt_solve(L, M, ld, beta, rdiag, n, m, y, v, u, lane);
    double* xd = sm + JV_oXD;
#pragma unroll
    for (int t = 0; t < QP_SLOTS; t++) {
      const int c = lane + 32 * t;
      if (c < nm) {
        const double val = c < n ? y[t] : 0.0;
        xd[c] = val;
        if (j.ox) j.ox[((size_t)env * D + d) * nm + c] = val;
      }
    }
    __syncwarp();
    if (j.otau && lane < na) {
      double s = dd[6 + lane] + dd[32 + 6 + lane];
      for (int k = 0; k < n; k++) s += TA[(size_t)lane * nm + k] * xd[k];
      j.otau[((size_t)env * D + d) * na + lane] = s;
    }
  }
}

/* K1 in tangent arithmetic seeded with one direction's q and v parts (tq, tv: this lane's component) */
template <int NV>
TSIDB_DEVNI void tick_jvp_k1(const DevConst& C, const double* mdl, Dual* ds, const double* sm, double tq, double tv, int lane) {
  if (lane < NV + 1) ds[SM_oQV + lane] = Dual(sm[SM_oQV + lane], tq);
  if (lane < NV) ds[SM_oQV + 32 + lane] = Dual(sm[SM_oQV + 32 + lane], tv);
  __syncwarp();
  k1_dynamics<NV>(C, mdl, ds, lane);
}

/* One env of tsidb_tick_jvp: tick_jvp_setup, then per direction its tangents staged, the tangent K1 when the direction
 * has a q or v part, and tick_jvp_dir. */
template <int NV>
TSIDB_DEV void tick_jvp_env(const DevConst& C, const double* mdl, Dual* ds, double* sm, double* qs, const TickArgs& a,
                            const JvpArgs& j, int env, int lane) {
  constexpr int nv = NV, na = NV - 6, nq = NV + 1;
  if (!tick_jvp_setup<NV>(C, mdl, sm, qs, a, j, env, lane)) return;
  const int D = j.n_dirs;
#pragma unroll 1
  for (int d = 0; d < D; d++) {
    const size_t row = j.shared ? (size_t)d : (size_t)env * D + d;
    const double tq = (j.dq && lane < nq) ? j.dq[row * nq + lane] : 0.0;
    const double tv = (j.dv && lane < nv) ? j.dv[row * nv + lane] : 0.0;
    sm[JV_oDQV + lane] = tq;
    sm[JV_oDQV + 32 + lane] = tv;
    const bool kin = __ballot_sync(FULL, tq != 0.0 || tv != 0.0) != 0;
    if (kin) tick_jvp_k1<NV>(C, mdl, ds, sm, tq, tv, lane);
    __syncwarp();
    tick_jvp_dir<NV>(C, mdl, ds, sm, qs, a, j, env, d, kin, lane);
  }
}

#ifndef TSIDB_EMU
/* class sort: slots ordered double support, single support, flight, so that the warps of a CTA round in
 * kernel F have equal trip counts and kernel A starts with the longest jobs. */
/* once per handle: the lane-indexed constants, laid out as the kernels stage them */
__global__ void tsidb_tables_kernel(int slot, double* out) {
  const DevConst& C = g_const[slot];
  stage_model(C, out + TBL_oMDL, threadIdx.x, blockDim.x);
  for (int i = threadIdx.x; i < 144; i += blockDim.x) out[TBL_oLF + i] = C.Lfinv[i / 12][i % 12];
  if (threadIdx.x < 32) {
    LaneConst K;
    lane_const_init(C, K, threadIdx.x);
    double* t = out + TBL_oLANE + threadIdx.x;
    for (int j = 0; j < 12; j++) t[j * 32] = K.Trow[j];
    for (int j = 0; j < 3; j++) t[(12 + j) * 32] = K.fric[j];
    t[15 * 32] = K.tmin; t[16 * 32] = K.tmax; t[17 * 32] = K.vmin; t[18 * 32] = K.vmax;
  }
}

/* Class sort with a longest-first order inside each class: the key of an env is (class, bucket), the bucket being its
 * iteration count in the PREVIOUS tick of this handle (a.pred, 4 iterations per bucket, most iterations first; all envs
 * share bucket 0 when there is no previous tick or the hint is off).  The persistent CTAs of the per-class kernels draw
 * slots in this order, so the longest active-set solves of a class start first and the kernel's tail shrinks; the order
 * of the slots never changes a result (every env is an independent problem). */
#define TSIDB_NBUCKET 8
#define TSIDB_NKEY (3 * TSIDB_NBUCKET)
__global__ void tsidb_classify_kernel(int n_envs, const uint8_t* mask, const int32_t* pred, int32_t* cls_pos, int32_t* counts,
                                      int32_t* bins) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  int key = -1;
  if (env < n_envs) {
    const int m = mask ? (mask[env] & 3) : 3;
    const int cls = 2 - ((m & 1) + ((m >> 1) & 1)); /* 0: DS, 1: SS, 2: flight */
    int bucket = 0;
    if (pred) {
      const int it = pred[env] >> 2;
      bucket = TSIDB_NBUCKET - 1 - (it < 0 ? 0 : (it > TSIDB_NBUCKET - 1 ? TSIDB_NBUCKET - 1 : it));
    }
    key = cls * TSIDB_NBUCKET + bucket;
  }
  /* warp-aggregated: one atomic per warp and key (and one per class for the class sizes) instead of one per env */
  const unsigned peers = __match_any_sync(FULL, key);
  const int leader = __ffs(peers) - 1;
  int base = 0;
  if (key >= 0 && lane == leader) {
    base = atomicAdd(&bins[key], __popc(peers));
    atomicAdd(&counts[key / TSIDB_NBUCKET], __popc(peers));
  }
  base = __shfl_sync(FULL, base, leader);
  if (key >= 0) cls_pos[env] = (key << 26) | (base + __popc(peers & ((1u << lane) - 1u)));
}
__global__ void tsidb_permute_kernel(int n_envs, const int32_t* cls_pos, const int32_t* bins, int32_t* perm) {
  __shared__ int32_t start[TSIDB_NKEY];
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int k = 0; k < TSIDB_NKEY; k++) { start[k] = acc; acc += bins[k]; }
  }
  __syncthreads();
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n_envs) return;
  const int cp = cls_pos[env], key = cp >> 26, pos = cp & 0x03ffffff;
  perm[start[key] + pos] = env;
}

template <int NV>
__global__ void __launch_bounds__(32 * TSIDB_WARPS_PER_BLOCK, TSIDB_D_CTAS_PER_SM)
tsidb_dynamics_kernel(const TickArgs a) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* sm = smem + wid * SM_PER_ENV;
  const DevConst& C = g_const[a.slot];
  double* mdl = smem + TSIDB_WARPS_PER_BLOCK * SM_PER_ENV;
  load_table(mdl, a.tables + TBL_oMDL, MDL_SIZE, threadIdx.x, blockDim.x);
  __syncthreads();
  /* rounds: in every round the CTA's warps take consecutive slots and move through the phases together
   * (PHASE_SYNC).  A warp without a slot of its own in the last round repeats the last slot (it must reach
   * the barriers); it stores the same values again. */
  const int per_round = gridDim.x * TSIDB_WARPS_PER_BLOCK;
  const int rounds = (a.n_envs + per_round - 1) / per_round;
  auto slot_of = [&](int r) {
    const int s_ = (r * gridDim.x + blockIdx.x) * TSIDB_WARPS_PER_BLOCK + wid;
    return s_ < a.n_envs ? s_ : a.n_envs - 1;
  };
  int slot = slot_of(0);
  int env = a.perm ? a.perm[slot] : slot;
  for (int r = 0; r < rounds; r++) {
    /* the warp's next env: its q, v are prefetched while this one is computed (not in kinematics-only calls, which
     * stage no references and so have no copy group to ride on; they still move on to the next slot) */
    const bool more = r + 1 < rounds;
    const int slot_n = more ? slot_of(r + 1) : slot;
    const int env_n = more ? (a.perm ? a.perm[slot_n] : slot_n) : -1;
    dynamics_env<NV>(C, mdl, sm, a, env, slot, lane, r > 0 && !a.kin_only, a.kin_only ? -1 : env_n);
    slot = slot_n;
    env = env_n;
  }
  if (lane == 0) bulk_store_wait_read(); /* shared memory must outlive the bulk stores that read it */
}

/* slot range of contact class NC (2: double support, 1: single support, 0: flight) in the class-sorted slot
 * order; without a contact mask every env is in double support */
template <int NC>
TSIDB_DEV void class_range(const TickArgs& a, int& start, int& count) {
  if (!a.perm) { start = 0; count = (NC == 2) ? a.n_envs : 0; return; }
  const int c0 = a.counter[1], c1 = a.counter[2], c2 = a.counter[3];
  start = (NC == 2) ? 0 : ((NC == 1) ? c0 : c0 + c1);
  count = (NC == 2) ? c0 : ((NC == 1) ? c1 : c2);
}

/* One launch per contact class: every size of the elimination is a compile-time constant and the lighter classes
 * fit more warps per SM.  A CTA is ONE warp (WARPS of them resident per SM) that pulls slots from the work counter
 * of its class and exits when the class is drained: its shared memory and registers are free at once for the
 * CTAs of whichever kernel is ready next (another class, the next stage, the next chunk of a host call), so a
 * kernel's tail does not idle the SM. */
template <int NV, int NC, int WARPS>
__global__ void __launch_bounds__(32 * TSIDB_E_CTA_WARPS, WARPS / TSIDB_E_CTA_WARPS)
tsidb_eliminate_kernel(const TickArgs a) {
  static_assert(WARPS % TSIDB_E_CTA_WARPS == 0, "CTA width divides the resident warps");
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  typedef EL<NV, NC> LE;
  double* sm = smem + wid * LE::per_env;
  const DevConst& C = g_const[a.slot];
  int start, count;
  class_range<NC>(a, start, count);
  if (count <= 0) return;
  /* the CTA's copy of the constant Lf^-1 (read with lane-dependent indices) */
  double* lfinv_sm = smem + TSIDB_E_CTA_WARPS * LE::per_env;
  load_table(lfinv_sm, a.tables + TBL_oLF, 144, threadIdx.x, blockDim.x);
  __syncthreads();
  int* counter = a.counter + 8 + NC;
  int k = 0;
  if (lane == 0) k = atomicAdd(counter, 1);
  k = __shfl_sync(FULL, k, 0);
  if (k >= count) return;
  if (lane == 0) mbar_init(sm + LE::oBar, 1);
  __syncwarp();
  unsigned parity = 0;
  while (k < count) {
    int kn = 0;
    if (lane == 0) kn = atomicAdd(counter, 1);
    kn = __shfl_sync(FULL, kn, 0);
    if (kn < count && lane == 0) bulk_prefetch_l2(a.ws3 + (size_t)(start + kn) * SE_IMAGE, SE_IMAGE * sizeof(double));
    eliminate_env<NV, NC>(C, lfinv_sm, sm, a, start + k, lane, parity);
    k = kn;
  }
}

/* one launch per contact class (sizes, strides and the shared-memory layout are compile-time; the lighter
 * classes fit more warps per SM); one-warp CTAs, each class pulls its slots from a work counter of its own because
 * the iteration counts vary from 1 to ~40 */
template <int NV, int NC, int WARPS>
__global__ void __launch_bounds__(32 * TSIDB_A_CTA_WARPS(NC), WARPS / TSIDB_A_CTA_WARPS(NC))
tsidb_activeset_kernel(const TickArgs a) {
  static_assert(WARPS % TSIDB_A_CTA_WARPS(NC) == 0, "CTA width divides the resident warps");
  extern __shared__ double smem[];
  typedef AL<NV, NC> LA;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* sm = smem + wid * LA::per_env;
  const DevConst& C = g_const[a.slot];
  int start, count;
  class_range<NC>(a, start, count);
  int* counter = a.counter + ((NC == 2) ? 0 : ((NC == 1) ? 4 : 5));
  /* the warp draws its next slot before it works on the current one, so that the next solver image can be pulled
   * into L2 and its env index read while the current env is being solved */
  int k = 0;
  if (lane == 0) k = atomicAdd(counter, 1);
  k = __shfl_sync(FULL, k, 0);
  if (k >= count) return;
  if (lane == 0) mbar_init(sm + LA::oBar, 1);
  __syncwarp();
  LaneConst K;
  lane_const_load(a.tables, K, lane);
  unsigned parity = 0;
  int env = a.perm ? a.perm[start + k] : start + k;
  while (k < count) {
    int kn = 0;
    if (lane == 0) kn = atomicAdd(counter, 1);
    kn = __shfl_sync(FULL, kn, 0);
    int envn = 0;
    if (kn < count) {
      if (lane == 0) bulk_prefetch_l2(a.ws + (size_t)(start + kn) * SA_IMAGE, LA::image * sizeof(double));
      envn = a.perm ? a.perm[start + kn] : start + kn;
    }
    activeset_env<NV, NC>(C, K, sm, a, env, start + k, lane, parity);
    k = kn;
    env = envn;
  }
}

/* QP export (tsidb_problem_data), after the dynamics kernel ran with slot == env: one warp per env on a persistent grid.
 * It is bound by its HBM writes (~93 KB per double-support robot/v1 env), so it does nothing but form and store rows. */
#define TSIDB_P_CTA_WARPS 4
#define TSIDB_P_CTAS_PER_SM 2
#define TSIDB_P_SMEM(NV) (((size_t)PT_SIZE + (size_t)TSIDB_P_CTA_WARPS * PB<NV>::per_env) * sizeof(double))
template <int NV>
__global__ void __launch_bounds__(32 * TSIDB_P_CTA_WARPS, TSIDB_P_CTAS_PER_SM)
tsidb_problem_kernel(const TickArgs a, const ProblemOut o) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* pt = smem;
  double* sm = smem + PT_SIZE + wid * PB<NV>::per_env;
  load_table(pt, a.tables + TBL_oPROB, PT_SIZE, threadIdx.x, blockDim.x);
  __syncthreads();
  const DevConst& C = g_const[a.slot];
  for (int env = blockIdx.x * TSIDB_P_CTA_WARPS + wid; env < a.n_envs; env += gridDim.x * TSIDB_P_CTA_WARPS)
    problem_env<NV>(C, pt, sm, a, o, env, lane);
}

/* Generic QP solve (tsidb_qp_solve): one one-warp CTA per env on a persistent grid.  The dynamic shared memory is
 * qp_layout(n_max, nin_max).per_env doubles, so the resident CTAs per SM follow from the call's strides. */
#define TSIDB_Q_MIN_CTAS 16 /* register cap: 128 per thread */
__global__ void __launch_bounds__(32, TSIDB_Q_MIN_CTAS) tsidb_qp_kernel(const QpArgs q) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31;
  for (int env = blockIdx.x; env < q.n_envs; env += gridDim.x) qp_env(q, smem, env, lane);
}

/* Adjoint of the generic QP solve (tsidb_qp_grad): one one-warp CTA per env on a persistent grid, dynamic shared memory
 * qg_layout(n_max, nin_max).per_env doubles (L and M, n_max x odd stride each, plus vectors). */
#define TSIDB_QG_MIN_CTAS 16 /* register cap: 128 per thread */
__global__ void __launch_bounds__(32, TSIDB_QG_MIN_CTAS) tsidb_qp_grad_kernel(const QpGradArgs a) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31;
  for (int env = blockIdx.x; env < a.n_envs; env += gridDim.x) qp_grad_env(a, smem, env, lane);
}

/* Adjoint of the reference terms (tsidb_refs_grad): the dynamics kernel's per-env shared memory and a CTA of warps sharing
 * the staged model table, one warp per env on a persistent grid, no images and no class sort.  12 warps per CTA and one
 * CTA per SM leave 168 registers per thread, which K1 followed by the adjoint needs to stay within the dynamics kernel's
 * spills (at 16 warps and 128 registers it spilled 688 bytes). */
#define TSIDB_R_CTA_WARPS 12
#define TSIDB_R_SMEM (((size_t)TSIDB_R_CTA_WARPS * SM_PER_ENV + MDL_SIZE) * sizeof(double))
template <int NV>
__global__ void __launch_bounds__(32 * TSIDB_R_CTA_WARPS, 1)
tsidb_refs_grad_kernel(const TickArgs a, const RefsGradArgs r) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* sm = smem + wid * SM_PER_ENV;
  const DevConst& C = g_const[a.slot];
  double* mdl = smem + TSIDB_R_CTA_WARPS * SM_PER_ENV;
  load_table(mdl, a.tables + TBL_oMDL, MDL_SIZE, threadIdx.x, blockDim.x);
  __syncthreads();
  for (int env = blockIdx.x * TSIDB_R_CTA_WARPS + wid; env < a.n_envs; env += gridDim.x * TSIDB_R_CTA_WARPS)
    refs_grad_env<NV>(C, mdl, sm, a, r, env, lane);
}

/* Adjoint of the export in the gains and weights (tsidb_gains_grad): shaped like the references' adjoint, one warp per
 * env on a persistent grid, 12-warp CTAs sharing the staged model table, one CTA per SM. */
#define TSIDB_G_CTA_WARPS 12
#define TSIDB_G_SMEM (((size_t)TSIDB_G_CTA_WARPS * SM_PER_ENV + MDL_SIZE) * sizeof(double))
template <int NV>
__global__ void __launch_bounds__(32 * TSIDB_G_CTA_WARPS, 1)
tsidb_gains_grad_kernel(const TickArgs a, const GainsGradArgs r) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* sm = smem + wid * SM_PER_ENV;
  const DevConst& C = g_const[a.slot];
  double* mdl = smem + TSIDB_G_CTA_WARPS * SM_PER_ENV;
  load_table(mdl, a.tables + TBL_oMDL, MDL_SIZE, threadIdx.x, blockDim.x);
  __syncthreads();
  for (int env = blockIdx.x * TSIDB_G_CTA_WARPS + wid; env < a.n_envs; env += gridDim.x * TSIDB_G_CTA_WARPS)
    gains_grad_env<NV>(C, mdl, sm, a, r, env, lane);
}

/* Adjoint of the export in q and v (tsidb_state_grad): one warp per env on a persistent grid, the CTA's warps sharing the
 * staged model table.  Per warp: the tangent workspace (K1_DUAL_SIZE Duals), whose start the double K1 and K2 use as
 * the dynamics kernel's env workspace, and the cotangents (SM_oRef doubles): 48 KB.  4 warps and one CTA per SM leave
 * 255 registers per thread, which the tangent K1 needs to stay within the dynamics kernel's spills. */
#define TSIDB_S_CTA_WARPS 4
#define TSIDB_S_PER_WARP (2 * K1_DUAL_SIZE + SM_oRef)
#define TSIDB_S_SMEM (((size_t)TSIDB_S_CTA_WARPS * TSIDB_S_PER_WARP + MDL_SIZE) * sizeof(double))
static_assert(2 * SM_oRef >= SM_PER_ENV && (TSIDB_S_PER_WARP % 2) == 0, "the env workspace fits the Dual view, 16-byte aligned");
template <int NV>
__global__ void __launch_bounds__(32 * TSIDB_S_CTA_WARPS, 1)
tsidb_state_grad_kernel(const TickArgs a, const StateGradArgs r) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* sm = smem + wid * TSIDB_S_PER_WARP;
  const DevConst& C = g_const[a.slot];
  double* mdl = smem + TSIDB_S_CTA_WARPS * TSIDB_S_PER_WARP;
  load_table(mdl, a.tables + TBL_oMDL, MDL_SIZE, threadIdx.x, blockDim.x);
  __syncthreads();
  for (int env = blockIdx.x * TSIDB_S_CTA_WARPS + wid; env < a.n_envs; env += gridDim.x * TSIDB_S_CTA_WARPS)
    state_grad_env<NV>(C, mdl, sm, sm + 2 * K1_DUAL_SIZE, a, r, env, lane);
}

/* Forward derivative of export + solve (tsidb_tick_jvp): one warp per env on a persistent grid, the CTA's warps sharing the
 * staged model table.  Per warp TSIDB_J_PER_WARP(n_max, nin_max) doubles of dynamic shared memory (tick_jvp_env): 101 KB
 * at the export's strides for robot/v1, so a CTA holds two warps and one CTA runs per SM; the host picks the warps per CTA
 * (up to TSIDB_J_MAX_WARPS) that fit the call's strides. */
#define TSIDB_J_MAX_WARPS 2
template <int NV>
__global__ void __launch_bounds__(32 * TSIDB_J_MAX_WARPS, 1)
tsidb_tick_jvp_kernel(const TickArgs a, const JvpArgs j) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, warps = blockDim.x >> 5;
  const int per_warp = TSIDB_J_PER_WARP(j.n_max, j.nin_max);
  double* w = smem + (size_t)wid * per_warp;
  const DevConst& C = g_const[a.slot];
  double* mdl = smem + (size_t)warps * per_warp;
  load_table(mdl, a.tables + TBL_oMDL, MDL_SIZE, threadIdx.x, blockDim.x);
  __syncthreads();
  for (int env = blockIdx.x * warps + wid; env < a.n_envs; env += gridDim.x * warps)
    tick_jvp_env<NV>(C, mdl, reinterpret_cast<Dual*>(w), w + JV_DUALS, w + JV_DUALS + JV_SIZE, a, j, env, lane);
}

/* ---- Small batches: the whole tick of one env in ONE launch ----
 * A CTA is one warp and takes one env through the three stages back to back (dynamics + assembly, elimination + basis,
 * active set + decode), branching on the env's contact class on the device: no class sort, no work counters, no
 * per-class launches, no launch gaps — a single robot's tick (the reference's operating point, ref:main.py:110-128)
 * is bound by the dependent chain (and the instruction fetch) of its ~12 k instructions; nine launches added a third.
 * The stage functions are the ones the batched kernels call.  !LOCAL: the hand-off images travel through global memory
 * (L2), so between the stages the warp orders its generic-proxy stores and completed bulk stores ahead of the next
 * stage's bulk (async-proxy) load (stage_handoff).  LOCAL: they stay in shared memory, see below. */
TSIDB_DEV void stage_handoff(int lane) {
  if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); /* bulk stores complete, not just read */
  __threadfence();
  asm volatile("fence.proxy.async;" ::: "memory");
  __syncwarp();
}
#define TSIDB_SMALL_SMEM_DOUBLES(NV)                                                                                     \
  ((a_layout(NV, 2).per_env > e_per_env(NV, 2) + 144 ? a_layout(NV, 2).per_env : e_per_env(NV, 2) + 144) > SM_PER_ENV + MDL_SIZE \
       ? (a_layout(NV, 2).per_env > e_per_env(NV, 2) + 144 ? a_layout(NV, 2).per_env : e_per_env(NV, 2) + 144)         \
       : SM_PER_ENV + MDL_SIZE)
/* LOCAL variant: the three stages own disjoint shared-memory regions (dynamics | elimination + Lf^-1 | active set); the
 * dynamics stage writes the assembly image into the elimination's region and its part of the solver image into the
 * active set's, the elimination adds x0 and the basis, and each stage works on its image IN PLACE: no store drain, no
 * fence, no bulk load between the stages.  70 KB per env instead of 27, so the host uses it for the smallest batches
 * only (TSIDB_SMALL_LOCAL_N). */
#define TSIDB_SMALL_oE(NV) (even_up(SM_PER_ENV + MDL_SIZE))
#define TSIDB_SMALL_oA(NV) (TSIDB_SMALL_oE(NV) + even_up(e_per_env(NV, 2) + 144))
#define TSIDB_SMALL_LOCAL_SMEM_DOUBLES(NV) (TSIDB_SMALL_oA(NV) + even_up(a_layout(NV, 2).per_env))
template <int NV, bool LOCAL>
__global__ void __launch_bounds__(32, 1) tsidb_tick_small_kernel(const TickArgs a_in) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x;
  const int env = blockIdx.x; /* slot == env: no class sort */
  const DevConst& C = g_const[a_in.slot];
  double* smE = LOCAL ? smem + TSIDB_SMALL_oE(NV) : smem;
  double* smA = LOCAL ? smem + TSIDB_SMALL_oA(NV) : smem;
  TickArgs a = a_in;
  if (LOCAL) { a.ws = smA; a.ws3 = smE; }
  const int slot = LOCAL ? 0 : env;
#if TSIDB_SMALL_PROFILE
  /* clock stamps of the stages of env 0 (tools/small_profile.py reads them back through tsidb_debug_terms) */
  long long stamp[8];
  int n_stamp = 0;
#define TSIDB_STAMP() do { __syncwarp(); stamp[n_stamp++] = clock64(); } while (0)
#else
#define TSIDB_STAMP() ((void)0)
#endif
  TSIDB_STAMP();
  {
    double* mdl = smem + SM_PER_ENV;
    load_table(mdl, a.tables + TBL_oMDL, MDL_SIZE, lane, 32);
    __syncwarp();
    TSIDB_STAMP();
    dynamics_env<NV, LOCAL>(C, mdl, smem, a, env, slot, lane);
  }
  if (LOCAL) __syncwarp(); else stage_handoff(lane);
  TSIDB_STAMP();
  const int mask = a.mask ? (a.mask[env] & 3) : 3;
  const int nc = (mask & 1) + ((mask >> 1) & 1);
  {
    double* lfinv_sm = smE + e_per_env(NV, 2);
    load_table(lfinv_sm, a.tables + TBL_oLF, 144, lane, 32);
    TSIDB_STAMP();
    unsigned parity = 0;
#define TSIDB_SMALL_E(NC_)                                                                 \
  {                                                                                          \
    double* bar = smE + EL<NV, NC_>::oBar;                                                   \
    if (!LOCAL && lane == 0) mbar_init(bar, 1);                                              \
    __syncwarp();                                                                            \
    eliminate_env<NV, NC_, LOCAL>(C, lfinv_sm, smE, a, slot, lane, parity);                  \
    if (!LOCAL && lane == 0) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory"); \
  }
    if (nc == 2) TSIDB_SMALL_E(2) else if (nc == 1) TSIDB_SMALL_E(1) else TSIDB_SMALL_E(0)
#undef TSIDB_SMALL_E
  }
  if (LOCAL) __syncwarp(); else stage_handoff(lane);
  TSIDB_STAMP();
  {
    LaneConst K;
    lane_const_load(a.tables, K, lane);
    TSIDB_STAMP();
    unsigned parity = 0;
#define TSIDB_SMALL_A(NC_)                                                                 \
  {                                                                                          \
    double* bar = smA + AL<NV, NC_>::oBar;                                                   \
    if (!LOCAL && lane == 0) mbar_init(bar, 1);                                              \
    __syncwarp();                                                                            \
    activeset_env<NV, NC_, LOCAL>(C, K, smA, a, env, slot, lane, parity);                    \
  }
    if (nc == 2) TSIDB_SMALL_A(2) else if (nc == 1) TSIDB_SMALL_A(1) else TSIDB_SMALL_A(0)
#undef TSIDB_SMALL_A
  }
  TSIDB_STAMP();
#if TSIDB_SMALL_PROFILE
  if (env == 0 && lane == 0)
    for (int k = 0; k < n_stamp; k++) a_in.ws3[k] = (double)(stamp[k] - stamp[0]);
#endif
#undef TSIDB_STAMP
}
#endif

#endif /* TSIDB_KERNELS_CUH_ */
