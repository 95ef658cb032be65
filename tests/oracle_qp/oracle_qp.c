/* oracle_qp.c — the CPU oracle's eiquadprog-fast (eq_solve of oracle/tsid_oracle.c) on a caller-supplied dense problem.
 * Test infrastructure (tests/oracle_qp.py): the oracle's source is compiled in as it stands, so the generic QP kernel is
 * checked against the very solver the tick's parity tests use. */
#include "../../oracle/tsid_oracle.c"

/* min 1/2 x'Hx + g'x s.t. CE x + ce0 = 0, CI x + ci0 >= 0 with dense, unpadded row-major arrays.  Returns the
 * TSIDB_STATUS_* oracle_tick reports for the same solver result, or -1 for sizes beyond the oracle's NMAX, NEQMAX and
 * NINMAX.  x [n], active [n] (CI rows of the working set in working-set order, -1 padded), lambda [n] (their
 * multipliers), lambda_eq [neq] are written for OPTIMAL and MAX_ITER_REACHED and zero (active -1) otherwise. */
int oracle_qp_solve(int n, int neq, int nin, const double* H, const double* g, const double* CE, const double* ce0,
                    const double* CI, const double* ci0, int max_iter, double* x, int* iters, int* active, double* lambda,
                    double* lambda_eq) {
  if (n < 1 || n > NMAX || neq < 0 || neq > NEQMAX || neq > n || nin < 0 || nin > NINMAX) return -1;
  qp_t* P = (qp_t*)calloc(1, sizeof(qp_t));
  eq_ws* w = (eq_ws*)malloc(sizeof(eq_ws));
  if (!P || !w) { free(P); free(w); return -1; }
  P->n = n; P->neq = neq; P->nin = nin;
  for (int i = 0; i < n * n; i++) P->H[i] = H[i];
  for (int i = 0; i < n; i++) P->g[i] = g[i];
  for (int i = 0; i < neq * n; i++) P->CE[i] = CE[i];
  for (int i = 0; i < neq; i++) P->ce0[i] = ce0[i];
  for (int i = 0; i < nin * n; i++) P->CI[i] = CI[i];
  for (int i = 0; i < nin; i++) P->ci0[i] = ci0[i];
  real xr[NMAX], u[NMAX + NEQMAX + 1];
  int A[NMAX + NEQMAX + 1], q = 0;
  const int st = eq_solve(P, max_iter, w, xr, iters, &q, u, A);
  int status;
  switch (st) { /* as oracle_tick maps it */
    case EQ_OPTIMAL: status = TSIDB_STATUS_OPTIMAL; break;
    case EQ_UNBOUNDED: status = TSIDB_STATUS_INFEASIBLE; break;
    case EQ_INFEASIBLE: status = TSIDB_STATUS_INFEASIBLE; break;
    case EQ_MAX_ITER: status = TSIDB_STATUS_MAX_ITER_REACHED; break;
    default: status = TSIDB_STATUS_ERROR; break;
  }
  const int out = st == EQ_OPTIMAL || st == EQ_MAX_ITER;
  for (int i = 0; i < n; i++) {
    x[i] = out ? (double)xr[i] : 0.0;
    active[i] = (out && neq + i < q) ? A[neq + i] : -1;
    lambda[i] = (out && neq + i < q) ? (double)u[neq + i] : 0.0;
  }
  for (int i = 0; i < neq; i++) lambda_eq[i] = out ? (double)u[i] : 0.0;
  free(P);
  free(w);
  return status;
}
