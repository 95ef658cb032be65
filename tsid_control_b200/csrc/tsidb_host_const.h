/* tsidb_host_const.h — host-side derivation of the per-handle constant block from the
 * C-ABI model/conf structs (include/tsidb.h).  Plain C++, no CUDA: used by tsidb.cu and by
 * the host emulation build under tests/emu.                                              */
#ifndef TSIDB_HOST_CONST_H_
#define TSIDB_HOST_CONST_H_
#include <math.h>
#include <string.h>

#include <string>

#include "../../include/tsidb.h"
#include "tsidb_const.h"

/* Gram matrix of the force regularisation, (W T)^T (W T): the derivative of the force block in w_force_reg */
static inline void tsidb_force_gram(const tsidb_conf* c, const double (*T)[12], double (*G)[12]) {
  for (int i = 0; i < 12; i++)
    for (int j = 0; j < 12; j++) {
      double s = 0.0;
      for (int r = 0; r < 6; r++) {
        const double wr = c->force_reg_weights[r];
        s += (wr * T[r][i]) * (wr * T[r][j]);
      }
      G[i][j] = s;
    }
}

/* force block of the Hessian, identical for every env and foot: w_freg (W T)^T (W T) + hreg I */
static inline void tsidb_force_hessian(const tsidb_conf* c, const double (*T)[12], double (*Hf)[12]) {
  double G[12][12];
  tsidb_force_gram(c, T, G);
  for (int i = 0; i < 12; i++)
    for (int j = 0; j < 12; j++) Hf[i][j] = c->w_force_reg * G[i][j] + (i == j ? c->hessian_reg : 0.0);
}

/* the force block's factor Lf, its inverse and the traces of DevConst from c and D->T (tsidb_create and tsidb_set_gains
 * both come here, so the two produce the same bits); false, D untouched: the block is not positive definite */
static inline bool tsidb_factor_force_block(const tsidb_conf* c, DevConst* D, std::string* err) {
  double Hf[12][12], Lf[12][12], Lfinv[12][12];
  memset(Lf, 0, sizeof Lf);
  memset(Lfinv, 0, sizeof Lfinv);
  tsidb_force_hessian(c, D->T, Hf);
  double Hf_trace = 0.0;
  for (int i = 0; i < 12; i++) Hf_trace += Hf[i][i];
  for (int j = 0; j < 12; j++) {
    double s = Hf[j][j];
    for (int k = 0; k < j; k++) s -= Lf[j][k] * Lf[j][k];
    if (!(s > 0.0)) { *err = "conf: force block of the Hessian is not positive definite"; return false; }
    Lf[j][j] = sqrt(s);
    for (int i = j + 1; i < 12; i++) {
      double t = Hf[i][j];
      for (int k = 0; k < j; k++) t -= Lf[i][k] * Lf[j][k];
      Lf[i][j] = t / Lf[j][j];
    }
  }
  /* inverse of the lower factor, column by column */
  for (int cidx = 0; cidx < 12; cidx++)
    for (int i = 0; i < 12; i++) {
      double s = (i == cidx) ? 1.0 : 0.0;
      for (int k = 0; k < i; k++) s -= Lf[i][k] * Lfinv[k][cidx];
      Lfinv[i][cidx] = s / Lf[i][i];
    }
  double Lfinv_trace = 0.0;
  for (int i = 0; i < 12; i++) Lfinv_trace += Lfinv[i][i];
  memcpy(D->Lf, Lf, sizeof Lf);
  memcpy(D->Lfinv, Lfinv, sizeof Lfinv);
  D->Hf_trace = Hf_trace;
  D->Lfinv_trace = Lfinv_trace;
  return true;
}

/* tsidb_gains <-> the gain and weight fields of tsidb_conf and DevConst */
static inline void tsidb_gains_of_conf(const tsidb_conf* c, tsidb_gains* g) {
  memcpy(g->kp_contact, c->kp_contact, sizeof g->kp_contact);
  memcpy(g->kd_contact, c->kd_contact, sizeof g->kd_contact);
  memcpy(g->kp_foot, c->kp_foot, sizeof g->kp_foot);
  memcpy(g->kd_foot, c->kd_foot, sizeof g->kd_foot);
  memcpy(g->kp_com, c->kp_com, sizeof g->kp_com);
  memcpy(g->kd_com, c->kd_com, sizeof g->kd_com);
  memcpy(g->kp_posture, c->kp_posture, sizeof g->kp_posture);
  memcpy(g->kd_posture, c->kd_posture, sizeof g->kd_posture);
  memcpy(g->kp_am, c->kp_am, sizeof g->kp_am);
  g->w_foot = c->w_foot; g->w_com = c->w_com; g->w_posture = c->w_posture; g->w_am = c->w_am;
  g->w_force_reg = c->w_force_reg;
}
static inline void tsidb_gains_to_conf(const tsidb_gains* g, tsidb_conf* c) {
  memcpy(c->kp_contact, g->kp_contact, sizeof g->kp_contact);
  memcpy(c->kd_contact, g->kd_contact, sizeof g->kd_contact);
  memcpy(c->kp_foot, g->kp_foot, sizeof g->kp_foot);
  memcpy(c->kd_foot, g->kd_foot, sizeof g->kd_foot);
  memcpy(c->kp_com, g->kp_com, sizeof g->kp_com);
  memcpy(c->kd_com, g->kd_com, sizeof g->kd_com);
  memcpy(c->kp_posture, g->kp_posture, sizeof g->kp_posture);
  memcpy(c->kd_posture, g->kd_posture, sizeof g->kd_posture);
  memcpy(c->kp_am, g->kp_am, sizeof g->kp_am);
  c->w_foot = g->w_foot; c->w_com = g->w_com; c->w_posture = g->w_posture; c->w_am = g->w_am;
  c->w_force_reg = g->w_force_reg;
}
static inline void tsidb_gains_to_devconst(const tsidb_gains* g, DevConst* D) {
  memcpy(D->kp_contact, g->kp_contact, sizeof D->kp_contact);
  memcpy(D->kd_contact, g->kd_contact, sizeof D->kd_contact);
  memcpy(D->kp_foot, g->kp_foot, sizeof D->kp_foot);
  memcpy(D->kd_foot, g->kd_foot, sizeof D->kd_foot);
  memcpy(D->kp_com, g->kp_com, sizeof D->kp_com);
  memcpy(D->kd_com, g->kd_com, sizeof D->kd_com);
  memcpy(D->kp_post, g->kp_posture, sizeof D->kp_post);
  memcpy(D->kd_post, g->kd_posture, sizeof D->kd_post);
  memcpy(D->kp_am, g->kp_am, sizeof D->kp_am);
  D->w_foot = g->w_foot; D->w_com = g->w_com; D->w_post = g->w_posture; D->w_am = g->w_am;
  D->w_freg = g->w_force_reg;
}

static inline bool tsidb_fill_devconst(const tsidb_model* m, const tsidb_conf* c, DevConst* D, std::string* err) {
  memset(D, 0, sizeof *D);
  const int nb = m->nb;
  if (nb < 2 || nb > 24) { *err = "model: nb out of range"; return false; }
  D->nb = nb; D->na = nb - 1; D->nv = nb + 5; D->nq = nb + 6;
  if (D->nv > TSIDB_NVX) { *err = "model: nv exceeds TSIDB_NVX (26) of this build"; return false; }
  /* tree tables */
  int nchild[24] = {0};
  D->maxdepth = 0;
  for (int b = 0; b < nb; b++) {
    D->parent[b] = m->parent[b];
    if (b == 0) { D->depth[0] = 0; continue; }
    if (m->parent[b] < 0 || m->parent[b] >= b) { *err = "model: parent must precede child"; return false; }
    D->depth[b] = D->depth[m->parent[b]] + 1;
    if (D->depth[b] > 7) { *err = "model: kinematic chains deeper than 7 joints are not supported"; return false; }
    if (D->depth[b] > D->maxdepth) D->maxdepth = D->depth[b];
    D->sibrank[b] = nchild[m->parent[b]]++;
  }
  for (int b = 1; b < nb; b++) {
    int cnt = nchild[m->parent[b]];
    if (cnt > D->maxsib[D->depth[b]]) D->maxsib[D->depth[b]] = cnt;
  }
  for (int f = 0; f < 2; f++) {
    D->foot_body[f] = m->foot_body[f];
    if (m->foot_body[f] <= 0 || m->foot_body[f] >= nb) { *err = "model: foot body out of range"; return false; }
    unsigned s = 0;
    for (int b = m->foot_body[f]; b >= 0; b = m->parent[b]) { s |= 1u << b; if (b == 0) break; }
    D->foot_support[f] = s;
    memcpy(D->fR[f], m->fR[f], sizeof(double) * 9);
    memcpy(D->fp[f], m->fp[f], sizeof(double) * 3);
  }
  memcpy(D->jR, m->jR, sizeof D->jR);
  memcpy(D->jp, m->jp, sizeof D->jp);
  memcpy(D->mass, m->mass, sizeof D->mass);
  memcpy(D->com, m->com, sizeof D->com);
  memcpy(D->inertia, m->inertia, sizeof D->inertia);
  memcpy(D->gravity, m->gravity, sizeof D->gravity);

  /* Contact6d: force generator, pyramid rows [UPSTREAM tsid Contact6d::updateForceGeneratorMatrix /
   * updateForceInequalityConstraints] */
  for (int i = 0; i < 4; i++) {
    const double p[3] = {c->contact_points[0][i], c->contact_points[1][i], c->contact_points[2][i]};
    for (int k = 0; k < 3; k++) D->T[k][3 * i + k] = 1.0;
    D->T[3][3 * i + 1] = -p[2]; D->T[3][3 * i + 2] = p[1];
    D->T[4][3 * i + 0] = p[2];  D->T[4][3 * i + 2] = -p[0];
    D->T[5][3 * i + 0] = -p[1]; D->T[5][3 * i + 1] = p[0];
  }
  {
    const double* n = c->contact_normal;
    auto cross = [](const double* a, const double* b, double* o) {
      o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
    };
    const double ex[3] = {1, 0, 0}, ey[3] = {0, 1, 0};
    double t1[3], t2[3];
    cross(n, ex, t1);
    if (sqrt(t1[0] * t1[0] + t1[1] * t1[1] + t1[2] * t1[2]) < 1e-5) cross(n, ey, t1);
    cross(n, t1, t2);
    const double n1 = sqrt(t1[0] * t1[0] + t1[1] * t1[1] + t1[2] * t1[2]);
    const double n2 = sqrt(t2[0] * t2[0] + t2[1] * t2[1] + t2[2] * t2[2]);
    for (int k = 0; k < 3; k++) {
      t1[k] /= n1; t2[k] /= n2;
      D->fric[0][k] = -t1[k] - c->mu * n[k];
      D->fric[1][k] = t1[k] - c->mu * n[k];
      D->fric[2][k] = -t2[k] - c->mu * n[k];
      D->fric[3][k] = t2[k] - c->mu * n[k];
      D->nrm[k] = n[k];
    }
  }
  D->fmin = c->fmin; D->fmax = c->fmax;
  memcpy(D->kp_contact, c->kp_contact, sizeof D->kp_contact);
  memcpy(D->kd_contact, c->kd_contact, sizeof D->kd_contact);
  memcpy(D->kp_foot, c->kp_foot, sizeof D->kp_foot);
  memcpy(D->kd_foot, c->kd_foot, sizeof D->kd_foot);
  memcpy(D->kp_com, c->kp_com, sizeof D->kp_com);
  memcpy(D->kd_com, c->kd_com, sizeof D->kd_com);
  memcpy(D->kp_post, c->kp_posture, sizeof D->kp_post);
  memcpy(D->kd_post, c->kd_posture, sizeof D->kd_post);
  memcpy(D->kp_am, c->kp_am, sizeof D->kp_am);
  D->w_foot = c->w_foot; D->w_com = c->w_com; D->w_post = c->w_posture; D->w_am = c->w_am;
  D->w_freg = c->w_force_reg; D->hreg = c->hessian_reg;
  D->use_am = c->w_am > 0.0 ? 1 : 0;
  D->use_tb = c->use_torque_bounds ? 1 : 0;
  D->use_jb = c->use_joint_bounds ? 1 : 0;
  D->max_iter = c->max_iter;
  memcpy(D->tau_min, c->tau_min, sizeof D->tau_min);
  memcpy(D->tau_max, c->tau_max, sizeof D->tau_max);
  memcpy(D->v_min, c->v_min, sizeof D->v_min);
  memcpy(D->v_max, c->v_max, sizeof D->v_max);
  D->jb_dt = c->joint_bounds_dt;
  /* one-sided rows of the reference's CI that exist without contacts (for the eiquadprog
   * termination threshold nIneq*eps*c1*c2*100) */
  D->nin_ref_fixed = 2 * ((D->use_tb ? D->na : 0) + (D->use_jb ? D->nv : 0));

  /* force block of the Hessian and its factor (identical for all envs and feet) */
  if (!tsidb_factor_force_block(c, D, err)) return false;
  /* neutral default references */
  for (int f = 0; f < 2; f++) {
    D->ref_foot[f][3] = D->ref_foot[f][7] = D->ref_foot[f][11] = 1.0;
    D->ref_contact[f][3] = D->ref_contact[f][7] = D->ref_contact[f][11] = 1.0;
  }
  return true;
}

/* the QP export's section of the global table (PT_* layout, tsidb_const.h), from a filled DevConst */
static inline void tsidb_fill_problem_table(const tsidb_conf* c, const DevConst* D, double* t) {
  memset(t, 0, PT_SIZE * sizeof(double));
  tsidb_force_hessian(c, D->T, reinterpret_cast<double(*)[12]>(t + PT_oHF));
  /* [UPSTREAM Contact6d::updateForceInequalityConstraints]: four pyramid rows per corner, then the total normal force */
  for (int i = 0; i < 4; i++)
    for (int k = 0; k < 3; k++) {
      for (int r = 0; r < 4; r++) t[PT_oB + (4 * i + r) * 12 + 3 * i + k] = D->fric[r][k];
      t[PT_oB + 16 * 12 + 3 * i + k] = D->nrm[k];
    }
  memcpy(t + PT_oT, D->T, 72 * sizeof(double));
  memcpy(t + PT_oTMIN, D->tau_min, 23 * sizeof(double));
  memcpy(t + PT_oTMAX, D->tau_max, 23 * sizeof(double));
  memcpy(t + PT_oVMIN, D->v_min, 23 * sizeof(double));
  memcpy(t + PT_oVMAX, D->v_max, 23 * sizeof(double));
}

#endif
