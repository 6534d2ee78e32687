/*
 * model_oracle.c -- CPU restatement of the lossy and Westervelt wave models (DESIGN.md section 4.5a).
 *
 * TEST INFRASTRUCTURE ONLY, like oracle/wave_oracle.c, which it includes unchanged: the stiffness applies,
 * the stage loop and the source below are that oracle's, so that with delta = beta = 0 wo_rk4_westervelt
 * reproduces wo_rk4 bit for bit (tests/test_models.py).  Its linear part is thereby pinned to the oracle,
 * which is pinned to the reference's own code.  The new terms are written out plainly and independently of
 * the CUDA path: un is kept explicitly, -c0^2 K un and -c0^2 K vn are two separate applies (not one apply
 * on un + s vn), kv is the plain quotient of the lumped system, g' is analytic.
 *
 * Lumped system per dof i (kappa = 2 beta / (rho0 c0^2), q = (delta / c0) m2):
 *   (m_i (1 - kappa p_i) + q_i) p_tt,i = [A p]_i + (delta / 1500^2) [A p_t]_i + kappa m_i p_t,i^2
 *                                        + (c0^2 g + delta g') m1_i - c0 m2_i p_t,i
 * with A = -1500^2 K the oracle's stiffness (c0 = 1500 hard-coded in skernel, as in the reference), so
 * that the second term is -delta K p_t.
 */
#include "../oracle/wave_oracle.c"

/* g(t) exactly as wo_rk4 forms it (LinearGLL.hpp:155-162) and its analytic derivative
 *   g'(t) = A (W' cos(w0 t) - W w0 sin(w0 t)),  W' = (f0 pi / 8) sin(f0 pi t / 4) inside the ramp, else 0 */
void wo_source(double t, double freq0, double p0, double c0, double* g, double* gdot)
{
  const double w0 = 2.0 * M_PI * freq0, T = 1.0 / freq0, alpha = 4.0;
  const int ramp = t < T * alpha;
  const double window = ramp ? 0.5 * (1.0 - cos(freq0 * M_PI * t / alpha)) : 1.0;
  const double wdot = ramp ? 0.5 * sin(freq0 * M_PI * t / alpha) * (freq0 * M_PI / alpha) : 0.0;
  *g = window * p0 * w0 / c0 * cos(w0 * t);
  *gdot = p0 * w0 / c0 * (wdot * cos(w0 * t) - window * w0 * sin(w0 * t));
}

static void model_stiffness(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                            const double* x, double* y, int sumfact, int nthreads)
{
  if (sumfact) wo_stiffness_apply_sumfact(P, ncells, ndofs, dofmap, G, x, y, nthreads);
  else wo_stiffness_apply_dense(P, ncells, ndofs, dofmap, G, x, y, nthreads);
}

/* kv = p_tt of the lumped system at time t for state (un, vn); b, bv: scratch vectors */
static void model_rhs(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                      const double* m, const double* m1, const double* m2, double c0, double freq0, double p0,
                      double delta, double beta, double rho0, double t, const double* un, const double* vn,
                      double* kv, double* b, double* bv, int sumfact, int nthreads)
{
  const size_t nb = sizeof(double) * ndofs;
  const double kappa = beta > 0 ? 2.0 * beta / (rho0 * c0 * c0) : 0.0;
  const double s = delta / (1500.0 * 1500.0);
  double g, gdot;
  wo_source(t, freq0, p0, c0, &g, &gdot);
  memset(b, 0, nb);
  memset(bv, 0, nb);
  model_stiffness(P, ncells, ndofs, dofmap, G, un, b, sumfact, nthreads);  /* A un */
  model_stiffness(P, ncells, ndofs, dofmap, G, vn, bv, sumfact, nthreads); /* A vn */
  for (int64_t k = 0; k < ndofs; ++k)
  {
    double r = b[k] + s * bv[k];
    r += (c0 * c0 * g + delta * gdot) * m1[k] - c0 * m2[k] * vn[k];
    r += kappa * m[k] * vn[k] * vn[k];
    kv[k] = r / (m[k] * (1.0 - kappa * un[k]) + delta / c0 * m2[k]);
  }
}

/* dv/dt = f1(t, u, v) of the lossy / Westervelt model */
void wo_f1_westervelt(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                      const double* m, const double* m1, const double* m2, double c0, double freq0, double p0,
                      double delta, double beta, double rho0, double t, const double* u, const double* v,
                      double* out, int sumfact, int nthreads)
{
  const size_t nb = sizeof(double) * ndofs;
  double *b = malloc(nb), *bv = malloc(nb);
  model_rhs(P, ncells, ndofs, dofmap, G, m, m1, m2, c0, freq0, p0, delta, beta, rho0, t, u, v, out, b, bv,
            sumfact, nthreads);
  free(b);
  free(bv);
}

/* rk4 of the lossy / Westervelt model: wo_rk4's stage loop (LinearGLL.hpp:241-270) with model_rhs as f1.
 * u_n, v_n: in = initial state, out = final state.  Returns the number of steps; *t_end the final time. */
int64_t wo_rk4_westervelt(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                          const double* m, const double* m1, const double* m2, double c0, double freq0, double p0,
                          double delta, double beta, double rho0, double t0, double tf, double dt,
                          int64_t max_steps, double* u_n, double* v_n, int sumfact, int nthreads, double* t_end)
{
  const double a_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const double b_runge[4] = {1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0};
  const double c_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const size_t nb = sizeof(double) * ndofs;
  double *u_ = malloc(nb), *v_ = malloc(nb), *un = malloc(nb), *vn = malloc(nb);
  double *u0 = malloc(nb), *v0 = malloc(nb), *ku = malloc(nb), *kv = malloc(nb), *b = malloc(nb), *bv = malloc(nb);
  memcpy(u_, u_n, nb);
  memcpy(v_, v_n, nb);
  memcpy(ku, u_, nb);
  memcpy(kv, v_, nb);
  double t = t0;
  int64_t step = 0;
  while (t < tf)
  {
    if (max_steps > 0 && step >= max_steps) break;
    dt = dt < tf - t ? dt : tf - t;
    memcpy(u0, u_, nb);
    memcpy(v0, v_, nb);
    for (int i = 0; i < 4; ++i)
    {
      memcpy(un, u0, nb);
      memcpy(vn, v0, nb);
      const double adt = dt * a_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) un[k] = ku[k] * adt + un[k];
      for (int64_t k = 0; k < ndofs; ++k) vn[k] = kv[k] * adt + vn[k];
      const double tn = t + c_runge[i] * dt;
      memcpy(ku, vn, nb);
      model_rhs(P, ncells, ndofs, dofmap, G, m, m1, m2, c0, freq0, p0, delta, beta, rho0, tn, un, vn, kv, b, bv,
                sumfact, nthreads);
      const double bdt = dt * b_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) u_[k] = ku[k] * bdt + u_[k];
      for (int64_t k = 0; k < ndofs; ++k) v_[k] = kv[k] * bdt + v_[k];
    }
    t += dt;
    step += 1;
  }
  memcpy(u_n, u_, nb);
  memcpy(v_n, v_, nb);
  if (t_end) *t_end = t;
  free(u_); free(v_); free(un); free(vn); free(u0); free(v0); free(ku); free(kv); free(b); free(bv);
  return step;
}

/* ---- source profiles (DESIGN.md section 4.5c) ----------------------------------------------------------------
 * The same model with a per-dof source g_k(t) = amp_k g(t - delay_k), g and g' of wo_source, both zero before
 * the delay.  model_rhs_profile is model_rhs with that source; with amp = 1 and delay = 0 it computes what
 * model_rhs computes, bit for bit (1 * g = g, t - 0 = t). */
static void model_rhs_profile(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                              const double* m, const double* m1, const double* m2, double c0, double freq0, double p0,
                              double delta, double beta, double rho0, const double* amp, const double* delay, double t,
                              const double* un, const double* vn, double* kv, double* b, double* bv, int sumfact,
                              int nthreads)
{
  const size_t nb = sizeof(double) * ndofs;
  const double kappa = beta > 0 ? 2.0 * beta / (rho0 * c0 * c0) : 0.0;
  const double s = delta / (1500.0 * 1500.0);
  memset(b, 0, nb);
  memset(bv, 0, nb);
  model_stiffness(P, ncells, ndofs, dofmap, G, un, b, sumfact, nthreads);  /* A un */
  model_stiffness(P, ncells, ndofs, dofmap, G, vn, bv, sumfact, nthreads); /* A vn */
  for (int64_t k = 0; k < ndofs; ++k)
  {
    double g = 0.0, gdot = 0.0;
    if (m1[k] != 0.0)
    {
      const double sk = t - delay[k];
      if (sk >= 0.0) wo_source(sk, freq0, p0, c0, &g, &gdot);
      else g = gdot = 0.0; /* the source has not started at this dof yet */
      g = amp[k] * g;
      gdot = amp[k] * gdot;
    }
    double r = b[k] + s * bv[k];
    r += (c0 * c0 * g + delta * gdot) * m1[k] - c0 * m2[k] * vn[k];
    r += kappa * m[k] * vn[k] * vn[k];
    kv[k] = r / (m[k] * (1.0 - kappa * un[k]) + delta / c0 * m2[k]);
  }
}

/* wo_f1_westervelt with a source profile amp[ndofs], delay[ndofs] */
void wo_f1_westervelt_profile(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                              const double* m, const double* m1, const double* m2, double c0, double freq0, double p0,
                              double delta, double beta, double rho0, const double* amp, const double* delay, double t,
                              const double* u, const double* v, double* out, int sumfact, int nthreads)
{
  const size_t nb = sizeof(double) * ndofs;
  double *b = malloc(nb), *bv = malloc(nb);
  model_rhs_profile(P, ncells, ndofs, dofmap, G, m, m1, m2, c0, freq0, p0, delta, beta, rho0, amp, delay, t, u, v,
                    out, b, bv, sumfact, nthreads);
  free(b);
  free(bv);
}

/* wo_rk4_westervelt with a source profile: the same stage loop, model_rhs_profile as f1 */
int64_t wo_rk4_westervelt_profile(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                                  const double* m, const double* m1, const double* m2, double c0, double freq0,
                                  double p0, double delta, double beta, double rho0, const double* amp,
                                  const double* delay, double t0, double tf, double dt, int64_t max_steps, double* u_n,
                                  double* v_n, int sumfact, int nthreads, double* t_end)
{
  const double a_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const double b_runge[4] = {1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0};
  const double c_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const size_t nb = sizeof(double) * ndofs;
  double *u_ = malloc(nb), *v_ = malloc(nb), *un = malloc(nb), *vn = malloc(nb);
  double *u0 = malloc(nb), *v0 = malloc(nb), *ku = malloc(nb), *kv = malloc(nb), *b = malloc(nb), *bv = malloc(nb);
  memcpy(u_, u_n, nb);
  memcpy(v_, v_n, nb);
  memcpy(ku, u_, nb);
  memcpy(kv, v_, nb);
  double t = t0;
  int64_t step = 0;
  while (t < tf)
  {
    if (max_steps > 0 && step >= max_steps) break;
    dt = dt < tf - t ? dt : tf - t;
    memcpy(u0, u_, nb);
    memcpy(v0, v_, nb);
    for (int i = 0; i < 4; ++i)
    {
      memcpy(un, u0, nb);
      memcpy(vn, v0, nb);
      const double adt = dt * a_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) un[k] = ku[k] * adt + un[k];
      for (int64_t k = 0; k < ndofs; ++k) vn[k] = kv[k] * adt + vn[k];
      const double tn = t + c_runge[i] * dt;
      memcpy(ku, vn, nb);
      model_rhs_profile(P, ncells, ndofs, dofmap, G, m, m1, m2, c0, freq0, p0, delta, beta, rho0, amp, delay, tn, un,
                        vn, kv, b, bv, sumfact, nthreads);
      const double bdt = dt * b_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) u_[k] = ku[k] * bdt + u_[k];
      for (int64_t k = 0; k < ndofs; ++k) v_[k] = kv[k] * bdt + v_[k];
    }
    t += dt;
    step += 1;
  }
  memcpy(u_n, u_, nb);
  memcpy(v_n, v_, nb);
  if (t_end) *t_end = t;
  free(u_); free(v_); free(un); free(vn); free(u0); free(v0); free(ku); free(kv); free(b); free(bv);
  return step;
}

/* ---- thermal model: Pennes bioheat equation (DESIGN.md section 4.5d) ------------------------------------------
 * State theta = T - T_art.  Lumped GLL system per dof i, written out plainly (one quotient, no precomputed scale,
 * r or f), with A = -1500^2 K the oracle's stiffness, so that (k / 1500^2) A theta = -k K theta:
 *   rhoC_i m_i theta_i' = (k / 1500^2) [A theta]_i - (wbCb_i m_i + h1 m1_i + h2 m2_i) theta_i
 *                         + h1 m1_i (T_ext1 - T_art) + h2 m2_i (T_ext2 - T_art) + s Q_i m_i
 * perf and Q may be NULL (0). */
void wo_rhs_pennes(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G, const double* m,
                   const double* m1, const double* m2, double k, const double* rhoc, const double* perf, double T_art,
                   double h1, double h2, double T_ext1, double T_ext2, const double* Q, double s, const double* theta,
                   double* out, int sumfact, int nthreads)
{
  memset(out, 0, sizeof(double) * ndofs);
  model_stiffness(P, ncells, ndofs, dofmap, G, theta, out, sumfact, nthreads); /* A theta */
  for (int64_t i = 0; i < ndofs; ++i)
  {
    const double wb = perf ? perf[i] : 0.0, q = Q ? Q[i] : 0.0;
    double num = k / (1500.0 * 1500.0) * out[i];
    num -= (wb * m[i] + h1 * m1[i] + h2 * m2[i]) * theta[i];
    num += h1 * m1[i] * (T_ext1 - T_art) + h2 * m2[i] * (T_ext2 - T_art) + s * q * m[i];
    out[i] = num / (rhoc[i] * m[i]);
  }
}

/* RK4 of the thermal model: the stage loop of wo_rk4_westervelt on theta alone.  After every step of size dt,
 * with T = T_art + theta:  cem43 += dt / 60 * R^(43 - T) (R = 0.5 for T >= 43, else 0.25) and
 * theta_max = max(theta_max, theta) (a NaN theta replaces the maximum).  theta, cem43, theta_max: in / out.
 * Returns the number of steps; *t_end the final time. */
int64_t wo_rk4_pennes(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G, const double* m,
                      const double* m1, const double* m2, double k, const double* rhoc, const double* perf,
                      double T_art, double h1, double h2, double T_ext1, double T_ext2, const double* Q, double s,
                      double t0, double tf, double dt, int64_t max_steps, double* theta, double* cem43,
                      double* theta_max, int sumfact, int nthreads, double* t_end)
{
  const double a_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const double b_runge[4] = {1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0};
  const size_t nb = sizeof(double) * ndofs;
  double *u_ = malloc(nb), *un = malloc(nb), *u0 = malloc(nb), *kv = malloc(nb);
  memcpy(u_, theta, nb);
  memset(kv, 0, nb);
  double t = t0;
  int64_t step = 0;
  while (t < tf)
  {
    if (max_steps > 0 && step >= max_steps) break;
    dt = dt < tf - t ? dt : tf - t;
    memcpy(u0, u_, nb);
    for (int i = 0; i < 4; ++i)
    {
      const double adt = dt * a_runge[i];
      for (int64_t j = 0; j < ndofs; ++j) un[j] = kv[j] * adt + u0[j];
      wo_rhs_pennes(P, ncells, ndofs, dofmap, G, m, m1, m2, k, rhoc, perf, T_art, h1, h2, T_ext1, T_ext2, Q, s, un,
                    kv, sumfact, nthreads);
      const double bdt = dt * b_runge[i];
      for (int64_t j = 0; j < ndofs; ++j) u_[j] = kv[j] * bdt + u_[j];
    }
    for (int64_t j = 0; j < ndofs; ++j)
    {
      const double T = T_art + u_[j];
      cem43[j] += dt / 60.0 * pow(T >= 43.0 ? 0.5 : 0.25, 43.0 - T);
      if (u_[j] > theta_max[j] || u_[j] != u_[j]) theta_max[j] = u_[j];
    }
    t += dt;
    step += 1;
  }
  memcpy(theta, u_, nb);
  if (t_end) *t_end = t;
  free(u_); free(un); free(u0); free(kv);
  return step;
}

/* ---- layered media (DESIGN.md section 4.5e) ------------------------------------------------------------------
 * Per-cell density, sound speed and nonlinearity enter the lumped system only through weights: G scaled per cell
 * by rho_ref / rho_c (passed in as G), the weighted lumped mass m, the weighted facet masses m1, m2 (passed in as
 * given) and a per-dof kappa.  model_rhs_medium is model_rhs with kappa[k] in place of the scalar kappa; with
 * kappa[k] equal to that scalar it computes what model_rhs computes, bit for bit. */

/* wo_boundary_facet_mass with facet f's contributions multiplied by fw[f] (written out like the oracle's loop) */
int wo_boundary_facet_mass_weighted(int P, int64_t nfacets, const int32_t* fcell, const int32_t* flocal,
                                    const int32_t* ftag, const double* x, const int32_t* xdofs, const int32_t* dofmap,
                                    const double* fw, double* m1, double* m2)
{
  const int n = P + 1, nd = n * n * n;
  double pts[WO_MAXN], wts[WO_MAXN];
  static const int F_AXIS[6] = {2, 1, 0, 0, 1, 2};
  static const int F_SIDE[6] = {0, 0, 0, 1, 1, 1};
  int* perm = (int*)malloc(sizeof(int) * nd);
  if (wo_gll(P, pts, wts) || wo_perm(P, perm)) { free(perm); return -1; }
  for (int64_t f = 0; f < nfacets; ++f)
  {
    const int64_t c = fcell[f];
    const int lf = flocal[f], tag = ftag[f];
    double* m = tag == 1 ? m1 : (tag == 2 ? m2 : NULL);
    if (!m) continue;
    const int ax = F_AXIS[lf], side = F_SIDE[lf];
    const int t1 = ax == 0 ? 1 : 0, t2 = ax == 2 ? 1 : 2;
    double coords[8][3];
    for (int v = 0; v < 8; ++v)
      for (int a = 0; a < 3; ++a) coords[v][a] = x[3 * (int64_t)xdofs[8 * c + v] + a];
    for (int ia = 0; ia < n; ++ia)
      for (int ib = 0; ib < n; ++ib)
      {
        int idx[3];
        idx[ax] = side;
        idx[t1] = ia;
        idx[t2] = ib;
        const double X[3] = {pts[idx[0]], pts[idx[1]], pts[idx[2]]};
        double d[3][8], J[3][3];
        cmap_dphi(X, d, 1);
        for (int i = 0; i < 3; ++i)
          for (int j = 0; j < 3; ++j)
          {
            double s = 0.0;
            for (int v = 0; v < 8; ++v) s += coords[v][i] * d[j][v];
            J[i][j] = s;
          }
        const double a0 = J[0][t1], a1 = J[1][t1], a2 = J[2][t1];
        const double b0 = J[0][t2], b1 = J[1][t2], b2 = J[2][t2];
        const double cx = a1 * b2 - a2 * b1, cy = a2 * b0 - a0 * b2, cz = a0 * b1 - a1 * b0;
        const double scale = sqrt(cx * cx + cy * cy + cz * cz);
        const int t = (idx[0] * n + idx[1]) * n + idx[2];
        m[dofmap[c * nd + perm[t]]] += fw[f] * (wts[ia] * wts[ib] * scale);
      }
  }
  free(perm);
  return 0;
}

static void model_rhs_medium(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                             const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                             double freq0, double p0, double delta, double t, const double* un, const double* vn,
                             double* kv, double* b, double* bv, int sumfact, int nthreads)
{
  const size_t nb = sizeof(double) * ndofs;
  const double s = delta / (1500.0 * 1500.0);
  double g, gdot;
  wo_source(t, freq0, p0, c0, &g, &gdot);
  memset(b, 0, nb);
  memset(bv, 0, nb);
  model_stiffness(P, ncells, ndofs, dofmap, G, un, b, sumfact, nthreads);  /* A un */
  model_stiffness(P, ncells, ndofs, dofmap, G, vn, bv, sumfact, nthreads); /* A vn */
  for (int64_t k = 0; k < ndofs; ++k)
  {
    double r = b[k] + s * bv[k];
    r += (c0 * c0 * g + delta * gdot) * m1[k] - c0 * m2[k] * vn[k];
    r += kappa[k] * m[k] * vn[k] * vn[k];
    kv[k] = r / (m[k] * (1.0 - kappa[k] * un[k]) + delta / c0 * m2[k]);
  }
}

/* dv/dt = f1(t, u, v) of the lossy / Westervelt model in a layered medium (kappa [ndofs]) */
void wo_f1_westervelt_medium(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                             const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                             double freq0, double p0, double delta, double t, const double* u, const double* v,
                             double* out, int sumfact, int nthreads)
{
  const size_t nb = sizeof(double) * ndofs;
  double *b = malloc(nb), *bv = malloc(nb);
  model_rhs_medium(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, t, u, v, out, b, bv, sumfact,
                   nthreads);
  free(b);
  free(bv);
}

/* wo_rk4_westervelt in a layered medium: the same stage loop, model_rhs_medium as f1 */
int64_t wo_rk4_westervelt_medium(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                                 const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                                 double freq0, double p0, double delta, double t0, double tf, double dt,
                                 int64_t max_steps, double* u_n, double* v_n, int sumfact, int nthreads, double* t_end)
{
  const double a_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const double b_runge[4] = {1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0};
  const double c_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const size_t nb = sizeof(double) * ndofs;
  double *u_ = malloc(nb), *v_ = malloc(nb), *un = malloc(nb), *vn = malloc(nb);
  double *u0 = malloc(nb), *v0 = malloc(nb), *ku = malloc(nb), *kv = malloc(nb), *b = malloc(nb), *bv = malloc(nb);
  memcpy(u_, u_n, nb);
  memcpy(v_, v_n, nb);
  memcpy(ku, u_, nb);
  memcpy(kv, v_, nb);
  double t = t0;
  int64_t step = 0;
  while (t < tf)
  {
    if (max_steps > 0 && step >= max_steps) break;
    dt = dt < tf - t ? dt : tf - t;
    memcpy(u0, u_, nb);
    memcpy(v0, v_, nb);
    for (int i = 0; i < 4; ++i)
    {
      memcpy(un, u0, nb);
      memcpy(vn, v0, nb);
      const double adt = dt * a_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) un[k] = ku[k] * adt + un[k];
      for (int64_t k = 0; k < ndofs; ++k) vn[k] = kv[k] * adt + vn[k];
      const double tn = t + c_runge[i] * dt;
      memcpy(ku, vn, nb);
      model_rhs_medium(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, tn, un, vn, kv, b, bv,
                       sumfact, nthreads);
      const double bdt = dt * b_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) u_[k] = ku[k] * bdt + u_[k];
      for (int64_t k = 0; k < ndofs; ++k) v_[k] = kv[k] * bdt + v_[k];
    }
    t += dt;
    step += 1;
  }
  memcpy(u_n, u_, nb);
  memcpy(v_n, v_, nb);
  if (t_end) *t_end = t;
  free(u_); free(v_); free(un); free(vn); free(u0); free(v0); free(ku); free(kv); free(b); free(bv);
  return step;
}

/* ---- relaxation absorption (DESIGN.md section 4.5f) ----------------------------------------------------------
 * M relaxation processes with times tau[nu] and per-dof strengths eps[nu * ndofs + k], memory variables
 * q[nu * ndofs + k], on the lumped system of model_rhs_medium:
 *   (m (1 - kappa p) + (delta / c0) m2) p_tt = r - m sum_nu q_nu'',   tau_nu q_nu' + q_nu = eps_nu p
 * with r the numerator of model_rhs_medium and q_nu'' = (eps_nu p_t - q_nu') / tau_nu.  Written out plainly: q_nu'
 * and q_nu'' divide by tau (no reciprocal), the sum is subtracted from the numerator, not folded into the quotient.
 * With M = 0 the stage loop and the quotient are those of wo_rk4_westervelt_medium, bit for bit. */
static void model_rhs_relax(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                            const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                            double freq0, double p0, double delta, int M, const double* tau, const double* eps, double t,
                            const double* un, const double* vn, const double* qn, double* kv, double* kq, double* b,
                            double* bv, int sumfact, int nthreads)
{
  const size_t nb = sizeof(double) * ndofs;
  const double s = delta / (1500.0 * 1500.0);
  double g, gdot;
  wo_source(t, freq0, p0, c0, &g, &gdot);
  memset(b, 0, nb);
  memset(bv, 0, nb);
  model_stiffness(P, ncells, ndofs, dofmap, G, un, b, sumfact, nthreads);  /* A un */
  model_stiffness(P, ncells, ndofs, dofmap, G, vn, bv, sumfact, nthreads); /* A vn */
  for (int64_t k = 0; k < ndofs; ++k)
  {
    double r = b[k] + s * bv[k];
    r += (c0 * c0 * g + delta * gdot) * m1[k] - c0 * m2[k] * vn[k];
    r += kappa[k] * m[k] * vn[k] * vn[k];
    if (M > 0)
    {
      double qdd = 0.0;
      for (int nu = 0; nu < M; ++nu)
      {
        const int64_t o = nu * ndofs + k;
        kq[o] = (eps[o] * un[k] - qn[o]) / tau[nu];
        qdd += (eps[o] * vn[k] - kq[o]) / tau[nu];
      }
      r -= m[k] * qdd;
    }
    kv[k] = r / (m[k] * (1.0 - kappa[k] * un[k]) + delta / c0 * m2[k]);
  }
}

/* dv/dt = f1(t, u, v; q) of the lossy / Westervelt model with relaxation at the memory variables q [M][ndofs] */
void wo_f1_westervelt_relax(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                            const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                            double freq0, double p0, double delta, int M, const double* tau, const double* eps, double t,
                            const double* u, const double* v, const double* q, double* out, int sumfact, int nthreads)
{
  const size_t nb = sizeof(double) * ndofs;
  double *b = malloc(nb), *bv = malloc(nb), *kq = malloc(nb * (M > 0 ? M : 1));
  model_rhs_relax(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, M, tau, eps, t, u, v, q, out, kq,
                  b, bv, sumfact, nthreads);
  free(b);
  free(bv);
  free(kq);
}

/* wo_rk4_westervelt_medium with relaxation: the same stage loop, with q [M][ndofs] (in / out) stepped by the same
 * tableau as u and v */
int64_t wo_rk4_westervelt_relax(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                                const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                                double freq0, double p0, double delta, int M, const double* tau, const double* eps,
                                double t0, double tf, double dt, int64_t max_steps, double* u_n, double* v_n,
                                double* q_n, int sumfact, int nthreads, double* t_end)
{
  const double a_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const double b_runge[4] = {1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0};
  const double c_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const size_t nb = sizeof(double) * ndofs, nq = nb * (M > 0 ? M : 1);
  const int64_t nqe = (int64_t)M * ndofs;
  double *u_ = malloc(nb), *v_ = malloc(nb), *un = malloc(nb), *vn = malloc(nb);
  double *u0 = malloc(nb), *v0 = malloc(nb), *ku = malloc(nb), *kv = malloc(nb), *b = malloc(nb), *bv = malloc(nb);
  double *q_ = malloc(nq), *qn = malloc(nq), *q0 = malloc(nq), *kq = malloc(nq);
  memcpy(u_, u_n, nb);
  memcpy(v_, v_n, nb);
  memcpy(ku, u_, nb);
  memcpy(kv, v_, nb);
  if (M > 0)
  {
    memcpy(q_, q_n, sizeof(double) * nqe);
    memset(kq, 0, sizeof(double) * nqe);
  }
  double t = t0;
  int64_t step = 0;
  while (t < tf)
  {
    if (max_steps > 0 && step >= max_steps) break;
    dt = dt < tf - t ? dt : tf - t;
    memcpy(u0, u_, nb);
    memcpy(v0, v_, nb);
    if (M > 0) memcpy(q0, q_, sizeof(double) * nqe);
    for (int i = 0; i < 4; ++i)
    {
      memcpy(un, u0, nb);
      memcpy(vn, v0, nb);
      const double adt = dt * a_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) un[k] = ku[k] * adt + un[k];
      for (int64_t k = 0; k < ndofs; ++k) vn[k] = kv[k] * adt + vn[k];
      for (int64_t k = 0; k < nqe; ++k) qn[k] = i == 0 ? q0[k] : kq[k] * adt + q0[k];
      const double tn = t + c_runge[i] * dt;
      memcpy(ku, vn, nb);
      model_rhs_relax(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, M, tau, eps, tn, un, vn, qn,
                      kv, kq, b, bv, sumfact, nthreads);
      const double bdt = dt * b_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) u_[k] = ku[k] * bdt + u_[k];
      for (int64_t k = 0; k < ndofs; ++k) v_[k] = kv[k] * bdt + v_[k];
      for (int64_t k = 0; k < nqe; ++k) q_[k] = kq[k] * bdt + q_[k];
    }
    t += dt;
    step += 1;
  }
  memcpy(u_n, u_, nb);
  memcpy(v_n, v_, nb);
  if (M > 0) memcpy(q_n, q_, sizeof(double) * nqe);
  if (t_end) *t_end = t;
  free(u_); free(v_); free(un); free(vn); free(u0); free(v0); free(ku); free(kv); free(b); free(bv);
  free(q_); free(qn); free(q0); free(kq);
  return step;
}

/* ---- perfectly matched layer (DESIGN.md section 4.5g) --------------------------------------------------------
 * The second-order PML of Grote and Sim (2010) on the lumped system of model_rhs_relax, with damping zeta[j * ndofs
 * + k] along physical axis j, psi [ndofs] and phi [ncells][nq][3] (points in tensor order t = (i0 n + i1) n + i2,
 * dof dofmap[c nq + perm[t]]).  PML cells: zeta > 0 at any of their dofs; PML dofs: the dofs of PML cells.  At the
 * stage state (p, p_t, psi, phi), with w = p + s p_t, chi = psi + s p, a_c = 1500^2 coeff[c] and the clamped 1-D
 * derivative table D of the stiffness:
 *   r_k += [D^T phi]_k - m_k (sum zeta p_t + sum zeta zeta p + zeta1 zeta2 zeta3 psi)_k   (PML dofs, before kappa)
 *   [D^T phi]_k = -sum_c sum_q grad^ l_k(xi_q) . (dJw_q K_q phi_q)
 *   psi' = p,   phi_l' = a_c (Gamma1_l (K^T grad^ w)_l + Gamma2_l (K^T grad^ chi)_l) - zeta_l phi_l
 * K = J^-1 [ncells][nq][3][3] (K[a][l] = dX_a / dx_l) and dJw = |detJ| w [ncells][nq], both in tensor order.  With
 * no PML cell every step is wo_rk4_westervelt_relax's, bit for bit. */
typedef struct
{
  const double *zeta, *K, *dJw, *coeff;
  int64_t ncells_pml;
  uint8_t *cell_on, *dof_on; /* [ncells], [ndofs] */
} pml_t;

static void pml_setup(pml_t* L, int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* zeta,
                      const double* K, const double* dJw, const double* coeff)
{
  const int nd = (P + 1) * (P + 1) * (P + 1);
  L->zeta = zeta, L->K = K, L->dJw = dJw, L->coeff = coeff;
  L->cell_on = calloc(ncells > 0 ? ncells : 1, 1);
  L->dof_on = calloc(ndofs > 0 ? ndofs : 1, 1);
  L->ncells_pml = 0;
  for (int64_t c = 0; c < ncells; ++c)
  {
    int on = 0;
    for (int t = 0; t < nd; ++t)
    {
      const int32_t d = dofmap[c * nd + t];
      on |= zeta[d] > 0 || zeta[ndofs + d] > 0 || zeta[2 * ndofs + d] > 0;
    }
    if (!on) continue;
    L->cell_on[c] = 1;
    L->ncells_pml += 1;
    for (int t = 0; t < nd; ++t) L->dof_on[dofmap[c * nd + t]] = 1;
  }
}

static void pml_free(pml_t* L)
{
  free(L->cell_on);
  free(L->dof_on);
}

/* tp[k] = the PML terms of dof k (PML dofs), kpsi, kphi: the layer's rates (0 off the layer) */
static void pml_terms(const pml_t* L, int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* m,
                      double s, const double* un, const double* vn, const double* psin, const double* phin, double* tp,
                      double* kpsi, double* kphi)
{
  const int n = P + 1, nd = n * n * n;
  double D[WO_MAXN * WO_MAXN];
  int* perm = malloc(sizeof(int) * nd);
  double* buf = malloc(sizeof(double) * nd * 5);
  double *W = buf, *X = buf + nd, *F = buf + 2 * nd; /* F [nd][3] */
  wo_deriv_1d(P, D, 1);
  wo_perm(P, perm);
  memset(tp, 0, sizeof(double) * ndofs);
  memset(kpsi, 0, sizeof(double) * ndofs);
  memset(kphi, 0, sizeof(double) * ncells * nd * 3);
  for (int64_t c = 0; c < ncells; ++c)
  {
    if (!L->cell_on[c]) continue;
    const int32_t* cd = dofmap + c * nd;
    const double a = 1500.0 * 1500.0 * L->coeff[c];
    for (int t = 0; t < nd; ++t)
    {
      const int32_t d = cd[perm[t]];
      W[t] = un[d] + s * vn[d];
      X[t] = psin[d] + s * un[d];
    }
    for (int i0 = 0; i0 < n; ++i0)
      for (int i1 = 0; i1 < n; ++i1)
        for (int i2 = 0; i2 < n; ++i2)
        {
          const int t = (i0 * n + i1) * n + i2;
          double gw[3] = {0, 0, 0}, gx[3] = {0, 0, 0};
          for (int q = 0; q < n; ++q)
          {
            gw[0] += D[i0 * n + q] * W[(q * n + i1) * n + i2];
            gw[1] += D[i1 * n + q] * W[(i0 * n + q) * n + i2];
            gw[2] += D[i2 * n + q] * W[(i0 * n + i1) * n + q];
            gx[0] += D[i0 * n + q] * X[(q * n + i1) * n + i2];
            gx[1] += D[i1 * n + q] * X[(i0 * n + q) * n + i2];
            gx[2] += D[i2 * n + q] * X[(i0 * n + i1) * n + q];
          }
          const double* k = L->K + (c * nd + t) * 9;
          const double* ph = phin + (c * nd + t) * 3;
          const double dj = L->dJw[c * nd + t];
          for (int d = 0; d < 3; ++d) F[t * 3 + d] = dj * (k[3 * d] * ph[0] + k[3 * d + 1] * ph[1] + k[3 * d + 2] * ph[2]);
          const int32_t dof = cd[perm[t]];
          const double z[3] = {L->zeta[dof], L->zeta[ndofs + dof], L->zeta[2 * ndofs + dof]};
          const double g1[3] = {z[1] + z[2] - z[0], z[0] + z[2] - z[1], z[0] + z[1] - z[2]};
          const double g2[3] = {z[1] * z[2], z[0] * z[2], z[0] * z[1]};
          for (int l = 0; l < 3; ++l)
          {
            const double pw = k[l] * gw[0] + k[3 + l] * gw[1] + k[6 + l] * gw[2];
            const double px = k[l] * gx[0] + k[3 + l] * gx[1] + k[6 + l] * gx[2];
            kphi[(c * nd + t) * 3 + l] = a * (g1[l] * pw + g2[l] * px) - z[l] * ph[l];
          }
        }
    for (int i0 = 0; i0 < n; ++i0)
      for (int i1 = 0; i1 < n; ++i1)
        for (int i2 = 0; i2 < n; ++i2)
        {
          double acc = 0.0;
          for (int q = 0; q < n; ++q)
            acc += D[q * n + i0] * F[((q * n + i1) * n + i2) * 3 + 0] + D[q * n + i1] * F[((i0 * n + q) * n + i2) * 3 + 1]
                   + D[q * n + i2] * F[((i0 * n + i1) * n + q) * 3 + 2];
          tp[cd[perm[(i0 * n + i1) * n + i2]]] -= acc;
        }
  }
  for (int64_t k = 0; k < ndofs; ++k)
  {
    if (!L->dof_on[k]) continue;
    const double z0 = L->zeta[k], z1 = L->zeta[ndofs + k], z2 = L->zeta[2 * ndofs + k];
    tp[k] -= m[k] * ((z0 + z1 + z2) * vn[k] + (z0 * z1 + z0 * z2 + z1 * z2) * un[k] + z0 * z1 * z2 * psin[k]);
    kpsi[k] = un[k];
  }
  free(buf);
  free(perm);
}

/* A volume source (DESIGN.md section 4.5h): n distinct dofs with weights q and delays, the term
 *   r_j += c0^2 q_j g(t - delay_j),   g of wo_source, g = 0 before the delay,
 * added after the boundary term, before the layer's, kappa and relaxation terms.  NULL or n = 0: no term. */
typedef struct
{
  int64_t n;
  const int32_t* dofs;
  const double *q, *delay;
} vsrc_t;

/* model_rhs_relax with the layer's terms tp added to the numerator (PML dofs), and a volume source S (nullable) */
static void model_rhs_pml(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                          const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                          double freq0, double p0, double delta, int M, const double* tau, const double* eps, double t,
                          const double* un, const double* vn, const double* qn, const pml_t* L, const double* psin,
                          const double* phin, const vsrc_t* S, double* kv, double* kq, double* kpsi, double* kphi,
                          double* tp, double* b, double* bv, int sumfact, int nthreads)
{
  const size_t nb = sizeof(double) * ndofs;
  const double s = delta / (1500.0 * 1500.0);
  double g, gdot;
  wo_source(t, freq0, p0, c0, &g, &gdot);
  memset(b, 0, nb);
  memset(bv, 0, nb);
  model_stiffness(P, ncells, ndofs, dofmap, G, un, b, sumfact, nthreads);  /* A un */
  model_stiffness(P, ncells, ndofs, dofmap, G, vn, bv, sumfact, nthreads); /* A vn */
  if (L->ncells_pml) pml_terms(L, P, ncells, ndofs, dofmap, m, s, un, vn, psin, phin, tp, kpsi, kphi);
  double* vs = NULL; /* the volume source's term at every dof, 0 off its dofs */
  if (S && S->n > 0)
  {
    vs = calloc(ndofs, sizeof(double));
    for (int64_t p = 0; p < S->n; ++p)
    {
      const double sp = t - S->delay[p];
      double gs = 0.0, gsdot;
      if (sp >= 0.0) wo_source(sp, freq0, p0, c0, &gs, &gsdot); /* g only: the term sits in the PDE */
      vs[S->dofs[p]] = (c0 * c0 * gs) * S->q[p];
    }
  }
  for (int64_t k = 0; k < ndofs; ++k)
  {
    double r = b[k] + s * bv[k];
    r += (c0 * c0 * g + delta * gdot) * m1[k] - c0 * m2[k] * vn[k];
    if (vs) r += vs[k];
    if (L->ncells_pml && L->dof_on[k]) r += tp[k];
    r += kappa[k] * m[k] * vn[k] * vn[k];
    if (M > 0)
    {
      double qdd = 0.0;
      for (int nu = 0; nu < M; ++nu)
      {
        const int64_t o = nu * ndofs + k;
        kq[o] = (eps[o] * un[k] - qn[o]) / tau[nu];
        qdd += (eps[o] * vn[k] - kq[o]) / tau[nu];
      }
      r -= m[k] * qdd;
    }
    kv[k] = r / (m[k] * (1.0 - kappa[k] * un[k]) + delta / c0 * m2[k]);
  }
  free(vs);
}

/* dv/dt = f1(t, u, v; q, psi, phi) of the lossy / Westervelt model with relaxation and a perfectly matched layer */
static void f1_pml(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G, const double* m,
                   const double* m1, const double* m2, const double* kappa, double c0, double freq0, double p0,
                   double delta, int M, const double* tau, const double* eps, const double* zeta, const double* K,
                   const double* dJw, const double* coeff, const vsrc_t* S, double t, const double* u, const double* v,
                   const double* q, const double* psi, const double* phi, double* out, int sumfact, int nthreads)
{
  const int nd = (P + 1) * (P + 1) * (P + 1);
  const size_t nb = sizeof(double) * ndofs, nphi = sizeof(double) * (ncells * nd * 3 + 1);
  double *b = malloc(nb), *bv = malloc(nb), *kq = malloc(nb * (M > 0 ? M : 1));
  double *tp = malloc(nb + 8), *kpsi = malloc(nb + 8), *kphi = malloc(nphi);
  pml_t L;
  pml_setup(&L, P, ncells, ndofs, dofmap, zeta, K, dJw, coeff);
  model_rhs_pml(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, M, tau, eps, t, u, v, q, &L, psi,
                phi, S, out, kq, kpsi, kphi, tp, b, bv, sumfact, nthreads);
  pml_free(&L);
  free(b); free(bv); free(kq); free(tp); free(kpsi); free(kphi);
}

/* wo_rk4_westervelt_relax with a perfectly matched layer: psi [ndofs] and phi [ncells][nq][3] (in / out) are stepped
 * by the same tableau as u, v and q */
static int64_t rk4_pml(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G, const double* m,
                       const double* m1, const double* m2, const double* kappa, double c0, double freq0, double p0,
                       double delta, int M, const double* tau, const double* eps, const double* zeta, const double* K,
                       const double* dJw, const double* coeff, const vsrc_t* S, double t0, double tf, double dt,
                       int64_t max_steps, double* u_n, double* v_n, double* q_n, double* psi_n, double* phi_n,
                       int sumfact, int nthreads, double* t_end)
{
  const double a_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const double b_runge[4] = {1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0};
  const double c_runge[4] = {0.0, 0.5, 0.5, 1.0};
  const int nd = (P + 1) * (P + 1) * (P + 1);
  const size_t nb = sizeof(double) * ndofs, nq = nb * (M > 0 ? M : 1);
  const int64_t nqe = (int64_t)M * ndofs, nph = ncells * nd * 3;
  double *u_ = malloc(nb), *v_ = malloc(nb), *un = malloc(nb), *vn = malloc(nb);
  double *u0 = malloc(nb), *v0 = malloc(nb), *ku = malloc(nb), *kv = malloc(nb), *b = malloc(nb), *bv = malloc(nb);
  double *q_ = malloc(nq), *qn = malloc(nq), *q0 = malloc(nq), *kq = malloc(nq);
  double *ps_ = malloc(nb + 8), *psn = malloc(nb + 8), *ps0 = malloc(nb + 8), *kps = malloc(nb + 8), *tp = malloc(nb + 8);
  const size_t nphb = sizeof(double) * (nph + 1);
  double *ph_ = malloc(nphb), *phn = malloc(nphb), *ph0 = malloc(nphb), *kph = malloc(nphb);
  pml_t L;
  pml_setup(&L, P, ncells, ndofs, dofmap, zeta, K, dJw, coeff);
  const int on = L.ncells_pml > 0;
  memcpy(u_, u_n, nb);
  memcpy(v_, v_n, nb);
  memcpy(ku, u_, nb);
  memcpy(kv, v_, nb);
  if (M > 0)
  {
    memcpy(q_, q_n, sizeof(double) * nqe);
    memset(kq, 0, sizeof(double) * nqe);
  }
  if (on)
  {
    memcpy(ps_, psi_n, nb);
    memcpy(ph_, phi_n, sizeof(double) * nph);
  }
  double t = t0;
  int64_t step = 0;
  while (t < tf)
  {
    if (max_steps > 0 && step >= max_steps) break;
    dt = dt < tf - t ? dt : tf - t;
    memcpy(u0, u_, nb);
    memcpy(v0, v_, nb);
    if (M > 0) memcpy(q0, q_, sizeof(double) * nqe);
    if (on)
    {
      memcpy(ps0, ps_, nb);
      memcpy(ph0, ph_, sizeof(double) * nph);
    }
    for (int i = 0; i < 4; ++i)
    {
      memcpy(un, u0, nb);
      memcpy(vn, v0, nb);
      const double adt = dt * a_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) un[k] = ku[k] * adt + un[k];
      for (int64_t k = 0; k < ndofs; ++k) vn[k] = kv[k] * adt + vn[k];
      for (int64_t k = 0; k < nqe; ++k) qn[k] = i == 0 ? q0[k] : kq[k] * adt + q0[k];
      if (on)
      {
        for (int64_t k = 0; k < ndofs; ++k) psn[k] = i == 0 ? ps0[k] : kps[k] * adt + ps0[k];
        for (int64_t k = 0; k < nph; ++k) phn[k] = i == 0 ? ph0[k] : kph[k] * adt + ph0[k];
      }
      const double tn = t + c_runge[i] * dt;
      memcpy(ku, vn, nb);
      model_rhs_pml(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, M, tau, eps, tn, un, vn, qn, &L,
                    psn, phn, S, kv, kq, kps, kph, tp, b, bv, sumfact, nthreads);
      const double bdt = dt * b_runge[i];
      for (int64_t k = 0; k < ndofs; ++k) u_[k] = ku[k] * bdt + u_[k];
      for (int64_t k = 0; k < ndofs; ++k) v_[k] = kv[k] * bdt + v_[k];
      for (int64_t k = 0; k < nqe; ++k) q_[k] = kq[k] * bdt + q_[k];
      if (on)
      {
        for (int64_t k = 0; k < ndofs; ++k) ps_[k] = kps[k] * bdt + ps_[k];
        for (int64_t k = 0; k < nph; ++k) ph_[k] = kph[k] * bdt + ph_[k];
      }
    }
    t += dt;
    step += 1;
  }
  memcpy(u_n, u_, nb);
  memcpy(v_n, v_, nb);
  if (M > 0) memcpy(q_n, q_, sizeof(double) * nqe);
  if (on)
  {
    memcpy(psi_n, ps_, nb);
    memcpy(phi_n, ph_, sizeof(double) * nph);
  }
  if (t_end) *t_end = t;
  pml_free(&L);
  free(u_); free(v_); free(un); free(vn); free(u0); free(v0); free(ku); free(kv); free(b); free(bv);
  free(q_); free(qn); free(q0); free(kq);
  free(ps_); free(psn); free(ps0); free(kps); free(tp);
  free(ph_); free(phn); free(ph0); free(kph);
  return step;
}

void wo_f1_westervelt_pml(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G, const double* m,
                          const double* m1, const double* m2, const double* kappa, double c0, double freq0, double p0,
                          double delta, int M, const double* tau, const double* eps, const double* zeta,
                          const double* K, const double* dJw, const double* coeff, double t, const double* u,
                          const double* v, const double* q, const double* psi, const double* phi, double* out,
                          int sumfact, int nthreads)
{
  f1_pml(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, M, tau, eps, zeta, K, dJw, coeff, NULL, t,
         u, v, q, psi, phi, out, sumfact, nthreads);
}

int64_t wo_rk4_westervelt_pml(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                              const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                              double freq0, double p0, double delta, int M, const double* tau, const double* eps,
                              const double* zeta, const double* K, const double* dJw, const double* coeff, double t0,
                              double tf, double dt, int64_t max_steps, double* u_n, double* v_n, double* q_n,
                              double* psi_n, double* phi_n, int sumfact, int nthreads, double* t_end)
{
  return rk4_pml(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, M, tau, eps, zeta, K, dJw, coeff,
                 NULL, t0, tf, dt, max_steps, u_n, v_n, q_n, psi_n, phi_n, sumfact, nthreads, t_end);
}

/* ---- volume sources (DESIGN.md section 4.5h) ------------------------------------------------------------------
 * wo_f1 / wo_rk4_westervelt_pml with a volume source: ns distinct dofs sdofs [ns], weights sq [ns] and delays
 * sdelay [ns] (see vsrc_t).  With ns = 0 they compute what wo_f1 / wo_rk4_westervelt_pml compute, bit for bit. */
void wo_f1_westervelt_source(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                             const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                             double freq0, double p0, double delta, int M, const double* tau, const double* eps,
                             const double* zeta, const double* K, const double* dJw, const double* coeff, int64_t ns,
                             const int32_t* sdofs, const double* sq, const double* sdelay, double t, const double* u,
                             const double* v, const double* q, const double* psi, const double* phi, double* out,
                             int sumfact, int nthreads)
{
  const vsrc_t S = {ns, sdofs, sq, sdelay};
  f1_pml(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, M, tau, eps, zeta, K, dJw, coeff, &S, t,
         u, v, q, psi, phi, out, sumfact, nthreads);
}

int64_t wo_rk4_westervelt_source(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap, const double* G,
                                 const double* m, const double* m1, const double* m2, const double* kappa, double c0,
                                 double freq0, double p0, double delta, int M, const double* tau, const double* eps,
                                 const double* zeta, const double* K, const double* dJw, const double* coeff,
                                 int64_t ns, const int32_t* sdofs, const double* sq, const double* sdelay, double t0,
                                 double tf, double dt, int64_t max_steps, double* u_n, double* v_n, double* q_n,
                                 double* psi_n, double* phi_n, int sumfact, int nthreads, double* t_end)
{
  const vsrc_t S = {ns, sdofs, sq, sdelay};
  return rk4_pml(P, ncells, ndofs, dofmap, G, m, m1, m2, kappa, c0, freq0, p0, delta, M, tau, eps, zeta, K, dJw, coeff,
                 &S, t0, tf, dt, max_steps, u_n, v_n, q_n, psi_n, phi_n, sumfact, nthreads, t_end);
}
