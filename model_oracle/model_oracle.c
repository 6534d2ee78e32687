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
