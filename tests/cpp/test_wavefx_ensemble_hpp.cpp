// Exercises the ensemble C++ wrappers (wave-fenics_b200/hpp/wavefx.hpp): StiffnessOperator<T>::
// apply_ensemble_device on member-interleaved device vectors against one apply per member, and
// LinearGLLEnsemble against one LinearGLLOpt per member.  Self-checking; prints "ensemble hpp ok" on
// success.  Needs a GPU to run, only a compiler to build.
#include "wavefx.hpp"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <random>

struct BoxMesh
{
  int P, N;
  std::vector<double> x;
  std::vector<std::int32_t> xdofs, dofmap, fcell, flocal, ftag;
  std::int64_t ndofs;
  wavefx::SpaceView view() const
  {
    wavefx::SpaceView V;
    V.degree = P;
    V.ncells = (std::int64_t)N * N * N;
    V.npoints = (std::int64_t)x.size() / 3;
    V.x = x.data();
    V.xdofs = xdofs.data();
    V.ndofs = V.size_local = ndofs;
    V.dofmap = dofmap.data();
    V.nfacets = (std::int64_t)fcell.size();
    V.facet_cell = fcell.data();
    V.facet_local = flocal.data();
    V.facet_tag = ftag.data();
    return V;
  }
};

static BoxMesh make_box(int N, int P, double L)
{
  BoxMesh m;
  m.P = P;
  m.N = N;
  const int n = P + 1, nd = n * n * n, M = P * N + 1;
  m.ndofs = (std::int64_t)M * M * M;
  for (int i = 0; i <= N; ++i)
    for (int j = 0; j <= N; ++j)
      for (int k = 0; k <= N; ++k)
      {
        m.x.push_back(L * i / N);
        m.x.push_back(L * j / N);
        m.x.push_back(L * k / N);
      }
  std::vector<std::int32_t> perm(nd);
  wavefx::check(wfx_compute_permutations(P, perm.data()));
  auto pos = [&](int a) { return a == 0 ? 0 : (a == 1 ? P : a - 1); };
  for (int cx = 0; cx < N; ++cx)
    for (int cy = 0; cy < N; ++cy)
      for (int cz = 0; cz < N; ++cz)
      {
        const std::int32_t c = (cx * N + cy) * N + cz;
        for (int v = 0; v < 8; ++v)
          m.xdofs.push_back(((cx + (v & 1)) * (N + 1) + (cy + ((v >> 1) & 1))) * (N + 1) + (cz + ((v >> 2) & 1)));
        std::vector<std::int32_t> cd(nd);
        for (int a = 0; a < n; ++a)
          for (int b = 0; b < n; ++b)
            for (int d = 0; d < n; ++d)
              cd[perm[(a * n + b) * n + d]] = ((cx * P + pos(a)) * M + (cy * P + pos(b))) * M + (cz * P + pos(d));
        m.dofmap.insert(m.dofmap.end(), cd.begin(), cd.end());
        if (cx == 0) { m.fcell.push_back(c); m.flocal.push_back(2); m.ftag.push_back(1); }
        if (cx == N - 1) { m.fcell.push_back(c); m.flocal.push_back(3); m.ftag.push_back(2); }
      }
  return m;
}

#define REQUIRE(cond)                                                              \
  do {                                                                             \
    if (!(cond)) { std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); return 1; } \
  } while (0)

static double rel_l2(const std::vector<double>& a, const std::vector<double>& b)
{
  double num = 0, den = 0;
  for (std::size_t i = 0; i < a.size(); ++i)
  {
    num += (a[i] - b[i]) * (a[i] - b[i]);
    den += b[i] * b[i];
  }
  return std::sqrt(num / den);
}

int main()
{
  const int P = 4, N = 3, nv = 3;
  const double L = 0.1;
  BoxMesh mesh = make_box(N, P, L);
  const wavefx::SpaceView V = mesh.view();
  const std::int64_t n = V.ndofs;
  auto ctx = std::make_shared<wavefx::Context>(0);
  auto geom = std::make_shared<wavefx::Geometry<double>>(ctx, V);
  std::map<std::string, double> params{{"c0", 1500.0}};
  wavefx::StiffnessOperator<double> K(geom, V, P, params, {}, WFX_STIFF_ENSEMBLE);

  // ensemble apply against one apply per member
  std::mt19937_64 rng(7);
  std::normal_distribution<double> nd;
  std::vector<double> X((std::size_t)(n * nv)), Y((std::size_t)(n * nv)), want((std::size_t)(n * nv));
  for (auto& v : X) v = nd(rng);
  void *dX = nullptr, *dY = nullptr, *dx = nullptr, *dy = nullptr;
  wavefx::check(wfx_malloc(ctx->get(), n * nv * 8, &dX));
  wavefx::check(wfx_malloc(ctx->get(), n * nv * 8, &dY));
  wavefx::check(wfx_malloc(ctx->get(), n * 8, &dx));
  wavefx::check(wfx_malloc(ctx->get(), n * 8, &dy));
  wavefx::check(wfx_memcpy_h2d(ctx->get(), dX, X.data(), n * nv * 8));
  K.apply_ensemble_device(nv, (const double*)dX, nullptr, (double*)dY, 0);
  wavefx::check(wfx_memcpy_d2h(ctx->get(), Y.data(), dY, n * nv * 8));
  std::vector<double> xm((std::size_t)n), ym((std::size_t)n);
  for (int m = 0; m < nv; ++m)
  {
    for (std::int64_t i = 0; i < n; ++i) xm[i] = X[i * nv + m];
    wavefx::check(wfx_memcpy_h2d(ctx->get(), dx, xm.data(), n * 8));
    K.apply_device((const double*)dx, (double*)dy, 0);
    wavefx::check(wfx_memcpy_d2h(ctx->get(), ym.data(), dy, n * 8));
    for (std::int64_t i = 0; i < n; ++i) want[i * nv + m] = ym[i];
  }
  REQUIRE(rel_l2(Y, want) < 1e-12);
  bool refused = false;
  try
  {
    K.apply_ensemble_device(9, (const double*)dX, nullptr, (double*)dY, 0);
  }
  catch (const std::runtime_error&)
  {
    refused = true;
  }
  REQUIRE(refused);
  for (void* p : {dX, dY, dx, dy}) wavefx::check(wfx_free(ctx->get(), p));

  // the ensemble model against one model per member
  const std::vector<double> f0s{0.5e6, 0.3e6}, p0s{6e4, 2e4};
  wavefx::LinearGLLEnsemble ens(ctx, V, P, 1500.0, f0s, p0s);
  REQUIRE(ens.size() == 2);
  ens.init();
  const double t0 = 0.0, dt = 2e-8, tf = 6.5 * dt; // the last step is a short one
  ens.set_probes({0, (std::int32_t)(n / 2)}, 100);
  const std::int64_t steps = ens.rk4(t0, tf, dt);
  REQUIRE(steps == 7);
  std::vector<double> ue, ve;
  ens.solution(ue, ve);
  std::vector<double> tp, vals;
  ens.probe_series(tp, vals);
  REQUIRE((std::int64_t)tp.size() == steps && (std::int64_t)vals.size() == steps * 2 * 2);
  for (int m = 0; m < 2; ++m)
  {
    int deg = P;
    double c0 = 1500.0, f0 = f0s[m], p0 = p0s[m];
    wavefx::LinearGLLOpt one(ctx, V, deg, c0, f0, p0);
    one.init();
    double a = t0, b = tf, h = dt;
    REQUIRE(one.rk4(a, b, h) == steps);
    std::vector<double> u1, v1;
    one.solution(u1, v1);
    std::vector<double> um((std::size_t)n), vm((std::size_t)n);
    for (std::int64_t i = 0; i < n; ++i) um[i] = ue[i * 2 + m], vm[i] = ve[i * 2 + m];
    double umax = 0;
    for (double v : u1) umax = std::max(umax, std::fabs(v));
    REQUIRE(umax > 0);
    REQUIRE(rel_l2(um, u1) < 1e-12 && rel_l2(vm, v1) < 1e-12);
    // the last probe record is the final state at the probed dofs
    REQUIRE(vals[((steps - 1) * 2 + 1) * 2 + m] == ue[(n / 2) * 2 + m]);
  }
  std::printf("ensemble hpp ok\n");
  return 0;
}
