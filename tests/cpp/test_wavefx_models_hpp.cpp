// Exercises the lossy / Westervelt C++ wrappers (wave-fenics_b200/hpp/wavefx.hpp): WesterveltGLLOpt with
// delta = beta = 0 against LinearGLLOpt (bit for bit), LossyGLLOpt and WesterveltGLLOpt runs with probes and a
// snapshot restart, and a refused parameter.  Self-checking; prints "models hpp ok" on success.  Needs a GPU
// to run, only a compiler to build.
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
  const int P = 3, N = 3;
  const double L = 0.1, c0 = 1500.0, f0 = 0.5e6, p0 = 6e4;
  BoxMesh mesh = make_box(N, P, L);
  const wavefx::SpaceView V = mesh.view();
  const std::int64_t n = V.ndofs;
  auto ctx = std::make_shared<wavefx::Context>(0);
  const double dt = 2e-8, tf = 30.5 * dt; // the last step is a short one

  // delta = beta = 0: the linear model, bit for bit
  std::vector<double> ul, vl, uw, vw;
  {
    int deg = P;
    double c = c0, f = f0, p = p0, a = 0.0, b = tf, h = dt;
    wavefx::LinearGLLOpt lin(ctx, V, deg, c, f, p);
    lin.init();
    REQUIRE(lin.rk4(a, b, h) == 31);
    lin.solution(ul, vl);
  }
  {
    wavefx::WesterveltGLLOpt w0(ctx, V, P, c0, f0, p0, 0.0, 0.0, 1.0);
    w0.init();
    double a = 0.0, b = tf, h = dt;
    REQUIRE(w0.rk4(a, b, h) == 31);
    w0.solution(uw, vw);
  }
  double umax = 0;
  for (double v : ul) umax = std::max(umax, std::fabs(v));
  REQUIRE(umax > 0 && uw == ul && vw == vl);

  // lossy: damped against the linear run, finite
  std::vector<double> us, vs;
  {
    wavefx::LossyGLLOpt lossy(ctx, V, P, c0, f0, p0, 1e-2);
    lossy.init();
    double a = 0.0, b = tf, h = dt;
    REQUIRE(lossy.rk4(a, b, h) == 31);
    lossy.solution(us, vs);
  }
  for (double v : us) REQUIRE(std::isfinite(v));
  REQUIRE(rel_l2(us, ul) > 1e-8 && rel_l2(us, ul) < 0.5);

  // Westervelt: probes, and a snapshot fed back through set_state resumes the run bit for bit
  wavefx::WesterveltGLLOpt wv(ctx, V, P, c0, f0, p0, 1e-2, 900.0, 1000.0);
  wv.init();
  wv.set_probes({0, (std::int32_t)(n / 2)}, 100);
  std::vector<double> su, sv;
  std::int64_t sstep = -1;
  double st = 0;
  wv.set_snapshot(20, [&](std::int64_t step, double t, const double* u, const double* v) {
    sstep = step, st = t;
    su.assign(u, u + n);
    sv.assign(v, v + n);
  });
  double a = 0.0, b = tf, h = dt;
  REQUIRE(wv.rk4(a, b, h) == 31);
  REQUIRE(sstep == 20);
  std::vector<double> ue, ve, tp, vals;
  wv.solution(ue, ve);
  wv.probe_series(tp, vals);
  REQUIRE(tp.size() == 31 && vals[30 * 2 + 1] == ue[n / 2]);
  wv.set_snapshot(0, nullptr);
  wv.set_state(su, sv);
  double a2 = st;
  REQUIRE(wv.rk4(a2, b, h) == 11);
  std::vector<double> u2, v2;
  wv.solution(u2, v2);
  REQUIRE(u2 == ue && v2 == ve);

  bool refused = false;
  try
  {
    wavefx::LossyGLLOpt bad(ctx, V, P, c0, f0, p0, -1.0);
  }
  catch (const std::runtime_error&)
  {
    refused = true;
  }
  REQUIRE(refused);
  std::printf("models hpp ok\n");
  return 0;
}
