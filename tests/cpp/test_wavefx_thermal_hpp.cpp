// Exercises the thermal C++ wrapper (wave-fenics_b200/hpp/wavefx.hpp): wavefx::PennesGLL at a constant temperature
// (the CEM43 dose in closed form), relaxation towards the perfusion equilibrium, a heat source from a wave model's
// harmonic maps, the stable step and a refused call.  Self-checking; prints "thermal hpp ok" on success.  Needs a GPU
// to run, only a compiler to build.
#include "wavefx.hpp"

#include <algorithm>
#include <cmath>
#include <cstdio>

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

int main()
{
  const int P = 3, N = 2;
  const double L = 0.01, k = 0.5, rhoc = 3.6e6, T_art = 37.0;
  BoxMesh mesh = make_box(N, P, L);
  const wavefx::SpaceView V = mesh.view();
  const std::int64_t n = V.ndofs;
  auto ctx = std::make_shared<wavefx::Context>(0);
  const std::vector<double> rhoC(n, rhoc), none;

  // insulated, no perfusion, 45 degC everywhere: CEM43 = N dt / 60 * 0.5^(43 - 45)
  {
    wavefx::PennesGLL th(ctx, V, P, k, rhoC, none, T_art);
    th.set_temperature(std::vector<double>(n, 45.0));
    REQUIRE(th.rk4(0.0, 5.0, 0.5) == 10);
    std::vector<double> cem, tmax, T;
    REQUIRE(th.dose(cem, tmax) == 10);
    for (std::int64_t i = 0; i < n; ++i)
      REQUIRE(std::abs(cem[i] / (5.0 / 60.0 * 4.0) - 1) < 1e-14 && std::abs(tmax[i] - 45.0) < 1e-12);
    th.temperature(T);
    REQUIRE(std::abs(T[0] - 45.0) < 1e-12);
    th.init();
    REQUIRE(th.dose(cem, tmax) == 0 && cem[0] == 0.0);
    REQUIRE(th.stable_dt() > 0.0);
    bool refused = false;
    try { th.set_heat_scale(-1.0); } catch (const std::runtime_error&) { refused = true; }
    REQUIRE(refused);
  }
  // uniform perfusion and Q with both Robin tags insulated (h = 0): T -> T_art + Q / wbCb
  {
    const double wb = 1e6, Q = 2e7;
    wavefx::PennesGLL th(ctx, V, P, k, rhoC, std::vector<double>(n, wb), T_art);
    th.init();
    th.set_heat_source(std::vector<double>(n, Q));
    const double r = wb / rhoc;
    th.rk4(0.0, 100.0 / r, th.stable_dt());
    std::vector<double> T;
    th.temperature(T);
    for (double x : T) REQUIRE(std::abs(x - (T_art + Q / wb)) < 1e-9 * (Q / wb));
  }
  // heat from a wave model's harmonic maps: non-negative and not zero
  {
    const double c0 = 1500.0, f0 = 0.5e6, p0 = 6e4;
    int deg = P;
    double cc = c0, ff = f0, pp = p0;
    wavefx::LinearGLLOpt wave(ctx, V, deg, cc, ff, pp);
    wave.init();
    wave.set_field_stats(true, 0.0, 2);
    double t0 = 0.0, dt = 2e-8, tf = 40 * dt;
    REQUIRE(wave.rk4(t0, tf, dt) >= 40);
    const std::array<double, 2> T_ext{20.0, T_art};
    wavefx::PennesGLL th(ctx, V, P, k, rhoC, none, T_art, {100.0, 0.0}, &T_ext);
    th.heat_from_wave(wave, 5.0, 1.1, 1000.0, c0);
    std::vector<double> q;
    th.heat_source(q);
    REQUIRE(*std::min_element(q.begin(), q.end()) >= 0.0 && *std::max_element(q.begin(), q.end()) > 0.0);
  }
  std::printf("thermal hpp ok\n");
  return 0;
}
