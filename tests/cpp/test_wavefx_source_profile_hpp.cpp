// Exercises the source-profile C++ wrappers (wave-fenics_b200/hpp/wavefx.hpp): set_source_profile on
// LinearGLLOpt, LossyGLLOpt (inherited) and LinearGLLEnsemble.  Identity profiles against unprofiled runs, clearing
// restores the unprofiled run bitwise, amplitudes scale the lossy model linearly, member profiles of an ensemble,
// and the refused calls.  Self-checking; prints "source profile hpp ok" on success.  Needs a GPU to run, only a
// compiler to build.
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

static double rel_diff(const std::vector<double>& a, const std::vector<double>& b, double scale = 1.0)
{
  double num = 0, den = 0;
  for (std::size_t i = 0; i < a.size(); ++i)
  {
    num += (a[i] - scale * b[i]) * (a[i] - scale * b[i]);
    den += scale * b[i] * scale * b[i];
  }
  return std::sqrt(num / den);
}

template <typename M>
static bool refused(M&& call)
{
  try { call(); } catch (const std::runtime_error&) { return true; }
  return false;
}

int main()
{
  int P = 3;
  const int N = 3;
  double L = 0.1, c0 = 1500.0, f0 = 0.5e6, p0 = 6e4;
  double t0 = 0.0, dt = 2e-8, tf = 30 * dt;
  BoxMesh mesh = make_box(N, P, L);
  const wavefx::SpaceView V = mesh.view();
  const std::int64_t n = V.ndofs;
  auto ctx = std::make_shared<wavefx::Context>(0);
  std::vector<double> u, v, uref, vref;

  // linear model: identity profile ~ unprofiled, cleared profile == unprofiled bitwise, zero amplitude == rest
  {
    wavefx::LinearGLLOpt lin(ctx, V, P, c0, f0, p0);
    lin.init();
    REQUIRE(lin.rk4(t0, tf, dt) == 30);
    lin.solution(uref, vref);
    lin.set_source_profile(std::vector<double>(n, 1.0), {});
    lin.init();
    lin.rk4(t0, tf, dt);
    lin.solution(u, v);
    REQUIRE(rel_diff(u, uref) < 1e-13 && rel_diff(v, vref) < 1e-13);
    lin.set_source_profile({}, {});
    lin.init();
    lin.rk4(t0, tf, dt);
    lin.solution(u, v);
    REQUIRE(u == uref && v == vref);
    lin.set_source_profile(std::vector<double>(n, 0.0), std::vector<double>(n, 3 * dt));
    lin.init();
    lin.rk4(t0, tf, dt);
    lin.solution(u, v);
    REQUIRE(std::all_of(u.begin(), u.end(), [](double x) { return x == 0.0; }));
    REQUIRE(refused([&] { lin.set_source_profile(std::vector<double>(n - 1, 1.0), {}); }));
    REQUIRE(refused([&] { lin.set_source_profile({}, std::vector<double>(n, -dt)); }));
    REQUIRE(refused([&] { lin.set_source_profile(std::vector<double>(n, NAN), {}); }));
  }

  // lossy model: the state is linear in the amplitude
  {
    wavefx::LossyGLLOpt lossy(ctx, V, P, c0, f0, p0, 1e-2);
    lossy.init();
    lossy.rk4(t0, tf, dt);
    lossy.solution(uref, vref);
    lossy.set_source_profile(std::vector<double>(n, 2.0), {});
    lossy.init();
    lossy.rk4(t0, tf, dt);
    lossy.solution(u, v);
    REQUIRE(rel_diff(u, uref, 2.0) < 1e-12 && rel_diff(v, vref, 2.0) < 1e-12);
  }

  // ensemble of two: member 0 with amplitude 1, member 1 switched off
  {
    wavefx::LinearGLLEnsemble ens(ctx, V, P, c0, {f0, 0.75e6}, {p0, 2 * p0});
    ens.init();
    ens.rk4(t0, tf, dt);
    ens.solution(uref, vref);
    std::vector<double> amp(2 * n);
    for (std::int64_t i = 0; i < n; ++i) amp[2 * i] = 1.0, amp[2 * i + 1] = 0.0;
    ens.set_source_profile(amp, {});
    ens.init();
    ens.rk4(t0, tf, dt);
    ens.solution(u, v);
    std::vector<double> u0(n), r0(n);
    for (std::int64_t i = 0; i < n; ++i)
    {
      u0[i] = u[2 * i];
      r0[i] = uref[2 * i];
      REQUIRE(u[2 * i + 1] == 0.0);
    }
    REQUIRE(rel_diff(u0, r0) < 1e-13);
    REQUIRE(refused([&] { ens.set_source_profile(std::vector<double>(n, 1.0), {}); }));
  }
  std::printf("source profile hpp ok\n");
  return 0;
}
