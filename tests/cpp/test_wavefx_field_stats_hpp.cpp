// Exercises the field-statistics C++ wrappers (wave-fenics_b200/hpp/wavefx.hpp): set_field_stats / field_stats on
// WesterveltGLLOpt (inherited from LinearGLLOpt) and on LinearGLLEnsemble, against probe series on every dof, and
// the refused calls.  Self-checking; prints "field stats hpp ok" on success.  Needs a GPU to run, only a compiler
// to build.
#include "wavefx.hpp"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <numeric>

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

// pmax / pmin of the field statistics against the probe records [nrec][entries] from record r0 on
static bool peaks_match(const wavefx::FieldStats& fs, const std::vector<double>& vals, std::int64_t entries,
                        std::int64_t r0, std::int64_t nrec)
{
  for (std::int64_t i = 0; i < entries; ++i)
  {
    double hi = -INFINITY, lo = INFINITY;
    for (std::int64_t r = r0; r < nrec; ++r)
    {
      hi = std::max(hi, vals[r * entries + i]);
      lo = std::min(lo, vals[r * entries + i]);
    }
    if (fs.pmax[i] != hi || fs.pmin[i] != lo) return false;
  }
  return true;
}

int main()
{
  const int P = 3, N = 3;
  const double L = 0.1, c0 = 1500.0, f0 = 0.5e6, p0 = 6e4, dt = 2e-8;
  BoxMesh mesh = make_box(N, P, L);
  const wavefx::SpaceView V = mesh.view();
  const std::int64_t n = V.ndofs;
  auto ctx = std::make_shared<wavefx::Context>(0);
  std::vector<std::int32_t> all(n);
  std::iota(all.begin(), all.end(), 0);

  // Westervelt model: 31 steps (the last a half step), the window starts at step 11
  {
    wavefx::WesterveltGLLOpt wv(ctx, V, P, c0, f0, p0, 1e-2, 900.0, 1000.0);
    wv.init();
    wv.set_probes(all, 40);
    wv.set_field_stats(true, 11 * dt, 2);
    double a = 0.0, b = 30.5 * dt, h = dt;
    REQUIRE(wv.rk4(a, b, h) == 31);
    wavefx::FieldStats fs;
    wv.field_stats(fs);
    std::vector<double> tp, vals;
    wv.probe_series(tp, vals);
    REQUIRE(tp.size() == 31 && fs.samples == 21 && fs.t_first == tp[10] && fs.t_last == tp[30]);
    REQUIRE(fs.harmonics.size() == (std::size_t)(2 * n));
    REQUIRE(peaks_match(fs, vals, n, 10, 31));
    // the fundamental at one dof against a direct sum over the probe records
    const std::int64_t i = n / 2;
    std::complex<double> s = 0;
    for (int r = 10; r < 31; ++r) s += vals[r * n + i] * std::exp(std::complex<double>(0, -2 * M_PI * f0 * tp[r]));
    s *= 2.0 / 21;
    REQUIRE(std::abs(fs.harmonics[i] - s) <= 1e-12 * std::max(std::abs(s), 1.0));
    REQUIRE(std::abs(s) > 0);
    // init resets them
    wv.init();
    wv.field_stats(fs);
    REQUIRE(fs.samples == 0 && fs.pmax[0] == -INFINITY && fs.pmin[0] == INFINITY && fs.harmonics[0] == 0.0);
    // off: field_stats is refused
    wv.set_field_stats(false);
    bool refused = false;
    try { wv.field_stats(fs); } catch (const std::runtime_error&) { refused = true; }
    REQUIRE(refused);
    refused = false;
    try { wv.set_field_stats(true, 0.0, WFX_HARMONICS_MAX + 1); } catch (const std::runtime_error&) { refused = true; }
    REQUIRE(refused);
    refused = false;
    try { wv.set_field_stats(true, NAN, 1); } catch (const std::runtime_error&) { refused = true; }
    REQUIRE(refused);
  }

  // ensemble of two: peaks per member against the member-interleaved probe records
  {
    wavefx::LinearGLLEnsemble ens(ctx, V, P, c0, {f0, 0.75e6}, {p0, 2 * p0});
    ens.init();
    ens.set_probes(all, 40);
    ens.set_field_stats(true, 0.0, 3);
    REQUIRE(ens.rk4(0.0, 25.5 * dt, dt) == 26);
    wavefx::FieldStats fs;
    ens.field_stats(fs);
    std::vector<double> tp, vals;
    ens.probe_series(tp, vals);
    REQUIRE(fs.samples == 26 && fs.harmonics.size() == (std::size_t)(3 * n * 2));
    REQUIRE(peaks_match(fs, vals, 2 * n, 0, 26));
    double hmax = 0;
    for (auto& z : fs.harmonics) hmax = std::max(hmax, std::abs(z));
    REQUIRE(hmax > 0 && std::isfinite(hmax));
  }
  std::printf("field stats hpp ok\n");
  return 0;
}
