// Exercises the relaxation methods of the C++ wrapper (wave-fenics_b200/hpp/wavefx.hpp): a WesterveltGLLOpt in a
// wavefx::Medium with set_relaxation, 15 steps, a checkpoint of u, v and the memory variables fed back through
// set_state and set_relaxation_state, 15 more steps.  The mesh, weights, relaxation and initial state come from raw
// fp64 / int32 files written by tests/test_relaxation.py (argv[1] names their directory); the final u and q are
// written back there for a bitwise comparison with the Python model.  Prints "relaxation hpp ok".  Needs a GPU to run,
// only a compiler to build.
#include "wavefx.hpp"

#include <cstdio>
#include <string>

template <typename T>
static std::vector<T> load(const std::string& dir, const char* name)
{
  std::vector<T> v;
  FILE* f = std::fopen((dir + "/" + name).c_str(), "rb");
  if (!f) throw std::runtime_error(std::string("cannot open ") + name);
  T x;
  while (std::fread(&x, sizeof(T), 1, f) == 1) v.push_back(x);
  std::fclose(f);
  return v;
}

static void save(const std::string& dir, const char* name, const std::vector<double>& v)
{
  FILE* f = std::fopen((dir + "/" + name).c_str(), "wb");
  if (!f || std::fwrite(v.data(), sizeof(double), v.size(), f) != v.size()) throw std::runtime_error("cannot write");
  std::fclose(f);
}

int main(int argc, char** argv)
{
  if (argc < 2)
  {
    std::fprintf(stderr, "usage: %s DIR\n", argv[0]);
    return 2;
  }
  const std::string dir = argv[1];
  try
  {
    // params: P, c0, f0, p0, delta, beta, rho0, dt, M
    const auto par = load<double>(dir, "params.f64");
    const auto x = load<double>(dir, "x.f64");
    const auto xdofs = load<std::int32_t>(dir, "xdofs.i32");
    const auto dofmap = load<std::int32_t>(dir, "dofmap.i32");
    const auto fcell = load<std::int32_t>(dir, "fcell.i32"), flocal = load<std::int32_t>(dir, "flocal.i32"),
               ftag = load<std::int32_t>(dir, "ftag.i32");
    const auto u0 = load<double>(dir, "u.f64"), v0 = load<double>(dir, "v.f64");
    const auto tau = load<double>(dir, "tau.f64"), eps = load<double>(dir, "eps.f64");
    wavefx::Medium med;
    med.stiffness = load<double>(dir, "stiffness.f64");
    med.mass = load<double>(dir, "mass.f64");
    med.facet = load<double>(dir, "facet.f64");
    med.kappa = load<double>(dir, "kappa.f64");
    const int P = (int)par[0];
    const double c0 = par[1], f0 = par[2], p0 = par[3], delta = par[4], beta = par[5], rho0 = par[6], dt = par[7];
    wavefx::SpaceView V;
    V.degree = P;
    V.ncells = (std::int64_t)xdofs.size() / 8;
    V.npoints = (std::int64_t)x.size() / 3;
    V.x = x.data();
    V.xdofs = xdofs.data();
    V.ndofs = V.size_local = (std::int64_t)u0.size();
    V.dofmap = dofmap.data();
    V.nfacets = (std::int64_t)fcell.size();
    V.facet_cell = fcell.data();
    V.facet_local = flocal.data();
    V.facet_tag = ftag.data();
    auto ctx = std::make_shared<wavefx::Context>(0);
    wavefx::WesterveltGLLOpt west(ctx, V, P, c0, f0, p0, delta, beta, rho0, med);
    west.set_relaxation(tau, eps);
    west.set_state(u0, v0);
    // 15 steps from t = 0 (the same count as the Python run: rk4 with max_steps)
    auto steps = [&](double t0) {
      std::int64_t n = 0;
      double t = 0;
      wavefx::check(wfx_wave_rk4(west.get(), t0, 1.0, dt, 15, &n, &t, nullptr));
      if (n != 15) throw std::runtime_error("expected 15 steps");
      return t;
    };
    const double t1 = steps(0.0);
    std::vector<double> u, v, q;
    west.solution(u, v);
    west.relaxation_state(q);
    west.set_state(u, v);
    west.set_relaxation_state(q);
    steps(t1);
    west.solution(u, v);
    west.relaxation_state(q);
    save(dir, "u.out.f64", u);
    save(dir, "q.out.f64", q);
    // a short eps and a short state are refused
    bool refused = false;
    try
    {
      west.set_relaxation(tau, std::vector<double>(eps.begin(), eps.end() - 1));
    }
    catch (const std::runtime_error&)
    {
      refused = true;
    }
    if (!refused) throw std::runtime_error("a short eps was accepted");
    refused = false;
    try
    {
      west.set_relaxation_state(std::vector<double>(q.begin(), q.end() - 1));
    }
    catch (const std::runtime_error&)
    {
      refused = true;
    }
    if (!refused) throw std::runtime_error("a short relaxation state was accepted");
  }
  catch (const std::exception& e)
  {
    std::fprintf(stderr, "relaxation hpp FAILED: %s\n", e.what());
    return 1;
  }
  std::printf("relaxation hpp ok\n");
  return 0;
}
